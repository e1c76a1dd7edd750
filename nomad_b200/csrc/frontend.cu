// Front of the conv feature encoder: conv0 (1 -> 512, k = 10, s = 5) + GroupNorm(512 groups) + GELU,
// and the LayerNorm(512) that follows the last conv.  All HBM-bound element-wise / reduction work.
//
// GroupNorm here normalises every (utterance, channel) over ALL conv0 frames of the utterance
// (fairseq ConvFeatureExtractionModel mode "default"; mirror torchaudio components.py:564-569).  The
// statistics of y[t, c] = sum_j w[c, j] x[5 t + j] are quadratic forms of the waveform's tap sums:
//     sum_t y      = sum_j  w_j  S_j          S_j    = sum_t x[5 t + j]
//     sum_t y^2    = sum_jj' w_j w_j' R_jj'    R_jj'  = sum_t x[5 t + j] x[5 t + j']
// so one cheap pass over the waveform (65 sums per utterance, fp64) replaces a stats pass over the
// 512-channel conv0 output, and normalisation folds into per-(utterance, channel) conv taps.
#include <cstdlib>

#include "kernels.cuh"

#ifndef NB_CONV0_BLOCKS
#define NB_CONV0_BLOCKS 3
#endif
#ifndef NB_CONV0_GELU_H2
#define NB_CONV0_GELU_H2 1
#endif

namespace nb {

// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) wave_stats_kernel(const float* __restrict__ wav,
                                                         const UttMeta* __restrict__ meta, int b0, int max_chunks,
                                                         double* __restrict__ part) {
    const int b = b0 + blockIdx.y, chunk = blockIdx.x;
    const UttMeta m = meta[b];
    const int t_begin = chunk * STAT_CHUNK;
    if (t_begin >= m.T0) return;
    const int t_end = min(m.T0, t_begin + STAT_CHUNK);
    const float* x = wav + m.wav_off;
    // fp64 throughout (the product of two fp32 samples is exact in fp64): the variance w^T R w / n - mean^2 of a
    // channel with strong stop-band rejection on band-limited input cancels most of the leading digits of R, which an
    // fp32 per-thread partial sum does not have to give (~0.2 G DFMA per 1024 utt-s: microseconds on B200)
    double acc[NSTAT];
#pragma unroll
    for (int i = 0; i < NSTAT; ++i) acc[i] = 0.0;
    for (int t = t_begin + threadIdx.x; t < t_end; t += blockDim.x) {
        double v[10];
#pragma unroll
        for (int j = 0; j < 10; ++j) v[j] = (double)__ldg(x + 5 * t + j);
        int idx = 10;
#pragma unroll
        for (int j = 0; j < 10; ++j) {
            acc[j] += v[j];
#pragma unroll
            for (int k = j; k < 10; ++k) { acc[idx] = fma(v[j], v[k], acc[idx]); ++idx; }
        }
    }
    __shared__ double red[8][NSTAT];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
    for (int i = 0; i < NSTAT; ++i) {
        double d = acc[i];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) d += __shfl_xor_sync(0xffffffffu, d, o);
        if (lane == 0) red[warp][i] = d;
    }
    __syncthreads();
    if (threadIdx.x < NSTAT) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < 8; ++w) s += red[w][threadIdx.x];
        part[((long long)b * max_chunks + chunk) * NSTAT + threadIdx.x] = s;
    }
}

int launch_wave_stats(cudaStream_t st, const float* wav, const UttMeta* meta, int b0, int nb, int max_chunks,
                      double* part) {
    dim3 grid(max_chunks, nb);
    wave_stats_kernel<<<grid, 256, 0, st>>>(wav, meta, b0, max_chunks, part);
    NB_LAUNCHED();
    return 0;
}

// ---------------------------------------------------------------------------------------------
// fold[b][c][0..9] = w[c][j] * rstd * gamma,  fold[b][c][10] = beta - mean * rstd * gamma
__global__ void __launch_bounds__(512) gn_fold_kernel(const double* __restrict__ part,
                                                      const UttMeta* __restrict__ meta, int b0, int max_chunks,
                                                      const float* __restrict__ w0, const float* __restrict__ gn_g,
                                                      const float* __restrict__ gn_b, float* __restrict__ fold,
                                                      float* __restrict__ stat_out, op_t* __restrict__ fold_h) {
    const int b = b0 + blockIdx.x;
    const UttMeta m = meta[b];
    __shared__ double s[NSTAT];
    if (threadIdx.x < NSTAT) {
        const int chunks = (m.T0 + STAT_CHUNK - 1) / STAT_CHUNK;
        double a = 0.0;
        for (int c = 0; c < chunks; ++c) a += part[((long long)b * max_chunks + c) * NSTAT + threadIdx.x];
        s[threadIdx.x] = a;
    }
    __syncthreads();
    const int c = threadIdx.x;
    double w[10];
#pragma unroll
    for (int j = 0; j < 10; ++j) w[j] = (double)w0[c * 10 + j];
    double sum = 0.0, sq = 0.0;
    int idx = 10;
#pragma unroll
    for (int j = 0; j < 10; ++j) {
        sum += w[j] * s[j];
#pragma unroll
        for (int k = j; k < 10; ++k) {
            const double r = w[j] * w[k] * s[idx++];
            sq += (k == j) ? r : 2.0 * r;
        }
    }
    const double inv_n = 1.0 / (double)m.T0;
    const double mean = sum * inv_n;
    double var = sq * inv_n - mean * mean;
    var = var > 0.0 ? var : 0.0;
    const double a = (double)gn_g[c] / sqrt(var + 1e-5);
    float* o = fold + ((long long)b * CONV_DIM + c) * 12;
#pragma unroll
    for (int j = 0; j < 10; ++j) o[j] = (float)(w[j] * a);
    o[10] = (float)((double)gn_b[c] - mean * a);
    o[11] = (float)a;  // gamma * rstd, folded into the saved GELU gradient for the loss backward
    if (fold_h != nullptr) {  // 16-bit taps for the tensor-core conv0 (B operands of two mma.sync k-steps, see there)
        uint32_t* h = reinterpret_cast<uint32_t*>(fold_h + ((long long)b * CONV_DIM + c) * 32);
        uint32_t hi[5], lo[5];
#pragma unroll
        for (int j = 0; j < 5; ++j) {
            const float t0 = (float)(w[2 * j] * a), t1 = (float)(w[2 * j + 1] * a);
            hi[j] = pack_op(t0, t1);
            const float2 hf = unpack_op(hi[j]);
            lo[j] = pack_op(t0 - hf.x, t1 - hf.y);
        }
        // k-step 1: [wh0..wh9 | wh0..wh5]      k-step 2: [wh6..wh9 | wl0..wl9 | 0 0]
#pragma unroll
        for (int j = 0; j < 5; ++j) h[j] = hi[j];
        h[5] = hi[0]; h[6] = hi[1]; h[7] = hi[2];
        h[8] = hi[3]; h[9] = hi[4];
#pragma unroll
        for (int j = 0; j < 5; ++j) h[10 + j] = lo[j];
        h[15] = 0u;
    }
    if (stat_out != nullptr) {
        stat_out[((long long)b * CONV_DIM + c) * 2 + 0] = (float)mean;
        stat_out[((long long)b * CONV_DIM + c) * 2 + 1] = (float)(1.0 / sqrt(var + 1e-5));
    }
}

int launch_gn_fold(cudaStream_t st, const double* part, const UttMeta* meta, int b0, int nb, int max_chunks,
                   const float* conv0_w, const float* gn_g, const float* gn_b, float* fold, float* stat_out,
                   op_t* fold_h) {
    gn_fold_kernel<<<nb, 512, 0, st>>>(part, meta, b0, max_chunks, conv0_w, gn_g, gn_b, fold, stat_out, fold_h);
    NB_LAUNCHED();
    return 0;
}

__global__ void __launch_bounds__(512) fold_unit_dgelu_gain_kernel(float* __restrict__ fold, int b0) {
    fold[((long long)(b0 + blockIdx.x) * CONV_DIM + threadIdx.x) * 12 + 11] = 1.f;
}

int launch_fold_unit_dgelu_gain(cudaStream_t st, float* fold, int b0, int nb) {
    fold_unit_dgelu_gain_kernel<<<nb, CONV_DIM, 0, st>>>(fold, b0);
    NB_LAUNCHED();
    return 0;
}

// ---------------------------------------------------------------------------------------------
// One block = 64 consecutive level-0 rows (always inside one utterance: rows0 is a multiple of 64),
// 256 threads x 2 channels.  out[row][c] = GELU(sum_j fold[c][j] x[5 t + j] + shift[c]) as op_t,
// zeros for the padding rows t >= T0.
static constexpr int C0_ROWS = 64;

__global__ void __launch_bounds__(256) conv0_apply_kernel(const float* __restrict__ wav,
                                                          const UttMeta* __restrict__ meta, int B, int blk0,
                                                          const float* __restrict__ fold, op_t* __restrict__ out,
                                                          op_t* __restrict__ aux_out) {
    const int blk = blk0 + blockIdx.x;
    const int row_base = blk * C0_ROWS;
    // utterance lookup: frame-level offsets are row offsets / 64
    const int b = find_utt_by_frame(meta, B, blk);
    const UttMeta m = meta[b];
    const int t_base = row_base - m.row0;
    __shared__ float xs[C0_ROWS * 5 + 8];
    const float* x = wav + m.wav_off;
    for (int i = threadIdx.x; i < C0_ROWS * 5 + 5; i += blockDim.x) {
        const long long s = (long long)t_base * 5 + i;
        xs[i] = (s < m.n) ? __ldg(x + s) : 0.f;
    }
    const int c = 2 * threadIdx.x;
    float w0[12], w1[12];
    {
        const float4* f = reinterpret_cast<const float4*>(fold + ((long long)b * CONV_DIM + c) * 12);
        const float4 a0 = __ldg(f), a1 = __ldg(f + 1), a2 = __ldg(f + 2), a3 = __ldg(f + 3), a4 = __ldg(f + 4),
                     a5 = __ldg(f + 5);
        w0[0] = a0.x; w0[1] = a0.y; w0[2] = a0.z; w0[3] = a0.w; w0[4] = a1.x; w0[5] = a1.y; w0[6] = a1.z;
        w0[7] = a1.w; w0[8] = a2.x; w0[9] = a2.y; w0[10] = a2.z; w0[11] = a2.w;
        w1[0] = a3.x; w1[1] = a3.y; w1[2] = a3.z; w1[3] = a3.w; w1[4] = a4.x; w1[5] = a4.y; w1[6] = a4.z;
        w1[7] = a4.w; w1[8] = a5.x; w1[9] = a5.y; w1[10] = a5.z; w1[11] = a5.w;
    }
    __syncthreads();
    uint32_t* o = reinterpret_cast<uint32_t*>(out + (long long)row_base * CONV_DIM + c);
    const int valid = m.T0 - t_base;  // rows of this block that are real frames
    if (aux_out == nullptr) {
        // sliding 10-sample window: frame t+1 reuses samples 5..9 of frame t, so 5 shared loads per frame
        float xw[10];
#pragma unroll
        for (int j = 0; j < 5; ++j) xw[5 + j] = xs[j];
#pragma unroll 4
        for (int t = 0; t < C0_ROWS; ++t) {
#pragma unroll
            for (int j = 0; j < 5; ++j) { xw[j] = xw[5 + j]; xw[5 + j] = xs[5 * t + 5 + j]; }
            uint32_t packed = 0u;
            if (t < valid) {
                float y0 = w0[10], y1 = w1[10];
#pragma unroll
                for (int j = 0; j < 10; ++j) {
                    y0 = fmaf(w0[j], xw[j], y0);
                    y1 = fmaf(w1[j], xw[j], y1);
                }
                packed = pack_op(gelu_act(y0), gelu_act(y1));
            }
            o[(long long)t * (CONV_DIM / 2)] = packed;
        }
    } else {
        uint32_t* ao = reinterpret_cast<uint32_t*>(aux_out + (long long)row_base * CONV_DIM + c);
#pragma unroll 2
        for (int t = 0; t < C0_ROWS; ++t) {
            uint32_t packed = 0u, gpacked = 0u;
            if (t < valid) {
                float y0 = w0[10], y1 = w1[10];
#pragma unroll
                for (int j = 0; j < 10; ++j) {
                    const float xv = xs[5 * t + j];
                    y0 = fmaf(w0[j], xv, y0);
                    y1 = fmaf(w1[j], xv, y1);
                }
                float g0, g1;
                y0 = gelu_erf_with_grad(y0, g0);
                y1 = gelu_erf_with_grad(y1, g1);
                packed = pack_op(y0, y1);
                gpacked = pack_op(g0 * w0[11], g1 * w1[11]);
            }
            o[(long long)t * (CONV_DIM / 2)] = packed;
            ao[(long long)t * (CONV_DIM / 2)] = gpacked;
        }
    }
}

// rows [T_l, rows_l) of each utterance at conv level l := 0
__global__ void __launch_bounds__(256) zero_pad_rows_kernel(op_t* __restrict__ buf, const UttMeta* __restrict__ meta,
                                                            int level) {
    const UttMeta m = meta[blockIdx.x];
    int T = m.T0;
    for (int l = 1; l <= level; ++l) T = (T - (l < 5 ? 3 : 2)) / 2 + 1;
    const long long r0 = ((long long)m.row0 >> level) + T, r1 = ((long long)m.row0 + m.rows0) >> level;
    uint4* p = reinterpret_cast<uint4*>(buf + r0 * CONV_DIM);
    const long long n = (r1 - r0) * (CONV_DIM / 8);
    for (long long i = threadIdx.x; i < n; i += blockDim.x) p[i] = make_uint4(0u, 0u, 0u, 0u);
}

int launch_zero_pad_rows(cudaStream_t st, op_t* buf, const UttMeta* meta, int B, int level) {
    zero_pad_rows_kernel<<<B, 256, 0, st>>>(buf, meta, level);
    NB_LAUNCHED();
    return 0;
}

// ---------------------------------------------------------------------------------------------
// Tensor-core conv0: the 10-tap stride-5 conv as mma.sync m16n8k16 (fp16 in, fp32 accumulate):
//   A[t][k] = x[5 t + k] (k < 16; taps 10..15 meet zero weights),  B[k][c] = folded taps (GroupNorm folded in).
// fp16 carries 11 bits, 16-bit PCM and trained band-pass taps need more: on real speech a plain fp16 product was
// measured 3-80x noisier than the fp16 rounding of the output (a filter's stop-band leakage scales with the
// quantisation of its taps and of the samples).  So samples and taps are split x = xh + xl, w = wh + wl and
// the product is xh wh + xl wh + xh wl (error ~2^-22, below fp32 accumulation noise): 30 products per output,
// packed into TWO k = 16 steps --
//   step 1: K slots 0..9 = xh_j wh_j,  10..15 = xl_j wh_j (j = 0..5)
//   step 2: K slots 0..3 = xl_j wh_j (j = 6..9),  4..13 = xh_j wl_j,  14..15 unused (zero taps).
// One block = 64 frames x 512 channels, warp w owns channels [64 w, 64 w + 64).  The scalar kernel above spends
// 20 of its ~27 instructions per element on FMAs and shared loads; here the FMAs are 32 mma per warp and what
// remains is the GELU.  Lanes of a quad trade halves so every store instruction writes full 32 B sectors.
__device__ __forceinline__ void mma_f16_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

template <int NT>  // 0: row-major tiles + quad shuffles (round 1); 2 / 4: channel-permuted groups of NT tiles, direct stores
__global__ void __launch_bounds__(256, NB_CONV0_BLOCKS) conv0_mma_kernel(const float* __restrict__ wav, const UttMeta* __restrict__ meta,
                                                        int B, int blk0, const float* __restrict__ fold,
                                                        const op_t* __restrict__ fold_h, op_t* __restrict__ out) {
    const int blk = blk0 + blockIdx.x;
    const int row_base = blk * C0_ROWS;
    const int b = find_utt_by_frame(meta, B, blk);
    const UttMeta m = meta[b];
    const int t_base = row_base - m.row0;
    __shared__ float xs[C0_ROWS * 5 + 16];
    const float* x = wav + m.wav_off;
    for (int i = threadIdx.x; i < C0_ROWS * 5 + 16; i += blockDim.x) {
        const long long s = (long long)t_base * 5 + i;
        xs[i] = (s < m.n) ? __ldg(x + s) : 0.f;
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int r = lane >> 2, q = lane & 3;
    __syncthreads();
    const int valid = m.T0 - t_base;
    // A fragments of the two k-steps for all four 16-row tiles of the block (32 registers, built once):
    // a[0], a[1] = K slots 2q, 2q+1 of rows r, r+8; a[2], a[3] = slots 2q+8, 2q+9
    uint32_t a1[4][4], a2[4][4];
#pragma unroll
    for (int mt = 0; mt < 4; ++mt) {
        const int ib[2] = {5 * (mt * 16 + r), 5 * (mt * 16 + r) + 40};  // first sample of rows r and r + 8
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const float* x = xs + ib[k];
            // step 1, slots 2q, 2q+1: xh[2q], xh[2q+1]
            a1[mt][k] = pack_op(x[2 * q], x[2 * q + 1]);
            // step 1, slots 2q+8, 2q+9: q = 0 -> xh[8], xh[9];  q >= 1 -> xl[2q-2], xl[2q-1]
            {
                const int o = q == 0 ? 8 : 2 * q - 2;
                const float x0 = x[o], x1 = x[o + 1];
                const uint32_t hh = pack_op(x0, x1);
                const float2 hf = unpack_op(hh);
                a1[mt][2 + k] = q == 0 ? hh : pack_op(x0 - hf.x, x1 - hf.y);
            }
            // step 2, slots 2q, 2q+1: q < 2 -> xl[6+2q], xl[7+2q];  q >= 2 -> xh[2q-4], xh[2q-3]
            {
                const int o = q < 2 ? 6 + 2 * q : 2 * q - 4;
                const float x0 = x[o], x1 = x[o + 1];
                const uint32_t hh = pack_op(x0, x1);
                const float2 hf = unpack_op(hh);
                a2[mt][k] = q < 2 ? pack_op(x0 - hf.x, x1 - hf.y) : hh;
            }
            // step 2, slots 2q+8, 2q+9 = xh[2q+4], xh[2q+5] (q = 3: slots 14, 15 meet zero taps)
            a2[mt][2 + k] = pack_op(x[2 * q + 4], x[2 * q + 5]);
        }
    }
    if constexpr (NT == 0) {
    op_t* obase = out + (long long)(row_base + r) * CONV_DIM + warp * 64 + 4 * q;
    const int src = (lane & ~3) | ((2 * q) & 3);
#pragma unroll 1
    for (int np = 0; np < 4; ++np) {  // pairs of channel tiles: 16 channels = 32 B per row per quad
        // B fragments + shifts of the two 8-channel tiles (streamed: they are L1-resident, the A side is not)
        uint32_t bf[2][2], bl[2][2];
        float sh[2][2];
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const int cb = warp * 64 + (2 * np + i) * 8;
            const uint32_t* h = reinterpret_cast<const uint32_t*>(fold_h + ((long long)b * CONV_DIM + cb + r) * 32);
            bf[i][0] = __ldg(h + q);
            bf[i][1] = __ldg(h + q + 4);
            bl[i][0] = __ldg(h + 8 + q);
            bl[i][1] = __ldg(h + 8 + q + 4);
            sh[i][0] = __ldg(fold + ((long long)b * CONV_DIM + cb + 2 * q) * 12 + 10);
            sh[i][1] = __ldg(fold + ((long long)b * CONV_DIM + cb + 2 * q + 1) * 12 + 10);
        }
#pragma unroll
        for (int mt = 0; mt < 4; ++mt) {
            float c0[4] = {sh[0][0], sh[0][1], sh[0][0], sh[0][1]};
            float c1[4] = {sh[1][0], sh[1][1], sh[1][0], sh[1][1]};
            mma_f16_16816(c0, a2[mt], bl[0][0], bl[0][1]);
            mma_f16_16816(c1, a2[mt], bl[1][0], bl[1][1]);
            mma_f16_16816(c0, a1[mt], bf[0][0], bf[0][1]);
            mma_f16_16816(c1, a1[mt], bf[1][0], bf[1][1]);
            // packed pairs: e = tile 2np (cols 2q, 2q+1), f = tile 2np+1, rows row0 / row1
#if NB_CONV0_GELU_H2
            uint32_t e0 = gelu_pair_h2(c0[0], c0[1]), e1 = gelu_pair_h2(c0[2], c0[3]);
            uint32_t f0 = gelu_pair_h2(c1[0], c1[1]), f1 = gelu_pair_h2(c1[2], c1[3]);
#else
            uint32_t e0 = pack_op(gelu_act(c0[0]), gelu_act(c0[1])), e1 = pack_op(gelu_act(c0[2]), gelu_act(c0[3]));
            uint32_t f0 = pack_op(gelu_act(c1[0]), gelu_act(c1[1])), f1 = pack_op(gelu_act(c1[2]), gelu_act(c1[3]));
#endif
            // lane q stores channels 4q..4q+3 of the 16: q<2 -> from tile 2np lanes (2q, 2q+1); q>=2 -> tile 2np+1
            const uint32_t a_e0 = __shfl_sync(0xffffffffu, e0, src), b_e0 = __shfl_sync(0xffffffffu, e0, src + 1);
            const uint32_t a_f0 = __shfl_sync(0xffffffffu, f0, src), b_f0 = __shfl_sync(0xffffffffu, f0, src + 1);
            const uint32_t a_e1 = __shfl_sync(0xffffffffu, e1, src), b_e1 = __shfl_sync(0xffffffffu, e1, src + 1);
            const uint32_t a_f1 = __shfl_sync(0xffffffffu, f1, src), b_f1 = __shfl_sync(0xffffffffu, f1, src + 1);
            uint2 v0 = q < 2 ? make_uint2(a_e0, b_e0) : make_uint2(a_f0, b_f0);
            uint2 v1 = q < 2 ? make_uint2(a_e1, b_e1) : make_uint2(a_f1, b_f1);
            const int row0 = mt * 16 + r, row1 = row0 + 8;
            if (row0 >= valid) v0 = make_uint2(0u, 0u);
            if (row1 >= valid) v1 = make_uint2(0u, 0u);
            *reinterpret_cast<uint2*>(obase + (long long)(mt * 16) * CONV_DIM + np * 16) = v0;
            *reinterpret_cast<uint2*>(obase + (long long)(mt * 16 + 8) * CONV_DIM + np * 16) = v1;
        }
    }
    } else {
    // Channel-permuted tiles: the MMA's N axis is only a labelling of output channels, so column j of tile i of a group of NT
    // tiles is made to carry channel 2 NT (j >> 1) + 2 i + (j & 1) of the group.  Lane q (which holds columns 2q, 2q+1 of every
    // tile) then owns the 2 NT CONSECUTIVE channels 2 NT q .. 2 NT q + 2 NT - 1 of a row: one 8 / 16-byte store, no shuffles.
    constexpr int GC = 8 * NT;  // channels per group
    op_t* obase = out + (long long)(row_base + r) * CONV_DIM + warp * 64 + 2 * NT * q;
#pragma unroll 1
    for (int np = 0; np < 64 / GC; ++np) {
        uint32_t bf[NT][2], bl[NT][2];
        float sh[NT][2];
        const int cb = warp * 64 + np * GC;
#pragma unroll
        for (int i = 0; i < NT; ++i) {
            const int cn = cb + 2 * NT * (r >> 1) + 2 * i + (r & 1);  // channel carried by column r of tile i
            const uint32_t* h = reinterpret_cast<const uint32_t*>(fold_h + ((long long)b * CONV_DIM + cn) * 32);
            bf[i][0] = __ldg(h + q);
            bf[i][1] = __ldg(h + q + 4);
            bl[i][0] = __ldg(h + 8 + q);
            bl[i][1] = __ldg(h + 8 + q + 4);
            const int cq = cb + 2 * NT * q + 2 * i;                   // channels of columns 2q, 2q+1 of tile i
            sh[i][0] = __ldg(fold + ((long long)b * CONV_DIM + cq) * 12 + 10);
            sh[i][1] = __ldg(fold + ((long long)b * CONV_DIM + cq + 1) * 12 + 10);
        }
#pragma unroll
        for (int mt = 0; mt < 4; ++mt) {
            uint32_t lo[NT], hi[NT];  // rows r / r + 8, channels 2 NT q + 2 i, + 1
#pragma unroll
            for (int i = 0; i < NT; ++i) {
                float c[4] = {sh[i][0], sh[i][1], sh[i][0], sh[i][1]};
                mma_f16_16816(c, a2[mt], bl[i][0], bl[i][1]);
                mma_f16_16816(c, a1[mt], bf[i][0], bf[i][1]);
#if NB_CONV0_GELU_H2
                lo[i] = gelu_pair_h2(c[0], c[1]);
                hi[i] = gelu_pair_h2(c[2], c[3]);
#else
                lo[i] = pack_op(gelu_act(c[0]), gelu_act(c[1]));
                hi[i] = pack_op(gelu_act(c[2]), gelu_act(c[3]));
#endif
            }
            const int row0 = mt * 16 + r, row1 = row0 + 8;
            const bool ok0 = row0 < valid, ok1 = row1 < valid;
            op_t* o0 = obase + (long long)(mt * 16) * CONV_DIM + np * GC;
            op_t* o1 = o0 + 8 * CONV_DIM;
            if constexpr (NT == 2) {
                *reinterpret_cast<uint2*>(o0) = ok0 ? make_uint2(lo[0], lo[1]) : make_uint2(0u, 0u);
                *reinterpret_cast<uint2*>(o1) = ok1 ? make_uint2(hi[0], hi[1]) : make_uint2(0u, 0u);
            } else {
                *reinterpret_cast<uint4*>(o0) = ok0 ? make_uint4(lo[0], lo[1], lo[2], lo[3]) : make_uint4(0u, 0u, 0u, 0u);
                *reinterpret_cast<uint4*>(o1) = ok1 ? make_uint4(hi[0], hi[1], hi[2], hi[3]) : make_uint4(0u, 0u, 0u, 0u);
            }
        }
    }
    }
}

// Variant 4: the A fragments (hi / lo split samples in mma layout) depend on (row tile, lane) only, not on the warp's channel
// range -- so warps 0..3 build one row tile each ONCE per block into shared memory (4 KB) instead of all 8 warps building all four
// (12 % of the kernel's instructions), and every warp reads the 8 registers of the tile it is working on with two LDS.128.
// That frees 24 registers: 64 per thread, FOUR blocks per SM (32 warps instead of 24) for a kernel bound by instruction latency.
template <int MINB>
__global__ void __launch_bounds__(256, MINB) conv0_mma_s_kernel(const float* __restrict__ wav, const UttMeta* __restrict__ meta,
                                                             int B, int blk0, const float* __restrict__ fold,
                                                             const op_t* __restrict__ fold_h, op_t* __restrict__ out) {
    const int blk = blk0 + blockIdx.x;
    const int row_base = blk * C0_ROWS;
    const int b = find_utt_by_frame(meta, B, blk);
    const UttMeta m = meta[b];
    const int t_base = row_base - m.row0;
    __shared__ float xs[C0_ROWS * 5 + 16];
    __shared__ uint4 frag[4][2][32];  // [row tile][k-step][lane]
    const float* x = wav + m.wav_off;
    for (int i = threadIdx.x; i < C0_ROWS * 5 + 16; i += blockDim.x) {
        const long long s = (long long)t_base * 5 + i;
        xs[i] = (s < m.n) ? __ldg(x + s) : 0.f;
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int r = lane >> 2, q = lane & 3;
    __syncthreads();
    const int valid = m.T0 - t_base;
    if (warp < 4) {
        const int mt = warp;
        uint32_t a1[4], a2[4];
        const int ib[2] = {5 * (mt * 16 + r), 5 * (mt * 16 + r) + 40};  // first sample of rows r and r + 8
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const float* x = xs + ib[k];
            a1[k] = pack_op(x[2 * q], x[2 * q + 1]);
            {
                const int o = q == 0 ? 8 : 2 * q - 2;
                const float x0 = x[o], x1 = x[o + 1];
                const uint32_t hh = pack_op(x0, x1);
                const float2 hf = unpack_op(hh);
                a1[2 + k] = q == 0 ? hh : pack_op(x0 - hf.x, x1 - hf.y);
            }
            {
                const int o = q < 2 ? 6 + 2 * q : 2 * q - 4;
                const float x0 = x[o], x1 = x[o + 1];
                const uint32_t hh = pack_op(x0, x1);
                const float2 hf = unpack_op(hh);
                a2[k] = q < 2 ? pack_op(x0 - hf.x, x1 - hf.y) : hh;
            }
            a2[2 + k] = pack_op(x[2 * q + 4], x[2 * q + 5]);
        }
        frag[mt][0][lane] = make_uint4(a1[0], a1[1], a1[2], a1[3]);
        frag[mt][1][lane] = make_uint4(a2[0], a2[1], a2[2], a2[3]);
    }
    __syncthreads();
    constexpr int NT = 2, GC = 8 * NT;
    op_t* obase = out + (long long)(row_base + r) * CONV_DIM + warp * 64 + 2 * NT * q;
#pragma unroll 1
    for (int np = 0; np < 64 / GC; ++np) {
        uint32_t bf[NT][2], bl[NT][2];
        float sh[NT][2];
        const int cb = warp * 64 + np * GC;
#pragma unroll
        for (int i = 0; i < NT; ++i) {
            const int cn = cb + 2 * NT * (r >> 1) + 2 * i + (r & 1);  // channel carried by column r of tile i
            const uint32_t* h = reinterpret_cast<const uint32_t*>(fold_h + ((long long)b * CONV_DIM + cn) * 32);
            bf[i][0] = __ldg(h + q);
            bf[i][1] = __ldg(h + q + 4);
            bl[i][0] = __ldg(h + 8 + q);
            bl[i][1] = __ldg(h + 8 + q + 4);
            const int cq = cb + 2 * NT * q + 2 * i;
            sh[i][0] = __ldg(fold + ((long long)b * CONV_DIM + cq) * 12 + 10);
            sh[i][1] = __ldg(fold + ((long long)b * CONV_DIM + cq + 1) * 12 + 10);
        }
#pragma unroll
        for (int mt = 0; mt < 4; ++mt) {
            const uint4 f1 = frag[mt][0][lane], f2 = frag[mt][1][lane];
            const uint32_t a1[4] = {f1.x, f1.y, f1.z, f1.w}, a2[4] = {f2.x, f2.y, f2.z, f2.w};
            uint32_t lo[NT], hi[NT];
#pragma unroll
            for (int i = 0; i < NT; ++i) {
                float c[4] = {sh[i][0], sh[i][1], sh[i][0], sh[i][1]};
                mma_f16_16816(c, a2, bl[i][0], bl[i][1]);
                mma_f16_16816(c, a1, bf[i][0], bf[i][1]);
                lo[i] = gelu_pair_h2(c[0], c[1]);
                hi[i] = gelu_pair_h2(c[2], c[3]);
            }
            const int row0 = mt * 16 + r, row1 = row0 + 8;
            op_t* o0 = obase + (long long)(mt * 16) * CONV_DIM + np * GC;
            *reinterpret_cast<uint2*>(o0) = row0 < valid ? make_uint2(lo[0], lo[1]) : make_uint2(0u, 0u);
            *reinterpret_cast<uint2*>(o0 + 8 * CONV_DIM) = row1 < valid ? make_uint2(hi[0], hi[1]) : make_uint2(0u, 0u);
        }
    }
}

int launch_conv0_apply(cudaStream_t st, const float* wav, const UttMeta* meta, int B, long long row_begin,
                       long long row_end, const float* fold, const op_t* fold_h, op_t* out, op_t* aux_out) {
    static const int use_mma = getenv("NOMAD_B200_CONV0_MMA") ? atoi(getenv("NOMAD_B200_CONV0_MMA")) : 4;  // 0 SIMT; 1 row-major tiles + shuffles 1.36-1.42 ms; 2 / 3 channel-permuted 1.27 / 1.45; 4 / 5 = 2 + shared A fragments at 4 / 3 blocks per SM 1.16 / 1.29
    const unsigned blocks = (unsigned)((row_end - row_begin) / C0_ROWS);
    const int blk0 = (int)(row_begin / C0_ROWS);
    if (blocks == 0) return 0;
    if (aux_out == nullptr && fold_h != nullptr && use_mma) {
        if (use_mma == 4) conv0_mma_s_kernel<4><<<blocks, 256, 0, st>>>(wav, meta, B, blk0, fold, fold_h, out);
        else if (use_mma == 5) conv0_mma_s_kernel<3><<<blocks, 256, 0, st>>>(wav, meta, B, blk0, fold, fold_h, out);
        else if (use_mma == 2) conv0_mma_kernel<2><<<blocks, 256, 0, st>>>(wav, meta, B, blk0, fold, fold_h, out);
        else if (use_mma == 3) conv0_mma_kernel<4><<<blocks, 256, 0, st>>>(wav, meta, B, blk0, fold, fold_h, out);
        else conv0_mma_kernel<0><<<blocks, 256, 0, st>>>(wav, meta, B, blk0, fold, fold_h, out);
        NB_LAUNCHED();
        return 0;
    }
    conv0_apply_kernel<<<blocks, 256, 0, st>>>(wav, meta, B, blk0, fold, out, aux_out);
    NB_LAUNCHED();
    return 0;
}

// ---------------------------------------------------------------------------------------------
// LayerNorm over 512 channels, op_t in -> op_t out, one warp per row (16 values per lane).
__global__ void __launch_bounds__(256) ln512_kernel(const op_t* __restrict__ in, long long rows,
                                                    const float* __restrict__ g, const float* __restrict__ bta,
                                                    op_t* __restrict__ out) {
    const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= rows) return;
    const int lane = threadIdx.x & 31;
    const uint4* p = reinterpret_cast<const uint4*>(in + row * CONV_DIM);
    float v[16];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const uint4 u = __ldg(p + lane + 32 * h);
        float2 f;
        f = unpack_op(u.x); v[8 * h + 0] = f.x; v[8 * h + 1] = f.y;
        f = unpack_op(u.y); v[8 * h + 2] = f.x; v[8 * h + 3] = f.y;
        f = unpack_op(u.z); v[8 * h + 4] = f.x; v[8 * h + 5] = f.y;
        f = unpack_op(u.w); v[8 * h + 6] = f.x; v[8 * h + 7] = f.y;
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) s += v[i];
    const float mean = warp_sum(s) * (1.0f / CONV_DIM);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) { const float d = v[i] - mean; q = fmaf(d, d, q); }
    const float rstd = rsqrtf(warp_sum(q) * (1.0f / CONV_DIM) + 1e-5f);
    uint4* o = reinterpret_cast<uint4*>(out + row * CONV_DIM);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int c0 = (lane + 32 * h) * 8;
        const float4 g0 = __ldg(reinterpret_cast<const float4*>(g + c0)), g1 = __ldg(reinterpret_cast<const float4*>(g + c0 + 4));
        const float4 b0 = __ldg(reinterpret_cast<const float4*>(bta + c0)), b1 = __ldg(reinterpret_cast<const float4*>(bta + c0 + 4));
        float r[8];
        r[0] = (v[8 * h + 0] - mean) * rstd * g0.x + b0.x; r[1] = (v[8 * h + 1] - mean) * rstd * g0.y + b0.y;
        r[2] = (v[8 * h + 2] - mean) * rstd * g0.z + b0.z; r[3] = (v[8 * h + 3] - mean) * rstd * g0.w + b0.w;
        r[4] = (v[8 * h + 4] - mean) * rstd * g1.x + b1.x; r[5] = (v[8 * h + 5] - mean) * rstd * g1.y + b1.y;
        r[6] = (v[8 * h + 6] - mean) * rstd * g1.z + b1.z; r[7] = (v[8 * h + 7] - mean) * rstd * g1.w + b1.w;
        o[lane + 32 * h] = make_uint4(pack_op(r[0], r[1]), pack_op(r[2], r[3]), pack_op(r[4], r[5]),
                                      pack_op(r[6], r[7]));
    }
}

int launch_ln512(cudaStream_t st, const op_t* in, long long rows, const float* g, const float* b, op_t* out) {
    if (rows <= 0) return 0;
    ln512_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, st>>>(in, rows, g, b, out);
    NB_LAUNCHED();
    return 0;
}

}  // namespace nb
