// fp32-class ("precise") scoring path: precision_mode = 1 of nomad_b200_create.
//
// The reference computes everything in fp32 (nomad.py:226-230; fairseq / ATen).  The default path of this library
// feeds the tensor cores fp16 operands (max-abs embedding error ~3.5e-4 against the fp32 reference: the north star's
// "bf16/tf32 class", <= 1e-3).  This file is the "fp32 mode" (<= 1e-5): every tensor-core operand is carried as TWO
// fp16 planes, x = hi + lo with hi = fp16(x), lo = fp16(x - hi) (~22 significant bits), and every GEMM runs three K
// segments into one TMEM accumulator, A_hi B_hi + A_lo B_hi + A_hi B_lo (gemm.cu, PREC instantiations) -- the same
// trick the distance kernel and conv0 already use.  Weights are stored times a power of two so that their lo planes
// stay in fp16's normal range; everything that is not a GEMM operand (residual stream, LayerNorm, softmax, GELU via
// libdevice erff, the QKV rows the attention kernel reads) stays fp32, and the attention core runs on the fp32 CUDA
// cores.  Nothing here is shared with the fp16 path except the GEMM mainloop, the GroupNorm statistics and the pooled
// head, so the two modes check each other in the GPU tests.
#include <cmath>
#include <cstring>

#include "precise.cuh"

namespace nb {

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// ------------------------------------------------------------------------------------------------ conv0
// out[row][c] = GELU(sum_j fold[c][j] x[5 t + j] + shift[c]) with the GroupNorm folded into the taps (frontend.cu),
// fp32 FMAs, libdevice erff, stored as hi + lo planes; zeros for the padding rows t >= T0.  pre_out (save mode, may be
// null): the GELU input, fp32.
__global__ void __launch_bounds__(256) conv0_precise_kernel(const float* __restrict__ wav, const UttMeta* __restrict__ meta,
                                                            int B, const float* __restrict__ fold, op_t* __restrict__ out_hi,
                                                            op_t* __restrict__ out_lo, float* __restrict__ pre_out) {
    const int blk = blockIdx.x;
    const int row_base = blk * 64;
    const int b = find_utt_by_frame(meta, B, blk);
    const UttMeta m = meta[b];
    const int t_base = row_base - m.row0;
    __shared__ float xs[64 * 5 + 8];
    const float* x = wav + m.wav_off;
    for (int i = threadIdx.x; i < 64 * 5 + 5; i += blockDim.x) {
        const long long s = (long long)t_base * 5 + i;
        xs[i] = (s < m.n) ? __ldg(x + s) : 0.f;
    }
    const int c = 2 * threadIdx.x;
    float w0[11], w1[11];
    {
        const float* f = fold + ((long long)b * CONV_DIM + c) * 12;
#pragma unroll
        for (int j = 0; j < 11; ++j) { w0[j] = __ldg(f + j); w1[j] = __ldg(f + 12 + j); }
    }
    __syncthreads();
    uint32_t* oh = reinterpret_cast<uint32_t*>(out_hi + (long long)row_base * CONV_DIM + c);
    uint32_t* ol = reinterpret_cast<uint32_t*>(out_lo + (long long)row_base * CONV_DIM + c);
    const int valid = m.T0 - t_base;
    for (int t = 0; t < 64; ++t) {
        uint32_t ph = 0u, pl = 0u;
        if (t < valid) {
            float y0 = w0[10], y1 = w1[10];
#pragma unroll
            for (int j = 0; j < 10; ++j) {
                const float xv = xs[5 * t + j];
                y0 = fmaf(w0[j], xv, y0);
                y1 = fmaf(w1[j], xv, y1);
            }
            if (pre_out != nullptr)
                *reinterpret_cast<float2*>(pre_out + (long long)(row_base + t) * CONV_DIM + c) = make_float2(y0, y1);
            y0 = gelu_erf_exact(y0);
            y1 = gelu_erf_exact(y1);
            ph = pack_op(y0, y1);
            const float2 f = unpack_op(ph);
            pl = pack_op(y0 - f.x, y1 - f.y);
        }
        oh[(long long)t * (CONV_DIM / 2)] = ph;
        ol[(long long)t * (CONV_DIM / 2)] = pl;
        if (pre_out != nullptr && t >= valid)
            *reinterpret_cast<float2*>(pre_out + (long long)(row_base + t) * CONV_DIM + c) = make_float2(0.f, 0.f);
    }
}

// save mode: GELU of the fp32 pre-activations `in` (n values, n % 8 == 0) to hi + lo planes and / or fp32 `out`
__global__ void __launch_bounds__(256) gelu_precise_kernel(const float* __restrict__ in, long long n, op_t* __restrict__ hi,
                                                           op_t* __restrict__ lo, float* __restrict__ out) {
    const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 8;
    if (i >= n) return;
    const float4 a = __ldg(reinterpret_cast<const float4*>(in + i)), b = __ldg(reinterpret_cast<const float4*>(in + i + 4));
    float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = gelu_erf_exact(v[j]);
    if (hi != nullptr) split_store8(v, hi + i, lo + i);
    if (out != nullptr) {
        *reinterpret_cast<float4*>(out + i) = make_float4(v[0], v[1], v[2], v[3]);
        *reinterpret_cast<float4*>(out + i + 4) = make_float4(v[4], v[5], v[6], v[7]);
    }
}
static int launch_gelu_precise(cudaStream_t st, const float* in, long long n, op_t* hi, op_t* lo, float* out) {
    gelu_precise_kernel<<<(unsigned)((n / 8 + 255) / 256), 256, 0, st>>>(in, n, hi, lo, out);
    NB_LAUNCHED();
    return 0;
}

// ------------------------------------------------------------------------------------------------ LayerNorm(512)
__global__ void __launch_bounds__(256) ln512_precise_kernel(const op_t* __restrict__ in_hi, const op_t* __restrict__ in_lo,
                                                            long long rows, const float* __restrict__ g,
                                                            const float* __restrict__ bta, op_t* __restrict__ out_hi,
                                                            op_t* __restrict__ out_lo) {
    const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= rows) return;
    const int lane = threadIdx.x & 31;
    float v[16];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const long long o = row * CONV_DIM + (lane + 32 * h) * 8;
        split_load8(in_hi + o, in_lo + o, v + 8 * h);
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) s += v[i];
    const float mean = warp_sum(s) * (1.0f / CONV_DIM);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) { const float d = v[i] - mean; q = fmaf(d, d, q); }
    const float rstd = 1.0f / sqrtf(warp_sum(q) * (1.0f / CONV_DIM) + 1e-5f);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int c0 = (lane + 32 * h) * 8;
        float r[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) r[i] = (v[8 * h + i] - mean) * rstd * __ldg(g + c0 + i) + __ldg(bta + c0 + i);
        split_store8(r, out_hi + row * CONV_DIM + c0, out_lo + row * CONV_DIM + c0);
    }
}

// ------------------------------------------------------------------------------------------------ positional conv staging
__global__ void __launch_bounds__(384) pos_scatter_precise_kernel(const float* __restrict__ x, const UttMeta* __restrict__ meta,
                                                                  int B, long long frames, long long pos_rows_alloc,
                                                                  op_t* __restrict__ g_hi, op_t* __restrict__ g_lo) {
    const long long f = (long long)blockIdx.x * 4 + threadIdx.x / 96;
    if (f >= frames) return;
    const int i = threadIdx.x % 96;  // 8-channel chunk
    const int b = find_utt_by_frame(meta, B, (int)f);
    const int t = (int)f - meta[b].frame0;
    if (t >= meta[b].T) return;
    const long long p = meta[b].pos0 + t;
    const float4* src = reinterpret_cast<const float4*>(x + f * EMBED + i * 8);
    const float4 a = __ldg(src), c = __ldg(src + 1);
    const float v[8] = {a.x, a.y, a.z, a.w, c.x, c.y, c.z, c.w};
    const int ch = i * 8, g = ch / POS_GC, cc = ch % POS_GC;
    const long long o = ((long long)g * pos_rows_alloc + p) * POS_GC + cc;
    split_store8(v, g_hi + o, g_lo + o);
}

// ------------------------------------------------------------------------------------------------ LayerNorm(768)
// one warp per frame; lane owns the 8-channel chunks {lane, lane + 32, lane + 64}
__device__ __forceinline__ void ln768_precise_row(float (&v)[24], const float* __restrict__ g, const float* __restrict__ bta,
                                                  int lane) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 24; ++i) s += v[i];
    const float mean = warp_sum(s) * (1.0f / EMBED);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < 24; ++i) { const float d = v[i] - mean; q = fmaf(d, d, q); }
    const float rstd = 1.0f / sqrtf(warp_sum(q) * (1.0f / EMBED) + 1e-5f);
#pragma unroll
    for (int h = 0; h < 3; ++h) {
        const int c0 = (lane + 32 * h) * 8;
#pragma unroll
        for (int i = 0; i < 8; ++i) v[8 * h + i] = (v[8 * h + i] - mean) * rstd * __ldg(g + c0 + i) + __ldg(bta + c0 + i);
    }
}
__device__ __forceinline__ void row768_precise_store(const float (&v)[24], bool valid, long long f, int lane,
                                                     float* __restrict__ x, op_t* __restrict__ xh, op_t* __restrict__ xl) {
#pragma unroll
    for (int h = 0; h < 3; ++h) {
        const int c0 = (lane + 32 * h) * 8;
        float r[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) r[i] = valid ? v[8 * h + i] : 0.f;
        float4* xo = reinterpret_cast<float4*>(x + f * EMBED + c0);
        xo[0] = make_float4(r[0], r[1], r[2], r[3]);
        xo[1] = make_float4(r[4], r[5], r[6], r[7]);
        split_store8(r, xh + f * EMBED + c0, xl + f * EMBED + c0);
    }
}

// x = LN(x0 + GELU(posconv)) on valid frames, 0 elsewhere; pos_y is fp32 in the padded row layout
__global__ void __launch_bounds__(256) pos_finish_ln_precise_kernel(const float* __restrict__ x0, const float* __restrict__ pos_y,
                                                                    const UttMeta* __restrict__ meta, int B, long long frames,
                                                                    const float* __restrict__ g, const float* __restrict__ bta,
                                                                    float* __restrict__ x, op_t* __restrict__ xh,
                                                                    op_t* __restrict__ xl) {
    const long long f = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (f >= frames) return;
    const int lane = threadIdx.x & 31;
    const int b = find_utt_by_frame(meta, B, (int)f);
    const int t = (int)f - meta[b].frame0;
    float v[24];
    const bool valid = t < meta[b].T;
    if (valid) {
        const long long m = (long long)meta[b].pos0 + t - POS_K / 2;
#pragma unroll
        for (int h = 0; h < 3; ++h) {
            const int c0 = (lane + 32 * h) * 8;
            const float4* xp = reinterpret_cast<const float4*>(x0 + f * EMBED + c0);
            const float4* yp = reinterpret_cast<const float4*>(pos_y + m * EMBED + c0);
            const float4 a = __ldg(xp), c = __ldg(xp + 1), ya = __ldg(yp), yc = __ldg(yp + 1);
            float* w = v + 8 * h;
            w[0] = a.x + ya.x; w[1] = a.y + ya.y; w[2] = a.z + ya.z; w[3] = a.w + ya.w;
            w[4] = c.x + yc.x; w[5] = c.y + yc.y; w[6] = c.z + yc.z; w[7] = c.w + yc.w;
        }
        ln768_precise_row(v, g, bta, lane);
    }
    row768_precise_store(v, valid, f, lane, x, xh, xl);
}

__global__ void __launch_bounds__(256) ln768_precise_kernel(const float* __restrict__ pre, const UttMeta* __restrict__ meta,
                                                            int B, long long frames, const float* __restrict__ g,
                                                            const float* __restrict__ bta, float* __restrict__ x,
                                                            op_t* __restrict__ xh, op_t* __restrict__ xl,
                                                            float* __restrict__ layer_out, int layer_T) {
    const long long f = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (f >= frames) return;
    const int lane = threadIdx.x & 31;
    const int b = find_utt_by_frame(meta, B, (int)f);
    const int t = (int)f - meta[b].frame0;
    float v[24];
    const bool valid = t < meta[b].T;
    if (valid) {
#pragma unroll
        for (int h = 0; h < 3; ++h) {
            const int c0 = (lane + 32 * h) * 8;
            const float4* xp = reinterpret_cast<const float4*>(pre + f * EMBED + c0);
            const float4 a = __ldg(xp), c = __ldg(xp + 1);
            float* w = v + 8 * h;
            w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w; w[4] = c.x; w[5] = c.y; w[6] = c.z; w[7] = c.w;
        }
        ln768_precise_row(v, g, bta, lane);
        if (layer_out != nullptr) {
            float* lo = layer_out + ((long long)b * layer_T + t) * EMBED;
#pragma unroll
            for (int h = 0; h < 3; ++h) {
                const int c0 = (lane + 32 * h) * 8;
                float4* o = reinterpret_cast<float4*>(lo + c0);
                o[0] = make_float4(v[8 * h], v[8 * h + 1], v[8 * h + 2], v[8 * h + 3]);
                o[1] = make_float4(v[8 * h + 4], v[8 * h + 5], v[8 * h + 6], v[8 * h + 7]);
            }
        }
    }
    row768_precise_store(v, valid, f, lane, x, xh, xl);
}

// ------------------------------------------------------------------------------------------------ attention core, fp32
// softmax(Q K^T) V per (utterance, head) on the fp32 cores: one CTA = 64 queries x one head, streaming 64-key tiles with
// an online softmax.  Thread (ty, tx) of the 16 x 16 layout owns queries 4 ty .. 4 ty + 3 and, in the two products,
// keys / output columns 4 tx .. 4 tx + 3 (4 x 4 register tiles fed by float4 shared loads).  q is already scaled by
// head_dim^-0.5 (folded into the QKV weights).  Output goes out as hi + lo planes (the out-projection's A operand);
// lse (save mode, may be null): frames x 12 log-sum-exp of the softmax rows.
static constexpr int PA_T = 64, PA_P = 68;  // tile edge, shared-memory row pitch (floats)
static constexpr int PA_SMEM = 4 * PA_T * PA_P * 4;

__global__ void __launch_bounds__(256) attention_precise_kernel(const float* __restrict__ qkv, const UttMeta* __restrict__ meta,
                                                                op_t* __restrict__ out_hi, op_t* __restrict__ out_lo,
                                                                float* __restrict__ lse) {
    const int b = blockIdx.z, h = blockIdx.y, q0 = blockIdx.x * PA_T;
    const int T = meta[b].T;
    if (q0 >= T) return;
    const long long f0 = meta[b].frame0;
    extern __shared__ __align__(16) float pa_sm[];
    float* Qt = pa_sm;                 // [d][q]
    float* Kt = Qt + PA_T * PA_P;      // [d][k]
    float* Vs = Kt + PA_T * PA_P;      // [k][d]
    float* Pt = Vs + PA_T * PA_P;      // [k][q]
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const float* base = qkv + f0 * (3 * EMBED) + h * HEAD_DIM;

    for (int idx = tid; idx < PA_T * 16; idx += 256) {
        const int r = idx >> 4, c4 = (idx & 15) * 4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (q0 + r < T) v = __ldg(reinterpret_cast<const float4*>(base + (long long)(q0 + r) * (3 * EMBED) + c4));
        Qt[(c4 + 0) * PA_P + r] = v.x; Qt[(c4 + 1) * PA_P + r] = v.y; Qt[(c4 + 2) * PA_P + r] = v.z; Qt[(c4 + 3) * PA_P + r] = v.w;
    }
    float o[4][4];
    float m_run[4], l_run[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        m_run[i] = -INFINITY;
        l_run[i] = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) o[i][j] = 0.f;
    }
    const int n_tiles = (T + PA_T - 1) / PA_T;
    for (int kt = 0; kt < n_tiles; ++kt) {
        const int k0 = kt * PA_T;
        __syncthreads();  // previous tile's P V product is done with Kt / Vs / Pt (and Qt is written, first time)
        for (int idx = tid; idx < PA_T * 16; idx += 256) {
            const int r = idx >> 4, c4 = (idx & 15) * 4;
            float4 kv = make_float4(0.f, 0.f, 0.f, 0.f), vv = kv;
            if (k0 + r < T) {
                const float* p = base + (long long)(k0 + r) * (3 * EMBED) + c4;
                kv = __ldg(reinterpret_cast<const float4*>(p + EMBED));
                vv = __ldg(reinterpret_cast<const float4*>(p + 2 * EMBED));
            }
            Kt[(c4 + 0) * PA_P + r] = kv.x; Kt[(c4 + 1) * PA_P + r] = kv.y; Kt[(c4 + 2) * PA_P + r] = kv.z; Kt[(c4 + 3) * PA_P + r] = kv.w;
            *reinterpret_cast<float4*>(Vs + r * PA_P + c4) = vv;
        }
        __syncthreads();
        float s[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) s[i][j] = 0.f;
#pragma unroll 8
        for (int d = 0; d < HEAD_DIM; ++d) {
            const float4 qa = *reinterpret_cast<const float4*>(Qt + d * PA_P + 4 * ty);
            const float4 ka = *reinterpret_cast<const float4*>(Kt + d * PA_P + 4 * tx);
            const float qv[4] = {qa.x, qa.y, qa.z, qa.w}, kv[4] = {ka.x, ka.y, ka.z, ka.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) s[i][j] = fmaf(qv[i], kv[j], s[i][j]);
        }
        float scale[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            float mx = -INFINITY;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (k0 + 4 * tx + j >= T) s[i][j] = -INFINITY;
                mx = fmaxf(mx, s[i][j]);
            }
#pragma unroll
            for (int w = 8; w > 0; w >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, w));  // the 16 tx lanes of this row group
            const float mn = fmaxf(m_run[i], mx);  // finite: every tile holds at least one valid key
            scale[i] = expf(m_run[i] - mn);
            m_run[i] = mn;
            float rs = 0.f;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                s[i][j] = expf(s[i][j] - mn);
                rs += s[i][j];
            }
#pragma unroll
            for (int w = 8; w > 0; w >>= 1) rs += __shfl_xor_sync(0xffffffffu, rs, w);
            l_run[i] = fmaf(l_run[i], scale[i], rs);
#pragma unroll
            for (int j = 0; j < 4; ++j) o[i][j] *= scale[i];
        }
#pragma unroll
        for (int j = 0; j < 4; ++j)
            *reinterpret_cast<float4*>(Pt + (4 * tx + j) * PA_P + 4 * ty) = make_float4(s[0][j], s[1][j], s[2][j], s[3][j]);
        __syncthreads();
#pragma unroll 8
        for (int k = 0; k < PA_T; ++k) {
            const float4 pa = *reinterpret_cast<const float4*>(Pt + k * PA_P + 4 * ty);
            const float4 va = *reinterpret_cast<const float4*>(Vs + k * PA_P + 4 * tx);
            const float pv[4] = {pa.x, pa.y, pa.z, pa.w}, vv[4] = {va.x, va.y, va.z, va.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) o[i][j] = fmaf(pv[i], vv[j], o[i][j]);
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int q = q0 + 4 * ty + i;
        if (q >= T) continue;
        const float inv = 1.0f / l_run[i];
        const float r0 = o[i][0] * inv, r1 = o[i][1] * inv, r2 = o[i][2] * inv, r3 = o[i][3] * inv;
        const uint32_t h0 = pack_op(r0, r1), h1 = pack_op(r2, r3);
        const float2 f0v = unpack_op(h0), f1v = unpack_op(h1);
        const long long off = (f0 + q) * EMBED + h * HEAD_DIM + 4 * tx;
        *reinterpret_cast<uint2*>(out_hi + off) = make_uint2(h0, h1);
        *reinterpret_cast<uint2*>(out_lo + off) = make_uint2(pack_op(r0 - f0v.x, r1 - f0v.y), pack_op(r2 - f1v.x, r3 - f1v.y));
        if (lse != nullptr && tx == 0) lse[(f0 + q) * HEADS + h] = m_run[i] + logf(l_run[i]);
    }
}

// ------------------------------------------------------------------------------------------------ workspace
size_t carve_precise(const Plan& p, void* base, PWorkspace* out, bool save) {
    size_t o = 0;
    auto take = [&](size_t bytes) {
        size_t at = o;
        o = align_up(o + bytes, 1024);
        return base ? (void*)((char*)base + at) : nullptr;
    };
    PWorkspace w;
    memset(&w, 0, sizeof(w));
    const size_t F = (size_t)p.frames;
    w.meta = (UttMeta*)take(sizeof(UttMeta) * p.B);
    w.stat_part = (double*)take(sizeof(double) * NSTAT * p.max_chunks * p.B);
    w.c0_fold = (float*)take(sizeof(float) * 12 * CONV_DIM * p.B);
    for (int i = 0; i < 2; ++i) {
        const size_t rows = (size_t)(i == 0 ? p.rows0 : p.rows0 / 2) + 8;
        w.y_hi[i] = (op_t*)take(2ull * CONV_DIM * rows);
        w.y_lo[i] = (op_t*)take(2ull * CONV_DIM * rows);
    }
    w.ln0_hi = w.y_hi[1];
    w.ln0_lo = w.y_lo[1];
    w.x0 = (float*)take(4ull * EMBED * F);
    w.x = (float*)take(4ull * EMBED * F);
    float* pre = (float*)take(4ull * EMBED * F);
    w.xh_hi = (op_t*)take(2ull * EMBED * F);
    w.xh_lo = (op_t*)take(2ull * EMBED * F);
    w.posg_hi = (op_t*)take(2ull * POS_G * POS_GC * (p.pos_rows + POS_K));
    w.posg_lo = (op_t*)take(2ull * POS_G * POS_GC * (p.pos_rows + POS_K));
    w.pos_y = (float*)take(4ull * EMBED * p.pos_rows);
    float* qkv = (float*)take(4ull * 3 * EMBED * F);
    op_t* attn_hi = (op_t*)take(2ull * EMBED * F);
    op_t* attn_lo = (op_t*)take(2ull * EMBED * F);
    w.ffn_hi = (op_t*)take(2ull * FFN * F);
    w.ffn_lo = (op_t*)take(2ull * FFN * F);
    for (int l = 0; l < LAYERS; ++l) {
        w.qkv[l] = qkv;
        w.attn_hi[l] = attn_hi;
        w.attn_lo[l] = attn_lo;
        w.pre1[l] = w.pre2[l] = pre;
    }
    if (save) {
        w.gn_stat = (float*)take(4ull * 2 * CONV_DIM * p.B);
        for (int l = 0; l < 7; ++l) w.u[l] = (float*)take(4ull * CONV_DIM * (size_t)(p.rows0 >> l));
        w.pos_pre = (float*)take(4ull * EMBED * p.pos_rows);
        for (int l = 0; l < LAYERS; ++l) {
            if (l > 0) {
                w.qkv[l] = (float*)take(4ull * 3 * EMBED * F);
                w.attn_hi[l] = (op_t*)take(2ull * EMBED * F);
                w.attn_lo[l] = (op_t*)take(2ull * EMBED * F);
                w.pre1[l] = (float*)take(4ull * EMBED * F);
            }
            w.pre2[l] = (float*)take(4ull * EMBED * F);
            w.lse[l] = (float*)take(4ull * HEADS * F);
            w.fc1_pre[l] = (float*)take(4ull * FFN * F);
        }
    }
    w.bytes = o;
    if (out) *out = w;
    return o;
}

size_t precise_workspace_bytes(const Plan& p) { return carve_precise(p, nullptr, nullptr, false); }

// ------------------------------------------------------------------------------------------------ forward
static GemmEpilogue epi_precise(int flags, const SplitW& w, const float* bias, const float* resid, float* out_f, op_t* out_h,
                                op_t* out_l, long long ld) {
    GemmEpilogue e = epi_linear(flags | EPI_PRECISE, bias, resid, out_f, out_h, ld);
    e.out_l = out_l;
    e.acc_scale = w.inv_scale;
    return e;
}

// wav (device, packed) -> residual stream after the 12th layer (ws.x), every utterance exactly as if alone (same masking
// rules as the fp16 path).  save: also keep what the waveform backward reads (PWorkspace); the arithmetic is the same.
static int forward_precise(Handle* h, const Plan& p, const PWorkspace& ws, const float* wav, cudaStream_t st, float* layers_out,
                           int layer_T, bool save) {
    const Weights& w = h->w;
    const PreciseWeights& pw = h->pw;
    const long long F = p.frames;
    {   // per-utterance geometry (pinned staging shared with the fp16 path)
        Workspace meta_only;
        memset(&meta_only, 0, sizeof(meta_only));
        meta_only.meta = ws.meta;
        Plan q = p;
        q.attn_items.clear();
        meta_only.attn_items = nullptr;
        NB_TRY(upload_meta(h, q, meta_only, st));
    }
    // rows just past a level's last utterance are read by the next conv (its last padding output rows): keep them finite
    for (int i = 0; i < 2; ++i) {
        for (int l = i; l < 6; l += 2) {
            NB_CUDA(cudaMemsetAsync(ws.y_hi[i] + (p.rows0 >> l) * CONV_DIM, 0, 2ull * CONV_DIM * 8, st));
            NB_CUDA(cudaMemsetAsync(ws.y_lo[i] + (p.rows0 >> l) * CONV_DIM, 0, 2ull * CONV_DIM * 8, st));
        }
    }
    NB_TRY(launch_wave_stats(st, wav, ws.meta, 0, p.B, p.max_chunks, ws.stat_part));
    NB_TRY(launch_gn_fold(st, ws.stat_part, ws.meta, 0, p.B, p.max_chunks, w.conv0_w, w.gn_g, w.gn_b, ws.c0_fold, ws.gn_stat, nullptr));
    conv0_precise_kernel<<<(unsigned)(p.rows0 / 64), 256, 0, st>>>(wav, ws.meta, p.B, ws.c0_fold, ws.y_hi[0], ws.y_lo[0], ws.u[0]);
    NB_LAUNCHED();
    for (int l = 1; l < 7; ++l) {
        const long long M = p.rows0 >> l;
        const int in = (l - 1) & 1, ot = l & 1;
        GemmOperand A{ws.y_hi[in], M, 2 * CONV_DIM, 0, 0, ws.y_lo[in]};
        GemmOperand Bw{pw.conv[l].hi, CONV_DIM, (long long)CONV_KERNEL[l] * CONV_DIM, 0, 0, pw.conv[l].lo};
        if (save) {  // pre-activation kept for the backward, GELU applied by a separate pass (same bits as the epilogue's)
            GemmEpilogue e = epi_precise(EPI_OUT_F32, pw.conv[l], nullptr, nullptr, ws.u[l], nullptr, nullptr, CONV_DIM);
            NB_TRY(gemm_h16(st, A, Bw, (int)M, CONV_DIM, CONV_KERNEL[l] * CONV_DIM, 1, e, 0));
            NB_TRY(launch_gelu_precise(st, ws.u[l], M * CONV_DIM, ws.y_hi[ot], ws.y_lo[ot], nullptr));
        } else {
            GemmEpilogue e = epi_precise(EPI_GELU | EPI_OUT_H16, pw.conv[l], nullptr, nullptr, nullptr, ws.y_hi[ot], ws.y_lo[ot], CONV_DIM);
            NB_TRY(gemm_h16(st, A, Bw, (int)M, CONV_DIM, CONV_KERNEL[l] * CONV_DIM, 1, e, 0));
        }
    }
    ln512_precise_kernel<<<(unsigned)((F + 7) / 8), 256, 0, st>>>(ws.y_hi[0], ws.y_lo[0], F, w.ln0_g, w.ln0_b, ws.ln0_hi, ws.ln0_lo);
    NB_LAUNCHED();
    {
        GemmOperand A{ws.ln0_hi, F, CONV_DIM, 0, 0, ws.ln0_lo};
        GemmOperand Bw{pw.proj.hi, EMBED, CONV_DIM, 0, 0, pw.proj.lo};
        GemmEpilogue e = epi_precise(EPI_BIAS | EPI_OUT_F32, pw.proj, w.proj_b, nullptr, ws.x0, nullptr, nullptr, EMBED);
        NB_TRY(gemm_h16(st, A, Bw, (int)F, EMBED, CONV_DIM, 1, e, 0));
    }
    {   // positional conv: 16 grouped overlapping-row GEMMs over the zero-padded per-group layout
        const long long rows_alloc = p.pos_rows + POS_K;
        NB_CUDA(cudaMemsetAsync(ws.posg_hi, 0, 2ull * POS_G * POS_GC * rows_alloc, st));
        NB_CUDA(cudaMemsetAsync(ws.posg_lo, 0, 2ull * POS_G * POS_GC * rows_alloc, st));
        pos_scatter_precise_kernel<<<(unsigned)((F + 3) / 4), 384, 0, st>>>(ws.x0, ws.meta, p.B, F, rows_alloc, ws.posg_hi, ws.posg_lo);
        NB_LAUNCHED();
        GemmOperand A{ws.posg_hi, p.pos_rows, POS_GC, rows_alloc * POS_GC, 0, ws.posg_lo};
        GemmOperand Bw{pw.pos.hi, POS_GC, (long long)POS_K * POS_GC, (long long)POS_GC * POS_K * POS_GC, 0, pw.pos.lo};
        GemmEpilogue e = epi_precise(save ? EPI_BIAS | EPI_OUT_F32 : EPI_BIAS | EPI_GELU | EPI_OUT_F32, pw.pos, w.pos_b, nullptr,
                                     save ? ws.pos_pre : ws.pos_y, nullptr, nullptr, EMBED);
        e.bias_bstride = POS_GC;
        e.out_bstride = POS_GC;
        NB_TRY(gemm_h16(st, A, Bw, (int)p.pos_rows, POS_GC, POS_K * POS_GC, POS_G, e, 0));
        if (save) NB_TRY(launch_gelu_precise(st, ws.pos_pre, p.pos_rows * EMBED, nullptr, nullptr, ws.pos_y));
        pos_finish_ln_precise_kernel<<<(unsigned)((F + 7) / 8), 256, 0, st>>>(ws.x0, ws.pos_y, ws.meta, p.B, F, w.lne_g, w.lne_b,
                                                                              ws.x, ws.xh_hi, ws.xh_lo);
        NB_LAUNCHED();
    }
    for (int l = 0; l < (save ? LAYERS : 1); ++l) {  // padded rows stay finite
        NB_CUDA(cudaMemsetAsync(ws.attn_hi[l], 0, 2ull * EMBED * F, st));
        NB_CUDA(cudaMemsetAsync(ws.attn_lo[l], 0, 2ull * EMBED * F, st));
    }
    static bool attr_set[64] = {false};
    if (bool* flag = device_once_flag(attr_set)) {
        NB_CUDA(cudaFuncSetAttribute(attention_precise_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PA_SMEM));
        *flag = true;
    }
    for (int l = 0; l < LAYERS; ++l) {
        const LayerWeights& L = w.layer[l];
        {
            GemmOperand A{ws.xh_hi, F, EMBED, 0, 0, ws.xh_lo};
            GemmOperand Bw{pw.qkv[l].hi, 3 * EMBED, EMBED, 0, 0, pw.qkv[l].lo};
            GemmEpilogue e = epi_precise(EPI_BIAS | EPI_OUT_F32, pw.qkv[l], L.b_qkv, nullptr, ws.qkv[l], nullptr, nullptr, 3 * EMBED);
            NB_TRY(gemm_h16(st, A, Bw, (int)F, 3 * EMBED, EMBED, 1, e, 0));
        }
        {
            dim3 grid((p.max_T + PA_T - 1) / PA_T, HEADS, p.B);
            attention_precise_kernel<<<grid, 256, PA_SMEM, st>>>(ws.qkv[l], ws.meta, ws.attn_hi[l], ws.attn_lo[l], ws.lse[l]);
            NB_LAUNCHED();
        }
        {
            GemmOperand A{ws.attn_hi[l], F, EMBED, 0, 0, ws.attn_lo[l]};
            GemmOperand Bw{pw.o[l].hi, EMBED, EMBED, 0, 0, pw.o[l].lo};
            GemmEpilogue e = epi_precise(EPI_BIAS | EPI_RESID | EPI_OUT_F32, pw.o[l], L.b_o, ws.x, ws.pre1[l], nullptr, nullptr, EMBED);
            NB_TRY(gemm_h16(st, A, Bw, (int)F, EMBED, EMBED, 1, e, 0));
        }
        ln768_precise_kernel<<<(unsigned)((F + 7) / 8), 256, 0, st>>>(ws.pre1[l], ws.meta, p.B, F, L.ln1_g, L.ln1_b, ws.x, ws.xh_hi,
                                                                      ws.xh_lo, nullptr, 0);
        NB_LAUNCHED();
        {
            GemmOperand A{ws.xh_hi, F, EMBED, 0, 0, ws.xh_lo};
            GemmOperand Bw{pw.fc1[l].hi, FFN, EMBED, 0, 0, pw.fc1[l].lo};
            if (save) {
                GemmEpilogue e = epi_precise(EPI_BIAS | EPI_OUT_F32, pw.fc1[l], L.b_fc1, nullptr, ws.fc1_pre[l], nullptr, nullptr, FFN);
                NB_TRY(gemm_h16(st, A, Bw, (int)F, FFN, EMBED, 1, e, 0));
                NB_TRY(launch_gelu_precise(st, ws.fc1_pre[l], F * FFN, ws.ffn_hi, ws.ffn_lo, nullptr));
            } else {
                GemmEpilogue e = epi_precise(EPI_BIAS | EPI_GELU | EPI_OUT_H16, pw.fc1[l], L.b_fc1, nullptr, nullptr, ws.ffn_hi, ws.ffn_lo, FFN);
                NB_TRY(gemm_h16(st, A, Bw, (int)F, FFN, EMBED, 1, e, 0));
            }
        }
        {
            GemmOperand A{ws.ffn_hi, F, FFN, 0, 0, ws.ffn_lo};
            GemmOperand Bw{pw.fc2[l].hi, EMBED, FFN, 0, 0, pw.fc2[l].lo};
            GemmEpilogue e = epi_precise(EPI_BIAS | EPI_RESID | EPI_OUT_F32, pw.fc2[l], L.b_fc2, ws.x, ws.pre2[l], nullptr, nullptr, EMBED);
            NB_TRY(gemm_h16(st, A, Bw, (int)F, EMBED, FFN, 1, e, 0));
        }
        float* lo = layers_out ? layers_out + (size_t)l * p.B * layer_T * EMBED : nullptr;
        ln768_precise_kernel<<<(unsigned)((F + 7) / 8), 256, 0, st>>>(ws.pre2[l], ws.meta, p.B, F, L.ln2_g, L.ln2_b, ws.x, ws.xh_hi,
                                                                      ws.xh_lo, lo, layer_T);
        NB_LAUNCHED();
    }
    return 0;
}

int embed_precise(Handle* h, const Plan& p, void* workspace, size_t workspace_bytes, const float* wav, cudaStream_t st,
                  float* layers_out, int layer_T, const float* head_wt, const float* head_b, float* emb_dev) {
    NB_CHECK(h->pw.built, "this handle was created without the fp32-class weights (precision_mode 1)");
    NB_CHECK(p.B <= 65535, "embed (fp32 mode): at most 65535 utterances per call (got %d); split the batch", p.B);
    PWorkspace ws;
    const size_t need = carve_precise(p, workspace, &ws, false);
    NB_CHECK(workspace_bytes >= need, "embed (fp32 mode): workspace too small (%zu < %zu bytes)", workspace_bytes, need);
    NB_TRY(forward_precise(h, p, ws, wav, st, layers_out, layer_T, false));
    if (emb_dev != nullptr) NB_TRY(launch_pool_head(st, ws.x, ws.meta, p.B, head_wt, head_b, emb_dev, nullptr));
    return 0;
}

int embed_precise_save(Handle* h, const Plan& p, void* saved, size_t saved_bytes, const float* wav, cudaStream_t st,
                       float* layers_out, int layer_T) {
    NB_CHECK(h->pw.built, "this handle was created without the fp32-class weights (precision_mode 1)");
    NB_CHECK(p.B <= 65535, "save-mode forward (fp32 mode): at most 65535 utterances per call (got %d)", p.B);
    PWorkspace ws;
    const size_t need = carve_precise(p, saved, &ws, true);
    NB_CHECK(saved_bytes >= need, "save-mode forward (fp32 mode): buffer too small (%zu < %zu bytes)", saved_bytes, need);
    return forward_precise(h, p, ws, wav, st, layers_out, layer_T, true);
}

}  // namespace nb
