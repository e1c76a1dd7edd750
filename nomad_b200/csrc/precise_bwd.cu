// fp32-class waveform backward (precision_mode 1): d loss / d wav through a save-mode forward of precise.cu.
//
// The chain is the one of backward_chain in loss.cu -- final LayerNorm, fc2^T x GELU', fc1^T + residual, LayerNorm,
// out-proj^T, attention, qkv^T + residual for each layer, then the encoder LayerNorm, the positional-conv dgrad (grouped
// GEMM with flipped taps), projection^T, LayerNorm(512) x feature_grad_mult, the conv1..6 dgrads and conv0 + GroupNorm
// -- in the arithmetic of the fp32-class forward: every tensor-core operand is a pair of hi + lo fp16 planes and every
// GEMM the three-segment PREC instantiation of gemm.cu (transposed weight planes built at create time, api.cu); every
// gradient a GEMM produces comes out in fp32, and the elementwise steps (GELU derivative from the saved fp32
// pre-activation with libdevice erff / expf, LayerNorm backward, the softmax backward) run in fp32 before the result is
// split into the next GEMM's planes.  Attention runs on the fp32 CUDA cores; its O is hi + lo, so D = rowsum(dO * O) is
// taken directly (no recomputed D as in the fp16 kernel).  Activation gradients carry the power-of-two scale S of the
// fp16 path (2^k upstream gradients still give exactly 2^k results); conv0 + GroupNorm reuse loss.cu's fp64-statistics
// kernel for the per-utterance constants.
#include <algorithm>
#include <cmath>
#include <cstring>

#include "precise.cuh"

namespace nb {

// loss.cu: per-utterance constants of the conv0 + GroupNorm backward (fp64 sums)
__global__ void conv0_bwd_consts_kernel(const double* __restrict__ sums, const UttMeta* __restrict__ meta,
                                        const float* __restrict__ w0, const float* __restrict__ stat, float* __restrict__ consts);

static inline size_t align_up_b(size_t v, size_t a) { return (v + a - 1) / a * a; }

__device__ __forceinline__ float dgelu_exact(float x) {
    return fmaf(x * 0.39894228040143267794f, expf(-0.5f * x * x), 0.5f * (1.0f + erff(x * 0.70710678118654752440f)));
}

// one warp per 768-wide row; lane owns the 8-channel chunks {lane, lane + 32, lane + 64}
__device__ __forceinline__ void ld_row24(float (&v)[24], const float* __restrict__ p, int lane) {
#pragma unroll
    for (int h = 0; h < 3; ++h) {
        const float4* q = reinterpret_cast<const float4*>(p + (lane + 32 * h) * 8);
        const float4 a = __ldg(q), c = __ldg(q + 1);
        float* w = v + 8 * h;
        w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w; w[4] = c.x; w[5] = c.y; w[6] = c.z; w[7] = c.w;
    }
}
// v -> xhat in place, returns rstd (fp32, 1 / sqrtf as the forward; rounded products so identical rows stay identical)
__device__ __forceinline__ float norm_row24(float (&v)[24]) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 24; ++i) s += v[i];
    const float mean = warp_sum(s) * (1.0f / EMBED);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < 24; ++i) { v[i] = __fsub_rn(v[i], mean); q = fmaf(v[i], v[i], q); }
    const float rstd = 1.0f / sqrtf(warp_sum(q) * (1.0f / EMBED) + 1e-5f);
#pragma unroll
    for (int i = 0; i < 24; ++i) v[i] = __fmul_rn(v[i], rstd);
    return rstd;
}
// LayerNorm backward in place: g (upstream) -> rstd * (g gamma - mean(g gamma) - xhat mean(g gamma xhat))
__device__ __forceinline__ void ln_bwd_row24(float (&g)[24], const float (&xh)[24], float rstd, const float* __restrict__ gam, int lane) {
    float gg[24];
    ld_row24(gg, gam, lane);
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < 24; ++i) {
        g[i] *= gg[i];
        s1 += g[i];
        s2 = fmaf(g[i], xh[i], s2);
    }
    s1 = warp_sum(s1) * (1.0f / EMBED);
    s2 = warp_sum(s2) * (1.0f / EMBED);
#pragma unroll
    for (int i = 0; i < 24; ++i) g[i] = rstd * (g[i] - s1 - xh[i] * s2);
}
__device__ __forceinline__ void st_row24(const float (&v)[24], float* __restrict__ f32, op_t* __restrict__ hi, op_t* __restrict__ lo,
                                         int lane) {
#pragma unroll
    for (int h = 0; h < 3; ++h) {
        const int c0 = (lane + 32 * h) * 8;
        const float* w = v + 8 * h;
        if (f32 != nullptr) {
            float4* o = reinterpret_cast<float4*>(f32 + c0);
            o[0] = make_float4(w[0], w[1], w[2], w[3]);
            o[1] = make_float4(w[4], w[5], w[6], w[7]);
        }
        if (hi != nullptr) split_store8(w, hi + c0, lo + c0);
    }
}

// ------------------------------------------------------------------------------------------------ LayerNorm(768) backward
// g = g_in + seed * sign((x_est - x_clean) gamma) [fused loss; clean row = f + frames] + S g_user[b, t] + S g_pool[b]
// (S = *scale, or 1 when scale is null), then the LayerNorm backward -> g_out (fp32) and hi + lo planes; zeros on
// padding rows.
__global__ void __launch_bounds__(256) ln768_bwd_precise_kernel(const float* __restrict__ g_in, const float* __restrict__ pre,
                                                                const UttMeta* __restrict__ meta, int B, long long frames,
                                                                const float* __restrict__ gam, float seed,
                                                                const float* __restrict__ g_user, int user_T,
                                                                const float* __restrict__ g_pool, const float* __restrict__ scale,
                                                                float* __restrict__ g_out, op_t* __restrict__ out_hi,
                                                                op_t* __restrict__ out_lo) {
    const long long f = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (f >= frames) return;
    const int lane = threadIdx.x & 31;
    const int b = find_utt_by_frame(meta, B, (int)f);
    const int t = (int)f - meta[b].frame0;
    float g[24];
    if (t >= meta[b].T) {
#pragma unroll
        for (int i = 0; i < 24; ++i) g[i] = 0.f;
        st_row24(g, g_out + f * EMBED, out_hi + f * EMBED, out_lo + f * EMBED, lane);
        return;
    }
    const float S = scale != nullptr ? __ldg(scale) : 1.0f;
    float xh[24];
    ld_row24(xh, pre + f * EMBED, lane);
    const float rstd = norm_row24(xh);
    if (g_in != nullptr) {
        ld_row24(g, g_in + f * EMBED, lane);
    } else {
#pragma unroll
        for (int i = 0; i < 24; ++i) g[i] = 0.f;
    }
    if (seed != 0.f) {
        float xc[24], gg[24];
        ld_row24(xc, pre + (f + frames) * EMBED, lane);
        norm_row24(xc);
        ld_row24(gg, gam, lane);
#pragma unroll
        for (int i = 0; i < 24; ++i) {
            const float d = __fsub_rn(xh[i], xc[i]) * gg[i];
            g[i] += d > 0.f ? seed : (d < 0.f ? -seed : 0.f);
        }
    }
    if (g_user != nullptr) {
        float u[24];
        ld_row24(u, g_user + ((long long)b * user_T + t) * EMBED, lane);
#pragma unroll
        for (int i = 0; i < 24; ++i) g[i] = fmaf(S, u[i], g[i]);
    }
    if (g_pool != nullptr) {
        float u[24];
        ld_row24(u, g_pool + (long long)b * EMBED, lane);
#pragma unroll
        for (int i = 0; i < 24; ++i) g[i] = fmaf(S, u[i], g[i]);
    }
    ln_bwd_row24(g, xh, rstd, gam, lane);
    st_row24(g, g_out + f * EMBED, out_hi + f * EMBED, out_lo + f * EMBED, lane);
}

// ------------------------------------------------------------------------------------------------ GELU' x, split
// out = g * gelu'(pre) as hi + lo planes, n values (n % 8 == 0)
__global__ void __launch_bounds__(256) mul_dgelu_split_kernel(const float* __restrict__ g, const float* __restrict__ pre, long long n,
                                                              op_t* __restrict__ hi, op_t* __restrict__ lo) {
    const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 8;
    if (i >= n) return;
    const float4 a = __ldg(reinterpret_cast<const float4*>(g + i)), b = __ldg(reinterpret_cast<const float4*>(g + i + 4));
    const float4 c = __ldg(reinterpret_cast<const float4*>(pre + i)), d = __ldg(reinterpret_cast<const float4*>(pre + i + 4));
    const float v[8] = {a.x * dgelu_exact(c.x), a.y * dgelu_exact(c.y), a.z * dgelu_exact(c.z), a.w * dgelu_exact(c.w),
                        b.x * dgelu_exact(d.x), b.y * dgelu_exact(d.y), b.z * dgelu_exact(d.z), b.w * dgelu_exact(d.w)};
    split_store8(v, hi + i, lo + i);
}

// conv level `level` (rows (row0 >> level) .. of each utterance, 512 channels): g * gelu'(u), zero on the rows t >= T_level;
// level 0 also multiplies by GroupNorm's gamma_c * rstd_c (fold[b][c][11]) and stays fp32 (f32_out), other levels go
// out as hi + lo planes.  One warp per row; f32_out may be g itself (each thread rewrites what it read).
__global__ void __launch_bounds__(256) conv_dgelu_precise_kernel(const float* g, const float* __restrict__ u,
                                                                 const UttMeta* __restrict__ meta, int B, long long rows, int level,
                                                                 const float* __restrict__ fold, float* f32_out,
                                                                 op_t* __restrict__ hi, op_t* __restrict__ lo) {
    const long long r = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (r >= rows) return;
    const int lane = threadIdx.x & 31;
    int lo_b = 0, hi_b = B - 1;
    while (lo_b < hi_b) {
        const int mid = (lo_b + hi_b + 1) >> 1;
        if ((long long)(meta[mid].row0 >> level) <= r) lo_b = mid; else hi_b = mid - 1;
    }
    const UttMeta m = meta[lo_b];
    int T = m.T0;
    for (int l = 1; l <= level; ++l) T = (T - (l < 5 ? 3 : 2)) / 2 + 1;  // CONV_KERNEL[l]
    const bool valid = r - (long long)(m.row0 >> level) < T;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int c0 = (lane + 32 * h) * 8;
        const long long o = r * CONV_DIM + c0;
        float v[8];
        if (valid) {
            const float4 a = *reinterpret_cast<const float4*>(g + o), b = *reinterpret_cast<const float4*>(g + o + 4);
            const float4 c = __ldg(reinterpret_cast<const float4*>(u + o)), d = __ldg(reinterpret_cast<const float4*>(u + o + 4));
            const float gv[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w}, uv[8] = {c.x, c.y, c.z, c.w, d.x, d.y, d.z, d.w};
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                v[i] = gv[i] * dgelu_exact(uv[i]);
                if (fold != nullptr) v[i] *= __ldg(fold + ((long long)lo_b * CONV_DIM + c0 + i) * 12 + 11);
            }
        } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = 0.f;
        }
        if (f32_out != nullptr) {
            *reinterpret_cast<float4*>(f32_out + o) = make_float4(v[0], v[1], v[2], v[3]);
            *reinterpret_cast<float4*>(f32_out + o + 4) = make_float4(v[4], v[5], v[6], v[7]);
        } else {
            split_store8(v, hi + o, lo + o);
        }
    }
}

// ------------------------------------------------------------------------------------------------ attention backward
// fp32 CUDA cores, 64 x 64 tiles, thread (ty, tx) of the 16 x 16 layout owning 4 x 4 register tiles (the layout of
// attention_precise_kernel).  P = exp(q.k - lse) (q carries head_dim^-0.5), dP = dO V^T, dS = P (dP - D),
// dV = P^T dO, dK = dS^T Q, dQ = dS K.  D[row][head] = rowsum(dO * O) with O = hi + lo.
static constexpr int PB_T = 64, PB_P = 68;
static constexpr int PB_KV_SMEM = 8 * PB_T * PB_P * 4 + 2 * PB_T * 4;
static constexpr int PB_Q_SMEM = 6 * PB_T * PB_P * 4;

__global__ void __launch_bounds__(256) attn_d_precise_kernel(const float* __restrict__ dO, const op_t* __restrict__ o_hi,
                                                             const op_t* __restrict__ o_lo, long long frames, float* __restrict__ D) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // (row, head)
    if (i >= frames * HEADS) return;
    const long long off = (i / HEADS) * EMBED + (i % HEADS) * HEAD_DIM;
    float s = 0.f;
#pragma unroll
    for (int c = 0; c < HEAD_DIM; c += 8) {
        float o[8];
        split_load8(o_hi + off + c, o_lo + off + c, o);
        const float4 a = __ldg(reinterpret_cast<const float4*>(dO + off + c)), b = __ldg(reinterpret_cast<const float4*>(dO + off + c + 4));
        s = fmaf(a.x, o[0], s); s = fmaf(a.y, o[1], s); s = fmaf(a.z, o[2], s); s = fmaf(a.w, o[3], s);
        s = fmaf(b.x, o[4], s); s = fmaf(b.y, o[5], s); s = fmaf(b.z, o[6], s); s = fmaf(b.w, o[7], s);
    }
    D[i] = s;
}

__device__ __forceinline__ void store4_split(op_t* hi, op_t* lo, float a, float b, float c, float d) {
    const uint32_t h0 = pack_op(a, b), h1 = pack_op(c, d);
    const float2 f0 = unpack_op(h0), f1 = unpack_op(h1);
    *reinterpret_cast<uint2*>(hi) = make_uint2(h0, h1);
    *reinterpret_cast<uint2*>(lo) = make_uint2(pack_op(a - f0.x, b - f0.y), pack_op(c - f1.x, d - f1.y));
}
// rows r of a [d][r] tile from 64 rows x 64 columns at src (row stride 2304), zero rows past n
__device__ __forceinline__ void load_t(float* dst, const float* src, int n, int tid) {
    for (int idx = tid; idx < PB_T * 16; idx += 256) {
        const int r = idx >> 4, c4 = (idx & 15) * 4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (r < n) v = __ldg(reinterpret_cast<const float4*>(src + (long long)r * (3 * EMBED) + c4));
        dst[(c4 + 0) * PB_P + r] = v.x; dst[(c4 + 1) * PB_P + r] = v.y; dst[(c4 + 2) * PB_P + r] = v.z; dst[(c4 + 3) * PB_P + r] = v.w;
    }
}
// the same rows kept as [r][d]; ld = row stride of src in floats
__device__ __forceinline__ void load_n(float* dst, const float* src, long long ld, int n, int tid) {
    for (int idx = tid; idx < PB_T * 16; idx += 256) {
        const int r = idx >> 4, c4 = (idx & 15) * 4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (r < n) v = __ldg(reinterpret_cast<const float4*>(src + (long long)r * ld + c4));
        *reinterpret_cast<float4*>(dst + r * PB_P + c4) = v;
    }
}
__device__ __forceinline__ void load_t_ld(float* dst, const float* src, long long ld, int n, int tid) {
    for (int idx = tid; idx < PB_T * 16; idx += 256) {
        const int r = idx >> 4, c4 = (idx & 15) * 4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (r < n) v = __ldg(reinterpret_cast<const float4*>(src + (long long)r * ld + c4));
        dst[(c4 + 0) * PB_P + r] = v.x; dst[(c4 + 1) * PB_P + r] = v.y; dst[(c4 + 2) * PB_P + r] = v.z; dst[(c4 + 3) * PB_P + r] = v.w;
    }
}
// acc[i][j] += sum_d X[d][4 a + i] Y[d][4 c + j] over the 64 rows of two [d][r] tiles
__device__ __forceinline__ void mm_tt(float (&acc)[4][4], const float* X, const float* Y, int a, int c) {
#pragma unroll 8
    for (int d = 0; d < HEAD_DIM; ++d) {
        const float4 x = *reinterpret_cast<const float4*>(X + d * PB_P + 4 * a);
        const float4 y = *reinterpret_cast<const float4*>(Y + d * PB_P + 4 * c);
        const float xv[4] = {x.x, x.y, x.z, x.w}, yv[4] = {y.x, y.y, y.z, y.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(xv[i], yv[j], acc[i][j]);
    }
}

// dK, dV: one CTA = 64 keys x one head, streaming the query tiles
__global__ void __launch_bounds__(256) attn_bwd_kv_precise_kernel(const float* __restrict__ qkv, const float* __restrict__ dO,
                                                                  const float* __restrict__ lse, const float* __restrict__ D,
                                                                  const UttMeta* __restrict__ meta, op_t* __restrict__ dqkv_hi,
                                                                  op_t* __restrict__ dqkv_lo) {
    const int b = blockIdx.z, h = blockIdx.y, k0 = blockIdx.x * PB_T;
    const int T = meta[b].T;
    if (k0 >= T) return;
    const long long f0 = meta[b].frame0;
    extern __shared__ __align__(16) float pb_sm[];
    float* Kt = pb_sm;
    float* Vt = Kt + PB_T * PB_P;
    float* Qt = Vt + PB_T * PB_P;
    float* dOt = Qt + PB_T * PB_P;
    float* Qs = dOt + PB_T * PB_P;
    float* dOs = Qs + PB_T * PB_P;
    float* Ps = dOs + PB_T * PB_P;   // [q][k]
    float* dSs = Ps + PB_T * PB_P;   // [q][k]
    float* lse_s = dSs + PB_T * PB_P;
    float* D_s = lse_s + PB_T;
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const float* base = qkv + f0 * (3 * EMBED) + h * HEAD_DIM;
    const int nk = min(PB_T, T - k0);
    load_t(Kt, base + (long long)k0 * (3 * EMBED) + EMBED, nk, tid);
    load_t(Vt, base + (long long)k0 * (3 * EMBED) + 2 * EMBED, nk, tid);
    float dk[4][4], dv[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) dk[i][j] = dv[i][j] = 0.f;
    for (int q0 = 0; q0 < T; q0 += PB_T) {
        const int nq = min(PB_T, T - q0);
        __syncthreads();  // previous tile's products are done with Qs / dOs / Ps / dSs
        load_t(Qt, base + (long long)q0 * (3 * EMBED), nq, tid);
        load_n(Qs, base + (long long)q0 * (3 * EMBED), 3 * EMBED, nq, tid);
        load_t_ld(dOt, dO + (f0 + q0) * EMBED + h * HEAD_DIM, EMBED, nq, tid);
        load_n(dOs, dO + (f0 + q0) * EMBED + h * HEAD_DIM, EMBED, nq, tid);
        if (tid < PB_T) {
            lse_s[tid] = tid < nq ? lse[(f0 + q0 + tid) * HEADS + h] : 0.f;
            D_s[tid] = tid < nq ? D[(f0 + q0 + tid) * HEADS + h] : 0.f;
        }
        __syncthreads();
        float s[4][4], dp[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) s[i][j] = dp[i][j] = 0.f;
        mm_tt(s, Kt, Qt, ty, tx);   // s[i][j]: key 4 ty + i, query 4 tx + j
        mm_tt(dp, Vt, dOt, ty, tx);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int q = 4 * tx + j;
            float p4[4], d4[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const bool ok = q < nq && 4 * ty + i < nk;
                p4[i] = ok ? expf(s[i][j] - lse_s[q]) : 0.f;
                d4[i] = p4[i] * (dp[i][j] - D_s[q]);
            }
            *reinterpret_cast<float4*>(Ps + q * PB_P + 4 * ty) = make_float4(p4[0], p4[1], p4[2], p4[3]);
            *reinterpret_cast<float4*>(dSs + q * PB_P + 4 * ty) = make_float4(d4[0], d4[1], d4[2], d4[3]);
        }
        __syncthreads();
#pragma unroll 4
        for (int q = 0; q < PB_T; ++q) {
            const float4 pa = *reinterpret_cast<const float4*>(Ps + q * PB_P + 4 * ty);
            const float4 sa = *reinterpret_cast<const float4*>(dSs + q * PB_P + 4 * ty);
            const float4 oa = *reinterpret_cast<const float4*>(dOs + q * PB_P + 4 * tx);
            const float4 qa = *reinterpret_cast<const float4*>(Qs + q * PB_P + 4 * tx);
            const float pv[4] = {pa.x, pa.y, pa.z, pa.w}, sv[4] = {sa.x, sa.y, sa.z, sa.w};
            const float ov[4] = {oa.x, oa.y, oa.z, oa.w}, qv[4] = {qa.x, qa.y, qa.z, qa.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    dv[i][c] = fmaf(pv[i], ov[c], dv[i][c]);
                    dk[i][c] = fmaf(sv[i], qv[c], dk[i][c]);
                }
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int k = 4 * ty + i;
        if (k >= nk) continue;
        const long long off = (f0 + k0 + k) * (3 * EMBED) + h * HEAD_DIM + 4 * tx;
        store4_split(dqkv_hi + off + EMBED, dqkv_lo + off + EMBED, dk[i][0], dk[i][1], dk[i][2], dk[i][3]);
        store4_split(dqkv_hi + off + 2 * EMBED, dqkv_lo + off + 2 * EMBED, dv[i][0], dv[i][1], dv[i][2], dv[i][3]);
    }
}

// dQ: one CTA = 64 queries x one head, streaming the key tiles
__global__ void __launch_bounds__(256) attn_bwd_q_precise_kernel(const float* __restrict__ qkv, const float* __restrict__ dO,
                                                                 const float* __restrict__ lse, const float* __restrict__ D,
                                                                 const UttMeta* __restrict__ meta, op_t* __restrict__ dqkv_hi,
                                                                 op_t* __restrict__ dqkv_lo) {
    const int b = blockIdx.z, h = blockIdx.y, q0 = blockIdx.x * PB_T;
    const int T = meta[b].T;
    if (q0 >= T) return;
    const long long f0 = meta[b].frame0;
    extern __shared__ __align__(16) float pb_sm[];
    float* Qt = pb_sm;
    float* dOt = Qt + PB_T * PB_P;
    float* Kt = dOt + PB_T * PB_P;
    float* Vt = Kt + PB_T * PB_P;
    float* Ks = Vt + PB_T * PB_P;    // [k][d]
    float* dSs = Ks + PB_T * PB_P;   // [k][q]
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const float* base = qkv + f0 * (3 * EMBED) + h * HEAD_DIM;
    const int nq = min(PB_T, T - q0);
    load_t(Qt, base + (long long)q0 * (3 * EMBED), nq, tid);
    load_t_ld(dOt, dO + (f0 + q0) * EMBED + h * HEAD_DIM, EMBED, nq, tid);
    float lq[4], dq_d[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int q = 4 * ty + i;
        lq[i] = q < nq ? __ldg(lse + (f0 + q0 + q) * HEADS + h) : 0.f;
        dq_d[i] = q < nq ? __ldg(D + (f0 + q0 + q) * HEADS + h) : 0.f;
    }
    float dq[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) dq[i][j] = 0.f;
    for (int k0 = 0; k0 < T; k0 += PB_T) {
        const int nk = min(PB_T, T - k0);
        __syncthreads();
        load_t(Kt, base + (long long)k0 * (3 * EMBED) + EMBED, nk, tid);
        load_t(Vt, base + (long long)k0 * (3 * EMBED) + 2 * EMBED, nk, tid);
        load_n(Ks, base + (long long)k0 * (3 * EMBED) + EMBED, 3 * EMBED, nk, tid);
        __syncthreads();
        float s[4][4], dp[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) s[i][j] = dp[i][j] = 0.f;
        mm_tt(s, Qt, Kt, ty, tx);   // s[i][j]: query 4 ty + i, key 4 tx + j
        mm_tt(dp, dOt, Vt, ty, tx);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float d4[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const bool ok = 4 * ty + i < nq && 4 * tx + j < nk;
                const float p = ok ? expf(s[i][j] - lq[i]) : 0.f;
                d4[i] = p * (dp[i][j] - dq_d[i]);
            }
            *reinterpret_cast<float4*>(dSs + (4 * tx + j) * PB_P + 4 * ty) = make_float4(d4[0], d4[1], d4[2], d4[3]);
        }
        __syncthreads();
#pragma unroll 4
        for (int k = 0; k < PB_T; ++k) {
            const float4 sa = *reinterpret_cast<const float4*>(dSs + k * PB_P + 4 * ty);
            const float4 ka = *reinterpret_cast<const float4*>(Ks + k * PB_P + 4 * tx);
            const float sv[4] = {sa.x, sa.y, sa.z, sa.w}, kv[4] = {ka.x, ka.y, ka.z, ka.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int c = 0; c < 4; ++c) dq[i][c] = fmaf(sv[i], kv[c], dq[i][c]);
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int q = 4 * ty + i;
        if (q >= nq) continue;
        const long long off = (f0 + q0 + q) * (3 * EMBED) + h * HEAD_DIM + 4 * tx;
        store4_split(dqkv_hi + off, dqkv_lo + off, dq[i][0], dq[i][1], dq[i][2], dq[i][3]);
    }
}

// ------------------------------------------------------------------------------------------------ positional conv
// encoder LayerNorm backward (z = x0 + GELU(pos_pre) recomputed) -> g_z (fp32), and g_z * gelu'(pos_pre) scattered into
// the grouped, zero-padded layout of the dgrad GEMM (hi + lo)
__global__ void __launch_bounds__(256) pos_bwd_prep_precise_kernel(const float* __restrict__ g_x, const float* __restrict__ x0,
                                                                   const float* __restrict__ pos_pre, const UttMeta* __restrict__ meta,
                                                                   int B, long long frames, const float* __restrict__ gam,
                                                                   long long pos_rows_alloc, float* __restrict__ g_z,
                                                                   op_t* __restrict__ pg_hi, op_t* __restrict__ pg_lo) {
    const long long f = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (f >= frames) return;
    const int lane = threadIdx.x & 31;
    const int b = find_utt_by_frame(meta, B, (int)f);
    const int t = (int)f - meta[b].frame0;
    float g[24];
    if (t >= meta[b].T) {
#pragma unroll
        for (int i = 0; i < 24; ++i) g[i] = 0.f;
        st_row24(g, g_z + f * EMBED, nullptr, nullptr, lane);
        return;
    }
    const long long m = (long long)meta[b].pos0 + t - POS_K / 2;  // row of this frame in pos_pre
    float z[24], u[24];
    ld_row24(z, x0 + f * EMBED, lane);
    ld_row24(u, pos_pre + m * EMBED, lane);
#pragma unroll
    for (int i = 0; i < 24; ++i) z[i] += gelu_erf_exact(u[i]);
    const float rstd = norm_row24(z);
    ld_row24(g, g_x + f * EMBED, lane);
    ln_bwd_row24(g, z, rstd, gam, lane);
    st_row24(g, g_z + f * EMBED, nullptr, nullptr, lane);
    const long long p = (long long)meta[b].pos0 + t;
#pragma unroll
    for (int h = 0; h < 3; ++h) {
        const int ch = (lane + 32 * h) * 8, grp = ch / POS_GC, cc = ch % POS_GC;
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = g[8 * h + i] * dgelu_exact(u[8 * h + i]);
        const long long o = ((long long)grp * pos_rows_alloc + p) * POS_GC + cc;
        split_store8(v, pg_hi + o, pg_lo + o);
    }
}

// g_x0 = g_z + dgrad[pos0 + t - 63] -> hi + lo (the projection dgrad's A operand); zeros on padding rows
__global__ void __launch_bounds__(256) pos_bwd_finish_precise_kernel(const float* __restrict__ g_z, const float* __restrict__ pos_dy,
                                                                     const UttMeta* __restrict__ meta, int B, long long frames,
                                                                     op_t* __restrict__ hi, op_t* __restrict__ lo) {
    const long long f = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (f >= frames) return;
    const int lane = threadIdx.x & 31;
    const int b = find_utt_by_frame(meta, B, (int)f);
    const int t = (int)f - meta[b].frame0;
    float r[24];
    if (t >= meta[b].T) {
#pragma unroll
        for (int i = 0; i < 24; ++i) r[i] = 0.f;
    } else {
        float y[24];
        ld_row24(r, g_z + f * EMBED, lane);
        ld_row24(y, pos_dy + ((long long)meta[b].pos0 + t - (POS_K / 2 - 1)) * EMBED, lane);
#pragma unroll
        for (int i = 0; i < 24; ++i) r[i] += y[i];
    }
    st_row24(r, nullptr, hi + f * EMBED, lo + f * EMBED, lane);
}

// ------------------------------------------------------------------------------------------------ LayerNorm(512)
// g_u6 = fgm * LN_bwd(g; y6 = GELU(u6)) * gelu'(u6) -> hi + lo; zeros on padding frames
__global__ void __launch_bounds__(256) ln512_bwd_precise_kernel(const float* __restrict__ g_in, const float* __restrict__ u6,
                                                                const UttMeta* __restrict__ meta, int B, long long rows,
                                                                const float* __restrict__ gam, float fgm, op_t* __restrict__ hi,
                                                                op_t* __restrict__ lo) {
    const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= rows) return;
    const int lane = threadIdx.x & 31;
    const int b = find_utt_by_frame(meta, B, (int)row);
    float x[16], g[16], u[16];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int c0 = (lane + 32 * h) * 8;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            u[8 * h + i] = __ldg(u6 + row * CONV_DIM + c0 + i);
            x[8 * h + i] = gelu_erf_exact(u[8 * h + i]);
            g[8 * h + i] = __ldg(g_in + row * CONV_DIM + c0 + i) * __ldg(gam + c0 + i);
        }
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) s += x[i];
    const float mean = warp_sum(s) * (1.0f / CONV_DIM);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) { x[i] -= mean; q = fmaf(x[i], x[i], q); }
    const float rstd = 1.0f / sqrtf(warp_sum(q) * (1.0f / CONV_DIM) + 1e-5f);
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) { x[i] *= rstd; s1 += g[i]; s2 = fmaf(g[i], x[i], s2); }
    s1 = warp_sum(s1) * (1.0f / CONV_DIM);
    s2 = warp_sum(s2) * (1.0f / CONV_DIM);
    const bool valid = (int)row - meta[b].frame0 < meta[b].T;
    const float k = rstd * fgm;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        float r[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) r[i] = valid ? k * (g[8 * h + i] - s1 - x[8 * h + i] * s2) * dgelu_exact(u[8 * h + i]) : 0.f;
        split_store8(r, hi + row * CONV_DIM + (lane + 32 * h) * 8, lo + row * CONV_DIM + (lane + 32 * h) * 8);
    }
}

// ------------------------------------------------------------------------------------------------ conv0 + GroupNorm
// loss.cu's conv0_bwd_stats_kernel with an fp32 G0: per (utt, channel) sums of G0 and G0 * uhat (fp64 atomics)
__global__ void __launch_bounds__(256) conv0_bwd_stats_precise_kernel(const float* __restrict__ G0, const float* __restrict__ wav,
                                                                      const UttMeta* __restrict__ meta, int B,
                                                                      const float* __restrict__ w0, const float* __restrict__ stat,
                                                                      double* __restrict__ sums) {
    const int row_base = blockIdx.x * 64;
    const int b = find_utt_by_frame(meta, B, blockIdx.x);
    const UttMeta m = meta[b];
    const int t_base = row_base - m.row0;
    const int valid = min(64, m.T0 - t_base);
    if (valid <= 0) return;
    __shared__ float xs[64 * 5 + 8];
    const float* x = wav + m.wav_off;
    for (int i = threadIdx.x; i < 64 * 5 + 5; i += blockDim.x) {
        const long long s = (long long)t_base * 5 + i;
        xs[i] = (s < m.n) ? __ldg(x + s) : 0.f;
    }
    const int c = 2 * threadIdx.x;
    float wa[10], wb[10];
#pragma unroll
    for (int j = 0; j < 10; ++j) { wa[j] = __ldg(w0 + c * 10 + j); wb[j] = __ldg(w0 + (c + 1) * 10 + j); }
    const float mean_a = stat[((long long)b * CONV_DIM + c) * 2], rstd_a = stat[((long long)b * CONV_DIM + c) * 2 + 1];
    const float mean_b = stat[((long long)b * CONV_DIM + c + 1) * 2], rstd_b = stat[((long long)b * CONV_DIM + c + 1) * 2 + 1];
    __syncthreads();
    float s1a = 0.f, s2a = 0.f, s1b = 0.f, s2b = 0.f;
    const float2* gp = reinterpret_cast<const float2*>(G0 + (long long)row_base * CONV_DIM + c);
    for (int t = 0; t < valid; ++t) {
        const float2 g = gp[(long long)t * (CONV_DIM / 2)];
        float ua = 0.f, ub = 0.f;
#pragma unroll
        for (int j = 0; j < 10; ++j) {
            const float xv = xs[5 * t + j];
            ua = fmaf(wa[j], xv, ua);
            ub = fmaf(wb[j], xv, ub);
        }
        ua = (ua - mean_a) * rstd_a;
        ub = (ub - mean_b) * rstd_b;
        s1a += g.x; s2a = fmaf(g.x, ua, s2a);
        s1b += g.y; s2b = fmaf(g.y, ub, s2b);
    }
    double* o = sums + ((long long)b * CONV_DIM + c) * 2;
    atomicAdd(o + 0, (double)s1a);
    atomicAdd(o + 1, (double)s2a);
    atomicAdd(o + 2, (double)s1b);
    atomicAdd(o + 3, (double)s2b);
}

// conv0 dgrad on the fp32 cores: V[r][j] = sum_c G0[r][c] w0[c][j] (j < 10; V rows are 16 wide), one warp per row
__global__ void __launch_bounds__(256) conv0_dgrad_precise_kernel(const float* __restrict__ G0, long long rows,
                                                                  const float* __restrict__ w0, float* __restrict__ V) {
    __shared__ float ws[CONV_DIM * 10];
    for (int i = threadIdx.x; i < CONV_DIM * 10; i += blockDim.x) ws[i] = __ldg(w0 + i);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    for (long long r = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); r < rows; r += (long long)gridDim.x * 8) {
        float acc[10];
#pragma unroll
        for (int j = 0; j < 10; ++j) acc[j] = 0.f;
        for (int i = 0; i < CONV_DIM / 32; ++i) {
            const int c = lane + 32 * i;
            const float g = __ldg(G0 + r * CONV_DIM + c);
#pragma unroll
            for (int j = 0; j < 10; ++j) acc[j] = fmaf(g, ws[c * 10 + j], acc[j]);
        }
#pragma unroll
        for (int j = 0; j < 10; ++j) acc[j] = warp_sum(acc[j]);
        if (lane < 10) {
            float v = acc[0];
#pragma unroll
            for (int j = 1; j < 10; ++j) v = lane == j ? acc[j] : v;
            V[r * 16 + lane] = v;
        }
    }
}

// Overlap-add of the 10 taps (stride 5) into the waveform gradient, times out_scale or / *scale_dev: loss.cu's
// conv0_bwd_finish_kernel, except that every thread of the block stages the constants before the threads past the
// utterance's end leave (the tail block of an utterance whose length is not a multiple of 256 needs all 110 of them).
__global__ void __launch_bounds__(256) conv0_bwd_finish_precise_kernel(const float* __restrict__ V, const float* __restrict__ wav,
                                                                       const UttMeta* __restrict__ meta,
                                                                       const float* __restrict__ consts, long long n_per_utt,
                                                                       float out_scale, const float* __restrict__ scale_dev,
                                                                       float* __restrict__ d_wav) {
    const int b = blockIdx.y;
    __shared__ float cs[112];
    if (threadIdx.x < 110) cs[threadIdx.x] = consts[(long long)b * 112 + threadIdx.x];
    __syncthreads();
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_per_utt) return;
    const UttMeta m = meta[b];
    const float* x = wav + m.wav_off;
    float acc = 0.f;
    const int t_hi = (int)(s / 5), j_lo = (int)(s % 5);
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const int t = t_hi - k, j = j_lo + 5 * k;
        if (t >= 0 && t < m.T0) {
            float v = V[((long long)m.row0 + t) * 16 + j] + cs[j];
#pragma unroll
            for (int jp = 0; jp < 10; ++jp) v = fmaf(-__ldg(x + 5 * t + jp), cs[10 + jp * 10 + j], v);
            acc += v;
        }
    }
    d_wav[(long long)b * n_per_utt + s] = acc * (scale_dev != nullptr ? 1.0f / __ldg(scale_dev) : out_scale);
}

// ------------------------------------------------------------------------------------------------ workspace
struct PBwd {
    float *g_a, *g_b, *g_c, *dO, *D, *tmp;   // tmp: fc2 dgrad output, pos dgrad output, conv dgrad outputs, G0
    op_t *gb_hi, *gb_lo, *gh_hi, *gh_lo, *dqkv_hi, *dqkv_lo, *pg_hi, *pg_lo, *gx_hi, *gx_lo;
    float* g_ln0;
    op_t *gu_hi[2], *gu_lo[2];                // conv-level gradients: 8 zero rows + rows, levels 6/4/2 in [0], 5/3/1 in [1]
    double* c0_sums;
    float *c0_consts, *c0_V;
};

static void bwd_geometry(const Plan& p, int B_bwd, long long* Fe, long long* R0e, long long* pos_rows_e) {
    *Fe = B_bwd < p.B ? p.utt[B_bwd].frame0 : p.frames;
    *R0e = B_bwd < p.B ? p.utt[B_bwd].row0 : p.rows0;
    *pos_rows_e = *Fe + (long long)POS_GAP * B_bwd + POS_K / 2;
}

static size_t carve_bwd(const Plan& p, int B_bwd, void* base, PBwd* out) {
    long long Fe, R0e, pr;
    bwd_geometry(p, B_bwd, &Fe, &R0e, &pr);
    size_t o = 0;
    auto take = [&](size_t bytes) {
        size_t at = o;
        o = align_up_b(o + bytes, 1024);
        return base ? (void*)((char*)base + at) : nullptr;
    };
    PBwd w;
    memset(&w, 0, sizeof(w));
    const size_t F = (size_t)Fe;
    w.g_a = (float*)take(4ull * EMBED * F);
    w.g_b = (float*)take(4ull * EMBED * F);
    w.g_c = (float*)take(4ull * EMBED * F);
    w.dO = (float*)take(4ull * EMBED * F);
    w.D = (float*)take(4ull * HEADS * F);
    size_t tmp = (size_t)FFN * F;
    tmp = std::max<size_t>(tmp, (size_t)EMBED * pr);
    tmp = std::max<size_t>(tmp, (size_t)CONV_DIM * R0e);
    w.tmp = (float*)take(4ull * tmp);
    w.gb_hi = (op_t*)take(2ull * EMBED * F);
    w.gb_lo = (op_t*)take(2ull * EMBED * F);
    w.gh_hi = (op_t*)take(2ull * FFN * F);
    w.gh_lo = (op_t*)take(2ull * FFN * F);
    w.dqkv_hi = (op_t*)take(2ull * 3 * EMBED * F);
    w.dqkv_lo = (op_t*)take(2ull * 3 * EMBED * F);
    w.pg_hi = (op_t*)take(2ull * POS_G * POS_GC * (pr + POS_K));
    w.pg_lo = (op_t*)take(2ull * POS_G * POS_GC * (pr + POS_K));
    w.gx_hi = (op_t*)take(2ull * EMBED * F);
    w.gx_lo = (op_t*)take(2ull * EMBED * F);
    w.g_ln0 = (float*)take(4ull * CONV_DIM * F);
    for (int i = 0; i < 2; ++i) {
        const size_t rows = (size_t)(R0e >> (2 - i)) + 16;  // level 2 / level 1 are the largest of each set
        w.gu_hi[i] = (op_t*)take(2ull * CONV_DIM * rows);
        w.gu_lo[i] = (op_t*)take(2ull * CONV_DIM * rows);
    }
    w.c0_sums = (double*)take(8ull * 2 * CONV_DIM * B_bwd);
    w.c0_consts = (float*)take(4ull * 112 * B_bwd);
    w.c0_V = (float*)take(4ull * 16 * R0e);
    if (out) *out = w;
    return o;
}

size_t precise_bwd_bytes(const Plan& p, int B_bwd) { return carve_bwd(p, B_bwd, nullptr, nullptr); }

static GemmEpilogue epi_split(int flags, const SplitW& w, const float* resid, float* out_f, long long ld) {
    GemmEpilogue e = epi_linear(flags | EPI_PRECISE, nullptr, resid, out_f, nullptr, ld);
    e.acc_scale = w.inv_scale;
    return e;
}

// ------------------------------------------------------------------------------------------------ the chain
int backward_precise(Handle* h, const Plan& p, void* saved, const PBwdArgs& a, const float* wav, int64_t N, float* d_wav,
                     void* workspace, size_t workspace_bytes, cudaStream_t st) {
    NB_CHECK(h->pw.built, "this handle was created without the fp32-class weights (precision_mode 1)");
    PWorkspace ws;
    carve_precise(p, saved, &ws, true);
    PBwd g;
    const size_t need = carve_bwd(p, a.B_bwd, workspace, &g);
    NB_CHECK(workspace_bytes >= need, "backward (fp32 mode): workspace too small (%zu < %zu bytes)", workspace_bytes, need);
    const Weights& w = h->w;
    const PreciseWeights& pw = h->pw;
    const int B = a.B_bwd;
    long long Fe, R0e, pos_rows_e;
    bwd_geometry(p, B, &Fe, &R0e, &pos_rows_e);
    const unsigned row_blocks = (unsigned)((Fe + 7) / 8);
    static bool attr_set[64] = {false};
    if (bool* flag = device_once_flag(attr_set)) {
        NB_CUDA(cudaFuncSetAttribute(attn_bwd_kv_precise_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PB_KV_SMEM));
        NB_CUDA(cudaFuncSetAttribute(attn_bwd_q_precise_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PB_Q_SMEM));
        *flag = true;
    }
    NB_CUDA(cudaMemsetAsync(g.dqkv_hi, 0, 2ull * 3 * EMBED * Fe, st));  // padding rows stay zero
    NB_CUDA(cudaMemsetAsync(g.dqkv_lo, 0, 2ull * 3 * EMBED * Fe, st));
    const float* g_running = nullptr;
    for (int l = a.top; l >= 0; --l) {
        const LayerWeights& W = w.layer[l];
        ln768_bwd_precise_kernel<<<row_blocks, 256, 0, st>>>(g_running, ws.pre2[l], ws.meta, B, Fe, W.ln2_g, a.seed_layer,
                                                             a.g_layers[l], a.user_T, l == LAYERS - 1 ? a.g_pool : nullptr,
                                                             a.scale_dev, g.g_b, g.gb_hi, g.gb_lo);
        NB_LAUNCHED();
        {   // fc2 dgrad, then times gelu'(fc1 pre-activation)
            GemmOperand A{g.gb_hi, Fe, EMBED, 0, 0, g.gb_lo};
            GemmOperand Bw{pw.fc2_t[l].hi, FFN, EMBED, 0, 0, pw.fc2_t[l].lo};
            NB_TRY(gemm_h16(st, A, Bw, (int)Fe, FFN, EMBED, 1, epi_split(EPI_OUT_F32, pw.fc2_t[l], nullptr, g.tmp, FFN), 0));
            const long long n = Fe * FFN;
            mul_dgelu_split_kernel<<<(unsigned)((n / 8 + 255) / 256), 256, 0, st>>>(g.tmp, ws.fc1_pre[l], n, g.gh_hi, g.gh_lo);
            NB_LAUNCHED();
        }
        {   // fc1 dgrad + residual branch
            GemmOperand A{g.gh_hi, Fe, FFN, 0, 0, g.gh_lo};
            GemmOperand Bw{pw.fc1_t[l].hi, EMBED, FFN, 0, 0, pw.fc1_t[l].lo};
            NB_TRY(gemm_h16(st, A, Bw, (int)Fe, EMBED, FFN, 1, epi_split(EPI_RESID | EPI_OUT_F32, pw.fc1_t[l], g.g_b, g.g_c, EMBED), 0));
        }
        ln768_bwd_precise_kernel<<<row_blocks, 256, 0, st>>>(g.g_c, ws.pre1[l], ws.meta, B, Fe, W.ln1_g, 0.f, nullptr, 0, nullptr,
                                                             nullptr, g.g_b, g.gb_hi, g.gb_lo);
        NB_LAUNCHED();
        {   // out_proj dgrad -> dO (fp32)
            GemmOperand A{g.gb_hi, Fe, EMBED, 0, 0, g.gb_lo};
            GemmOperand Bw{pw.o_t[l].hi, EMBED, EMBED, 0, 0, pw.o_t[l].lo};
            NB_TRY(gemm_h16(st, A, Bw, (int)Fe, EMBED, EMBED, 1, epi_split(EPI_OUT_F32, pw.o_t[l], nullptr, g.dO, EMBED), 0));
        }
        {
            const long long n = Fe * HEADS;
            attn_d_precise_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(g.dO, ws.attn_hi[l], ws.attn_lo[l], Fe, g.D);
            NB_LAUNCHED();
            dim3 grid((p.max_T + PB_T - 1) / PB_T, HEADS, B);
            attn_bwd_kv_precise_kernel<<<grid, 256, PB_KV_SMEM, st>>>(ws.qkv[l], g.dO, ws.lse[l], g.D, ws.meta, g.dqkv_hi, g.dqkv_lo);
            NB_LAUNCHED();
            attn_bwd_q_precise_kernel<<<grid, 256, PB_Q_SMEM, st>>>(ws.qkv[l], g.dO, ws.lse[l], g.D, ws.meta, g.dqkv_hi, g.dqkv_lo);
            NB_LAUNCHED();
        }
        {   // fused q/k/v dgrad + residual branch -> gradient wrt this layer's input
            GemmOperand A{g.dqkv_hi, Fe, 3 * EMBED, 0, 0, g.dqkv_lo};
            GemmOperand Bw{pw.qkv_t[l].hi, EMBED, 3 * EMBED, 0, 0, pw.qkv_t[l].lo};
            NB_TRY(gemm_h16(st, A, Bw, (int)Fe, EMBED, 3 * EMBED, 1, epi_split(EPI_RESID | EPI_OUT_F32, pw.qkv_t[l], g.g_b, g.g_a, EMBED), 0));
        }
        g_running = g.g_a;
    }
    {   // encoder LayerNorm + positional conv
        const long long rows_alloc = pos_rows_e + POS_K;
        NB_CUDA(cudaMemsetAsync(g.pg_hi, 0, 2ull * POS_G * POS_GC * rows_alloc, st));
        NB_CUDA(cudaMemsetAsync(g.pg_lo, 0, 2ull * POS_G * POS_GC * rows_alloc, st));
        pos_bwd_prep_precise_kernel<<<row_blocks, 256, 0, st>>>(g.g_a, ws.x0, ws.pos_pre, ws.meta, B, Fe, w.lne_g, rows_alloc, g.g_b,
                                                                g.pg_hi, g.pg_lo);
        NB_LAUNCHED();
        GemmOperand A{g.pg_hi, pos_rows_e, POS_GC, rows_alloc * POS_GC, 0, g.pg_lo};
        GemmOperand Bw{pw.pos_t.hi, POS_GC, (long long)POS_K * POS_GC, (long long)POS_GC * POS_K * POS_GC, 0, pw.pos_t.lo};
        GemmEpilogue e = epi_split(EPI_OUT_F32, pw.pos_t, nullptr, g.tmp, EMBED);
        e.out_bstride = POS_GC;
        NB_TRY(gemm_h16(st, A, Bw, (int)pos_rows_e, POS_GC, POS_K * POS_GC, POS_G, e, 0));
        pos_bwd_finish_precise_kernel<<<row_blocks, 256, 0, st>>>(g.g_b, g.tmp, ws.meta, B, Fe, g.gx_hi, g.gx_lo);
        NB_LAUNCHED();
    }
    {   // feature projection dgrad
        GemmOperand A{g.gx_hi, Fe, EMBED, 0, 0, g.gx_lo};
        GemmOperand Bw{pw.proj_t.hi, CONV_DIM, EMBED, 0, 0, pw.proj_t.lo};
        NB_TRY(gemm_h16(st, A, Bw, (int)Fe, CONV_DIM, EMBED, 1, epi_split(EPI_OUT_F32, pw.proj_t, nullptr, g.g_ln0, CONV_DIM), 0));
    }
    // conv stack.  Gradient planes start 8 rows into their allocation so that "row -1" reads zeros.
    op_t *gh[7], *gl[7];
    for (int i = 0; i < 2; ++i) {
        NB_CUDA(cudaMemsetAsync(g.gu_hi[i], 0, 2ull * CONV_DIM * 8, st));
        NB_CUDA(cudaMemsetAsync(g.gu_lo[i], 0, 2ull * CONV_DIM * 8, st));
    }
    for (int l = 1; l < 7; ++l) {
        gh[l] = g.gu_hi[(l & 1) ? 1 : 0] + 8 * CONV_DIM;
        gl[l] = g.gu_lo[(l & 1) ? 1 : 0] + 8 * CONV_DIM;
    }
    ln512_bwd_precise_kernel<<<row_blocks, 256, 0, st>>>(g.g_ln0, ws.u[6], ws.meta, B, Fe, w.ln0_g, a.feature_grad_mult, gh[6], gl[6]);
    NB_LAUNCHED();
    for (int l = 6; l >= 1; --l) {
        const long long M = R0e >> l;
        const SplitW& wt = pw.conv_t[l];
        if (CONV_KERNEL[l] == 2) {  // rows 2m and 2m+1 of level l-1 in one GEMM: N = 1024 = (tap, cin)
            GemmOperand A{gh[l], M, CONV_DIM, 0, 0, gl[l]};
            GemmOperand Bw{wt.hi, 2 * CONV_DIM, CONV_DIM, 0, 0, wt.lo};
            NB_TRY(gemm_h16(st, A, Bw, (int)M, 2 * CONV_DIM, CONV_DIM, 1, epi_split(EPI_OUT_F32, wt, nullptr, g.tmp, 2 * CONV_DIM), 0));
        } else {
            {   // even rows 2m: taps 2 (from row m-1) and 0 (row m), overlapping rows starting one row early
                GemmOperand A{gh[l] - CONV_DIM, M, CONV_DIM, 0, 0, gl[l] - CONV_DIM};
                GemmOperand Bw{pw.conv_te[l].hi, CONV_DIM, 2 * CONV_DIM, 0, 0, pw.conv_te[l].lo};
                NB_TRY(gemm_h16(st, A, Bw, (int)M, CONV_DIM, 2 * CONV_DIM, 1,
                                epi_split(EPI_OUT_F32, pw.conv_te[l], nullptr, g.tmp, 2 * CONV_DIM), 0));
            }
            {   // odd rows 2m+1: tap 1
                GemmOperand A{gh[l], M, CONV_DIM, 0, 0, gl[l]};
                GemmOperand Bw{wt.hi + (size_t)CONV_DIM * CONV_DIM, CONV_DIM, CONV_DIM, 0, 0, wt.lo + (size_t)CONV_DIM * CONV_DIM};
                NB_TRY(gemm_h16(st, A, Bw, (int)M, CONV_DIM, CONV_DIM, 1,
                                epi_split(EPI_OUT_F32, wt, nullptr, g.tmp + CONV_DIM, 2 * CONV_DIM), 0));
            }
        }
        const long long rows = R0e >> (l - 1);
        // level 0: G0 = dL/du0 * gamma * rstd in fp32, in place
        conv_dgelu_precise_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, st>>>(
            g.tmp, ws.u[l - 1], ws.meta, B, rows, l - 1, l == 1 ? ws.c0_fold : nullptr, l == 1 ? g.tmp : nullptr,
            l == 1 ? nullptr : gh[l - 1], l == 1 ? nullptr : gl[l - 1]);
        NB_LAUNCHED();
    }
    // conv0 + GroupNorm backward: g.tmp = G0
    NB_CUDA(cudaMemsetAsync(g.c0_sums, 0, 8ull * 2 * CONV_DIM * B, st));
    conv0_bwd_stats_precise_kernel<<<(unsigned)(R0e / 64), 256, 0, st>>>(g.tmp, wav, ws.meta, B, w.conv0_w, ws.gn_stat, g.c0_sums);
    NB_LAUNCHED();
    conv0_bwd_consts_kernel<<<B, 128, 0, st>>>(g.c0_sums, ws.meta, w.conv0_w, ws.gn_stat, g.c0_consts);
    NB_LAUNCHED();
    conv0_dgrad_precise_kernel<<<(unsigned)std::min<long long>((R0e + 7) / 8, 148 * 16), 256, 0, st>>>(g.tmp, R0e, w.conv0_w, g.c0_V);
    NB_LAUNCHED();
    dim3 fgrid((unsigned)((N + 255) / 256), B);
    conv0_bwd_finish_precise_kernel<<<fgrid, 256, 0, st>>>(g.c0_V, wav, ws.meta, g.c0_consts, N, a.out_scale, a.scale_dev, d_wav);
    NB_LAUNCHED();
    return 0;
}

}  // namespace nb
