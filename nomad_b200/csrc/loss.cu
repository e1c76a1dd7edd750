// NOMAD loss (reference nomad.py:142-146, 243-282) forward + backward to the estimate waveform.
//
// The 2B utterances (B estimates followed by B clean references, all N samples) run through ONE forward
// pass in "save" mode; the loss is the sum of 13 mean-L1 terms between the two halves; the backward
// walks the estimate half only (dgrad chain, no weight gradients).  All gradient tensors carry a
// power-of-two scale S (chosen so the L1 seeds are O(1)) to stay inside fp16's normal range; the final
// kernel divides it out.  fairseq's GradMultiply(feature_grad_mult) on the conv features is applied at
// the LayerNorm(512) boundary.
#include <cmath>
#include <cstdlib>
#include <cstring>

#include "../../include/nomad_b200.h"
#include "precise.cuh"

namespace nb {

int launch_attention_bwd(cudaStream_t st, const op_t* qkv, const op_t* attn_out, const op_t* d_out, const float* lse,
                         float* D, const UttMeta* meta, int B, int max_T, long long frames, op_t* d_qkv, bool consistent_d);

// ---------------------------------------------------------------------------------------------
struct Row768f {
    float v[24];
};
__device__ __forceinline__ void load_row768(Row768f& r, const float* __restrict__ p, int lane) {
#pragma unroll
    for (int h = 0; h < 3; ++h) {
        const float4* xp = reinterpret_cast<const float4*>(p + (lane + 32 * h) * 8);
        const float4 a = __ldg(xp), c = __ldg(xp + 1);
        float* v = r.v + 8 * h;
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = c.x; v[5] = c.y; v[6] = c.z; v[7] = c.w;
    }
}
__device__ __forceinline__ void load_vec768(Row768f& r, const float* __restrict__ p, int lane) { load_row768(r, p, lane); }
// x -> xhat (in place), returns rstd
__device__ __forceinline__ float normalise768(Row768f& r) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 24; ++i) s += r.v[i];
    const float mean = warp_sum(s) * (1.0f / EMBED);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < 24; ++i) { r.v[i] = __fsub_rn(r.v[i], mean); q = fmaf(r.v[i], r.v[i], q); }
    const float rstd = rsqrtf(warp_sum(q) * (1.0f / EMBED) + 1e-5f);
    // explicit rounding: the compiler must not contract this product into a later (est - clean) subtraction,
    // or identical inputs stop giving an exactly zero L1 term / zero gradient sign
#pragma unroll
    for (int i = 0; i < 24; ++i) r.v[i] = __fmul_rn(r.v[i], rstd);
    return rstd;
}
__device__ __forceinline__ void store_row768(const Row768f& r, float* __restrict__ x, op_t* __restrict__ xh, int lane) {
#pragma unroll
    for (int h = 0; h < 3; ++h) {
        const int c0 = (lane + 32 * h) * 8;
        const float* v = r.v + 8 * h;
        if (x != nullptr) {
            float4* xo = reinterpret_cast<float4*>(x + c0);
            xo[0] = make_float4(v[0], v[1], v[2], v[3]);
            xo[1] = make_float4(v[4], v[5], v[6], v[7]);
        }
        if (xh != nullptr)
            *reinterpret_cast<uint4*>(xh + c0) =
                make_uint4(pack_op(v[0], v[1]), pack_op(v[2], v[3]), pack_op(v[4], v[5]), pack_op(v[6], v[7]));
    }
}

// ---------------------------------------------------------------------------------------------
// One L1 term between the two halves of a layer output x = LN(pre):  acc += sum |x_est - x_clean|
__global__ void __launch_bounds__(256) l1_layer_kernel(const float* __restrict__ pre, const UttMeta* __restrict__ meta,
                                                       int B_est, long long frames_est, const float* __restrict__ g,
                                                       double* __restrict__ acc) {
    const long long f = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    float tot = 0.f;
    if (f < frames_est) {
        const int b = find_utt_by_frame(meta, B_est, (int)f);
        if ((int)f - meta[b].frame0 < meta[b].T) {
            Row768f e, c, gg;
            load_row768(e, pre + f * EMBED, lane);
            load_row768(c, pre + (f + frames_est) * EMBED, lane);
            load_vec768(gg, g, lane);
            normalise768(e);
            normalise768(c);
#pragma unroll
            for (int i = 0; i < 24; ++i) tot += fabsf(__fsub_rn(e.v[i], c.v[i]) * gg.v[i]);  // beta cancels
        }
    }
    tot = warp_sum(tot);
    __shared__ float red[8];
    if (lane == 0) red[threadIdx.x >> 5] = tot;
    __syncthreads();
    if (threadIdx.x == 0) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) s += red[w];
        if (s != 0.f) atomicAdd(acc, (double)s);
    }
}

// ---------------------------------------------------------------------------------------------
// LayerNorm(768) backward on the estimate rows, with the optional L1 seed of this layer's output and an
// optional per-utterance broadcast gradient (mean-pool of the head).
//   g = g_in + seed * sign(x_est - x_clean) + g_pool[utt]
//   g_pre = rstd * (g*gamma - mean(g*gamma) - xhat * mean(g*gamma*xhat))
__global__ void __launch_bounds__(256) ln768_bwd_kernel(const float* __restrict__ g_in, const float* __restrict__ pre,
                                                        const UttMeta* __restrict__ meta, int B_est, long long frames_est,
                                                        const float* __restrict__ gam, float seed,
                                                        const float* __restrict__ g_pool, float* __restrict__ g_out,
                                                        op_t* __restrict__ g_out_h) {
    const long long f = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (f >= frames_est) return;
    const int lane = threadIdx.x & 31;
    const int b = find_utt_by_frame(meta, B_est, (int)f);
    Row768f out;
    if ((int)f - meta[b].frame0 >= meta[b].T) {
#pragma unroll
        for (int i = 0; i < 24; ++i) out.v[i] = 0.f;
        store_row768(out, g_out ? g_out + f * EMBED : nullptr, g_out_h ? g_out_h + f * EMBED : nullptr, lane);
        return;
    }
    Row768f xh, gg, g;
    load_row768(xh, pre + f * EMBED, lane);
    load_vec768(gg, gam, lane);
    const float rstd = normalise768(xh);
    if (g_in != nullptr) {
        load_row768(g, g_in + f * EMBED, lane);
    } else {
#pragma unroll
        for (int i = 0; i < 24; ++i) g.v[i] = 0.f;
    }
    if (seed != 0.f) {
        Row768f xc;
        load_row768(xc, pre + (f + frames_est) * EMBED, lane);
        normalise768(xc);
#pragma unroll
        for (int i = 0; i < 24; ++i) {
            const float d = __fsub_rn(xh.v[i], xc.v[i]) * gg.v[i];  // x_est - x_clean (beta cancels)
            g.v[i] += d > 0.f ? seed : (d < 0.f ? -seed : 0.f);
        }
    }
    if (g_pool != nullptr) {
        Row768f gp;
        load_vec768(gp, g_pool + (long long)b * EMBED, lane);
#pragma unroll
        for (int i = 0; i < 24; ++i) g.v[i] += gp.v[i];
    }
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < 24; ++i) {
        g.v[i] *= gg.v[i];
        s1 += g.v[i];
        s2 = fmaf(g.v[i], xh.v[i], s2);
    }
    s1 = warp_sum(s1) * (1.0f / EMBED);
    s2 = warp_sum(s2) * (1.0f / EMBED);
#pragma unroll
    for (int i = 0; i < 24; ++i) out.v[i] = rstd * (g.v[i] - s1 - xh.v[i] * s2);
    store_row768(out, g_out ? g_out + f * EMBED : nullptr, g_out_h ? g_out_h + f * EMBED : nullptr, lane);
}

// The same backward with caller-given upstream gradients (nomad_b200_layers_bwd): g_user is the gradient wrt this
// layer's output in the caller's (B, T, 768) layout (row b * user_T + t, may be null); S is read from the device.
//   g = g_in + S * g_user[b, t] + S * g_pool[utt]
__global__ void __launch_bounds__(256) ln768_bwd_user_kernel(const float* __restrict__ g_in, const float* __restrict__ pre,
                                                             const UttMeta* __restrict__ meta, int B, long long frames,
                                                             const float* __restrict__ gam, const float* __restrict__ g_user,
                                                             int user_T, const float* __restrict__ g_pool,
                                                             const float* __restrict__ scale, float* __restrict__ g_out,
                                                             op_t* __restrict__ g_out_h) {
    const long long f = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (f >= frames) return;
    const int lane = threadIdx.x & 31;
    const int b = find_utt_by_frame(meta, B, (int)f);
    const int t = (int)f - meta[b].frame0;
    Row768f out;
    if (t >= meta[b].T) {
#pragma unroll
        for (int i = 0; i < 24; ++i) out.v[i] = 0.f;
        store_row768(out, g_out + f * EMBED, g_out_h + f * EMBED, lane);
        return;
    }
    const float S = __ldg(scale);
    Row768f xh, gg, g;
    load_row768(xh, pre + f * EMBED, lane);
    load_vec768(gg, gam, lane);
    const float rstd = normalise768(xh);
    if (g_in != nullptr) {
        load_row768(g, g_in + f * EMBED, lane);
    } else {
#pragma unroll
        for (int i = 0; i < 24; ++i) g.v[i] = 0.f;
    }
    if (g_user != nullptr) {
        Row768f gu;
        load_row768(gu, g_user + ((long long)b * user_T + t) * EMBED, lane);
#pragma unroll
        for (int i = 0; i < 24; ++i) g.v[i] = fmaf(S, gu.v[i], g.v[i]);
    }
    if (g_pool != nullptr) {
        Row768f gp;
        load_vec768(gp, g_pool + (long long)b * EMBED, lane);
#pragma unroll
        for (int i = 0; i < 24; ++i) g.v[i] = fmaf(S, gp.v[i], g.v[i]);
    }
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < 24; ++i) {
        g.v[i] *= gg.v[i];
        s1 += g.v[i];
        s2 = fmaf(g.v[i], xh.v[i], s2);
    }
    s1 = warp_sum(s1) * (1.0f / EMBED);
    s2 = warp_sum(s2) * (1.0f / EMBED);
#pragma unroll
    for (int i = 0; i < 24; ++i) out.v[i] = rstd * (g.v[i] - s1 - xh.v[i] * s2);
    store_row768(out, g_out + f * EMBED, g_out_h + f * EMBED, lane);
}

// Power-of-two gradient scale of the autograd backward, chosen on the device: S with max|g| * S in [1, 2) over every
// upstream gradient given (S = 1 when they are all zero or not finite).  state[0] = running max as float bits (|g| >= 0
// orders like its bits), state[1] = finished blocks; both zeroed by the caller.  The last block writes S.
struct ScaleSources {
    const float* p[LAYERS + 1];
    long long n[LAYERS + 1];
};
__global__ void __launch_bounds__(256) grad_scale_kernel(ScaleSources src, unsigned* __restrict__ state, float* __restrict__ scale) {
    unsigned m = 0;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (int a = 0; a < LAYERS + 1; ++a) {
        const float* p = src.p[a];
        if (p == nullptr) continue;
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < src.n[a]; i += stride)
            m = max(m, __float_as_uint(fabsf(__ldg(p + i))));
    }
    m = __reduce_max_sync(0xffffffffu, m);
    __shared__ unsigned red[8];
    __shared__ bool last;
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) m = max(m, red[w]);
        atomicMax(state, m);
        __threadfence();
        last = atomicAdd(state + 1, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (last && threadIdx.x == 0) {
        const float mx = __uint_as_float(atomicMax(state, 0u));
        float S = 1.f;
        if (mx > 0.f && mx <= 3.402823466e38f) S = ldexpf(1.f, min(max(-ilogbf(mx), -126), 127));
        *scale = S;
    }
}

// Head backward from an explicit upstream gradient g_emb of e = normalize(W relu(pooled) + b) (the forward's snapshot of
// the head): gy[b] = d<g_emb, e> / d y, unscaled.  y is recomputed in the forward kernel's order.
__global__ void __launch_bounds__(256) head_emb_bwd_kernel(const float* __restrict__ pooled, const float* __restrict__ head_wt,
                                                           const float* __restrict__ head_b, const float* __restrict__ g_emb,
                                                           float* __restrict__ gy) {
    const int b = blockIdx.x, tid = threadIdx.x;
    __shared__ float pr[EMBED];
    __shared__ float red[2][8];
    for (int k = tid; k < EMBED; k += 256) pr[k] = fmaxf(pooled[(long long)b * EMBED + k], 0.f);
    __syncthreads();
    float y = head_b[tid];
    for (int k = 0; k < EMBED; ++k) y = fmaf(pr[k], __ldg(head_wt + k * EMB + tid), y);
    const float sq = warp_sum(y * y);
    if ((tid & 31) == 0) red[0][tid >> 5] = sq;
    __syncthreads();
    float n = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) n += red[0][w];
    n = fmaxf(sqrtf(n), 1e-12f);
    const float e = y / n, ge = g_emb[(long long)b * EMB + tid];
    const float dp = warp_sum(ge * e);
    if ((tid & 31) == 0) red[1][tid >> 5] = dp;
    __syncthreads();
    float dot = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) dot += red[1][w];
    gy[(long long)b * EMB + tid] = (ge - e * dot) / n;  // backward of y / max(||y||, eps)
}

// ---------------------------------------------------------------------------------------------
// Head term: e = normalize(W relu(pooled) + b) for both halves; acc += sum |e_est - e_clean|;
// g_pool[b][k] = d(term) / d x[t, k] for every valid frame t of estimate b (already divided by T).
__global__ void __launch_bounds__(256) head_bwd_kernel(const float* __restrict__ pooled, const UttMeta* __restrict__ meta,
                                                       int B_est, const float* __restrict__ head_wt,
                                                       const float* __restrict__ head_w, const float* __restrict__ head_b,
                                                       float seed, double* __restrict__ acc, float* __restrict__ g_pool) {
    const int b = blockIdx.x, tid = threadIdx.x;
    __shared__ float pe[EMBED], pc[EMBED], gy[EMB];
    __shared__ float red[3][8];
    for (int k = tid; k < EMBED; k += 256) {
        pe[k] = pooled[(long long)b * EMBED + k];
        pc[k] = pooled[(long long)(b + B_est) * EMBED + k];
    }
    __syncthreads();
    float ye = head_b[tid], yc = ye;
    for (int k = 0; k < EMBED; ++k) {
        const float w = __ldg(head_wt + k * EMB + tid);
        ye = fmaf(fmaxf(pe[k], 0.f), w, ye);
        yc = fmaf(fmaxf(pc[k], 0.f), w, yc);
    }
    float se = warp_sum(ye * ye), sc = warp_sum(yc * yc);
    if ((tid & 31) == 0) { red[0][tid >> 5] = se; red[1][tid >> 5] = sc; }
    __syncthreads();
    float ne = 0.f, nc = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) { ne += red[0][w]; nc += red[1][w]; }
    ne = fmaxf(sqrtf(ne), 1e-12f);
    nc = fmaxf(sqrtf(nc), 1e-12f);
    const float ee = ye / ne, ec = yc / nc;
    const float d = ee - ec;
    const float ge = d > 0.f ? seed : (d < 0.f ? -seed : 0.f);
    float l1 = warp_sum(fabsf(d)), dot = warp_sum(ge * ee);
    __syncthreads();
    if ((tid & 31) == 0) { red[0][tid >> 5] = l1; red[2][tid >> 5] = dot; }
    __syncthreads();
    float l1t = 0.f, dott = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) { l1t += red[0][w]; dott += red[2][w]; }
    if (tid == 0) atomicAdd(acc, (double)l1t);
    gy[tid] = (ge - ee * dott) / ne;  // backward of x / max(||x||, eps)
    __syncthreads();
    const float invT = 1.0f / (float)meta[b].T;
    for (int k = tid; k < EMBED; k += 256) {
        float a = 0.f;
        for (int o = 0; o < EMB; ++o) a = fmaf(gy[o], __ldg(head_w + (long long)o * EMBED + k), a);
        g_pool[(long long)b * EMBED + k] = pe[k] > 0.f ? a * invT : 0.f;
    }
}

// ---------------------------------------------------------------------------------------------
// Positional-conv backward, step 1: encoder LayerNorm backward (z = x0 + pos_y recomputed) -> g_z (fp32),
// and scatter of g_z * gelu'(pos pre-activation) into the grouped, zero-padded layout for the dgrad GEMM.
__global__ void __launch_bounds__(256) pos_bwd_prep_kernel(const float* __restrict__ g_x, const float* __restrict__ x0,
                                                           const op_t* __restrict__ pos_y, const op_t* __restrict__ pos_aux,
                                                           const UttMeta* __restrict__ meta, int B_est, long long frames_est,
                                                           const float* __restrict__ gam, long long pos_rows_alloc,
                                                           float* __restrict__ g_z, op_t* __restrict__ pos_g) {
    const long long f = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (f >= frames_est) return;
    const int lane = threadIdx.x & 31;
    const int b = find_utt_by_frame(meta, B_est, (int)f);
    const int t = (int)f - meta[b].frame0;
    Row768f out;
    if (t >= meta[b].T) {
#pragma unroll
        for (int i = 0; i < 24; ++i) out.v[i] = 0.f;
        store_row768(out, g_z + f * EMBED, nullptr, lane);
        return;
    }
    const long long m = (long long)meta[b].pos0 + t - POS_K / 2;  // row of this frame in pos_y / pos_aux
    Row768f z, g, gg;
    load_row768(z, x0 + f * EMBED, lane);
    float aux[24];
#pragma unroll
    for (int h = 0; h < 3; ++h) {
        const int c0 = (lane + 32 * h) * 8;
        const uint4 y = __ldg(reinterpret_cast<const uint4*>(pos_y + m * EMBED + c0));
        const uint4 a = __ldg(reinterpret_cast<const uint4*>(pos_aux + m * EMBED + c0));
        float2 t0 = unpack_op(y.x), t1 = unpack_op(y.y), t2 = unpack_op(y.z), t3 = unpack_op(y.w);
        float* v = z.v + 8 * h;
        v[0] += t0.x; v[1] += t0.y; v[2] += t1.x; v[3] += t1.y; v[4] += t2.x; v[5] += t2.y; v[6] += t3.x; v[7] += t3.y;
        t0 = unpack_op(a.x); t1 = unpack_op(a.y); t2 = unpack_op(a.z); t3 = unpack_op(a.w);
        float* q = aux + 8 * h;
        q[0] = t0.x; q[1] = t0.y; q[2] = t1.x; q[3] = t1.y; q[4] = t2.x; q[5] = t2.y; q[6] = t3.x; q[7] = t3.y;
    }
    const float rstd = normalise768(z);
    load_row768(g, g_x + f * EMBED, lane);
    load_vec768(gg, gam, lane);
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < 24; ++i) {
        g.v[i] *= gg.v[i];
        s1 += g.v[i];
        s2 = fmaf(g.v[i], z.v[i], s2);
    }
    s1 = warp_sum(s1) * (1.0f / EMBED);
    s2 = warp_sum(s2) * (1.0f / EMBED);
#pragma unroll
    for (int i = 0; i < 24; ++i) out.v[i] = rstd * (g.v[i] - s1 - z.v[i] * s2);
    store_row768(out, g_z + f * EMBED, nullptr, lane);
    const long long p = (long long)meta[b].pos0 + t;
#pragma unroll
    for (int h = 0; h < 3; ++h) {
        const int ch = (lane + 32 * h) * 8, grp = ch / POS_GC, cc = ch % POS_GC;
        const float* v = out.v + 8 * h;
        const float* q = aux + 8 * h;
        *reinterpret_cast<uint4*>(pos_g + ((long long)grp * pos_rows_alloc + p) * POS_GC + cc) =
            make_uint4(pack_op(v[0] * q[0], v[1] * q[1]), pack_op(v[2] * q[2], v[3] * q[3]),
                       pack_op(v[4] * q[4], v[5] * q[5]), pack_op(v[6] * q[6], v[7] * q[7]));
    }
}

// step 2 (after the dgrad GEMM): g_x0 = g_z + dgrad[pos0 + t - 63]  -> 16-bit operand of the projection dgrad
__global__ void __launch_bounds__(256) pos_bwd_finish_kernel(const float* __restrict__ g_z, const op_t* __restrict__ pos_dy,
                                                             const UttMeta* __restrict__ meta, int B_est,
                                                             long long frames_est, op_t* __restrict__ g_x0h) {
    const long long f = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (f >= frames_est) return;
    const int lane = threadIdx.x & 31;
    const int b = find_utt_by_frame(meta, B_est, (int)f);
    const int t = (int)f - meta[b].frame0;
    Row768f r;
    if (t >= meta[b].T) {
#pragma unroll
        for (int i = 0; i < 24; ++i) r.v[i] = 0.f;
    } else {
        load_row768(r, g_z + f * EMBED, lane);
        const long long m = (long long)meta[b].pos0 + t - (POS_K / 2 - 1);
#pragma unroll
        for (int h = 0; h < 3; ++h) {
            const uint4 y = __ldg(reinterpret_cast<const uint4*>(pos_dy + m * EMBED + (lane + 32 * h) * 8));
            const float2 t0 = unpack_op(y.x), t1 = unpack_op(y.y), t2 = unpack_op(y.z), t3 = unpack_op(y.w);
            float* v = r.v + 8 * h;
            v[0] += t0.x; v[1] += t0.y; v[2] += t1.x; v[3] += t1.y; v[4] += t2.x; v[5] += t2.y; v[6] += t3.x; v[7] += t3.y;
        }
    }
    store_row768(r, nullptr, g_x0h + f * EMBED, lane);
}

// ---------------------------------------------------------------------------------------------
// LayerNorm(512) backward fused with GradMultiply and the GELU gradient of conv layer 6:
//   g_u6 = fgm * LN_bwd(g; y6) * gelu'(u6)      (aux6 is zero on padding rows)
__global__ void __launch_bounds__(256) ln512_bwd_kernel(const float* __restrict__ g_in, const op_t* __restrict__ y6,
                                                        const op_t* __restrict__ aux6, long long rows,
                                                        const float* __restrict__ gam, float fgm, op_t* __restrict__ g_u6) {
    const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= rows) return;
    const int lane = threadIdx.x & 31;
    float x[16], g[16], a[16];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int c0 = (lane + 32 * h) * 8;
        const uint4 u = __ldg(reinterpret_cast<const uint4*>(y6 + row * CONV_DIM + c0));
        const uint4 w = __ldg(reinterpret_cast<const uint4*>(aux6 + row * CONV_DIM + c0));
        float2 f;
        f = unpack_op(u.x); x[8 * h + 0] = f.x; x[8 * h + 1] = f.y;
        f = unpack_op(u.y); x[8 * h + 2] = f.x; x[8 * h + 3] = f.y;
        f = unpack_op(u.z); x[8 * h + 4] = f.x; x[8 * h + 5] = f.y;
        f = unpack_op(u.w); x[8 * h + 6] = f.x; x[8 * h + 7] = f.y;
        f = unpack_op(w.x); a[8 * h + 0] = f.x; a[8 * h + 1] = f.y;
        f = unpack_op(w.y); a[8 * h + 2] = f.x; a[8 * h + 3] = f.y;
        f = unpack_op(w.z); a[8 * h + 4] = f.x; a[8 * h + 5] = f.y;
        f = unpack_op(w.w); a[8 * h + 6] = f.x; a[8 * h + 7] = f.y;
        const float4 g0 = __ldg(reinterpret_cast<const float4*>(g_in + row * CONV_DIM + c0));
        const float4 g1 = __ldg(reinterpret_cast<const float4*>(g_in + row * CONV_DIM + c0 + 4));
        const float4 m0 = __ldg(reinterpret_cast<const float4*>(gam + c0)), m1 = __ldg(reinterpret_cast<const float4*>(gam + c0 + 4));
        g[8 * h + 0] = g0.x * m0.x; g[8 * h + 1] = g0.y * m0.y; g[8 * h + 2] = g0.z * m0.z; g[8 * h + 3] = g0.w * m0.w;
        g[8 * h + 4] = g1.x * m1.x; g[8 * h + 5] = g1.y * m1.y; g[8 * h + 6] = g1.z * m1.z; g[8 * h + 7] = g1.w * m1.w;
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) s += x[i];
    const float mean = warp_sum(s) * (1.0f / CONV_DIM);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) { x[i] -= mean; q = fmaf(x[i], x[i], q); }
    const float rstd = rsqrtf(warp_sum(q) * (1.0f / CONV_DIM) + 1e-5f);
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) { x[i] *= rstd; s1 += g[i]; s2 = fmaf(g[i], x[i], s2); }
    s1 = warp_sum(s1) * (1.0f / CONV_DIM);
    s2 = warp_sum(s2) * (1.0f / CONV_DIM);
    const float k = rstd * fgm;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        float r[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) r[i] = k * (g[8 * h + i] - s1 - x[8 * h + i] * s2) * a[8 * h + i];
        *reinterpret_cast<uint4*>(g_u6 + row * CONV_DIM + (lane + 32 * h) * 8) =
            make_uint4(pack_op(r[0], r[1]), pack_op(r[2], r[3]), pack_op(r[4], r[5]), pack_op(r[6], r[7]));
    }
}

// ---------------------------------------------------------------------------------------------
// conv0 + GroupNorm backward.  G0[t, c] = (dL/du0)[t, c] * gamma_c * rstd_c is produced by the level-1
// dgrad GEMM (aux0 carries gelu' * gamma * rstd).  With uhat = (conv0 - mean) * rstd:
//   dL/dconv0[t, c] = G0 - mean_t(G0) - uhat * mean_t(G0 * uhat)
// Pass 1: per (utt, channel) sums of G0 and G0 * uhat.
__global__ void __launch_bounds__(256) conv0_bwd_stats_kernel(const op_t* __restrict__ G0, const float* __restrict__ wav,
                                                              const UttMeta* __restrict__ meta, int B_est,
                                                              const float* __restrict__ w0, const float* __restrict__ stat,
                                                              double* __restrict__ sums) {
    const int row_base = blockIdx.x * 64;
    const int b = find_utt_by_frame(meta, B_est, blockIdx.x);
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
    const uint32_t* gp = reinterpret_cast<const uint32_t*>(G0 + (long long)row_base * CONV_DIM + c);
    for (int t = 0; t < valid; ++t) {
        const float2 g = unpack_op(gp[(long long)t * (CONV_DIM / 2)]);
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

// With the conv encoder's forward saved for its parameter gradients (aux0 = gelu' alone), the level-1 dgrad wrote
// dL/du0; G0 = dL/du0 * gamma_c * rstd_c per (utterance, channel), in place.  One block per 64 level-0 rows.
__global__ void __launch_bounds__(256) conv0_gain_fold_kernel(op_t* __restrict__ G0, const UttMeta* __restrict__ meta, int B,
                                                              const float* __restrict__ gn_g, const float* __restrict__ stat) {
    const int b = find_utt_by_frame(meta, B, blockIdx.x);
    const UttMeta m = meta[b];
    const int t_base = blockIdx.x * 64 - m.row0;
    const int valid = min(64, m.T0 - t_base);
    const int c = 2 * threadIdx.x;
    const float ga = __ldg(gn_g + c) * stat[((long long)b * CONV_DIM + c) * 2 + 1];
    const float gb = __ldg(gn_g + c + 1) * stat[((long long)b * CONV_DIM + c + 1) * 2 + 1];
    uint32_t* gp = reinterpret_cast<uint32_t*>(G0 + (long long)blockIdx.x * 64 * CONV_DIM + c);
    for (int t = 0; t < valid; ++t) {
        const float2 g = unpack_op(gp[(long long)t * (CONV_DIM / 2)]);
        gp[(long long)t * (CONV_DIM / 2)] = pack_op(g.x * ga, g.y * gb);
    }
}

// Per-utterance constants of the dgrad:  val(t, j) = V[t, j] - c1[j] + c2[j] - sum_j' x[5t + j'] Q[j'][j]
//   c1[j] = sum_c m1_c w[c,j];  c2[j] = sum_c mean_c rstd_c m2_c w[c,j];  Q[j'][j] = sum_c w[c,j'] rstd_c m2_c w[c,j]
// consts[b] = { cc[10] = c2 - c1, Q[100] }
__global__ void __launch_bounds__(128) conv0_bwd_consts_kernel(const double* __restrict__ sums, const UttMeta* __restrict__ meta,
                                                               const float* __restrict__ w0, const float* __restrict__ stat,
                                                               float* __restrict__ consts) {
    const int b = blockIdx.x, tid = threadIdx.x;
    if (tid >= 110) return;
    const double invT = 1.0 / (double)meta[b].T0;
    double a = 0.0;
    if (tid < 10) {
        const int j = tid;
        for (int c = 0; c < CONV_DIM; ++c) {
            const double m1 = sums[((long long)b * CONV_DIM + c) * 2] * invT, m2 = sums[((long long)b * CONV_DIM + c) * 2 + 1] * invT;
            const double mean = stat[((long long)b * CONV_DIM + c) * 2], rstd = stat[((long long)b * CONV_DIM + c) * 2 + 1];
            a += (mean * rstd * m2 - m1) * (double)w0[c * 10 + j];
        }
    } else {
        const int jp = (tid - 10) / 10, j = (tid - 10) % 10;
        for (int c = 0; c < CONV_DIM; ++c) {
            const double m2 = sums[((long long)b * CONV_DIM + c) * 2 + 1] * invT;
            const double rstd = stat[((long long)b * CONV_DIM + c) * 2 + 1];
            a += (double)w0[c * 10 + jp] * rstd * m2 * (double)w0[c * 10 + j];
        }
    }
    consts[(long long)b * 112 + tid] = (float)a;
}

// Overlap-add of the 10 taps (stride 5) into the waveform gradient, times out_scale (= 1 / S), or times 1 / *scale_dev
// when the scale was chosen on the device (scale_dev non-null).
__global__ void __launch_bounds__(256) conv0_bwd_finish_kernel(const float* __restrict__ V, const float* __restrict__ wav,
                                                               const UttMeta* __restrict__ meta, const float* __restrict__ consts,
                                                               long long n_per_utt, float out_scale,
                                                               const float* __restrict__ scale_dev, float* __restrict__ d_wav) {
    const int b = blockIdx.y;
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_per_utt) return;
    const UttMeta m = meta[b];
    __shared__ float cs[112];
    if (threadIdx.x < 110) cs[threadIdx.x] = consts[(long long)b * 112 + threadIdx.x];
    __syncthreads();
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

__global__ void loss_finalize_kernel(const double* __restrict__ acc, double inv_layer, double inv_head, float* __restrict__ loss) {
    double s = 0.0;
    for (int i = 0; i < LAYERS; ++i) s += acc[i] * inv_layer;
    s += acc[LAYERS] * inv_head;
    *loss = (float)s;
}

// ---------------------------------------------------------------------------------------------
struct LossBufs {
    double* acc;        // [13] L1 sums
    float* pooled;      // [2B][768] pre-ReLU mean-pooled features
    float* emb;         // [2B][256] (not used by the loss value itself; keeps pool_head's contract)
    // backward (estimate half)
    float* g_pool;      // [B][768]
    float* g_a;         // frames_e x 768 fp32 (gradient wrt a layer output / running)
    float* g_b;         // frames_e x 768 fp32 (LN backward output, residual branch)
    op_t* g_bh;         // 16-bit copy
    float* g_c;         // frames_e x 768 fp32
    op_t* g_h;          // frames_e x 3072
    op_t* g_attn;       // frames_e x 768
    op_t* g_qkv;        // frames_e x 2304
    float* D;           // frames_e x 12
    op_t* pos_g;        // grouped padded layout (reuses geometry of the forward one, estimate half)
    op_t* pos_dy;       // [pos_rows_e][768]
    op_t* g_x0h;        // frames_e x 768
    float* g_ln0;       // frames_e x 512
    op_t* gu_a;         // conv-level gradients, levels 6/4/2/0: 8 zero rows + (rows0_e + 8) x 512
    op_t* gu_b;         // levels 5/3/1
    double* c0_sums;    // [B][512][2]
    float* c0_consts;   // [B][112]
    float* c0_V;        // rows0_e x 16
    size_t bytes;
};

static size_t carve_loss(const Plan& p, int B_est, long long frames_e, long long rows0_e, long long pos_rows_e,
                         bool with_grad, void* base, LossBufs* out) {
    size_t o = 0;
    auto take = [&](size_t bytes) {
        size_t at = o;
        o = (o + bytes + 1023) / 1024 * 1024;
        return base ? (void*)((char*)base + at) : nullptr;
    };
    LossBufs L;
    memset(&L, 0, sizeof(L));
    L.acc = (double*)take(sizeof(double) * 16);
    L.pooled = (float*)take(4ull * EMBED * p.B);
    L.emb = (float*)take(4ull * EMB * p.B);
    L.g_pool = (float*)take(4ull * EMBED * B_est);
    if (with_grad) {
        L.g_a = (float*)take(4ull * EMBED * frames_e);
        L.g_b = (float*)take(4ull * EMBED * frames_e);
        L.g_bh = (op_t*)take(2ull * EMBED * frames_e);
        L.g_c = (float*)take(4ull * EMBED * frames_e);
        L.g_h = (op_t*)take(2ull * FFN * frames_e);
        L.g_attn = (op_t*)take(2ull * EMBED * frames_e);
        L.g_qkv = (op_t*)take(2ull * 3 * EMBED * frames_e);
        L.D = (float*)take(4ull * HEADS * frames_e);
        L.pos_g = (op_t*)take(2ull * POS_G * POS_GC * (pos_rows_e + POS_K));
        L.pos_dy = (op_t*)take(2ull * EMBED * pos_rows_e);
        L.g_x0h = (op_t*)take(2ull * EMBED * frames_e);
        L.g_ln0 = (float*)take(4ull * CONV_DIM * frames_e);
        L.gu_a = (op_t*)take(2ull * CONV_DIM * (rows0_e + 16));
        L.gu_b = (op_t*)take(2ull * CONV_DIM * (rows0_e / 2 + 16));
        L.c0_sums = (double*)take(8ull * 2 * CONV_DIM * B_est);
        L.c0_consts = (float*)take(4ull * 112 * B_est);
        L.c0_V = (float*)take(4ull * 16 * rows0_e);
    }
    L.bytes = o;
    if (out) *out = L;
    return o;
}

static int loss_plan(int B, int64_t N, Plan* p) {
    NB_CHECK(B > 0 && N >= NOMAD_B200_MIN_SAMPLES, "loss: need B > 0 and N >= %d samples", NOMAD_B200_MIN_SAMPLES);
    std::vector<int64_t> off(2 * (size_t)B + 1);
    for (int b = 0; b <= 2 * B; ++b) off[b] = (int64_t)b * N;
    return make_plan(off.data(), 2 * B, p);
}

}  // namespace nb

using namespace nb;

extern "C" {

// core workspace of one loss step (forward in save mode + backward buffers), without the CUDA-graph staging area
static size_t loss_core_bytes(int B, int64_t N, int with_grad) {
    Plan p;
    if (loss_plan(B, N, &p)) return 0;
    const size_t fwd = carve_workspace(p, nullptr, nullptr, true);
    const long long frames_e = p.frames / 2, rows0_e = p.rows0 / 2;
    const long long pos_rows_e = frames_e + (long long)POS_GAP * B + POS_K / 2;
    return fwd + carve_loss(p, B, frames_e, rows0_e, pos_rows_e, with_grad != 0, nullptr, nullptr) + 2048;
}
static size_t loss_stage_bytes(int B, int64_t N) { return ((size_t)3 * B * N * 4 + 4096 + 1023) / 1024 * 1024; }

size_t nomad_b200_loss_workspace_bytes(int B, int64_t N, int with_grad) {
    const size_t core = loss_core_bytes(B, N, with_grad);
    if (core == 0) return 0;
    // + estimate / clean / gradient / loss staging: the step is replayed as a CUDA graph over fixed addresses
    return (core + 1023) / 1024 * 1024 + loss_stage_bytes(B, N);
}

// fp32-class step: [save-mode forward of the 2B utterances | L1 sums, pooled features, head gradient | backward scratch]
static size_t loss_precise_bytes(const Plan& p, int B, bool with_grad, size_t* fwd, size_t* mid) {
    *fwd = carve_precise(p, nullptr, nullptr, true);
    *mid = carve_loss(p, B, 0, 0, 0, false, nullptr, nullptr);
    return *fwd + *mid + (with_grad ? precise_bwd_bytes(p, B) : 0);
}

size_t nomad_b200_loss_workspace_bytes_mode(int B, int64_t N, int with_grad, int precision_mode) {
    if (precision_mode != NOMAD_B200_PRECISION_FP32) return nomad_b200_loss_workspace_bytes(B, N, with_grad);
    Plan p;
    if (loss_plan(B, N, &p)) return 0;
    size_t fwd, mid;
    return loss_precise_bytes(p, B, with_grad != 0, &fwd, &mid);
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// Backward of the encoder for the first B utterances of the batch (frames [0, Fe)): gradient wrt every layer input down
// to the waveform (dgrad chain).  `seed_layer`: L1 seed of every layer output against the second half of the batch (the
// loss path; 0 = none); L.g_pool: per-utterance gradient of the mean-pooled top layer.  `tc` (triplet fine-tuning,
// triplet section below): also produce the parameter gradients of everything after the conv feature encoder, and stop
// there when the encoder is frozen; when it is trained, go on through conv layers 6..1 (weight gradients from each
// level's pre-GELU gradient) and stop at conv0 + GroupNorm, whose parameter gradients replace the waveform gradient.  `ug` (autograd path, nomad_b200_layers_bwd): caller-given upstream gradients of the layer outputs and the
// pooled head instead of the L1 seeds, under a scale S that lives on the device.  Both (nomad_b200_layers_bwd_params):
// the parameter gradients from the caller's gradients, and the waveform gradient too when d_est_dev is non-null.
struct TrainCtx;
struct UserGrads {
    const float* g_layers[LAYERS];  // gradient wrt layer l's output, B x T x 768 (caller layout), or null
    int T;                          // frames per utterance of that layout
    const float* g_pool;            // [B][768] unscaled pooled-feature gradient of the head, or null
    const float* scale;             // device: S
    int top;                        // highest layer that receives a gradient; the layers above it are skipped
    bool scaled_out;                // the waveform gradient keeps S (parameter path: every output carries S)
};
static int train_hook_layer(Handle* h, const Workspace& ws, const LossBufs& L, TrainCtx* tc, int l, int stage, int B,
                            long long Fe, const float* g_running, cudaStream_t st);
static int train_hook_front(Handle* h, const Workspace& ws, const LossBufs& L, TrainCtx* tc, int stage, int B, long long Fe,
                            long long pos_rows_e, cudaStream_t st);
static bool train_conv(const TrainCtx* tc);
static int train_hook_conv(TrainCtx* tc, int l, const op_t* gu, const op_t* y_in, long long y_rows, long long M, cudaStream_t st);
static int train_hook_conv0(TrainCtx* tc, const Workspace& ws, const op_t* D0, const float* wav, int B, long long R0,
                            const Weights& w, cudaStream_t st);

static int backward_chain(Handle* h, const Workspace& ws, const LossBufs& L, int B, long long Fe, long long R0e,
                          long long pos_rows_e, int T, float seed_layer, float feature_grad_mult, float S,
                          const float* est_dev, int64_t N, float* d_est_dev, cudaStream_t st, TrainCtx* tc,
                          const UserGrads* ug = nullptr) {
    const Weights& w = h->w;
    const int impl = h->gemm_impl;
    const unsigned row_blocks = (unsigned)((Fe + 7) / 8);
    auto epi_grad = [&](int flags, const float* resid, float* out_f, op_t* out_h, const op_t* aux, long long ld) {
        GemmEpilogue e = epi_linear(flags, nullptr, resid, out_f, out_h, ld);
        e.aux = aux;
        return e;
    };
    NB_CUDA(cudaMemsetAsync(L.g_qkv, 0, 2ull * 3 * EMBED * Fe, st));
    const float* g_running = nullptr;  // gradient wrt the current layer's output from the layers above
    for (int l = ug != nullptr ? ug->top : LAYERS - 1; l >= 0; --l) {
        const LayerWeights& W = w.layer[l];
        const LayerBufs& Lb = ws.layer[l];
        // final_layer_norm backward (+ L1 seed of this layer's output, + pooled-head gradient on the top layer)
        if (ug != nullptr) {
            ln768_bwd_user_kernel<<<row_blocks, 256, 0, st>>>(g_running, Lb.pre2, ws.meta, B, Fe, W.ln2_g, ug->g_layers[l],
                                                              ug->T, l == LAYERS - 1 ? ug->g_pool : nullptr, ug->scale,
                                                              L.g_b, L.g_bh);
        } else {
            ln768_bwd_kernel<<<row_blocks, 256, 0, st>>>(g_running, Lb.pre2, ws.meta, B, Fe, W.ln2_g, seed_layer,
                                                         l == LAYERS - 1 ? L.g_pool : nullptr, L.g_b, L.g_bh);
        }
        NB_LAUNCHED();
        if (tc) NB_TRY(train_hook_layer(h, ws, L, tc, l, 0, B, Fe, g_running, st));  // LN2 params, fc2 weight + bias
        {   // fc2 dgrad, times gelu'(fc1 pre-activation)
            GemmOperand A{L.g_bh, Fe, EMBED, 0, 0};
            GemmOperand Bw{W.wt_fc2, FFN, EMBED, 0, 0};
            GemmEpilogue e = epi_grad(EPI_MUL_AUX | EPI_OUT_H16, nullptr, nullptr, L.g_h, Lb.ffn_aux, FFN);
            NB_TRY(gemm_h16(st, A, Bw, (int)Fe, FFN, EMBED, 1, e, impl));
        }
        {   // fc1 dgrad + residual branch
            GemmOperand A{L.g_h, Fe, FFN, 0, 0};
            GemmOperand Bw{W.wt_fc1, EMBED, FFN, 0, 0};
            GemmEpilogue e = epi_grad(EPI_RESID | EPI_OUT_F32, L.g_b, L.g_c, nullptr, nullptr, EMBED);
            NB_TRY(gemm_h16(st, A, Bw, (int)Fe, EMBED, FFN, 1, e, impl));
        }
        if (tc) NB_TRY(train_hook_layer(h, ws, L, tc, l, 1, B, Fe, g_running, st));  // fc1 weight + bias (L.g_h is ready)
        // self_attn_layer_norm backward
        ln768_bwd_kernel<<<row_blocks, 256, 0, st>>>(L.g_c, Lb.pre1, ws.meta, B, Fe, W.ln1_g, 0.f, nullptr, L.g_b, L.g_bh);
        NB_LAUNCHED();
        if (tc) NB_TRY(train_hook_layer(h, ws, L, tc, l, 2, B, Fe, g_running, st));  // LN1 params, out_proj weight + bias
        {   // out_proj dgrad
            GemmOperand A{L.g_bh, Fe, EMBED, 0, 0};
            GemmOperand Bw{W.wt_o, EMBED, EMBED, 0, 0};
            GemmEpilogue e = epi_grad(EPI_OUT_H16, nullptr, nullptr, L.g_attn, nullptr, EMBED);
            NB_TRY(gemm_h16(st, A, Bw, (int)Fe, EMBED, EMBED, 1, e, impl));
        }
        NB_TRY(launch_attention_bwd(st, Lb.qkv, Lb.attn, L.g_attn, Lb.lse, L.D, ws.meta, B, T, Fe, L.g_qkv, tc != nullptr));
        if (tc) NB_TRY(train_hook_layer(h, ws, L, tc, l, 3, B, Fe, g_running, st));  // fused q/k/v weight + bias
        {   // fused q/k/v dgrad + residual branch -> gradient wrt this layer's input
            GemmOperand A{L.g_qkv, Fe, 3 * EMBED, 0, 0};
            GemmOperand Bw{W.wt_qkv, EMBED, 3 * EMBED, 0, 0};
            GemmEpilogue e = epi_grad(EPI_RESID | EPI_OUT_F32, L.g_b, L.g_a, nullptr, nullptr, EMBED);
            NB_TRY(gemm_h16(st, A, Bw, (int)Fe, EMBED, 3 * EMBED, 1, e, impl));
        }
        g_running = L.g_a;
    }
    // encoder LayerNorm + positional conv backward
    {
        const long long rows_alloc = pos_rows_e + POS_K;
        NB_CUDA(cudaMemsetAsync(L.pos_g, 0, 2ull * POS_G * POS_GC * rows_alloc, st));
        if (tc) NB_TRY(train_hook_front(h, ws, L, tc, 0, B, Fe, pos_rows_e, st));  // encoder LayerNorm params (reads L.g_a)
        pos_bwd_prep_kernel<<<row_blocks, 256, 0, st>>>(L.g_a, ws.x0, ws.pos_y, ws.pos_aux, ws.meta, B, Fe, w.lne_g,
                                                        rows_alloc, L.g_b, L.pos_g);
        NB_LAUNCHED();
        if (tc) NB_TRY(train_hook_front(h, ws, L, tc, 1, B, Fe, pos_rows_e, st));  // positional conv weight + bias
        if (impl == 0) {
            NB_TRY(launch_posconv(st, L.pos_g, rows_alloc, pos_rows_e, w.pos_wt, nullptr, 0, L.pos_dy, nullptr));
        } else {
            GemmOperand A{L.pos_g, pos_rows_e, POS_GC, rows_alloc * POS_GC, 0};
            GemmOperand Bw{w.pos_wt, POS_GC, (long long)POS_K * POS_GC, (long long)POS_GC * POS_K * POS_GC, 0};
            GemmEpilogue e = epi_grad(EPI_OUT_H16, nullptr, nullptr, L.pos_dy, nullptr, EMBED);
            e.out_bstride = POS_GC;
            NB_TRY(gemm_h16(st, A, Bw, (int)pos_rows_e, POS_GC, POS_K * POS_GC, POS_G, e, impl));
        }
        pos_bwd_finish_kernel<<<row_blocks, 256, 0, st>>>(L.g_b, L.pos_dy, ws.meta, B, Fe, L.g_x0h);
        NB_LAUNCHED();
        if (tc) NB_TRY(train_hook_front(h, ws, L, tc, 2, B, Fe, pos_rows_e, st));  // projection weight + bias
    }
    {   // feature projection dgrad
        GemmOperand A{L.g_x0h, Fe, EMBED, 0, 0};
        GemmOperand Bw{w.proj_wt, CONV_DIM, EMBED, 0, 0};
        GemmEpilogue e = epi_grad(EPI_OUT_F32, nullptr, L.g_ln0, nullptr, nullptr, CONV_DIM);
        NB_TRY(gemm_h16(st, A, Bw, (int)Fe, CONV_DIM, EMBED, 1, e, impl));
    }
    if (tc) {
        NB_TRY(train_hook_front(h, ws, L, tc, 3, B, Fe, pos_rows_e, st));  // LayerNorm(512) params
        if (!train_conv(tc) && d_est_dev == nullptr) return 0;              // conv encoder frozen, no waveform gradient
    }
    // conv stack backward.  Gradient buffers start 8 rows into their allocation so that "row -1" reads zeros.
    NB_CUDA(cudaMemsetAsync(L.gu_a, 0, 2ull * CONV_DIM * 8, st));
    NB_CUDA(cudaMemsetAsync(L.gu_b, 0, 2ull * CONV_DIM * 8, st));
    op_t* gu[7];
    for (int l = 0; l < 7; ++l) gu[l] = ((l & 1) ? L.gu_b : L.gu_a) + 8 * CONV_DIM;
    ln512_bwd_kernel<<<row_blocks, 256, 0, st>>>(L.g_ln0, ws.y[6], ws.aux[6], Fe, w.ln0_g, feature_grad_mult, gu[6]);
    NB_LAUNCHED();
    for (int l = 6; l >= 1; --l) {
        const long long M = R0e >> l;  // rows at level l (estimate half)
        if (tc && train_conv(tc)) NB_TRY(train_hook_conv(tc, l, gu[l], ws.y[l - 1], (R0e >> (l - 1)) + 8, M, st));  // before gu[l] is reused
        if (CONV_KERNEL[l] == 2) {
            // rows 2m and 2m+1 of level l-1 in one GEMM: N = 1024 = (tap, cin)
            GemmOperand A{gu[l], M, CONV_DIM, 0, 0};
            GemmOperand Bw{w.conv_wt[l], 2 * CONV_DIM, CONV_DIM, 0, 0};
            GemmEpilogue e = epi_grad(EPI_MUL_AUX | EPI_OUT_H16, nullptr, nullptr, gu[l - 1], ws.aux[l - 1], 2 * CONV_DIM);
            NB_TRY(gemm_h16(st, A, Bw, (int)M, 2 * CONV_DIM, CONV_DIM, 1, e, impl));
        } else {
            {   // even rows 2m: taps 2 (from row m-1) and 0 (row m): overlapping rows starting one row early
                GemmOperand A{gu[l] - CONV_DIM, M, CONV_DIM, 0, 0};
                GemmOperand Bw{w.conv_wte[l], CONV_DIM, 2 * CONV_DIM, 0, 0};
                GemmEpilogue e = epi_grad(EPI_MUL_AUX | EPI_OUT_H16, nullptr, nullptr, gu[l - 1], ws.aux[l - 1], 2 * CONV_DIM);
                NB_TRY(gemm_h16(st, A, Bw, (int)M, CONV_DIM, 2 * CONV_DIM, 1, e, impl));
            }
            {   // odd rows 2m+1: tap 1
                GemmOperand A{gu[l], M, CONV_DIM, 0, 0};
                GemmOperand Bw{w.conv_wt[l] + (size_t)CONV_DIM * CONV_DIM, CONV_DIM, CONV_DIM, 0, 0};
                GemmEpilogue e = epi_grad(EPI_MUL_AUX | EPI_OUT_H16, nullptr, nullptr, gu[l - 1] + CONV_DIM,
                                          ws.aux[l - 1] + CONV_DIM, 2 * CONV_DIM);
                NB_TRY(gemm_h16(st, A, Bw, (int)M, CONV_DIM, CONV_DIM, 1, e, impl));
            }
        }
    }
    if (tc && train_conv(tc)) {
        NB_TRY(train_hook_conv0(tc, ws, gu[0], est_dev, B, R0e, h->w, st));  // reads gu[0] = dL/du0 (aux0_raw)
        if (d_est_dev == nullptr) return 0;
    }
    if (ws.aux0_raw) {  // gu[0] = dL/du0 without the GroupNorm gamma * rstd that the waveform backward expects
        conv0_gain_fold_kernel<<<(unsigned)(R0e / 64), 256, 0, st>>>(gu[0], ws.meta, B, w.gn_g, ws.gn_stat);
        NB_LAUNCHED();
    }
    // conv0 + GroupNorm backward: gu[0] = G0
    NB_CUDA(cudaMemsetAsync(L.c0_sums, 0, 8ull * 2 * CONV_DIM * B, st));
    conv0_bwd_stats_kernel<<<(unsigned)(R0e / 64), 256, 0, st>>>(gu[0], est_dev, ws.meta, B, w.conv0_w, ws.gn_stat, L.c0_sums);
    NB_LAUNCHED();
    conv0_bwd_consts_kernel<<<B, 128, 0, st>>>(L.c0_sums, ws.meta, w.conv0_w, ws.gn_stat, L.c0_consts);
    NB_LAUNCHED();
    {
        GemmOperand A{gu[0], R0e, CONV_DIM, 0, 0};
        GemmOperand Bw{w.conv0_wh, 16, CONV_DIM, 0, 0};
        GemmEpilogue e = epi_grad(EPI_OUT_F32, nullptr, L.c0_V, nullptr, nullptr, 16);
        NB_TRY(gemm_h16(st, A, Bw, (int)R0e, 16, CONV_DIM, 1, e, impl));
    }
    dim3 fgrid((unsigned)((N + 255) / 256), B);
    conv0_bwd_finish_kernel<<<fgrid, 256, 0, st>>>(L.c0_V, est_dev, ws.meta, L.c0_consts, N, 1.0f / S,
                                                   ug != nullptr && !ug->scaled_out ? ug->scale : nullptr, d_est_dev);
    NB_LAUNCHED();
    return 0;
}

// =============================================================================================================
// Triplet fine-tuning step (reference src/training/train_triplet.py:112-133, conv feature encoder frozen as in
// src/config/train_triplet.yaml `freeze_convnet: True`): embeddings of anchors / positives / negatives ->
// TripletMarginLoss(margin, p = 2, eps = 1e-6) -> gradients of EVERY trainable parameter (LayerNorm(512), feature
// projection, positional conv, encoder LayerNorm, the 12 transformer layers, the embedding head).  The activation
// gradients are the dgrad chain above; each weight gradient dW = dY^T X is a tensor-core GEMM over the token dimension
// (both operands transposed into K-major first: two bandwidth-trivial passes), bias / LayerNorm gradients are column
// reductions.  All gradients carry the power-of-two scale S of the chain; the caller divides it out.  With
// `freeze_convnet: False` (nomad_b200_triplet_conv_fwd_bwd) the conv feature encoder's gradients follow as well (split-K
// GEMMs for conv1-6, per-channel sums for conv0 + GroupNorm; see the conv section below).

// flat gradient buffer (fp32): per layer [qkv_w 2304x768 | qkv_b | o_w | o_b | fc1_w | fc1_b | fc2_w | fc2_b | ln1_g | ln1_b |
// ln2_g | ln2_b], then [enc_ln_g | enc_ln_b | pos_w 16x48x6144 (folded weight, layout [g][n][tap*48+c]) | pos_b |
// proj_w 768x512 | proj_b | ln0_g | ln0_b | head_w 256x768 | head_b]
struct TrainLayout {
    static constexpr long long QKV_W = 0, QKV_B = QKV_W + 2304LL * 768, O_W = QKV_B + 2304, O_B = O_W + 768LL * 768,
                               FC1_W = O_B + 768, FC1_B = FC1_W + 3072LL * 768, FC2_W = FC1_B + 3072,
                               FC2_B = FC2_W + 768LL * 3072, LN1_G = FC2_B + 768, LN1_B = LN1_G + 768, LN2_G = LN1_B + 768,
                               LN2_B = LN2_G + 768, LAYER = LN2_B + 768;
    static constexpr long long ENC_G = LAYER * LAYERS, ENC_B = ENC_G + 768, POS_W = ENC_B + 768,
                               POS_B = POS_W + (long long)POS_G * POS_GC * POS_K * POS_GC, PROJ_W = POS_B + 768,
                               PROJ_B = PROJ_W + 768LL * 512, LN0_G = PROJ_B + 768, LN0_B = LN0_G + 512, HEAD_W = LN0_B + 512,
                               HEAD_B = HEAD_W + 256LL * 768, TOTAL = HEAD_B + 256;
};

struct TrainCtx {
    float* grads;     // TrainLayout::TOTAL floats, zeroed
    op_t* tA;         // 3072 x Fp: transposed dY
    op_t* tB;         // 3072 x Fp: transposed X
    op_t* xh_tmp;     // F x 768: recomputed LayerNorm output (GEMM input of the layer being differentiated)
    float* x_tmp;     // F x 768 fp32 scratch for the recomputation kernels
    float* gy;        // [3B][256] gradient wrt the un-normalised head output
    long long Fp;     // tokens rounded up to 8 (K of the weight-gradient GEMMs)
    // conv feature encoder training (nomad_b200_triplet_conv_fwd_bwd); conv_grads == nullptr: encoder frozen
    float* conv_grads;  // ConvLayout::TOTAL floats
    op_t* ctA;          // [splits][512][Ks]: a level's pre-GELU gradient, transposed (K = rows, split into K slices)
    op_t* ctB;          // [splits][k * 512][Ks]: the overlapping-row view of the level's input, transposed the same way
    float* part;        // [splits][512][k * 512] fp32 partial weight gradients of the K slices
    double* c0_sums;    // [3B][512][12] per (utterance, channel): sum D, sum D uhat, sum D x[5t + j]
    int max_chunks;     // wave-stats chunks per utterance (Plan::max_chunks)
    const UserGrads* ug;  // autograd parameter path (nomad_b200_layers_bwd_params): the caller's output gradients, or null
};

// flat conv-encoder gradient buffer (fp32), each tensor in the checkpoint's (out, in, tap) order:
// [conv0 512x1x10 | GroupNorm weight 512 | GroupNorm bias 512 | conv1..6 512x512xk]
struct ConvLayout {
    static constexpr long long C0_W = 0, GN_G = C0_W + 512 * 10, GN_B = GN_G + 512, L1 = GN_B + 512,
                               TOTAL = L1 + 4 * 512LL * 512 * 3 + 2 * 512LL * 512 * 2;
    static long long level(int l) { return L1 + 512LL * 512 * 3 * std::min(l - 1, 4) + 512LL * 512 * 2 * std::max(l - 5, 0); }
};
// K slices of a conv weight-gradient GEMM: M (512) x N (512 k) is only 16-24 output tiles, while K = rows of the level
// reaches ~4e5 at 8 triplets x 10 s; the slices run as the GEMM's batch and one pass sums their fp32 partials
static constexpr int CONV_SPLIT_MAX = 24;
static int conv_splits(long long M, long long* Ks) {
    const int s = (int)std::min<long long>(CONV_SPLIT_MAX, std::max<long long>(1, (M + 4095) / 4096));
    *Ks = ((M + s - 1) / s + 63) / 64 * 64;
    return s;
}

// in [rows][cols] (16-bit) -> out[z][cols][rows_p] with out[z][c][r] = in[r + z][c] (zero past the end): copy z is the
// transpose shifted by z rows (copies = 1: the plain transpose, columns rows..rows_p-1 zero)
__global__ void __launch_bounds__(256) transpose_h16_kernel(const op_t* __restrict__ in, long long rows, int cols,
                                                            long long rows_p, op_t* __restrict__ out) {
    __shared__ op_t tile[64][66];
    const long long r0 = (long long)blockIdx.x * 64;
    const int c0 = blockIdx.y * 64, z = blockIdx.z;
    for (int i = threadIdx.x; i < 64 * 64; i += 256) {
        const int r = i >> 6, c = i & 63;
        tile[r][c] = (r0 + r + z < rows && c0 + c < cols) ? in[(r0 + r + z) * cols + c0 + c] : f2op(0.f);
    }
    __syncthreads();
    op_t* o = out + (long long)z * cols * rows_p;
    for (int i = threadIdx.x; i < 64 * 64; i += 256) {
        const int c = i >> 6, r = i & 63;
        if (c0 + c < cols && r0 + r < rows_p) o[(long long)(c0 + c) * rows_p + r0 + r] = tile[r][c];
    }
}
static int launch_transpose(cudaStream_t st, const op_t* in, long long rows, int cols, long long rows_p, op_t* out, int copies = 1) {
    dim3 grid((unsigned)((rows_p + 63) / 64), (unsigned)((cols + 63) / 64), copies);
    transpose_h16_kernel<<<grid, 256, 0, st>>>(in, rows, cols, rows_p, out);
    NB_LAUNCHED();
    return 0;
}
// dW[No][Ki] (fp32) = sum_t dY[t][no] X[t][ki]
static int wgrad(cudaStream_t st, TrainCtx* tc, const op_t* dY, int No, const op_t* X, int Ki, long long F, float* dW) {
    NB_TRY(launch_transpose(st, dY, F, No, tc->Fp, tc->tA));
    NB_TRY(launch_transpose(st, X, F, Ki, tc->Fp, tc->tB));
    GemmOperand A{tc->tA, No, tc->Fp, 0, 0};
    GemmOperand Bw{tc->tB, Ki, tc->Fp, 0, 0};
    GemmEpilogue e = epi_linear(EPI_OUT_F32, nullptr, nullptr, dW, nullptr, Ki);
    return gemm_h16(st, A, Bw, No, Ki, (int)tc->Fp, 1, e, 0);
}
// out[c] += sum over rows of in[r][c]
template <typename T>
__global__ void __launch_bounds__(256) colsum_kernel(const T* __restrict__ in, long long rows, int cols, float* __restrict__ out) {
    const int c = blockIdx.x * 64 + (threadIdx.x & 63);
    const int g = threadIdx.x >> 6;
    float s = 0.f;
    if (c < cols)
        for (long long r = (long long)blockIdx.y * 4 + g; r < rows; r += 4LL * gridDim.y) s += (float)in[r * cols + c];
    __shared__ float red[4][64];
    red[g][threadIdx.x & 63] = s;
    __syncthreads();
    if (g == 0 && c < cols) atomicAdd(out + c, red[0][threadIdx.x] + red[1][threadIdx.x] + red[2][threadIdx.x] + red[3][threadIdx.x]);
}
template <typename T>
static int launch_colsum(cudaStream_t st, const T* in, long long rows, int cols, float* out) {
    dim3 grid((unsigned)((cols + 63) / 64), 32);
    colsum_kernel<T><<<grid, 256, 0, st>>>(in, rows, cols, out);
    NB_LAUNCHED();
    return 0;
}
// LayerNorm(768) parameter gradients: with g = gradient wrt the LayerNorm OUTPUT (g_in rows + g_pool[utt] broadcast, either
// may be null) and xhat the normalised input: d_gamma += g * xhat, d_beta += g.  `pos_y` non-null: the input row is
// x[f] + pos_y[pos row of f] (the encoder LayerNorm).  USER (autograd parameter path): the incoming gradient is
// g_in + S * g_user[b, t] + S * g_pool[utt] as ln768_bwd_user_kernel forms it (g_user in the caller's layout, row
// b * user_T + t, may be null; S read from the device).
template <bool USER>
__global__ void __launch_bounds__(256) ln768_param_grad_kernel(const float* __restrict__ g_in, const float* __restrict__ g_pool,
                                                               const float* __restrict__ pre, const op_t* __restrict__ pos_y,
                                                               const UttMeta* __restrict__ meta, int B, long long frames,
                                                               float* __restrict__ d_gamma, float* __restrict__ d_beta,
                                                               const float* __restrict__ g_user, int user_T,
                                                               const float* __restrict__ scale) {
    __shared__ float sg[EMBED], sb[EMBED];
    for (int i = threadIdx.x; i < EMBED; i += 256) { sg[i] = 0.f; sb[i] = 0.f; }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    float ag[24], ab[24];
#pragma unroll
    for (int i = 0; i < 24; ++i) { ag[i] = 0.f; ab[i] = 0.f; }
    for (long long f = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); f < frames; f += 8LL * gridDim.x) {
        const int b = find_utt_by_frame(meta, B, (int)f);
        const int t = (int)f - meta[b].frame0;
        if (t >= meta[b].T) continue;
        Row768f x, g;
        load_row768(x, pre + f * EMBED, lane);
        if (pos_y != nullptr) {
            const long long m = (long long)meta[b].pos0 + t - POS_K / 2;
#pragma unroll
            for (int h = 0; h < 3; ++h) {
                const uint4 y = __ldg(reinterpret_cast<const uint4*>(pos_y + m * EMBED + (lane + 32 * h) * 8));
                const float2 t0 = unpack_op(y.x), t1 = unpack_op(y.y), t2 = unpack_op(y.z), t3 = unpack_op(y.w);
                float* v = x.v + 8 * h;
                v[0] += t0.x; v[1] += t0.y; v[2] += t1.x; v[3] += t1.y; v[4] += t2.x; v[5] += t2.y; v[6] += t3.x; v[7] += t3.y;
            }
        }
        normalise768(x);
        if (g_in != nullptr) {
            load_row768(g, g_in + f * EMBED, lane);
        } else {
#pragma unroll
            for (int i = 0; i < 24; ++i) g.v[i] = 0.f;
        }
        if (USER) {
            const float S = __ldg(scale);
            if (g_user != nullptr) {
                Row768f gu;
                load_row768(gu, g_user + ((long long)b * user_T + t) * EMBED, lane);
#pragma unroll
                for (int i = 0; i < 24; ++i) g.v[i] = fmaf(S, gu.v[i], g.v[i]);
            }
            if (g_pool != nullptr) {
                Row768f gp;
                load_vec768(gp, g_pool + (long long)b * EMBED, lane);
#pragma unroll
                for (int i = 0; i < 24; ++i) g.v[i] = fmaf(S, gp.v[i], g.v[i]);
            }
        } else if (g_pool != nullptr) {
            Row768f gp;
            load_vec768(gp, g_pool + (long long)b * EMBED, lane);
#pragma unroll
            for (int i = 0; i < 24; ++i) g.v[i] += gp.v[i];
        }
#pragma unroll
        for (int i = 0; i < 24; ++i) { ag[i] = fmaf(g.v[i], x.v[i], ag[i]); ab[i] += g.v[i]; }
    }
#pragma unroll
    for (int h = 0; h < 3; ++h)
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            atomicAdd(&sg[(lane + 32 * h) * 8 + i], ag[8 * h + i]);
            atomicAdd(&sb[(lane + 32 * h) * 8 + i], ab[8 * h + i]);
        }
    __syncthreads();
    for (int i = threadIdx.x; i < EMBED; i += 256) { atomicAdd(d_gamma + i, sg[i]); atomicAdd(d_beta + i, sb[i]); }
}
static int launch_ln768_param_grad(cudaStream_t st, const float* g_in, const float* g_pool, const float* pre, const op_t* pos_y,
                                   const UttMeta* meta, int B, long long frames, float* dg, float* db) {
    const unsigned blocks = (unsigned)std::min<long long>((frames + 7) / 8, 296);
    ln768_param_grad_kernel<false><<<blocks, 256, 0, st>>>(g_in, g_pool, pre, pos_y, meta, B, frames, dg, db, nullptr, 0, nullptr);
    NB_LAUNCHED();
    return 0;
}
static int launch_ln768_param_grad_user(cudaStream_t st, const float* g_in, const float* g_user, int user_T, const float* g_pool,
                                        const float* scale, const float* pre, const UttMeta* meta, int B, long long frames,
                                        float* dg, float* db) {
    const unsigned blocks = (unsigned)std::min<long long>((frames + 7) / 8, 296);
    ln768_param_grad_kernel<true><<<blocks, 256, 0, st>>>(g_in, g_pool, pre, nullptr, meta, B, frames, dg, db, g_user, user_T,
                                                          scale);
    NB_LAUNCHED();
    return 0;
}
// LayerNorm(512) parameter gradients from g (fp32, wrt the LayerNorm output) and the conv features y6 (16-bit)
__global__ void __launch_bounds__(256) ln512_param_grad_kernel(const float* __restrict__ g, const op_t* __restrict__ y6,
                                                               const UttMeta* __restrict__ meta, int B, long long rows,
                                                               float* __restrict__ d_gamma, float* __restrict__ d_beta) {
    __shared__ float sg[CONV_DIM], sb[CONV_DIM];
    for (int i = threadIdx.x; i < CONV_DIM; i += 256) { sg[i] = 0.f; sb[i] = 0.f; }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    float ag[16], ab[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) { ag[i] = 0.f; ab[i] = 0.f; }
    for (long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); row < rows; row += 8LL * gridDim.x) {
        const int b = find_utt_by_frame(meta, B, (int)row);
        if ((int)row - meta[b].frame0 >= meta[b].T) continue;
        float x[16], gg[16];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int c0 = (lane + 32 * h) * 8;
            const uint4 u = __ldg(reinterpret_cast<const uint4*>(y6 + row * CONV_DIM + c0));
            float2 f;
            f = unpack_op(u.x); x[8 * h + 0] = f.x; x[8 * h + 1] = f.y;
            f = unpack_op(u.y); x[8 * h + 2] = f.x; x[8 * h + 3] = f.y;
            f = unpack_op(u.z); x[8 * h + 4] = f.x; x[8 * h + 5] = f.y;
            f = unpack_op(u.w); x[8 * h + 6] = f.x; x[8 * h + 7] = f.y;
            const float4 g0 = __ldg(reinterpret_cast<const float4*>(g + row * CONV_DIM + c0));
            const float4 g1 = __ldg(reinterpret_cast<const float4*>(g + row * CONV_DIM + c0 + 4));
            gg[8 * h + 0] = g0.x; gg[8 * h + 1] = g0.y; gg[8 * h + 2] = g0.z; gg[8 * h + 3] = g0.w;
            gg[8 * h + 4] = g1.x; gg[8 * h + 5] = g1.y; gg[8 * h + 6] = g1.z; gg[8 * h + 7] = g1.w;
        }
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < 16; ++i) s += x[i];
        const float mean = warp_sum(s) * (1.0f / CONV_DIM);
        float q = 0.f;
#pragma unroll
        for (int i = 0; i < 16; ++i) { x[i] -= mean; q = fmaf(x[i], x[i], q); }
        const float rstd = rsqrtf(warp_sum(q) * (1.0f / CONV_DIM) + 1e-5f);
#pragma unroll
        for (int i = 0; i < 16; ++i) { ag[i] = fmaf(gg[i], x[i] * rstd, ag[i]); ab[i] += gg[i]; }
    }
#pragma unroll
    for (int h = 0; h < 2; ++h)
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            atomicAdd(&sg[(lane + 32 * h) * 8 + i], ag[8 * h + i]);
            atomicAdd(&sb[(lane + 32 * h) * 8 + i], ab[8 * h + i]);
        }
    __syncthreads();
    for (int i = threadIdx.x; i < CONV_DIM; i += 256) { atomicAdd(d_gamma + i, sg[i]); atomicAdd(d_beta + i, sb[i]); }
}
// Positional-conv weight gradient: dW[g][n][tap][c] = sum_p dY[g][p][n] X[g][p - 64 + tap][c] over the zero-padded
// grouped layouts (dY = the scattered g_z * gelu' rows of pos_bwd_prep_kernel, X = the forward's scattered input).
// One block per (group, tap); thread (n, c-octet) owns 8 outputs; rows staged through shared memory 64 at a time.
__global__ void __launch_bounds__(288) pos_wgrad_kernel(const op_t* __restrict__ dy, const op_t* __restrict__ x,
                                                        long long rows_alloc, long long pos_rows, float* __restrict__ dw) {
    const int g = blockIdx.y, tap = blockIdx.x;
    const int n = threadIdx.x / 6, c0 = (threadIdx.x % 6) * 8;
    __shared__ float sdy[64][POS_GC], sx[64][POS_GC];
    float acc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = 0.f;
    const op_t* dyg = dy + (long long)g * rows_alloc * POS_GC;
    const op_t* xg = x + (long long)g * rows_alloc * POS_GC;
    for (long long p0 = POS_K / 2; p0 < pos_rows + POS_K / 2; p0 += 64) {
        __syncthreads();
        for (int i = threadIdx.x; i < 64 * POS_GC; i += 288) {
            const int r = i / POS_GC, c = i % POS_GC;
            const long long p = p0 + r, q = p - POS_K / 2 + tap;
            sdy[r][c] = p < rows_alloc ? op2f(dyg[p * POS_GC + c]) : 0.f;
            sx[r][c] = q < rows_alloc ? op2f(xg[q * POS_GC + c]) : 0.f;
        }
        __syncthreads();
#pragma unroll 4
        for (int r = 0; r < 64; ++r) {
            const float d = sdy[r][n];
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[i] = fmaf(d, sx[r][c0 + i], acc[i]);
        }
    }
    float* o = dw + ((long long)(g * POS_GC + n)) * (POS_K * POS_GC) + (long long)tap * POS_GC + c0;
#pragma unroll
    for (int i = 0; i < 8; ++i) o[i] = acc[i];
}
// column sums of the grouped layout: bias[g * 48 + n] = sum_p dY[g][p][n]
__global__ void __launch_bounds__(256) pos_bias_grad_kernel(const op_t* __restrict__ dy, long long rows_alloc, float* __restrict__ db) {
    const int g = blockIdx.x;
    const int n = threadIdx.x % POS_GC, part = threadIdx.x / POS_GC;  // 5 row partitions (240 threads active)
    __shared__ float red[5][POS_GC];
    if (part < 5) {
        float s = 0.f;
        for (long long p = part; p < rows_alloc; p += 5) s += op2f(dy[((long long)g * rows_alloc + p) * POS_GC + n]);
        red[part][n] = s;
    }
    __syncthreads();
    if (threadIdx.x < POS_GC) db[g * POS_GC + threadIdx.x] = red[0][threadIdx.x] + red[1][threadIdx.x] + red[2][threadIdx.x] + red[3][threadIdx.x] + red[4][threadIdx.x];
}

// Triplet head: e = normalize(W relu(pooled) + b) for anchor / positive / negative i; loss_i = max(||e_a - e_p + eps|| -
// ||e_a - e_n + eps|| + margin, 0) (torch.nn.TripletMarginLoss: pairwise_distance adds eps = 1e-6 to the difference);
// gy[u][o] = S/B * d loss_i / d y_u[o] with y the un-normalised head output.  One block of 256 threads per triplet.
__global__ void __launch_bounds__(256) triplet_head_kernel(const float* __restrict__ pooled, int B, const float* __restrict__ head_wt,
                                                           const float* __restrict__ head_b, float margin, float scale,
                                                           double* __restrict__ loss_acc, float* __restrict__ gy) {
    const int i = blockIdx.x, tid = threadIdx.x;
    __shared__ float pl[3][EMBED];
    __shared__ float red[4][8];
    for (int k = tid; k < EMBED; k += 256)
#pragma unroll
        for (int u = 0; u < 3; ++u) pl[u][k] = fmaxf(pooled[((long long)u * B + i) * EMBED + k], 0.f);
    __syncthreads();
    float y[3] = {head_b[tid], head_b[tid], head_b[tid]};
    for (int k = 0; k < EMBED; ++k) {
        const float w = __ldg(head_wt + k * EMB + tid);
#pragma unroll
        for (int u = 0; u < 3; ++u) y[u] = fmaf(pl[u][k], w, y[u]);
    }
    auto block_sum = [&](float v, int slot) {
        v = warp_sum(v);
        __syncthreads();
        if ((tid & 31) == 0) red[slot][tid >> 5] = v;
        __syncthreads();
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) t += red[slot][w];
        return t;
    };
    float nrm[3], e[3];
#pragma unroll
    for (int u = 0; u < 3; ++u) {
        nrm[u] = fmaxf(sqrtf(block_sum(y[u] * y[u], u)), 1e-12f);
        e[u] = y[u] / nrm[u];
    }
    const float dp = e[0] - e[1] + 1e-6f, dn = e[0] - e[2] + 1e-6f;
    const float d_ap = sqrtf(block_sum(dp * dp, 0)), d_an = sqrtf(block_sum(dn * dn, 1));
    const float li = d_ap - d_an + margin;
    if (tid == 0 && li > 0.f) atomicAdd(loss_acc, (double)li);
    float ge[3] = {0.f, 0.f, 0.f};
    if (li > 0.f) {
        const float a = dp / fmaxf(d_ap, 1e-20f), c = dn / fmaxf(d_an, 1e-20f);
        ge[0] = scale * (a - c);
        ge[1] = -scale * a;
        ge[2] = scale * c;
    }
#pragma unroll
    for (int u = 0; u < 3; ++u) {
        const float dot = block_sum(ge[u] * e[u], 2);
        gy[((long long)u * B + i) * EMB + tid] = (ge[u] - e[u] * dot) / nrm[u];  // backward of y / max(||y||, eps)
    }
}
// head parameter gradients and the pooled-feature gradient from gy; DEV_SCALE: times the scale S on the device (the
// autograd parameter path, whose gy is unscaled)
template <bool DEV_SCALE>
__global__ void __launch_bounds__(256) head_param_grad_kernel(const float* __restrict__ gy, const float* __restrict__ pooled, int n_utt,
                                                              float* __restrict__ dW, float* __restrict__ db,
                                                              const float* __restrict__ scale) {
    const int o = blockIdx.x;  // output row of the head
    const float S = DEV_SCALE ? __ldg(scale) : 1.f;
    float bsum = 0.f;
    for (int k = threadIdx.x; k < EMBED; k += 256) {
        float a = 0.f;
        for (int u = 0; u < n_utt; ++u) a = fmaf(gy[(long long)u * EMB + o], fmaxf(pooled[(long long)u * EMBED + k], 0.f), a);
        dW[(long long)o * EMBED + k] = DEV_SCALE ? a * S : a;
    }
    if (threadIdx.x == 0) {
        for (int u = 0; u < n_utt; ++u) bsum += gy[(long long)u * EMB + o];
        db[o] = DEV_SCALE ? bsum * S : bsum;
    }
}
__global__ void __launch_bounds__(256) head_pool_grad_kernel(const float* __restrict__ gy, const float* __restrict__ pooled,
                                                             const UttMeta* __restrict__ meta, const float* __restrict__ head_wt,
                                                             float* __restrict__ g_pool) {
    const int u = blockIdx.x;
    __shared__ float g[EMB];
    g[threadIdx.x] = gy[(long long)u * EMB + threadIdx.x];
    __syncthreads();
    const float invT = 1.0f / (float)meta[u].T;
    for (int k = threadIdx.x; k < EMBED; k += 256) {
        float a = 0.f;
        for (int o = 0; o < EMB; ++o) a = fmaf(g[o], __ldg(head_wt + (long long)k * EMB + o), a);
        g_pool[(long long)u * EMBED + k] = pooled[(long long)u * EMBED + k] > 0.f ? a * invT : 0.f;
    }
}
__global__ void triplet_loss_finalize_kernel(const double* __restrict__ acc, double inv_b, float* __restrict__ loss) {
    *loss = (float)(acc[0] * inv_b);
}

// ---- conv feature encoder (trained only with nomad_b200_triplet_conv_fwd_bwd) ----------------------------------------
// K-major operands of the conv weight gradient dW_l[n][tap * 512 + c] = sum_m gu[m][n] y[2m + tap][c]:
// out[s][z * 512 + c][r] = in[stride * m + z][c] with m = s * Ks + r (zero for m >= M or past in_rows), z < gridDim.z.
// stride 1, one tap: the transposed gradient; stride 2, k taps: the overlapping-row view of the level's input.
__global__ void __launch_bounds__(256) conv_wgrad_transpose_kernel(const op_t* __restrict__ in, long long in_rows, int stride,
                                                                   long long M, long long Ks, op_t* __restrict__ out) {
    __shared__ op_t tile[64][66];
    const long long m0 = (long long)blockIdx.x * 64;
    const int c0 = blockIdx.y * 64, z = blockIdx.z, taps = gridDim.z;
    for (int i = threadIdx.x; i < 64 * 64; i += 256) {
        const int r = i >> 6, c = i & 63;
        const long long m = m0 + r, src = stride * m + z;
        tile[r][c] = (m < M && src < in_rows) ? in[src * CONV_DIM + c0 + c] : f2op(0.f);
    }
    __syncthreads();
    const long long s = m0 / Ks, r0 = m0 - s * Ks;  // Ks % 64 == 0: the 64 rows stay in one slice
    op_t* o = out + (s * taps * CONV_DIM + (long long)z * CONV_DIM) * Ks + r0;
    for (int i = threadIdx.x; i < 64 * 64; i += 256) {
        const int c = i >> 6, r = i & 63;
        o[(long long)(c0 + c) * Ks + r] = tile[r][c];
    }
}
// dW[o][c][tap] (checkpoint order) = sum over slices of part[s][o][tap * 512 + c]
__global__ void __launch_bounds__(256) conv_wgrad_reduce_kernel(const float* __restrict__ part, int splits, int k,
                                                                float* __restrict__ dw) {
    const long long n = (long long)CONV_DIM * k * CONV_DIM;
    const long long i = (long long)blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    float a = 0.f;
    for (int s = 0; s < splits; ++s) a += part[s * n + i];
    const int o = (int)(i / (k * CONV_DIM)), rem = (int)(i % (k * CONV_DIM)), tap = rem / CONV_DIM, c = rem % CONV_DIM;
    dw[((long long)o * CONV_DIM + c) * k + tap] = a;
}

// conv0 + GroupNorm parameter gradients, pass 1.  D = dL/du0 (u0 = GroupNorm output; the forward saved gelu' itself for
// level 0, so the level-1 dgrad wrote D), uhat = (conv0 - mean) * rstd:  per (utt, channel) fp64 sums of D, D * uhat and
// D * x[5t + j] (j < 10).  One block = 4 x 64 level-0 rows (a 64-row group never straddles two utterances).
static constexpr int C0W_SUMS = 12;
__global__ void __launch_bounds__(256) conv0_wgrad_stats_kernel(const op_t* __restrict__ D, const float* __restrict__ wav,
                                                                const UttMeta* __restrict__ meta, int B, long long groups,
                                                                const float* __restrict__ w0, const float* __restrict__ stat,
                                                                double* __restrict__ sums) {
    __shared__ float xs[64 * 5 + 8];
    const int c = 2 * threadIdx.x;
    float wa[10], wb[10];
#pragma unroll
    for (int j = 0; j < 10; ++j) { wa[j] = __ldg(w0 + c * 10 + j); wb[j] = __ldg(w0 + (c + 1) * 10 + j); }
    float acc[2][C0W_SUMS];
    int cur = -1;
    float mean_a = 0.f, rstd_a = 0.f, mean_b = 0.f, rstd_b = 0.f;
    auto flush = [&]() {
        if (cur < 0) return;
        double* o = sums + ((long long)cur * CONV_DIM + c) * C0W_SUMS;
#pragma unroll
        for (int i = 0; i < C0W_SUMS; ++i) {
            atomicAdd(o + i, (double)acc[0][i]);
            atomicAdd(o + C0W_SUMS + i, (double)acc[1][i]);
        }
    };
    for (int q = 0; q < 4; ++q) {
        const long long grp = (long long)blockIdx.x * 4 + q;
        if (grp >= groups) break;
        const int b = find_utt_by_frame(meta, B, (int)grp);
        const UttMeta m = meta[b];
        const int t_base = (int)(grp * 64) - m.row0;
        const int valid = min(64, m.T0 - t_base);
        if (valid <= 0) continue;
        if (b != cur) {
            flush();
            cur = b;
#pragma unroll
            for (int i = 0; i < C0W_SUMS; ++i) { acc[0][i] = 0.f; acc[1][i] = 0.f; }
            mean_a = stat[((long long)b * CONV_DIM + c) * 2]; rstd_a = stat[((long long)b * CONV_DIM + c) * 2 + 1];
            mean_b = stat[((long long)b * CONV_DIM + c + 1) * 2]; rstd_b = stat[((long long)b * CONV_DIM + c + 1) * 2 + 1];
        }
        __syncthreads();
        const float* x = wav + m.wav_off;
        for (int i = threadIdx.x; i < 64 * 5 + 5; i += blockDim.x) {
            const long long s = (long long)t_base * 5 + i;
            xs[i] = (s < m.n) ? __ldg(x + s) : 0.f;
        }
        __syncthreads();
        const uint32_t* gp = reinterpret_cast<const uint32_t*>(D + grp * 64 * CONV_DIM + c);
        for (int t = 0; t < valid; ++t) {
            const float2 g = unpack_op(gp[(long long)t * (CONV_DIM / 2)]);
            float ua = 0.f, ub = 0.f;
#pragma unroll
            for (int j = 0; j < 10; ++j) {
                const float xv = xs[5 * t + j];
                ua = fmaf(wa[j], xv, ua);
                ub = fmaf(wb[j], xv, ub);
                acc[0][2 + j] = fmaf(g.x, xv, acc[0][2 + j]);
                acc[1][2 + j] = fmaf(g.y, xv, acc[1][2 + j]);
            }
            ua = (ua - mean_a) * rstd_a;
            ub = (ub - mean_b) * rstd_b;
            acc[0][0] += g.x; acc[0][1] = fmaf(g.x, ua, acc[0][1]);
            acc[1][0] += g.y; acc[1][1] = fmaf(g.y, ub, acc[1][1]);
        }
    }
    flush();
}

// pass 2 (one thread per channel, fp64): with a = gamma rstd, G0 = a D, m1 = mean_t G0, m2 = mean_t G0 uhat and the
// waveform's tap sums S_j / cross-products C_kj (the forward's wave-stats partials):
//   dW0[c][j] = sum_b  a P_j - m1 S_j - m2 rstd (sum_k w_k C_kj - mean S_j),  P_j = sum_t D x[5t + j]
//   d gamma_c = sum_b sum_t D uhat,  d beta_c = sum_b sum_t D
// (dL/dconv0 = G0 - m1 - uhat m2, times x[5t + j] summed over t; sum_t uhat x[5t + j] = rstd (sum_k w_k C_kj - mean S_j)).
__global__ void __launch_bounds__(512) conv0_param_grad_kernel(const double* __restrict__ sums, const double* __restrict__ part,
                                                               const UttMeta* __restrict__ meta, int B, int max_chunks,
                                                               const float* __restrict__ w0, const float* __restrict__ gn_g,
                                                               float* __restrict__ dw0, float* __restrict__ d_gamma,
                                                               float* __restrict__ d_beta) {
    const int c = threadIdx.x;
    __shared__ double st[NSTAT], cr[10][10];
    double w[10], dw[10], dg = 0.0, db = 0.0;
#pragma unroll
    for (int j = 0; j < 10; ++j) { w[j] = (double)w0[c * 10 + j]; dw[j] = 0.0; }
    for (int b = 0; b < B; ++b) {
        const UttMeta m = meta[b];
        __syncthreads();
        if (c < NSTAT) {
            const int chunks = (m.T0 + STAT_CHUNK - 1) / STAT_CHUNK;
            double a = 0.0;
            for (int k = 0; k < chunks; ++k) a += part[((long long)b * max_chunks + k) * NSTAT + c];
            st[c] = a;
        }
        __syncthreads();
        if (c < 100) {  // C_jk from the upper triangle (wave_stats_kernel's order)
            const int j = c / 10, k = c % 10, lo = min(j, k), hi = max(j, k);
            cr[j][k] = st[10 + lo * 10 - lo * (lo - 1) / 2 + (hi - lo)];
        }
        __syncthreads();
        // GroupNorm statistics (gn_fold_kernel's arithmetic up to the summation order): wc_j = sum_k w_k C_kj
        double wc[10], sum = 0.0, sq = 0.0;
#pragma unroll
        for (int j = 0; j < 10; ++j) {
            double a = 0.0;
            for (int k = 0; k < 10; ++k) a += w[k] * cr[k][j];
            wc[j] = a;
            sum += w[j] * st[j];
            sq += w[j] * a;
        }
        const double inv_n = 1.0 / (double)m.T0;
        const double mean = sum * inv_n;
        double var = sq * inv_n - mean * mean;
        var = var > 0.0 ? var : 0.0;
        const double rstd = 1.0 / sqrt(var + 1e-5);
        const double a = (double)gn_g[c] * rstd;
        const double* q = sums + ((long long)b * CONV_DIM + c) * C0W_SUMS;
        db += q[0];
        dg += q[1];
        const double m1 = a * q[0] * inv_n, m2 = a * q[1] * inv_n;
#pragma unroll
        for (int j = 0; j < 10; ++j) dw[j] += a * q[2 + j] - m1 * st[j] - m2 * rstd * (wc[j] - mean * st[j]);
    }
#pragma unroll
    for (int j = 0; j < 10; ++j) dw0[c * 10 + j] = (float)dw[j];
    d_gamma[c] = (float)dg;
    d_beta[c] = (float)db;
}

// ---- hooks called from backward_chain --------------------------------------------------------------------------
static bool train_conv(const TrainCtx* tc) { return tc->conv_grads != nullptr; }

// weight gradient of conv level l (1..6) from its pre-GELU gradient gu (M rows) and its input y_in (y_rows rows)
static int train_hook_conv(TrainCtx* tc, int l, const op_t* gu, const op_t* y_in, long long y_rows, long long M, cudaStream_t st) {
    const int k = CONV_KERNEL[l];
    long long Ks;
    const int splits = conv_splits(M, &Ks);
    const unsigned tiles = (unsigned)(splits * Ks / 64);
    conv_wgrad_transpose_kernel<<<dim3(tiles, CONV_DIM / 64, 1), 256, 0, st>>>(gu, M, 1, M, Ks, tc->ctA);
    NB_LAUNCHED();
    conv_wgrad_transpose_kernel<<<dim3(tiles, CONV_DIM / 64, k), 256, 0, st>>>(y_in, y_rows, 2, M, Ks, tc->ctB);
    NB_LAUNCHED();
    const int Ki = k * CONV_DIM;
    GemmOperand A{tc->ctA, CONV_DIM, Ks, CONV_DIM * Ks, 0};
    GemmOperand Bw{tc->ctB, Ki, Ks, Ki * Ks, 0};
    GemmEpilogue e = epi_linear(EPI_OUT_F32, nullptr, nullptr, tc->part, nullptr, Ki);
    e.out_bstride = (long long)CONV_DIM * Ki;
    NB_TRY(gemm_h16(st, A, Bw, CONV_DIM, Ki, (int)Ks, splits, e, 0));
    conv_wgrad_reduce_kernel<<<(unsigned)((CONV_DIM * Ki + 255) / 256), 256, 0, st>>>(tc->part, splits, k,
                                                                                     tc->conv_grads + ConvLayout::level(l));
    NB_LAUNCHED();
    return 0;
}

static int train_hook_conv0(TrainCtx* tc, const Workspace& ws, const op_t* D0, const float* wav, int B, long long R0,
                            const Weights& w, cudaStream_t st) {
    NB_CUDA(cudaMemsetAsync(tc->c0_sums, 0, 8ull * C0W_SUMS * CONV_DIM * B, st));
    const long long groups = R0 / 64;
    conv0_wgrad_stats_kernel<<<(unsigned)((groups + 3) / 4), 256, 0, st>>>(D0, wav, ws.meta, B, groups, w.conv0_w, ws.gn_stat,
                                                                         tc->c0_sums);
    NB_LAUNCHED();
    float* G = tc->conv_grads;
    conv0_param_grad_kernel<<<1, CONV_DIM, 0, st>>>(tc->c0_sums, ws.stat_part, ws.meta, B, tc->max_chunks, w.conv0_w, w.gn_g,
                                                    G + ConvLayout::C0_W, G + ConvLayout::GN_G, G + ConvLayout::GN_B);
    NB_LAUNCHED();
    return 0;
}

static int train_hook_layer(Handle* h, const Workspace& ws, const LossBufs& L, TrainCtx* tc, int l, int stage, int B,
                            long long Fe, const float* g_running, cudaStream_t st) {
    const Weights& w = h->w;
    const LayerWeights& W = w.layer[l];
    const LayerBufs& Lb = ws.layer[l];
    float* G = tc->grads + TrainLayout::LAYER * l;
    if (stage == 0) {  // final_layer_norm params (incoming: g_running + pooled gradient on the top layer); fc2
        if (tc->ug != nullptr) {  // + the caller's gradient of this layer's output, both under S
            const UserGrads& ug = *tc->ug;
            NB_TRY(launch_ln768_param_grad_user(st, g_running, ug.g_layers[l], ug.T, l == LAYERS - 1 ? ug.g_pool : nullptr,
                                                ug.scale, Lb.pre2, ws.meta, B, Fe, G + TrainLayout::LN2_G, G + TrainLayout::LN2_B));
        } else {
            NB_TRY(launch_ln768_param_grad(st, g_running, l == LAYERS - 1 ? L.g_pool : nullptr, Lb.pre2, nullptr, ws.meta, B, Fe,
                                           G + TrainLayout::LN2_G, G + TrainLayout::LN2_B));
        }
        NB_TRY(wgrad(st, tc, L.g_bh, EMBED, Lb.ffn_h, FFN, Fe, G + TrainLayout::FC2_W));
        NB_TRY(launch_colsum<float>(st, L.g_b, Fe, EMBED, G + TrainLayout::FC2_B));
    } else if (stage == 1) {  // fc1: input = LayerNorm1(pre1), recomputed
        NB_TRY(launch_ln768(st, Lb.pre1, ws.meta, B, Fe, W.ln1_g, W.ln1_b, nullptr, tc->xh_tmp, nullptr, nullptr, 0));
        NB_TRY(wgrad(st, tc, L.g_h, FFN, tc->xh_tmp, EMBED, Fe, G + TrainLayout::FC1_W));
        NB_TRY(launch_colsum<op_t>(st, L.g_h, Fe, FFN, G + TrainLayout::FC1_B));
    } else if (stage == 2) {  // self_attn_layer_norm params (incoming L.g_c); out_proj
        NB_TRY(launch_ln768_param_grad(st, L.g_c, nullptr, Lb.pre1, nullptr, ws.meta, B, Fe, G + TrainLayout::LN1_G,
                                       G + TrainLayout::LN1_B));
        NB_TRY(wgrad(st, tc, L.g_bh, EMBED, Lb.attn, EMBED, Fe, G + TrainLayout::O_W));
        NB_TRY(launch_colsum<float>(st, L.g_b, Fe, EMBED, G + TrainLayout::O_B));
    } else {  // fused q/k/v: input = this layer's input (previous final_layer_norm output / encoder LayerNorm output)
        if (l > 0) {
            NB_TRY(launch_ln768(st, ws.layer[l - 1].pre2, ws.meta, B, Fe, w.layer[l - 1].ln2_g, w.layer[l - 1].ln2_b, nullptr,
                                tc->xh_tmp, nullptr, nullptr, 0));
        } else {
            NB_TRY(launch_pos_finish_ln(st, ws.x0, ws.pos_y, ws.meta, B, Fe, w.lne_g, w.lne_b, tc->x_tmp, tc->xh_tmp));
        }
        NB_TRY(wgrad(st, tc, L.g_qkv, 3 * EMBED, tc->xh_tmp, EMBED, Fe, G + TrainLayout::QKV_W));
        NB_TRY(launch_colsum<op_t>(st, L.g_qkv, Fe, 3 * EMBED, G + TrainLayout::QKV_B));
    }
    return 0;
}

static int train_hook_front(Handle* h, const Workspace& ws, const LossBufs& L, TrainCtx* tc, int stage, int B, long long Fe,
                            long long pos_rows_e, cudaStream_t st) {
    const Weights& w = h->w;
    float* G = tc->grads;
    const long long rows_alloc = pos_rows_e + POS_K;
    if (stage == 0) {  // encoder LayerNorm params: input x0 + pos_y, incoming gradient L.g_a
        NB_TRY(launch_ln768_param_grad(st, L.g_a, nullptr, ws.x0, ws.pos_y, ws.meta, B, Fe, G + TrainLayout::ENC_G, G + TrainLayout::ENC_B));
    } else if (stage == 1) {  // positional conv (folded weight) + bias: dY = L.pos_g, X = ws.pos_g
        // dW[g][n][tap][c] = sum_p dY[g][p][n] X[g][p - 64 + tap][c]: per group, transpose both padded layouts to
        // [48][rows] (K-major over the rows) and run ONE shared-operand tensor-core GEMM batched over the 128 taps, the
        // B operand's K origin shifted per tap.  TMA wants 16-byte aligned origins, so X is kept as 8 transposes
        // pre-shifted by 0..7 rows: tap = 8 q + r reads copy r at origin 8 q - 64 (outside the row reads zero).
        static const int pos_simt = getenv("NOMAD_B200_POS_WGRAD_SIMT") ? atoi(getenv("NOMAD_B200_POS_WGRAD_SIMT")) : 0;
        const long long Rp = (rows_alloc + 7) / 8 * 8;
        if (pos_simt || 8 * (long long)POS_GC * Rp > (long long)FFN * tc->Fp) {  // scratch too small: CUDA-core fallback
            dim3 grid(POS_K, POS_G);
            pos_wgrad_kernel<<<grid, 288, 0, st>>>(L.pos_g, ws.pos_g, rows_alloc, pos_rows_e, G + TrainLayout::POS_W);
            NB_LAUNCHED();
        } else {
            for (int g = 0; g < POS_G; ++g) {
                NB_TRY(launch_transpose(st, L.pos_g + (long long)g * rows_alloc * POS_GC, rows_alloc, POS_GC, Rp, tc->tA));
                NB_TRY(launch_transpose(st, ws.pos_g + (long long)g * rows_alloc * POS_GC, rows_alloc, POS_GC, Rp, tc->tB, 8));
                GemmOperand A{tc->tA, POS_GC, Rp, 0, 0};
                GemmOperand Bw{tc->tB, POS_GC, Rp, (long long)POS_GC * Rp, 0};
                GemmEpilogue e = epi_linear(EPI_OUT_F32, nullptr, nullptr, G + TrainLayout::POS_W + (long long)g * POS_GC * POS_K * POS_GC,
                                            nullptr, (long long)POS_K * POS_GC);
                e.out_bstride = POS_GC;  // batch = tap: columns [tap * 48, tap * 48 + 48) of the [n][tap * 48 + c] rows
                NB_TRY(gemm_h16_corr(st, A, Bw, POS_GC, POS_GC, (int)Rp, POS_K, -(POS_K / 2), 8, 8, e));
            }
        }
        pos_bias_grad_kernel<<<POS_G, 256, 0, st>>>(L.pos_g, rows_alloc, G + TrainLayout::POS_B);
        NB_LAUNCHED();
    } else if (stage == 2) {  // feature projection: dY = L.g_x0h, X = LayerNorm(512) output
        NB_TRY(wgrad(st, tc, L.g_x0h, EMBED, ws.ln0_out, CONV_DIM, Fe, G + TrainLayout::PROJ_W));
        NB_TRY(launch_colsum<op_t>(st, L.g_x0h, Fe, EMBED, G + TrainLayout::PROJ_B));
    } else {  // LayerNorm(512) params: incoming L.g_ln0, input = conv features (level 6)
        const unsigned blocks = (unsigned)std::min<long long>((Fe + 7) / 8, 296);
        ln512_param_grad_kernel<<<blocks, 256, 0, st>>>(L.g_ln0, ws.y[6], ws.meta, B, Fe, G + TrainLayout::LN0_G, G + TrainLayout::LN0_B);
        NB_LAUNCHED();
    }
    return 0;
}

static size_t train_extra_bytes(long long F, int n_utt) {
    const long long Fp = (F + 7) / 8 * 8;
    auto al = [](size_t v) { return (v + 1023) / 1024 * 1024; };
    return al(2ull * FFN * Fp) * 2 + al(2ull * EMBED * F) + al(4ull * EMBED * F) + al(4ull * EMB * n_utt) + 4096;
}

// phase 0: the whole step; 1: only the per-call metadata upload (the part of a step that cannot live in a CUDA graph:
// it goes through the handle's pinned staging ring); 2: the whole step except that upload (what the graph holds)
static int loss_run(nomad_b200_handle* hh, const float* est_dev, const float* clean_dev, int B, int64_t N,
                    float feature_grad_mult, float* loss_dev, float* d_est_dev, void* workspace_dev, size_t workspace_bytes,
                    cudaStream_t st, int phase) {
    Handle* h = &hh->h;
    const bool with_grad = d_est_dev != nullptr;
    const Weights& w = h->w;
    const int impl = h->gemm_impl;

    Plan p;
    NB_TRY(loss_plan(B, N, &p));
    // utterances 0..B-1 = estimates, B..2B-1 = clean; both addressed relative to est_dev
    const long long clean_off = (long long)(((intptr_t)clean_dev - (intptr_t)est_dev) / 4);
    for (int b = 0; b < B; ++b) {
        p.utt[b].wav_off = (long long)b * N;
        p.utt[B + b].wav_off = clean_off + (long long)b * N;
    }
    const long long F = p.frames, Fe = F / 2, R0e = p.rows0 / 2;
    const long long pos_rows_e = Fe + (long long)POS_GAP * B + POS_K / 2;
    const int T = p.max_T;
    Workspace ws;
    const size_t fwd_bytes = carve_workspace(p, workspace_dev, &ws, true);
    LossBufs L;
    const size_t loss_bytes = carve_loss(p, B, Fe, R0e, pos_rows_e, with_grad, (char*)workspace_dev + fwd_bytes, &L);
    NB_CHECK(workspace_bytes >= fwd_bytes + loss_bytes, "loss: workspace too small (%zu < %zu bytes)", workspace_bytes,
             fwd_bytes + loss_bytes);
    NB_CHECK(((uintptr_t)workspace_dev & 1023) == 0, "loss: workspace must be 1024-byte aligned");

    // ------------------------------------------------------------------ forward (both halves, save mode)
    if (phase != 2) NB_TRY(upload_meta(h, p, ws, st));
    if (phase == 1) return 0;
    NB_CUDA(cudaMemsetAsync(L.acc, 0, sizeof(double) * 16, st));
    NB_TRY(forward_encoder(h, p, ws, est_dev, st, nullptr, 0));
    NB_TRY(launch_pool_head(st, ws.x, ws.meta, p.B, w.loss_head_wt, w.loss_head_b, L.emb, L.pooled));
    const unsigned row_blocks = (unsigned)((Fe + 7) / 8);
    for (int l = 0; l < LAYERS; ++l) {
        l1_layer_kernel<<<row_blocks, 256, 0, st>>>(ws.layer[l].pre2, ws.meta, B, Fe, w.layer[l].ln2_g, L.acc + l);
        NB_LAUNCHED();
    }
    // gradient scale: power of two with S / (B T 768) in [1, 2)
    const double numel = (double)B * T * EMBED;
    const float S = with_grad ? (float)std::exp2(std::ceil(std::log2(numel))) : 0.f;
    const float seed_layer = (float)(S / numel), seed_head = (float)(S / ((double)B * EMB));
    // head term (13th): value always, pooled-feature gradient when a backward follows (seed 0 otherwise)
    head_bwd_kernel<<<B, 256, 0, st>>>(L.pooled, ws.meta, B, w.loss_head_wt, w.loss_head_w, w.loss_head_b, seed_head,
                                       L.acc + LAYERS, L.g_pool);
    NB_LAUNCHED();
    loss_finalize_kernel<<<1, 1, 0, st>>>(L.acc, 1.0 / numel, 1.0 / ((double)B * EMB), loss_dev);
    NB_LAUNCHED();
    if (getenv("NOMAD_B200_DEBUG_LOSS")) {  // per-term L1 sums, for debugging only (synchronises)
        double hacc[16];
        NB_CUDA(cudaStreamSynchronize(st));
        NB_CUDA(cudaMemcpy(hacc, L.acc, sizeof(hacc), cudaMemcpyDeviceToHost));
        for (int i = 0; i < 13; ++i) fprintf(stderr, "[nomad_b200] L1 term %2d: sum |diff| = %.9g\n", i, hacc[i]);
    }
    if (!with_grad) return 0;

    // ------------------------------------------------------------------ backward (estimate half)
    return backward_chain(h, ws, L, B, Fe, R0e, pos_rows_e, T, seed_layer, feature_grad_mult, S, est_dev, N, d_est_dev, st, nullptr);
}

// The fused loss step on a handle in NOMAD_B200_PRECISION_FP32: the fp32-class save-mode forward of both halves, the same
// L1 / head kernels as loss_run on its pre-LayerNorm sums and residual stream, and the fp32-class waveform backward of
// the estimate half.  Always eager (the step is dominated by its split-operand GEMMs, not by launch gaps).
static int loss_run_precise(Handle* h, const float* est_dev, const float* clean_dev, int B, int64_t N, float feature_grad_mult,
                            float* loss_dev, float* d_est_dev, void* workspace_dev, size_t workspace_bytes, cudaStream_t st) {
    const bool with_grad = d_est_dev != nullptr;
    const Weights& w = h->w;
    Plan p;
    NB_TRY(loss_plan(B, N, &p));
    const long long clean_off = (long long)(((intptr_t)clean_dev - (intptr_t)est_dev) / 4);
    for (int b = 0; b < B; ++b) {
        p.utt[b].wav_off = (long long)b * N;
        p.utt[B + b].wav_off = clean_off + (long long)b * N;
    }
    size_t fwd, mid;
    const size_t need = loss_precise_bytes(p, B, with_grad, &fwd, &mid);
    NB_CHECK(workspace_bytes >= need, "loss (fp32 mode): workspace too small (%zu < %zu bytes); size it with "
             "nomad_b200_loss_workspace_bytes_mode", workspace_bytes, need);
    char* base = (char*)workspace_dev;
    PWorkspace ws;
    carve_precise(p, base, &ws, true);
    LossBufs L;
    carve_loss(p, B, 0, 0, 0, false, base + fwd, &L);
    const long long Fe = p.frames / 2;
    const int T = p.max_T;
    NB_CUDA(cudaMemsetAsync(L.acc, 0, sizeof(double) * 16, st));
    NB_TRY(embed_precise_save(h, p, base, fwd, est_dev, st, nullptr, 0));
    NB_TRY(launch_pool_head(st, ws.x, ws.meta, p.B, w.loss_head_wt, w.loss_head_b, L.emb, L.pooled));
    const unsigned row_blocks = (unsigned)((Fe + 7) / 8);
    for (int l = 0; l < LAYERS; ++l) {
        l1_layer_kernel<<<row_blocks, 256, 0, st>>>(ws.pre2[l], ws.meta, B, Fe, w.layer[l].ln2_g, L.acc + l);
        NB_LAUNCHED();
    }
    const double numel = (double)B * T * EMBED;
    const float S = with_grad ? (float)std::exp2(std::ceil(std::log2(numel))) : 0.f;
    head_bwd_kernel<<<B, 256, 0, st>>>(L.pooled, ws.meta, B, w.loss_head_wt, w.loss_head_w, w.loss_head_b,
                                       (float)(S / ((double)B * EMB)), L.acc + LAYERS, L.g_pool);
    NB_LAUNCHED();
    loss_finalize_kernel<<<1, 1, 0, st>>>(L.acc, 1.0 / numel, 1.0 / ((double)B * EMB), loss_dev);
    NB_LAUNCHED();
    if (!with_grad) return 0;
    PBwdArgs a;
    memset(&a, 0, sizeof(a));
    a.B_bwd = B;
    a.top = LAYERS - 1;
    a.g_pool = L.g_pool;
    a.seed_layer = (float)(S / numel);
    a.out_scale = 1.0f / S;
    a.feature_grad_mult = feature_grad_mult;
    return backward_precise(h, p, base, a, est_dev, N, d_est_dev, base + fwd + mid, workspace_bytes - fwd - mid, st);
}

extern "C" {

// The step is ~250 small launches for B = 32 x 2 s (profiles/r02_loss_trace_before.log: 8 % of the step was launch gaps):
// after one eager call per (B, N, grad, feature_grad_mult, workspace) the launch sequence is captured into a CUDA graph
// over fixed addresses -- inputs are copied into a staging area at the end of the caller's workspace, results copied
// out -- and replayed.  NOMAD_B200_LOSS_GRAPH=0 keeps every call eager.
int nomad_b200_loss_fwd_bwd(nomad_b200_handle* hh, const float* est_dev, const float* clean_dev, int B, int64_t N,
                            float feature_grad_mult, float* loss_dev, float* d_est_dev, void* workspace_dev,
                            size_t workspace_bytes, void* stream) {
    NB_CHECK(hh != nullptr, "null nomad_b200 handle");
    Handle* h = &hh->h;
    NB_CHECK(est_dev && clean_dev && loss_dev && workspace_dev, "loss: null pointer");
    NB_CHECK(h->has_loss_head, "loss: call nomad_b200_set_loss_head first (LossNetLayers has its own head, nomad.py:238-241)");
    NB_CHECK((((uintptr_t)est_dev | (uintptr_t)clean_dev) & 3) == 0, "loss: waveform pointers must be 4-byte aligned");
    NB_CHECK(((uintptr_t)workspace_dev & 1023) == 0, "loss: workspace must be 1024-byte aligned");
    NB_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (h->precision == NOMAD_B200_PRECISION_FP32)
        return loss_run_precise(h, est_dev, clean_dev, B, N, feature_grad_mult, loss_dev, d_est_dev, workspace_dev, workspace_bytes, st);
    const int with_grad = d_est_dev != nullptr ? 1 : 0;
    static const int use_graph = getenv("NOMAD_B200_LOSS_GRAPH") ? atoi(getenv("NOMAD_B200_LOSS_GRAPH")) : 1;
    const size_t core = (loss_core_bytes(B, N, with_grad) + 1023) / 1024 * 1024;
    NB_CHECK(core != 0, "loss: %s", nomad_b200_last_error());
    const bool graph_ok = use_graph && h->gemm_impl == 0 && !getenv("NOMAD_B200_DEBUG_LOSS") && !gemm_profile_active() &&
                          workspace_bytes >= core + loss_stage_bytes(B, N);
    if (!graph_ok)
        return loss_run(hh, est_dev, clean_dev, B, N, feature_grad_mult, loss_dev, d_est_dev, workspace_dev, workspace_bytes, st, 0);

    const size_t bn = (size_t)B * N;
    float* s_est = (float*)((char*)workspace_dev + core);
    float* s_clean = s_est + bn;
    float* s_grad = s_clean + bn;
    float* s_loss = s_grad + bn;
    NB_CUDA(cudaMemcpyAsync(s_est, est_dev, bn * 4, cudaMemcpyDeviceToDevice, st));
    NB_CUDA(cudaMemcpyAsync(s_clean, clean_dev, bn * 4, cudaMemcpyDeviceToDevice, st));
    LossGraphEntry* ent = nullptr;
    for (auto& e : h->loss_graphs)
        if (e.mode == h->precision && e.B == B && e.N == N && e.with_grad == with_grad && e.fgm == feature_grad_mult &&
            e.ws == workspace_dev)
            ent = &e;
    if (ent == nullptr) {  // first call with this shape: eager (also performs the one-off per-kernel attribute set-up)
        if (h->loss_graphs.size() >= 8) {
            for (auto& e : h->loss_graphs)
                if (e.exec) cudaGraphExecDestroy(e.exec);
            h->loss_graphs.clear();
        }
        h->loss_graphs.push_back(LossGraphEntry{h->precision, B, (long long)N, with_grad, feature_grad_mult, workspace_dev, nullptr, 0, false});
        NB_TRY(loss_run(hh, s_est, s_clean, B, N, feature_grad_mult, s_loss, with_grad ? s_grad : nullptr, workspace_dev, core, st, 0));
    } else if (ent->exec == nullptr && !ent->failed) {  // second call: capture on the handle's own stream, then launch
        if (!h->graph_stream) NB_CUDA(cudaStreamCreateWithFlags(&h->graph_stream, cudaStreamNonBlocking));
        NB_TRY(loss_run(hh, s_est, s_clean, B, N, feature_grad_mult, s_loss, with_grad ? s_grad : nullptr, workspace_dev, core, st, 1));
        const long long n0 = nomad_b200_launch_count();
        cudaGraph_t graph = nullptr;
        NB_CUDA(cudaStreamBeginCapture(h->graph_stream, cudaStreamCaptureModeThreadLocal));
        const int rc = loss_run(hh, s_est, s_clean, B, N, feature_grad_mult, s_loss, with_grad ? s_grad : nullptr, workspace_dev,
                                core, h->graph_stream, 2);
        const cudaError_t ce = cudaStreamEndCapture(h->graph_stream, &graph);
        ent->kernels = nomad_b200_launch_count() - n0;
        if (rc == 0 && ce == cudaSuccess && graph != nullptr &&
            cudaGraphInstantiate(&ent->exec, graph, 0) == cudaSuccess) {
            cudaGraphDestroy(graph);
            NB_CUDA(cudaGraphLaunch(ent->exec, st));
        } else {  // capture not possible here: stay eager for this shape
            if (graph) cudaGraphDestroy(graph);
            cudaGetLastError();
            ent->exec = nullptr;
            ent->failed = true;
            count_launches(-ent->kernels);
            NB_TRY(loss_run(hh, s_est, s_clean, B, N, feature_grad_mult, s_loss, with_grad ? s_grad : nullptr, workspace_dev, core, st, 2));
        }
    } else if (ent->exec != nullptr) {
        NB_TRY(loss_run(hh, s_est, s_clean, B, N, feature_grad_mult, s_loss, with_grad ? s_grad : nullptr, workspace_dev, core, st, 1));
        NB_CUDA(cudaGraphLaunch(ent->exec, st));
        count_launches(ent->kernels);
    } else {
        NB_TRY(loss_run(hh, s_est, s_clean, B, N, feature_grad_mult, s_loss, with_grad ? s_grad : nullptr, workspace_dev, core, st, 0));
    }
    NB_CUDA(cudaMemcpyAsync(loss_dev, s_loss, 4, cudaMemcpyDeviceToDevice, st));
    if (with_grad) NB_CUDA(cudaMemcpyAsync(d_est_dev, s_grad, bn * 4, cudaMemcpyDeviceToDevice, st));
    return 0;
}

}  // extern "C"

// ---- triplet fine-tuning step: C ABI ---------------------------------------------------------------------------
extern "C" {

int64_t nomad_b200_triplet_grad_floats(void) { return TrainLayout::TOTAL; }

// segment i of the flat gradient buffer: name, offset and element count; returns 0 while i is valid, 1 past the end
int nomad_b200_triplet_grad_segment(int i, char* name, int name_cap, int64_t* offset, int64_t* numel) {
    static const struct { const char* n; long long off, cnt; } per_layer[12] = {
        {"qkv.weight", TrainLayout::QKV_W, 2304LL * 768}, {"qkv.bias", TrainLayout::QKV_B, 2304},
        {"self_attn.out_proj.weight", TrainLayout::O_W, 768LL * 768}, {"self_attn.out_proj.bias", TrainLayout::O_B, 768},
        {"fc1.weight", TrainLayout::FC1_W, 3072LL * 768}, {"fc1.bias", TrainLayout::FC1_B, 3072},
        {"fc2.weight", TrainLayout::FC2_W, 768LL * 3072}, {"fc2.bias", TrainLayout::FC2_B, 768},
        {"self_attn_layer_norm.weight", TrainLayout::LN1_G, 768}, {"self_attn_layer_norm.bias", TrainLayout::LN1_B, 768},
        {"final_layer_norm.weight", TrainLayout::LN2_G, 768}, {"final_layer_norm.bias", TrainLayout::LN2_B, 768}};
    static const struct { const char* n; long long off, cnt; } global[10] = {
        {"ssl_model.encoder.layer_norm.weight", TrainLayout::ENC_G, 768}, {"ssl_model.encoder.layer_norm.bias", TrainLayout::ENC_B, 768},
        {"ssl_model.encoder.pos_conv.0.folded_weight", TrainLayout::POS_W, (long long)POS_G * POS_GC * POS_K * POS_GC},
        {"ssl_model.encoder.pos_conv.0.bias", TrainLayout::POS_B, 768},
        {"ssl_model.post_extract_proj.weight", TrainLayout::PROJ_W, 768LL * 512}, {"ssl_model.post_extract_proj.bias", TrainLayout::PROJ_B, 768},
        {"ssl_model.layer_norm.weight", TrainLayout::LN0_G, 512}, {"ssl_model.layer_norm.bias", TrainLayout::LN0_B, 512},
        {"embedding_layer.1.weight", TrainLayout::HEAD_W, 256LL * 768}, {"embedding_layer.1.bias", TrainLayout::HEAD_B, 256}};
    if (i < 0 || name == nullptr || offset == nullptr || numel == nullptr) return 1;
    if (i < 12 * LAYERS) {
        const int l = i / 12, k = i % 12;
        snprintf(name, name_cap, "ssl_model.encoder.layers.%d.%s", l, per_layer[k].n);
        *offset = TrainLayout::LAYER * l + per_layer[k].off;
        *numel = per_layer[k].cnt;
        return 0;
    }
    i -= 12 * LAYERS;
    if (i >= 10) return 1;
    snprintf(name, name_cap, "%s", global[i].n);
    *offset = global[i].off;
    *numel = global[i].cnt;
    return 0;
}

static int triplet_plan(int B, int64_t N, Plan* p) {
    NB_CHECK(B > 0 && N >= NOMAD_B200_MIN_SAMPLES, "triplet: need B > 0 and N >= %d samples", NOMAD_B200_MIN_SAMPLES);
    std::vector<int64_t> off(3 * (size_t)B + 1);
    for (int b = 0; b <= 3 * B; ++b) off[b] = (int64_t)b * N;
    return make_plan(off.data(), 3 * B, p);
}

size_t nomad_b200_triplet_workspace_bytes(int B, int64_t N) {
    Plan p;
    if (triplet_plan(B, N, &p)) return 0;
    const size_t fwd = carve_workspace(p, nullptr, nullptr, true, true);
    const long long pos_rows = p.frames + (long long)POS_GAP * 3 * B + POS_K / 2;
    return fwd + carve_loss(p, 3 * B, p.frames, p.rows0, pos_rows, true, nullptr, nullptr) + train_extra_bytes(p.frames, 3 * B) + 4096;
}

}  // extern "C"

// extra scratch of the conv-encoder step: [ctA | ctB | part | c0_sums], carved from `base` (sizes only when null)
static size_t carve_conv_train(long long R0, int U, void* base, TrainCtx* tc) {
    const long long rows = R0 / 2 + 64LL * CONV_SPLIT_MAX;  // level 1 (the largest) plus the slices' padding
    size_t o = 0;
    auto take = [&](size_t bytes) {
        size_t at = o;
        o = (o + bytes + 1023) / 1024 * 1024;
        return base ? (void*)((char*)base + at) : nullptr;
    };
    void* a = take(2ull * CONV_DIM * rows);
    void* b = take(2ull * 3 * CONV_DIM * rows);
    void* part = take(4ull * CONV_SPLIT_MAX * CONV_DIM * 3 * CONV_DIM);
    void* sums = take(8ull * C0W_SUMS * CONV_DIM * U);
    if (tc) {
        tc->ctA = (op_t*)a;
        tc->ctB = (op_t*)b;
        tc->part = (float*)part;
        tc->c0_sums = (double*)sums;
    }
    return o;
}

// wav_dev: 3B x N fp32 (anchors, then positives, then negatives); loss_dev: 1 float; grads_dev:
// nomad_b200_triplet_grad_floats() floats (zeroed here) = grad_scale_out[0] * d loss / d parameter.  conv_grads_dev non-null:
// the conv feature encoder is trained too (its gradients, times fgm, go there) and the workspace holds the conv scratch.
static int triplet_run(nomad_b200_handle* hh, const float* wav_dev, int B, int64_t N, float margin, float fgm, float* loss_dev,
                       float* grads_dev, float* conv_grads_dev, float* grad_scale_out, void* workspace_dev, size_t workspace_bytes,
                       void* stream) {
    NB_CHECK(hh != nullptr, "null nomad_b200 handle");
    Handle* h = &hh->h;
    NB_CHECK(wav_dev && loss_dev && grads_dev && grad_scale_out && workspace_dev, "triplet: null pointer");
    NB_CHECK(h->gemm_impl == 0, "triplet: tensor-core GEMMs only");
    NB_CHECK(((uintptr_t)workspace_dev & 1023) == 0, "triplet: workspace must be 1024-byte aligned");
    NB_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    const Weights& w = h->w;
    Plan p;
    NB_TRY(triplet_plan(B, N, &p));
    const int U = 3 * B;
    const long long F = p.frames, R0 = p.rows0;
    const long long pos_rows = F + (long long)POS_GAP * U + POS_K / 2;
    Workspace ws;
    const size_t fwd_bytes = carve_workspace(p, workspace_dev, &ws, true, true);
    LossBufs L;
    const size_t loss_bytes = carve_loss(p, U, F, R0, pos_rows, true, (char*)workspace_dev + fwd_bytes, &L);
    const size_t extra = train_extra_bytes(F, U);
    const size_t conv_bytes = conv_grads_dev != nullptr ? carve_conv_train(R0, U, nullptr, nullptr) : 0;
    NB_CHECK(workspace_bytes >= fwd_bytes + loss_bytes + extra + conv_bytes, "triplet: workspace too small (%zu < %zu bytes)",
             workspace_bytes, fwd_bytes + loss_bytes + extra + conv_bytes);
    TrainCtx tc;
    memset(&tc, 0, sizeof(tc));
    {
        auto al = [](size_t v) { return (v + 1023) / 1024 * 1024; };
        char* q = (char*)workspace_dev + fwd_bytes + loss_bytes;
        tc.Fp = (F + 7) / 8 * 8;
        tc.tA = (op_t*)q; q += al(2ull * FFN * tc.Fp);
        tc.tB = (op_t*)q; q += al(2ull * FFN * tc.Fp);
        tc.xh_tmp = (op_t*)q; q += al(2ull * EMBED * F);
        tc.x_tmp = (float*)q; q += al(4ull * EMBED * F);
        tc.gy = (float*)q;
        tc.grads = grads_dev;
    }
    if (conv_grads_dev != nullptr) {
        NB_CHECK(((uintptr_t)conv_grads_dev & 15) == 0, "triplet: conv gradient buffer must be 16-byte aligned");
        carve_conv_train(R0, U, (char*)workspace_dev + fwd_bytes + loss_bytes + extra, &tc);
        tc.conv_grads = conv_grads_dev;
        tc.max_chunks = p.max_chunks;
        ws.aux0_raw = true;
    }
    NB_TRY(upload_meta(h, p, ws, st));
    NB_CUDA(cudaMemsetAsync(grads_dev, 0, sizeof(float) * TrainLayout::TOTAL, st));
    NB_CUDA(cudaMemsetAsync(L.acc, 0, sizeof(double) * 16, st));
    NB_TRY(forward_encoder(h, p, ws, wav_dev, st, nullptr, 0));
    NB_TRY(launch_pool_head(st, ws.x, ws.meta, U, w.head_wt, w.head_b, L.emb, L.pooled));
    // gradient scale: power of two so that the 16-bit activation gradients sit in fp16's normal range
    const float S = (float)std::exp2(std::ceil(std::log2((double)B * p.max_T)) + 10.0);
    triplet_head_kernel<<<B, 256, 0, st>>>(L.pooled, B, w.head_wt, w.head_b, margin, S / (float)B, L.acc, tc.gy);
    NB_LAUNCHED();
    triplet_loss_finalize_kernel<<<1, 1, 0, st>>>(L.acc, 1.0 / (double)B, loss_dev);
    NB_LAUNCHED();
    head_param_grad_kernel<false><<<EMB, 256, 0, st>>>(tc.gy, L.pooled, U, grads_dev + TrainLayout::HEAD_W,
                                                       grads_dev + TrainLayout::HEAD_B, nullptr);
    NB_LAUNCHED();
    head_pool_grad_kernel<<<U, 256, 0, st>>>(tc.gy, L.pooled, ws.meta, w.head_wt, L.g_pool);
    NB_LAUNCHED();
    *grad_scale_out = S;
    return backward_chain(h, ws, L, U, F, R0, pos_rows, p.max_T, 0.f, conv_grads_dev != nullptr ? fgm : 1.0f, S, wav_dev, N,
                          nullptr, st, &tc);
}

extern "C" {

int nomad_b200_triplet_fwd_bwd(nomad_b200_handle* hh, const float* wav_dev, int B, int64_t N, float margin, float* loss_dev,
                               float* grads_dev, float* grad_scale_out, void* workspace_dev, size_t workspace_bytes, void* stream) {
    return triplet_run(hh, wav_dev, B, N, margin, 1.0f, loss_dev, grads_dev, nullptr, grad_scale_out, workspace_dev,
                       workspace_bytes, stream);
}

int64_t nomad_b200_triplet_conv_grad_floats(void) { return ConvLayout::TOTAL; }

int nomad_b200_triplet_conv_grad_segment(int i, char* name, int name_cap, int64_t* offset, int64_t* numel) {
    if (i < 0 || i >= 9 || name == nullptr || offset == nullptr || numel == nullptr) return 1;
    const char* P = "ssl_model.feature_extractor.conv_layers.";
    if (i < 3) {
        static const char* leaf[3] = {"0.0.weight", "0.2.weight", "0.2.bias"};
        static const long long off[3] = {ConvLayout::C0_W, ConvLayout::GN_G, ConvLayout::GN_B}, cnt[3] = {512 * 10, 512, 512};
        snprintf(name, name_cap, "%s%s", P, leaf[i]);
        *offset = off[i];
        *numel = cnt[i];
        return 0;
    }
    const int l = i - 2;
    snprintf(name, name_cap, "%s%d.0.weight", P, l);
    *offset = ConvLayout::level(l);
    *numel = 512LL * 512 * CONV_KERNEL[l];
    return 0;
}

size_t nomad_b200_triplet_conv_workspace_bytes(int B, int64_t N) {
    const size_t base = nomad_b200_triplet_workspace_bytes(B, N);
    if (base == 0) return 0;
    Plan p;
    if (triplet_plan(B, N, &p)) return 0;
    return base + carve_conv_train(p.rows0, 3 * B, nullptr, nullptr);
}

int nomad_b200_triplet_conv_fwd_bwd(nomad_b200_handle* hh, const float* wav_dev, int B, int64_t N, float margin,
                                    float feature_grad_mult, float* loss_dev, float* grads_dev, float* conv_grads_dev,
                                    float* grad_scale_out, void* workspace_dev, size_t workspace_bytes, void* stream) {
    NB_CHECK(conv_grads_dev != nullptr, "triplet_conv: null conv gradient buffer");
    return triplet_run(hh, wav_dev, B, N, margin, feature_grad_mult, loss_dev, grads_dev, conv_grads_dev, grad_scale_out,
                       workspace_dev, workspace_bytes, stream);
}

}  // extern "C"

// ---- autograd through LossNetLayers / TripletModel: save-mode forward + backward from arbitrary upstream gradients ----
// The saved buffer is [record | save-mode Workspace | pooled features B x 768 | head output B x 256 | head snapshot:
// transposed weight 768 x 256, bias 256].  The backward re-derives the Plan from (B, N) and re-carves the same Workspace
// over it, so every pointer (metadata included) comes back as the forward left it; the backward only reads it.  The
// record holds what the forward saved for (NOMAD_B200_SAVE_* flags; PARAMS makes the Workspace larger): the parameter
// backward reads it back first and refuses what the forward did not save for.
struct SavedTail {
    float* pooled;
    float* emb;
    float* head_wt;
    float* head_b;
};
struct SavedRecord {
    uint32_t magic;
    int32_t flags, head, B;
    int64_t N;
    int32_t mode;  // precision_mode of the forward: 1 = the fp32-class layout of precise.cu (flags 0 only)
};
static constexpr uint32_t SAVED_MAGIC = 0x4e425356u;
static constexpr size_t SAVED_RECORD_BYTES = 1024;

static int layers_plan(int B, int64_t N, Plan* p) {
    NB_CHECK(B > 0, "layers: need B > 0 utterances");
    NB_CHECK(N >= NOMAD_B200_MIN_SAMPLES,
             "layers: N = %lld samples; the conv feature encoder needs at least %d (kernel size can't be greater than "
             "actual input size)", (long long)N, NOMAD_B200_MIN_SAMPLES);
    std::vector<int64_t> off((size_t)B + 1);
    for (int b = 0; b <= B; ++b) off[b] = (int64_t)b * N;
    return make_plan(off.data(), B, p);
}

// mode 1: [record | fp32-class save-mode forward (carve_precise) | tail]; `ws` is then not filled
static size_t carve_saved(const Plan& p, int flags, void* base, Workspace* ws, SavedTail* tail, int mode = 0) {
    size_t o = SAVED_RECORD_BYTES;
    if (mode == NOMAD_B200_PRECISION_FP32) {
        o += carve_precise(p, nullptr, nullptr, true);
    } else {
        o += carve_workspace(p, base ? (char*)base + SAVED_RECORD_BYTES : nullptr, ws, true, (flags & NOMAD_B200_SAVE_PARAMS) != 0);
        if (ws) ws->aux0_raw = (flags & NOMAD_B200_SAVE_CONV) != 0;
    }
    auto take = [&](size_t bytes) {
        size_t at = o;
        o = (o + bytes + 1023) / 1024 * 1024;
        return base ? (float*)((char*)base + at) : nullptr;
    };
    SavedTail t;
    t.pooled = take(4ull * EMBED * p.B);
    t.emb = take(4ull * EMB * p.B);
    t.head_wt = take(4ull * EMBED * EMB);
    t.head_b = take(4ull * EMB);
    if (tail) *tail = t;
    return o;
}

// backward scratch: [LossBufs | gy B x 256 | scale state: max bits, block counter, S]
static size_t carve_layers_bwd(const Plan& p, void* base, LossBufs* L, float** gy, unsigned** state) {
    const size_t lb = carve_loss(p, p.B, p.frames, p.rows0, p.pos_rows, true, base, L);
    const size_t gy_bytes = (4ull * EMB * p.B + 1023) / 1024 * 1024;
    if (base) {
        *gy = (float*)((char*)base + lb);
        *state = (unsigned*)((char*)base + lb + gy_bytes);
    }
    return lb + gy_bytes + 1024;
}

// parameter backward scratch: [carve_layers_bwd | TrainCtx buffers (train_extra_bytes) | conv scratch when CONV]
static size_t carve_params_bwd(const Plan& p, int flags, void* base, LossBufs* L, float** gy, unsigned** state, TrainCtx* tc) {
    const size_t lb = carve_layers_bwd(p, base, L, gy, state);
    const size_t extra = train_extra_bytes(p.frames, p.B);
    if (base) {
        auto al = [](size_t v) { return (v + 1023) / 1024 * 1024; };
        char* q = (char*)base + lb;
        tc->Fp = (p.frames + 7) / 8 * 8;
        tc->tA = (op_t*)q; q += al(2ull * FFN * tc->Fp);
        tc->tB = (op_t*)q; q += al(2ull * FFN * tc->Fp);
        tc->xh_tmp = (op_t*)q; q += al(2ull * EMBED * p.frames);
        tc->x_tmp = (float*)q; q += al(4ull * EMBED * p.frames);
        tc->gy = (float*)q;
    }
    const size_t conv = (flags & NOMAD_B200_SAVE_CONV) ? carve_conv_train(p.rows0, p.B, base ? (char*)base + lb + extra : nullptr, tc) : 0;
    return lb + extra + conv;
}

// fp32-class backward scratch: [backward_precise scratch | g_pool B x 768 | gy B x 256 | scale state]
static size_t carve_layers_bwd_precise(const Plan& p, void* base, float** g_pool, float** gy, unsigned** state, size_t* bwd) {
    auto al = [](size_t v) { return (v + 1023) / 1024 * 1024; };
    const size_t b = precise_bwd_bytes(p, p.B), gp = al(4ull * EMBED * p.B), gyb = al(4ull * EMB * p.B);
    if (base) {
        *bwd = b;
        *g_pool = (float*)((char*)base + b);
        *gy = (float*)((char*)base + b + gp);
        *state = (unsigned*)((char*)base + b + gp + gyb);
    }
    return b + gp + gyb + 1024;
}

extern "C" {

size_t nomad_b200_layers_saved_bytes(int B, int64_t N) { return nomad_b200_layers_saved_bytes_ex(B, N, 0); }

size_t nomad_b200_layers_saved_bytes_ex(int B, int64_t N, int flags) {
    Plan p;
    if (layers_plan(B, N, &p)) return 0;
    return carve_saved(p, flags, nullptr, nullptr, nullptr);
}

size_t nomad_b200_layers_bwd_workspace_bytes(int B, int64_t N) {
    Plan p;
    if (layers_plan(B, N, &p)) return 0;
    return carve_layers_bwd(p, nullptr, nullptr, nullptr, nullptr);
}

size_t nomad_b200_layers_saved_bytes_mode(int B, int64_t N, int precision_mode) {
    Plan p;
    if (layers_plan(B, N, &p)) return 0;
    return carve_saved(p, 0, nullptr, nullptr, nullptr, precision_mode == NOMAD_B200_PRECISION_FP32 ? 1 : 0);
}

size_t nomad_b200_layers_bwd_workspace_bytes_mode(int B, int64_t N, int precision_mode) {
    Plan p;
    if (layers_plan(B, N, &p)) return 0;
    if (precision_mode != NOMAD_B200_PRECISION_FP32) return carve_layers_bwd(p, nullptr, nullptr, nullptr, nullptr);
    return carve_layers_bwd_precise(p, nullptr, nullptr, nullptr, nullptr, nullptr);
}

size_t nomad_b200_layers_bwd_params_workspace_bytes(int B, int64_t N, int flags) {
    Plan p;
    if (layers_plan(B, N, &p)) return 0;
    return carve_params_bwd(p, flags, nullptr, nullptr, nullptr, nullptr, nullptr);
}

int nomad_b200_layers_fwd_save(nomad_b200_handle* hh, const float* wav_dev, int B, int64_t N, int head, float* layers_dev,
                               float* emb_dev, void* saved_dev, size_t saved_bytes, void* stream) {
    return nomad_b200_layers_fwd_save_ex(hh, wav_dev, B, N, head, layers_dev, emb_dev, saved_dev, saved_bytes, 0, stream);
}

int nomad_b200_layers_fwd_save_ex(nomad_b200_handle* hh, const float* wav_dev, int B, int64_t N, int head, float* layers_dev,
                                  float* emb_dev, void* saved_dev, size_t saved_bytes, int flags, void* stream) {
    NB_CHECK(hh != nullptr, "null nomad_b200 handle");
    Handle* h = &hh->h;
    NB_CHECK(wav_dev && saved_dev, "layers_fwd_save: null pointer");
    NB_CHECK(head == 0 || head == 1, "layers_fwd_save: head must be 0 (NOMAD head) or 1 (loss head)");
    NB_CHECK(head == 0 || h->has_loss_head, "layers_fwd_save: head 1 needs nomad_b200_set_loss_head first");
    NB_CHECK((flags & ~(NOMAD_B200_SAVE_PARAMS | NOMAD_B200_SAVE_CONV)) == 0, "layers_fwd_save: unknown flags %d", flags);
    NB_CHECK(((uintptr_t)wav_dev & 3) == 0, "layers_fwd_save: waveform pointer must be 4-byte aligned");
    NB_CHECK(((uintptr_t)saved_dev & 1023) == 0, "layers_fwd_save: saved buffer must be 1024-byte aligned");
    NB_CUDA(cudaSetDevice(h->device));
    Plan p;
    NB_TRY(layers_plan(B, N, &p));
    // parameter gradients (flags != 0) keep the fp16-operand arithmetic in either mode
    const int mode = flags == 0 && h->precision == NOMAD_B200_PRECISION_FP32 ? NOMAD_B200_PRECISION_FP32 : NOMAD_B200_PRECISION_FP16;
    Workspace ws;
    SavedTail t;
    const size_t need = carve_saved(p, flags, saved_dev, &ws, &t, mode);
    NB_CHECK(saved_bytes >= need, "layers_fwd_save: saved buffer too small (%zu < %zu bytes)%s", saved_bytes, need,
             mode ? "; the handle is in fp32 mode: size it with nomad_b200_layers_saved_bytes_mode" : "");
    cudaStream_t st = (cudaStream_t)stream;
    const Weights& w = h->w;
    // pageable source: staged by the call itself, nothing to keep alive
    const SavedRecord rec{SAVED_MAGIC, flags, head, B, (int64_t)N, mode};
    NB_CUDA(cudaMemcpyAsync(saved_dev, &rec, sizeof(rec), cudaMemcpyHostToDevice, st));
    NB_CUDA(cudaMemcpyAsync(t.head_wt, head ? w.loss_head_wt : w.head_wt, 4ull * EMBED * EMB, cudaMemcpyDeviceToDevice, st));
    NB_CUDA(cudaMemcpyAsync(t.head_b, head ? w.loss_head_b : w.head_b, 4ull * EMB, cudaMemcpyDeviceToDevice, st));
    if (mode == NOMAD_B200_PRECISION_FP32) {
        char* fwd = (char*)saved_dev + SAVED_RECORD_BYTES;
        NB_TRY(embed_precise_save(h, p, fwd, carve_precise(p, nullptr, nullptr, true), wav_dev, st, layers_dev, p.max_T));
        PWorkspace pws;
        carve_precise(p, fwd, &pws, true);
        return launch_pool_head(st, pws.x, pws.meta, p.B, t.head_wt, t.head_b, emb_dev ? emb_dev : t.emb, t.pooled);
    }
    NB_TRY(upload_meta(h, p, ws, st));
    NB_TRY(forward_encoder(h, p, ws, wav_dev, st, layers_dev, p.max_T));
    NB_TRY(launch_pool_head(st, ws.x, ws.meta, p.B, t.head_wt, t.head_b, emb_dev ? emb_dev : t.emb, t.pooled));
    return 0;
}

}  // extern "C"

// Backward of one saved forward from the caller's output gradients.  grads_dev null (nomad_b200_layers_bwd): the waveform
// gradient only, S divided out.  grads_dev non-null (nomad_b200_layers_bwd_params): every parameter gradient as well
// (TrainLayout; conv_grads_dev: ConvLayout, which needs a CONV forward), the waveform gradient only when d_wav_dev is
// non-null; every output is multiplied by S and S goes to scale_out.
static int layers_backward(Handle* h, const Plan& p, int flags, int head, const void* saved_dev, const float* wav_dev, int64_t N,
                           const float* const* g_layers, const float* g_emb, float feature_grad_mult, float* d_wav_dev,
                           float* grads_dev, float* conv_grads_dev, float* scale_out, void* workspace_dev,
                           size_t workspace_bytes, cudaStream_t st) {
    const int B = p.B;
    const bool params = grads_dev != nullptr;
    Workspace ws;
    SavedTail t;
    carve_saved(p, flags, (void*)saved_dev, &ws, &t);
    LossBufs L;
    float* gy = nullptr;
    unsigned* state = nullptr;
    TrainCtx tc;
    memset(&tc, 0, sizeof(tc));
    const size_t need = params ? carve_params_bwd(p, flags, workspace_dev, &L, &gy, &state, &tc)
                               : carve_layers_bwd(p, workspace_dev, &L, &gy, &state);
    NB_CHECK(workspace_bytes >= need, "layers_bwd: workspace too small (%zu < %zu bytes)", workspace_bytes, need);

    UserGrads ug;
    memset(&ug, 0, sizeof(ug));
    ug.T = p.max_T;
    ug.top = -1;
    ug.scaled_out = params;
    ScaleSources src;
    memset(&src, 0, sizeof(src));
    const long long layer_n = (long long)B * p.max_T * EMBED;
    for (int l = 0; l < LAYERS; ++l) {
        ug.g_layers[l] = g_layers != nullptr ? g_layers[l] : nullptr;
        src.p[l] = ug.g_layers[l];
        src.n[l] = layer_n;
        if (ug.g_layers[l] != nullptr) ug.top = l;
    }
    float* scale = scale_out != nullptr ? scale_out : (float*)(state + 2);
    ug.scale = scale;
    if (ug.top < 0 && g_emb == nullptr) {  // no output is used: the gradient is zero
        if (d_wav_dev != nullptr) NB_CUDA(cudaMemsetAsync(d_wav_dev, 0, 4ull * B * N, st));
        if (!params) return 0;
        NB_CUDA(cudaMemsetAsync(grads_dev, 0, sizeof(float) * TrainLayout::TOTAL, st));
        if (conv_grads_dev != nullptr) NB_CUDA(cudaMemsetAsync(conv_grads_dev, 0, sizeof(float) * ConvLayout::TOTAL, st));
        NB_CUDA(cudaMemsetAsync(state, 0, 2 * sizeof(unsigned), st));
        grad_scale_kernel<<<1, 256, 0, st>>>(src, state, scale);  // no sources: S = 1
        NB_LAUNCHED();
        return 0;
    }
    if (params) NB_CUDA(cudaMemsetAsync(grads_dev, 0, sizeof(float) * TrainLayout::TOTAL, st));
    if (g_emb != nullptr) {  // head: g_emb -> gy -> pooled-feature gradient (ReLU mask, / T), with the snapshotted head
        head_emb_bwd_kernel<<<B, 256, 0, st>>>(t.pooled, t.head_wt, t.head_b, g_emb, gy);
        NB_LAUNCHED();
        head_pool_grad_kernel<<<B, 256, 0, st>>>(gy, t.pooled, ws.meta, t.head_wt, L.g_pool);
        NB_LAUNCHED();
        ug.g_pool = L.g_pool;
        ug.top = LAYERS - 1;
        src.p[LAYERS] = L.g_pool;
        src.n[LAYERS] = (long long)B * EMBED;
    }
    NB_CUDA(cudaMemsetAsync(state, 0, 2 * sizeof(unsigned), st));
    grad_scale_kernel<<<2 * 148, 256, 0, st>>>(src, state, scale);
    NB_LAUNCHED();
    if (params) {
        // the NOMAD head's own gradient (gy is unscaled: S from the device); the loss head (head 1) is not trained here
        if (g_emb != nullptr && head == 0) {
            head_param_grad_kernel<true><<<EMB, 256, 0, st>>>(gy, t.pooled, B, grads_dev + TrainLayout::HEAD_W,
                                                              grads_dev + TrainLayout::HEAD_B, scale);
            NB_LAUNCHED();
        }
        tc.grads = grads_dev;
        tc.conv_grads = conv_grads_dev;
        tc.max_chunks = p.max_chunks;
        tc.ug = &ug;
    }
    return backward_chain(h, ws, L, B, p.frames, p.rows0, p.pos_rows, p.max_T, 0.f, feature_grad_mult, 1.f, wav_dev, N,
                          d_wav_dev, st, params ? &tc : nullptr, &ug);
}

// The same for a buffer saved in fp32 mode: head and gradient scale as above, then backward_precise.
static int layers_backward_precise(Handle* h, const Plan& p, const void* saved_dev, const float* wav_dev, int64_t N,
                                   const float* const* g_layers, const float* g_emb, float feature_grad_mult, float* d_wav_dev,
                                   void* workspace_dev, size_t workspace_bytes, cudaStream_t st) {
    const int B = p.B;
    SavedTail t;
    carve_saved(p, 0, (void*)saved_dev, nullptr, &t, NOMAD_B200_PRECISION_FP32);
    void* fwd = (char*)saved_dev + SAVED_RECORD_BYTES;
    PWorkspace ws;
    carve_precise(p, fwd, &ws, true);
    float *g_pool = nullptr, *gy = nullptr;
    unsigned* state = nullptr;
    size_t bwd = 0;
    const size_t need = carve_layers_bwd_precise(p, workspace_dev, &g_pool, &gy, &state, &bwd);
    NB_CHECK(workspace_bytes >= need, "layers_bwd (fp32 mode): workspace too small (%zu < %zu bytes); size it with "
             "nomad_b200_layers_bwd_workspace_bytes_mode", workspace_bytes, need);
    PBwdArgs a;
    memset(&a, 0, sizeof(a));
    a.B_bwd = B;
    a.top = -1;
    a.user_T = p.max_T;
    a.feature_grad_mult = feature_grad_mult;
    ScaleSources src;
    memset(&src, 0, sizeof(src));
    for (int l = 0; l < LAYERS; ++l) {
        a.g_layers[l] = g_layers != nullptr ? g_layers[l] : nullptr;
        src.p[l] = a.g_layers[l];
        src.n[l] = (long long)B * p.max_T * EMBED;
        if (a.g_layers[l] != nullptr) a.top = l;
    }
    if (a.top < 0 && g_emb == nullptr) {  // no output is used: the gradient is zero
        NB_CUDA(cudaMemsetAsync(d_wav_dev, 0, 4ull * B * N, st));
        return 0;
    }
    if (g_emb != nullptr) {
        head_emb_bwd_kernel<<<B, 256, 0, st>>>(t.pooled, t.head_wt, t.head_b, g_emb, gy);
        NB_LAUNCHED();
        head_pool_grad_kernel<<<B, 256, 0, st>>>(gy, t.pooled, ws.meta, t.head_wt, g_pool);
        NB_LAUNCHED();
        a.g_pool = g_pool;
        a.top = LAYERS - 1;
        src.p[LAYERS] = g_pool;
        src.n[LAYERS] = (long long)B * EMBED;
    }
    float* scale = (float*)(state + 2);
    NB_CUDA(cudaMemsetAsync(state, 0, 2 * sizeof(unsigned), st));
    grad_scale_kernel<<<2 * 148, 256, 0, st>>>(src, state, scale);
    NB_LAUNCHED();
    a.scale_dev = scale;
    a.out_scale = 1.f;
    return backward_precise(h, p, fwd, a, wav_dev, N, d_wav_dev, workspace_dev, bwd, st);
}

extern "C" {

int nomad_b200_layers_bwd(nomad_b200_handle* hh, const void* saved_dev, size_t saved_bytes, const float* wav_dev, int B,
                          int64_t N, const float* const* g_layers, const float* g_emb, float feature_grad_mult,
                          float* d_wav_dev, void* workspace_dev, size_t workspace_bytes, void* stream) {
    NB_CHECK(hh != nullptr, "null nomad_b200 handle");
    Handle* h = &hh->h;
    NB_CHECK(saved_dev && wav_dev && d_wav_dev && workspace_dev, "layers_bwd: null pointer");
    NB_CHECK(((uintptr_t)saved_dev & 1023) == 0 && ((uintptr_t)workspace_dev & 1023) == 0,
             "layers_bwd: saved buffer and workspace must be 1024-byte aligned");
    NB_CHECK(((uintptr_t)wav_dev & 3) == 0 && ((uintptr_t)d_wav_dev & 3) == 0, "layers_bwd: waveform pointers must be 4-byte aligned");
    NB_CHECK(((uintptr_t)g_emb & 15) == 0, "layers_bwd: g_emb must be 16-byte aligned");
    for (int l = 0; g_layers != nullptr && l < LAYERS; ++l)
        NB_CHECK(((uintptr_t)g_layers[l] & 15) == 0, "layers_bwd: g_layers[%d] must be 16-byte aligned", l);
    NB_CUDA(cudaSetDevice(h->device));
    Plan p;
    NB_TRY(layers_plan(B, N, &p));
    cudaStream_t st = (cudaStream_t)stream;
    int mode = NOMAD_B200_PRECISION_FP16;
    if (h->pw.built) {  // the handle can save either layout: read the record back (one stream synchronisation)
        NB_CHECK(saved_bytes >= SAVED_RECORD_BYTES, "layers_bwd: saved buffer too small");
        SavedRecord rec;
        NB_CUDA(cudaMemcpyAsync(&rec, saved_dev, sizeof(rec), cudaMemcpyDeviceToHost, st));
        NB_CUDA(cudaStreamSynchronize(st));
        NB_CHECK(rec.magic == SAVED_MAGIC && rec.B == B && rec.N == (int64_t)N,
                 "layers_bwd: the saved buffer is not from a nomad_b200_layers_fwd_save of this B x N");
        NB_CHECK(rec.mode == h->precision,
                 "layers_bwd: the saved buffer was written in precision_mode %d but the handle is now in mode %d; switch "
                 "back with nomad_b200_set_precision before the backward, or run the forward again", rec.mode, h->precision);
        mode = rec.mode;
    }
    const size_t need_saved = carve_saved(p, 0, nullptr, nullptr, nullptr, mode);
    NB_CHECK(saved_bytes >= need_saved, "layers_bwd: saved buffer too small (%zu < %zu bytes): not from a forward of this B x N?",
             saved_bytes, need_saved);
    if (mode == NOMAD_B200_PRECISION_FP32)
        return layers_backward_precise(h, p, saved_dev, wav_dev, N, g_layers, g_emb, feature_grad_mult, d_wav_dev, workspace_dev,
                                       workspace_bytes, st);
    return layers_backward(h, p, 0, 0, saved_dev, wav_dev, N, g_layers, g_emb, feature_grad_mult, d_wav_dev, nullptr, nullptr,
                           nullptr, workspace_dev, workspace_bytes, st);
}

int nomad_b200_layers_bwd_params(nomad_b200_handle* hh, const void* saved_dev, size_t saved_bytes, const float* wav_dev, int B,
                                 int64_t N, const float* const* g_layers, const float* g_emb, float feature_grad_mult,
                                 float* d_wav_dev, float* grads_dev, float* conv_grads_dev, float* grad_scale_dev,
                                 void* workspace_dev, size_t workspace_bytes, void* stream) {
    NB_CHECK(hh != nullptr, "null nomad_b200 handle");
    Handle* h = &hh->h;
    NB_CHECK(saved_dev && wav_dev && grad_scale_dev && workspace_dev, "layers_bwd_params: null pointer");
    NB_CHECK(d_wav_dev != nullptr || grads_dev != nullptr, "layers_bwd_params: nothing to compute (d_wav and grads both NULL)");
    NB_CHECK(conv_grads_dev == nullptr || grads_dev != nullptr, "layers_bwd_params: conv_grads needs grads too");
    NB_CHECK(((uintptr_t)saved_dev & 1023) == 0 && ((uintptr_t)workspace_dev & 1023) == 0,
             "layers_bwd_params: saved buffer and workspace must be 1024-byte aligned");
    NB_CHECK(((uintptr_t)wav_dev & 3) == 0 && ((uintptr_t)d_wav_dev & 3) == 0 && ((uintptr_t)grad_scale_dev & 3) == 0,
             "layers_bwd_params: waveform and scale pointers must be 4-byte aligned");
    NB_CHECK((((uintptr_t)g_emb | (uintptr_t)grads_dev | (uintptr_t)conv_grads_dev) & 15) == 0,
             "layers_bwd_params: g_emb, grads and conv_grads must be 16-byte aligned");
    for (int l = 0; g_layers != nullptr && l < LAYERS; ++l)
        NB_CHECK(((uintptr_t)g_layers[l] & 15) == 0, "layers_bwd_params: g_layers[%d] must be 16-byte aligned", l);
    NB_CUDA(cudaSetDevice(h->device));
    Plan p;
    NB_TRY(layers_plan(B, N, &p));
    NB_CHECK(saved_bytes >= SAVED_RECORD_BYTES, "layers_bwd_params: saved buffer too small");
    cudaStream_t st = (cudaStream_t)stream;
    SavedRecord rec;
    NB_CUDA(cudaMemcpyAsync(&rec, saved_dev, sizeof(rec), cudaMemcpyDeviceToHost, st));
    NB_CUDA(cudaStreamSynchronize(st));
    NB_CHECK(rec.magic == SAVED_MAGIC && rec.B == B && rec.N == (int64_t)N,
             "layers_bwd_params: the saved buffer is not from a nomad_b200_layers_fwd_save(_ex) of this B x N");
    NB_CHECK(rec.mode == NOMAD_B200_PRECISION_FP16,
             "layers_bwd_params: the buffer holds an fp32-class forward (parameter gradients run the fp16-operand path: save "
             "with NOMAD_B200_SAVE_PARAMS, or use nomad_b200_layers_bwd for the waveform gradient)");
    NB_CHECK(grads_dev == nullptr || (rec.flags & NOMAD_B200_SAVE_PARAMS),
             "layers_bwd_params: parameter gradients need a forward saved with NOMAD_B200_SAVE_PARAMS");
    NB_CHECK(conv_grads_dev == nullptr || (rec.flags & NOMAD_B200_SAVE_CONV),
             "layers_bwd_params: conv encoder gradients need a forward saved with NOMAD_B200_SAVE_CONV");
    const size_t need_saved = carve_saved(p, rec.flags, nullptr, nullptr, nullptr);
    NB_CHECK(saved_bytes >= need_saved, "layers_bwd_params: saved buffer too small (%zu < %zu bytes)", saved_bytes, need_saved);
    return layers_backward(h, p, rec.flags, rec.head, saved_dev, wav_dev, N, g_layers, g_emb, feature_grad_mult, d_wav_dev,
                           grads_dev, conv_grads_dev, grad_scale_dev, workspace_dev, workspace_bytes, st);
}

}  // extern "C"
