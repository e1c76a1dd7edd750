// fp32-class ("precise") path, shared by its forward (precise.cu) and its waveform backward (precise_bwd.cu).
#pragma once
#include "kernels.cuh"

namespace nb {

// 8 fp32 values -> 8 hi + 8 lo halves (16 bytes each)
__device__ __forceinline__ void split_store8(const float* v, op_t* hi, op_t* lo) {
    uint32_t h[4], l[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        h[i] = pack_op(v[2 * i], v[2 * i + 1]);
        const float2 f = unpack_op(h[i]);
        l[i] = pack_op(v[2 * i] - f.x, v[2 * i + 1] - f.y);
    }
    *reinterpret_cast<uint4*>(hi) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4*>(lo) = make_uint4(l[0], l[1], l[2], l[3]);
}
__device__ __forceinline__ void split_load8(const op_t* hi, const op_t* lo, float* v) {
    const uint4 h = __ldg(reinterpret_cast<const uint4*>(hi)), l = __ldg(reinterpret_cast<const uint4*>(lo));
    const uint32_t hh[4] = {h.x, h.y, h.z, h.w}, ll[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float2 a = unpack_op(hh[i]), b = unpack_op(ll[i]);
        v[2 * i] = a.x + b.x;
        v[2 * i + 1] = a.y + b.y;
    }
}

// Device buffers of one fp32-class forward.  Scoring mode: the per-layer pointers alias one scratch set.  Save mode
// (the waveform backward follows): everything the backward reads gets its own storage -- the GroupNorm statistics, each
// conv level's pre-activation u[l] (fp32; its GELU derivative is recomputed from it), the projection output x0, the
// positional-conv pre-activation, and per layer the fp32 QKV rows, the attention output (hi + lo), its log-sum-exp,
// the two pre-LayerNorm sums and the fc1 pre-activation.
struct PWorkspace {
    UttMeta* meta;
    double* stat_part;
    float* c0_fold;
    op_t *y_hi[2], *y_lo[2];    // conv levels ping-pong: even levels in [0], odd levels in [1]
    op_t *ln0_hi, *ln0_lo;      // alias y[1] (level 6 lives in y[0])
    float *x0, *x;
    op_t *xh_hi, *xh_lo;
    op_t *posg_hi, *posg_lo;
    float* pos_y;
    op_t *ffn_hi, *ffn_lo;
    float* qkv[LAYERS];
    op_t *attn_hi[LAYERS], *attn_lo[LAYERS];
    float *pre1[LAYERS], *pre2[LAYERS];
    // save mode only (nullptr otherwise)
    float* gn_stat;             // [B][512][2] mean, rstd of the raw conv0 output
    float* u[7];                // level l: (rows0 >> l) x 512 pre-activations (level 0: GroupNorm-affine output)
    float* pos_pre;             // [pos_rows][768] positional conv + bias, before the GELU
    float* lse[LAYERS];         // frames x 12
    float* fc1_pre[LAYERS];     // frames x 3072
    size_t bytes;
};
size_t carve_precise(const Plan& p, void* base, PWorkspace* out, bool save);

// save-mode forward: layers_out (12 x B x layer_T x 768) may be null; the final residual stream is left in ws.x
int embed_precise_save(Handle* h, const Plan& p, void* saved, size_t saved_bytes, const float* wav, cudaStream_t st,
                       float* layers_out, int layer_T);

// Waveform backward of the first B_bwd utterances of a save-mode forward (precise_bwd.cu), the order of backward_chain
// in loss.cu.  Upstream gradients: seed_layer != 0 = the fused loss's L1 signs against utterances B_bwd.. (g_pool already
// scaled); otherwise g_layers (B x user_T x 768, caller layout) and g_pool, both times the S at scale_dev.  d_wav =
// result * out_scale, or / *scale_dev when scale_dev is non-null.
struct PBwdArgs {
    int B_bwd;
    const float* g_layers[LAYERS];
    int top;                    // highest layer that receives a gradient
    int user_T;
    const float* g_pool;
    const float* scale_dev;
    float seed_layer;
    float out_scale;
    float feature_grad_mult;
};
size_t precise_bwd_bytes(const Plan& p, int B_bwd);
int backward_precise(Handle* h, const Plan& p, void* saved, const PBwdArgs& a, const float* wav, int64_t N, float* d_wav,
                     void* workspace, size_t workspace_bytes, cudaStream_t st);

}  // namespace nb
