// Device-side rebuild of the kernel-ready weights from fp32 master tensors that already live on the GPU: the step after
// the optimiser update of the triplet fine-tuning loop (reference src/training/train_triplet.py:129-130, `optimizer.step()`).
// nomad_b200_create does the same preparation on the host from host tensors (api.cu: build_weights: fp16 conversion, q-scale,
// q/k/v fusion, transposes for the dgrad GEMMs, LayerNorm folds, weight-norm fold of the positional conv); repeating that per
// training step would cost seconds.  Here it is a handful of bandwidth-bound kernels (~190 MB of fp32 read, ~0.5 GB written).
// nomad_b200_refresh_weights rebuilds everything after the conv feature encoder, which the reference's default
// configuration freezes (`freeze_convnet: True`); with `freeze_convnet: False` nomad_b200_refresh_conv_weights rebuilds the
// encoder's buffers too.  The fp32-class weight planes (precision_mode 1) are not rebuilt: fine-tuning runs the fp16-operand
// path.
#include <cstdlib>
#include <cstring>
#include <string>
#include <unordered_map>

#include "../../include/nomad_b200.h"
#include "kernels.cuh"

namespace nb {

// src [R][C] fp32 (rows scaled by `scale` for r < scaled_rows) -> dst [R][C] fp16 (+ dst_off rows) and, if dst_t, dst_t [C][R_total]
__global__ void __launch_bounds__(256) rf_convert_kernel(const float* __restrict__ src, int R, int C, float scale, int scaled_rows,
                                                         op_t* __restrict__ dst, op_t* __restrict__ dst_t, int row_off, int R_total) {
    __shared__ float tile[32][33];
    const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
    for (int i = ty; i < 32; i += 8) {
        const int r = r0 + i, c = c0 + tx;
        float v = 0.f;
        if (r < R && c < C) {
            v = src[(long long)r * C + c] * (r < scaled_rows ? scale : 1.0f);
            dst[(long long)(row_off + r) * C + c] = f2op(v);
        }
        tile[i][tx] = v;
    }
    if (dst_t == nullptr) return;
    __syncthreads();
    for (int i = ty; i < 32; i += 8) {
        const int c = c0 + i, r = r0 + tx;
        if (r < R && c < C) dst_t[(long long)c * R_total + row_off + r] = f2op(tile[tx][i]);
    }
}
// LayerNorm fold (api.cu: upload_folded): Wf[n][k] = fp16(W[n][k] * sc * gamma[k]), s[n] = sum_k Wf[n][k] (of the ROUNDED values),
// c[n] = sum_k W[n][k] * sc * beta[k] + b[n] * sc; one warp per output row
__global__ void __launch_bounds__(256) rf_fold_kernel(const float* __restrict__ W, const float* __restrict__ b, int N, int K, float sc,
                                                      const float* __restrict__ gamma, const float* __restrict__ beta,
                                                      op_t* __restrict__ Wf, float* __restrict__ s, float* __restrict__ c, int row_off) {
    const int n = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (n >= N) return;
    double ss = 0.0, cs = 0.0;  // fp64 sums like the host build (api.cu: upload_folded), so both give the same fp32 vectors
    for (int k = lane; k < K; k += 32) {
        const float w = W[(long long)n * K + k];
        const op_t q = f2op(__fmul_rn(__fmul_rn(w, sc), gamma[k]));
        Wf[(long long)(row_off + n) * K + k] = q;
        ss += (double)op2f(q);
        cs += (double)w * (double)sc * (double)beta[k];
    }
    for (int o = 16; o > 0; o >>= 1) {
        ss += __shfl_xor_sync(0xffffffffu, ss, o);
        cs += __shfl_xor_sync(0xffffffffu, cs, o);
    }
    if (lane == 0) {
        s[row_off + n] = (float)ss;
        c[row_off + n] = (float)(cs + (double)b[n] * (double)sc);
    }
}
__global__ void rf_copy_scale_kernel(const float* __restrict__ src, int n, float scale, float* __restrict__ dst) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i < n) dst[i] = src[i] * scale;
}
// head: W [256][768] -> head_wt [768][256] fp32
__global__ void rf_transpose_f32_kernel(const float* __restrict__ src, int R, int C, float* __restrict__ dst) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i < R * C) dst[(long long)(i % C) * R + i / C] = src[i];
}
// positional conv: per-tap norms of weight_v over (out, in), then the two grouped layouts of w = g * v / ||v||
__global__ void __launch_bounds__(256) rf_pos_norm_kernel(const float* __restrict__ v, const float* __restrict__ g, double* __restrict__ scale) {
    const int k = blockIdx.x;  // tap
    double a = 0.0;
    for (int i = threadIdx.x; i < 768 * POS_GC; i += 256) {
        const double x = v[(long long)i * POS_K + k];
        a += x * x;
    }
    __shared__ double red[256];
    red[threadIdx.x] = a;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) scale[k] = (double)g[k] / sqrt(red[0]);
}
__global__ void __launch_bounds__(256) rf_pos_fold_kernel(const float* __restrict__ v, const double* __restrict__ scale,
                                                          op_t* __restrict__ fw, op_t* __restrict__ bw) {
    const long long i = (long long)blockIdx.x * 256 + threadIdx.x;  // index into v: ((g*48 + n)*48 + c)*128 + k
    if (i >= (long long)768 * POS_GC * POS_K) return;
    const int k = (int)(i % POS_K);
    const int c = (int)((i / POS_K) % POS_GC);
    const int on = (int)(i / ((long long)POS_K * POS_GC));  // g * 48 + n
    const int g = on / POS_GC, n = on % POS_GC;
    const op_t q = f2op((float)((double)v[i] * scale[k]));
    fw[(long long)on * (POS_K * POS_GC) + (long long)k * POS_GC + c] = q;
    bw[(long long)(g * POS_GC + c) * (POS_K * POS_GC) + (long long)(POS_K - 1 - k) * POS_GC + n] = q;
}

// conv layer with k taps: W (cout, cin, tap) fp32 -> conv_w [cout][tap * 512 + cin], conv_wt [tap][cin][cout] and, for
// k = 3, conv_wte [cin][tap 2: cout | tap 0: cout] (api.cu: build_weights)
__global__ void __launch_bounds__(256) rf_conv_kernel(const float* __restrict__ W, int k, op_t* __restrict__ fw,
                                                      op_t* __restrict__ bw, op_t* __restrict__ ew) {
    const long long i = (long long)blockIdx.x * 256 + threadIdx.x;
    if (i >= 512LL * 512 * k) return;
    const int j = (int)(i % k), c = (int)((i / k) % 512), o = (int)(i / (512LL * k));
    const op_t v = f2op(W[i]);
    fw[(long long)o * (k * 512) + j * 512 + c] = v;
    bw[((long long)j * 512 + c) * 512 + o] = v;
    if (ew != nullptr && j != 1) ew[(long long)c * 1024 + (j == 2 ? 0 : 512) + o] = v;
}
// conv0 taps w[c][j] -> conv0_wh [16][512] (rows 10..15 stay zero)
__global__ void rf_conv0_kernel(const float* __restrict__ W, op_t* __restrict__ wh) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i < 512 * 10) wh[(i % 10) * 512 + i / 10] = f2op(W[i]);
}

static int convert(cudaStream_t st, const float* src, int R, int C, float scale, int scaled_rows, op_t* dst, op_t* dst_t,
                   int row_off, int R_total) {
    dim3 grid((C + 31) / 32, (R + 31) / 32);
    rf_convert_kernel<<<grid, 256, 0, st>>>(src, R, C, scale, scaled_rows, dst, dst_t, row_off, R_total);
    NB_LAUNCHED();
    return 0;
}
static int copy_f32(cudaStream_t st, const float* src, int n, float scale, float* dst) {
    rf_copy_scale_kernel<<<(n + 255) / 256, 256, 0, st>>>(src, n, scale, dst);
    NB_LAUNCHED();
    return 0;
}

}  // namespace nb

using namespace nb;

extern "C" int nomad_b200_refresh_weights(nomad_b200_handle* hh, const nomad_b200_tensor* tensors_dev, int n_tensors, void* stream) {
    NB_CHECK(hh != nullptr && tensors_dev != nullptr && n_tensors > 0, "refresh_weights: bad arguments");
    Handle* h = &hh->h;
    NB_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    std::unordered_map<std::string, const nomad_b200_tensor*> map;
    for (int i = 0; i < n_tensors; ++i)
        if (tensors_dev[i].name && tensors_dev[i].data) map[tensors_dev[i].name] = &tensors_dev[i];
    auto get = [&](const std::string& name, long long numel) -> const float* {
        auto it = map.find(name);
        if (it == map.end()) { set_error("refresh_weights: missing tensor %s", name.c_str()); return nullptr; }
        if (it->second->numel != numel) { set_error("refresh_weights: tensor %s has %lld elements, expected %lld", name.c_str(), (long long)it->second->numel, numel); return nullptr; }
        return it->second->data;
    };
#define RGET(var, name, numel) const float* var = get(name, numel); if (!var) return 1;
    Weights& w = h->w;
    const std::string P = "ssl_model.";
    const float qs = 0.125f;
    RGET(l0g, P + "layer_norm.weight", 512); RGET(l0b, P + "layer_norm.bias", 512);
    NB_TRY(copy_f32(st, l0g, 512, 1.f, w.ln0_g)); NB_TRY(copy_f32(st, l0b, 512, 1.f, w.ln0_b));
    RGET(pw, P + "post_extract_proj.weight", 768LL * 512); RGET(pb, P + "post_extract_proj.bias", 768);
    NB_TRY(convert(st, pw, 768, 512, 1.f, 0, w.proj_w, w.proj_wt, 0, 768));
    NB_TRY(copy_f32(st, pb, 768, 1.f, w.proj_b));
    RGET(pv, P + "encoder.pos_conv.0.weight_v", 768LL * POS_GC * POS_K); RGET(pg, P + "encoder.pos_conv.0.weight_g", POS_K);
    RGET(pbias, P + "encoder.pos_conv.0.bias", 768);
    {
        double* scale = w.pos_scale_tmp;
        if (scale == nullptr) {
            void* d = nullptr;
            NB_CUDA(cudaMalloc(&d, sizeof(double) * POS_K));
            h->allocs.push_back(d);
            scale = w.pos_scale_tmp = (double*)d;
        }
        rf_pos_norm_kernel<<<POS_K, 256, 0, st>>>(pv, pg, scale);
        NB_LAUNCHED();
        const long long n = (long long)768 * POS_GC * POS_K;
        rf_pos_fold_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(pv, scale, w.pos_w, w.pos_wt);
        NB_LAUNCHED();
        NB_TRY(copy_f32(st, pbias, 768, 1.f, w.pos_b));
    }
    RGET(leg, P + "encoder.layer_norm.weight", 768); RGET(leb, P + "encoder.layer_norm.bias", 768);
    NB_TRY(copy_f32(st, leg, 768, 1.f, w.lne_g)); NB_TRY(copy_f32(st, leb, 768, 1.f, w.lne_b));
    const float *prev_g2 = nullptr, *prev_b2 = nullptr;
    for (int l = 0; l < LAYERS; ++l) {
        LayerWeights& L = w.layer[l];
        const std::string Q = P + "encoder.layers." + std::to_string(l) + ".";
        RGET(wq, Q + "self_attn.q_proj.weight", 768LL * 768); RGET(wk, Q + "self_attn.k_proj.weight", 768LL * 768);
        RGET(wv, Q + "self_attn.v_proj.weight", 768LL * 768);
        RGET(bq, Q + "self_attn.q_proj.bias", 768); RGET(bk, Q + "self_attn.k_proj.bias", 768); RGET(bv, Q + "self_attn.v_proj.bias", 768);
        RGET(wo, Q + "self_attn.out_proj.weight", 768LL * 768); RGET(bo, Q + "self_attn.out_proj.bias", 768);
        RGET(w1, Q + "fc1.weight", 3072LL * 768); RGET(b1, Q + "fc1.bias", 3072);
        RGET(w2, Q + "fc2.weight", 768LL * 3072); RGET(b2, Q + "fc2.bias", 768);
        RGET(g1, Q + "self_attn_layer_norm.weight", 768); RGET(e1, Q + "self_attn_layer_norm.bias", 768);
        RGET(g2, Q + "final_layer_norm.weight", 768); RGET(e2, Q + "final_layer_norm.bias", 768);
        // fused q|k|v (q rows carry head_dim^-0.5) + the transposed copy [768][2304] for the dgrad GEMM
        NB_TRY(convert(st, wq, 768, 768, qs, 768, L.w_qkv, L.wt_qkv, 0, 2304));
        NB_TRY(convert(st, wk, 768, 768, 1.f, 0, L.w_qkv, L.wt_qkv, 768, 2304));
        NB_TRY(convert(st, wv, 768, 768, 1.f, 0, L.w_qkv, L.wt_qkv, 1536, 2304));
        NB_TRY(copy_f32(st, bq, 768, qs, L.b_qkv)); NB_TRY(copy_f32(st, bk, 768, 1.f, L.b_qkv + 768));
        NB_TRY(copy_f32(st, bv, 768, 1.f, L.b_qkv + 1536));
        NB_TRY(convert(st, wo, 768, 768, 1.f, 0, L.w_o, L.wt_o, 0, 768));
        NB_TRY(convert(st, w1, 3072, 768, 1.f, 0, L.w_fc1, L.wt_fc1, 0, 3072));
        NB_TRY(convert(st, w2, 768, 3072, 1.f, 0, L.w_fc2, L.wt_fc2, 0, 768));
        NB_TRY(copy_f32(st, bo, 768, 1.f, L.b_o)); NB_TRY(copy_f32(st, b1, 3072, 1.f, L.b_fc1)); NB_TRY(copy_f32(st, b2, 768, 1.f, L.b_fc2));
        NB_TRY(copy_f32(st, g1, 768, 1.f, L.ln1_g)); NB_TRY(copy_f32(st, e1, 768, 1.f, L.ln1_b));
        NB_TRY(copy_f32(st, g2, 768, 1.f, L.ln2_g)); NB_TRY(copy_f32(st, e2, 768, 1.f, L.ln2_b));
        // LayerNorm folds of the scoring path: FC1 with this layer's self_attn_layer_norm, QKV with the previous final_layer_norm
        rf_fold_kernel<<<(3072 + 7) / 8, 256, 0, st>>>(w1, b1, 3072, 768, 1.f, g1, e1, L.w_fc1_f, L.s_fc1, L.c_fc1, 0);
        NB_LAUNCHED();
        if (l > 0) {
            rf_fold_kernel<<<96, 256, 0, st>>>(wq, bq, 768, 768, qs, prev_g2, prev_b2, L.w_qkv_f, L.s_qkv, L.c_qkv, 0);
            NB_LAUNCHED();
            rf_fold_kernel<<<96, 256, 0, st>>>(wk, bk, 768, 768, 1.f, prev_g2, prev_b2, L.w_qkv_f, L.s_qkv, L.c_qkv, 768);
            NB_LAUNCHED();
            rf_fold_kernel<<<96, 256, 0, st>>>(wv, bv, 768, 768, 1.f, prev_g2, prev_b2, L.w_qkv_f, L.s_qkv, L.c_qkv, 1536);
            NB_LAUNCHED();
        }
        prev_g2 = g2;
        prev_b2 = e2;
    }
    RGET(hw, "embedding_layer.1.weight", 256LL * 768); RGET(hb, "embedding_layer.1.bias", 256);
    rf_transpose_f32_kernel<<<(256 * 768 + 255) / 256, 256, 0, st>>>(hw, 256, 768, w.head_wt);
    NB_LAUNCHED();
    NB_TRY(copy_f32(st, hb, 256, 1.f, w.head_b));
#undef RGET
    NB_CHECK(!h->pw.built || h->precision == NOMAD_B200_PRECISION_FP16,
             "refresh_weights: the fp32-class weight planes are not rebuilt; switch the handle to precision_mode 0 for fine-tuning");
    return 0;
}

extern "C" int nomad_b200_refresh_conv_weights(nomad_b200_handle* hh, const nomad_b200_tensor* tensors_dev, int n_tensors,
                                               void* stream) {
    NB_CHECK(hh != nullptr && tensors_dev != nullptr && n_tensors > 0, "refresh_conv_weights: bad arguments");
    Handle* h = &hh->h;
    NB_CHECK(!h->pw.built || h->precision == NOMAD_B200_PRECISION_FP16,
             "refresh_conv_weights: the fp32-class weight planes are not rebuilt; switch the handle to precision_mode 0 for fine-tuning");
    NB_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    std::unordered_map<std::string, const nomad_b200_tensor*> map;
    for (int i = 0; i < n_tensors; ++i)
        if (tensors_dev[i].name && tensors_dev[i].data) map[tensors_dev[i].name] = &tensors_dev[i];
    const std::string P = "ssl_model.feature_extractor.conv_layers.";
    const float* src[9];
    const char* leaf[3] = {"0.0.weight", "0.2.weight", "0.2.bias"};
    for (int i = 0; i < 9; ++i) {
        const std::string name = i < 3 ? P + leaf[i] : P + std::to_string(i - 2) + ".0.weight";
        const long long numel = i == 0 ? 512 * 10 : i < 3 ? 512 : 512LL * 512 * CONV_KERNEL[i - 2];
        auto it = map.find(name);
        NB_CHECK(it != map.end(), "refresh_conv_weights: missing tensor %s", name.c_str());
        NB_CHECK(it->second->numel == numel, "refresh_conv_weights: tensor %s has %lld elements, expected %lld", name.c_str(),
                 (long long)it->second->numel, numel);
        src[i] = it->second->data;
    }
    Weights& w = h->w;
    NB_TRY(copy_f32(st, src[0], 512 * 10, 1.f, w.conv0_w));
    NB_TRY(copy_f32(st, src[1], 512, 1.f, w.gn_g));
    NB_TRY(copy_f32(st, src[2], 512, 1.f, w.gn_b));
    rf_conv0_kernel<<<(512 * 10 + 255) / 256, 256, 0, st>>>(src[0], w.conv0_wh);
    NB_LAUNCHED();
    for (int l = 1; l < 7; ++l) {
        const int k = CONV_KERNEL[l];
        rf_conv_kernel<<<(unsigned)((512LL * 512 * k + 255) / 256), 256, 0, st>>>(src[l + 2], k, w.conv_w[l], w.conv_wt[l],
                                                                                  k == 3 ? w.conv_wte[l] : nullptr);
        NB_LAUNCHED();
    }
    return 0;
}

// Test hook: copy one kernel-ready weight buffer to the host (synchronous).  which: "pos_w" | "pos_wt" | "l<k>.w_fc1_f" |
// "l<k>.s_fc1" | "l<k>.c_fc1" | "l<k>.w_qkv_f" | "l<k>.s_qkv" | "l<k>.c_qkv" | "l<k>.w_qkv" | "l<k>.wt_fc2" | "head_wt" |
// conv encoder: "conv0_w" | "gn_g" | "gn_b" | "conv0_wh" | "c<l>.w" | "c<l>.wt" | "c<l>.wte" (l = 1..6; wte for k = 3)
extern "C" int nomad_b200_debug_read_weight(nomad_b200_handle* hh, const char* which, void* dst_host, size_t bytes) {
    NB_CHECK(hh && which && dst_host, "debug_read_weight: bad arguments");
    Weights& w = hh->h.w;
    const void* src = nullptr;
    std::string s(which);
    if (s == "pos_w") src = w.pos_w;
    else if (s == "pos_wt") src = w.pos_wt;
    else if (s == "head_wt") src = w.head_wt;
    else if (s == "conv0_w") src = w.conv0_w;
    else if (s == "gn_g") src = w.gn_g;
    else if (s == "gn_b") src = w.gn_b;
    else if (s == "conv0_wh") src = w.conv0_wh;
    else if (s.size() > 2 && s[0] == 'c' && s[1] >= '1' && s[1] <= '6' && s[2] == '.') {
        const int l = s[1] - '0';
        const std::string f = s.substr(3);
        if (f == "w") src = w.conv_w[l]; else if (f == "wt") src = w.conv_wt[l]; else if (f == "wte") src = w.conv_wte[l];
    }
    else if (s.size() > 2 && s[0] == 'l') {
        const size_t dot = s.find('.');
        NB_CHECK(dot != std::string::npos, "debug_read_weight: bad name %s", which);
        const int l = atoi(s.substr(1, dot - 1).c_str());
        NB_CHECK(l >= 0 && l < LAYERS, "debug_read_weight: bad layer in %s", which);
        const std::string f = s.substr(dot + 1);
        LayerWeights& L = w.layer[l];
        if (f == "w_fc1_f") src = L.w_fc1_f; else if (f == "s_fc1") src = L.s_fc1; else if (f == "c_fc1") src = L.c_fc1;
        else if (f == "w_qkv_f") src = L.w_qkv_f; else if (f == "s_qkv") src = L.s_qkv; else if (f == "c_qkv") src = L.c_qkv;
        else if (f == "w_qkv") src = L.w_qkv; else if (f == "wt_fc2") src = L.wt_fc2;
    }
    NB_CHECK(src != nullptr, "debug_read_weight: unknown buffer %s", which);
    NB_CUDA(cudaDeviceSynchronize());
    NB_CUDA(cudaMemcpy(dst_host, src, bytes, cudaMemcpyDeviceToHost));
    return 0;
}
