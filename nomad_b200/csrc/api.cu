// Handle, weight preparation, batch planning and the forward pass behind the C ABI.
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <string>
#include <unordered_map>

#include "../../include/nomad_b200.h"
#include "kernels.cuh"

namespace nb {

// ================================================================================================
// Plan
static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

int make_plan(const int64_t* off, int B, Plan* p) {
    NB_CHECK(off != nullptr && B > 0, "embed: need B > 0 utterances and their sample offsets");
    p->B = B;
    p->utt.resize(B);
    long long row = 0;
    int max_T0 = 0;
    p->max_T = 0;
    p->uniform = true;
    for (int b = 0; b < B; ++b) {
        const long long n = off[b + 1] - off[b];
        NB_CHECK(n >= NOMAD_B200_MIN_SAMPLES,
                 "utterance %d has %lld samples; the conv feature encoder needs at least %d (kernel size can't be "
                 "greater than actual input size)", b, n, NOMAD_B200_MIN_SAMPLES);
        NB_CHECK(n < (1LL << 30), "utterance %d is too long (%lld samples)", b, n);
        long long t = n;
        int T[7];
        for (int l = 0; l < 7; ++l) {
            t = (t - CONV_KERNEL[l]) / CONV_STRIDE[l] + 1;
            T[l] = (int)t;
        }
        UttMeta& m = p->utt[b];
        m.wav_off = off[b];
        m.n = (int)n;
        m.T0 = T[0];
        m.rows0 = (T[0] + 63) / 64 * 64;
        NB_CHECK(row + m.rows0 < (1LL << 31) - 4096, "batch too large: more than 2^31 conv0 rows; split the batch");
        m.row0 = (int)row;
        m.T = T[6];
        m.frame0 = m.row0 / 64;
        m.frames = m.rows0 / 64;
        m.pos0 = m.frame0 + POS_GAP * b + POS_K / 2;
        NB_CHECK(m.T >= 1 && m.T <= m.frames, "internal: frame bookkeeping (T=%d frames=%d)", m.T, m.frames);
        row += m.rows0;
        if (T[0] > max_T0) max_T0 = T[0];
        if (m.T > p->max_T) p->max_T = m.T;
        if (n != off[1] - off[0]) p->uniform = false;
    }
    p->total_samples = off[B] - off[0];
    p->rows0 = row;
    p->frames = row / 64;
    p->pos_rows = p->frames + (long long)POS_GAP * B + POS_K / 2;
    p->max_chunks = (max_T0 + STAT_CHUNK - 1) / STAT_CHUNK;
    build_attention_items(*p, &p->attn_items);
    return 0;
}

size_t carve_workspace(const Plan& p, void* base, Workspace* ws, bool save, bool train) {
    size_t o = 0;
    auto take = [&](size_t bytes) {
        size_t at = o;
        o = align_up(o + bytes, 1024);
        return base ? (void*)((char*)base + at) : nullptr;
    };
    Workspace w;
    memset(&w, 0, sizeof(w));
    w.save = save;
    w.train = train;
    const size_t F = (size_t)p.frames;
    w.meta = (UttMeta*)take(sizeof(UttMeta) * p.B);
    w.attn_items = (uint32_t*)take(sizeof(uint32_t) * p.attn_items.size());
    w.stat_part = (double*)take(sizeof(double) * NSTAT * p.max_chunks * p.B);
    w.c0_fold = (float*)take(sizeof(float) * 12 * CONV_DIM * p.B);
    w.c0_fold_h = (op_t*)take(2ull * 32 * CONV_DIM * p.B);
    w.gn_stat = save ? (float*)take(sizeof(float) * 2 * CONV_DIM * p.B) : nullptr;
    if (!save) {
        op_t* act_a = (op_t*)take(2ull * CONV_DIM * (p.rows0 + 8));
        op_t* act_b = (op_t*)take(2ull * CONV_DIM * (p.rows0 / 2 + 8));
        for (int l = 0; l < 7; ++l) {
            w.y[l] = (l & 1) ? act_b : act_a;
            w.aux[l] = nullptr;
        }
        w.ln0_out = act_b;  // level 6 lives in act_a
    } else {
        for (int l = 0; l < 7; ++l) {
            w.y[l] = (op_t*)take(2ull * CONV_DIM * ((p.rows0 >> l) + 8));
            w.aux[l] = (op_t*)take(2ull * CONV_DIM * ((p.rows0 >> l) + 8));
        }
        w.ln0_out = (op_t*)take(2ull * CONV_DIM * (F + 8));
    }
    w.ln_stats = (float*)take(4ull * 2 * 2 * F);  // two alternating slots
    w.ln_part = save ? nullptr : (float*)take(sizeof(float) * 2 * 2 * LN_PARTS * F);
    w.x = (float*)take(4ull * EMBED * F);
    w.xh = (op_t*)take(2ull * EMBED * F);
    w.pos_g = (op_t*)take(2ull * POS_G * POS_GC * (p.pos_rows + POS_K));
    w.pos_y = (op_t*)take(2ull * EMBED * p.pos_rows);
    w.pos_aux = save ? (op_t*)take(2ull * EMBED * p.pos_rows) : nullptr;
    w.ffn_h = (op_t*)take(2ull * FFN * F);
    if (!save) {
        float* pre = (float*)take(4ull * EMBED * F);
        op_t* qkv = (op_t*)take(2ull * 3 * EMBED * F);
        op_t* attn = (op_t*)take(2ull * EMBED * F);
        w.x0 = pre;
        for (int l = 0; l < LAYERS; ++l) w.layer[l] = LayerBufs{qkv, attn, nullptr, pre, nullptr, pre, nullptr};
    } else {
        w.x0 = (float*)take(4ull * EMBED * F);
        for (int l = 0; l < LAYERS; ++l) {
            LayerBufs& L = w.layer[l];
            L.qkv = (op_t*)take(2ull * 3 * EMBED * F);
            L.attn = (op_t*)take(2ull * EMBED * F);
            L.lse = (float*)take(4ull * HEADS * F);
            L.pre1 = (float*)take(4ull * EMBED * F);
            L.ffn_aux = (op_t*)take(2ull * FFN * F);
            L.pre2 = (float*)take(4ull * EMBED * F);
            L.ffn_h = train ? (op_t*)take(2ull * FFN * F) : nullptr;
        }
    }
    w.bytes = o;
    if (ws) *ws = w;
    return o;
}

// ================================================================================================
// Weights
struct TensorTable {
    std::unordered_map<std::string, const nomad_b200_tensor*> map;
    const float* get(const std::string& name, int64_t numel) {
        auto it = map.find(name);
        if (it == map.end()) {
            set_error("checkpoint is missing tensor %s", name.c_str());
            return nullptr;
        }
        if (it->second->numel != numel) {
            set_error("checkpoint tensor %s has %lld elements, expected %lld", name.c_str(),
                      (long long)it->second->numel, (long long)numel);
            return nullptr;
        }
        return it->second->data;
    }
};

template <typename T>
static int upload(Handle* h, const std::vector<T>& host, T** dev) {
    void* d = nullptr;
    NB_CUDA(cudaMalloc(&d, host.size() * sizeof(T)));
    h->allocs.push_back(d);
    NB_CUDA(cudaMemcpy(d, host.data(), host.size() * sizeof(T), cudaMemcpyHostToDevice));
    *dev = (T*)d;
    return 0;
}
static int upload_f32(Handle* h, const float* src, size_t n, float** dev) {
    std::vector<float> v(src, src + n);
    return upload(h, v, dev);
}
static std::vector<op_t> to_op(const float* src, size_t n, float scale = 1.0f) {
    std::vector<op_t> v(n);
    for (size_t i = 0; i < n; ++i) v[i] = f2op(src[i] * scale);
    return v;
}
// [rows][cols] -> op_t [cols][rows]
static std::vector<op_t> transpose_op(const std::vector<op_t>& src, size_t rows, size_t cols) {
    std::vector<op_t> v(src.size());
    for (size_t r = 0; r < rows; ++r)
        for (size_t c = 0; c < cols; ++c) v[c * rows + r] = src[r * cols + c];
    return v;
}

// LayerNorm folded into the consuming Linear (EPI_LN_FOLD): W' = W diag(gamma) as op_t, s[n] = sum_k W'[n][k] of
// the ROUNDED values (what the tensor core multiplies), c[n] = sum_k W[n][k] beta[k] + bias[n].  `scale` is applied
// to rows [0, scaled_rows) (the q rows of the fused QKV weight carry head_dim^-0.5).
static int upload_folded(Handle* h, const float* const* w_parts, const float* const* b_parts, int n_parts, int rows_per_part,
                         int K, const float* gamma, const float* beta, float scale0, op_t** w_f, float** s_out,
                         float** c_out) {
    const int N = n_parts * rows_per_part;
    std::vector<op_t> wf((size_t)N * K);
    std::vector<float> sv(N), cv(N);
    for (int part = 0; part < n_parts; ++part) {
        const float sc = part == 0 ? scale0 : 1.0f;
        for (int r = 0; r < rows_per_part; ++r) {
            const float* wr = w_parts[part] + (size_t)r * K;
            const size_t n = (size_t)part * rows_per_part + r;
            double ssum = 0.0, csum = 0.0;
            for (int k = 0; k < K; ++k) {
                const op_t q = f2op(wr[k] * sc * gamma[k]);
                wf[n * K + k] = q;
                ssum += (double)op2f(q);
                csum += (double)wr[k] * sc * (double)beta[k];
            }
            sv[n] = (float)ssum;
            cv[n] = (float)(csum + (double)b_parts[part][r] * sc);
        }
    }
    NB_TRY(upload(h, wf, w_f));
    NB_TRY(upload(h, sv, s_out));
    NB_TRY(upload(h, cv, c_out));
    return 0;
}

#define GET(var, name, numel)                         \
    const float* var = tt.get(name, numel);           \
    if (!var) return 1;

static int build_weights(Handle* h, TensorTable& tt) {
    Weights& w = h->w;
    const std::string P = "ssl_model.";
    // --- conv feature encoder
    GET(c0, P + "feature_extractor.conv_layers.0.0.weight", 512 * 10);
    NB_TRY(upload_f32(h, c0, 512 * 10, &w.conv0_w));
    GET(gng, P + "feature_extractor.conv_layers.0.2.weight", 512);
    GET(gnb, P + "feature_extractor.conv_layers.0.2.bias", 512);
    NB_TRY(upload_f32(h, gng, 512, &w.gn_g));
    NB_TRY(upload_f32(h, gnb, 512, &w.gn_b));
    w.conv_w[0] = nullptr;
    w.conv_wt[0] = nullptr;
    for (int l = 0; l < 7; ++l) w.conv_wte[l] = nullptr;
    {
        std::vector<op_t> t((size_t)16 * 512, f2op(0.f));
        for (int c = 0; c < 512; ++c)
            for (int j = 0; j < 10; ++j) t[(size_t)j * 512 + c] = f2op(c0[c * 10 + j]);
        NB_TRY(upload(h, t, &w.conv0_wh));
    }
    for (int l = 1; l < 7; ++l) {
        const int k = CONV_KERNEL[l];
        GET(cw, P + "feature_extractor.conv_layers." + std::to_string(l) + ".0.weight", 512LL * 512 * k);
        // (cout, cin, tap) -> [cout][tap * 512 + cin]
        std::vector<op_t> fw((size_t)512 * 512 * k), bw((size_t)512 * 512 * k);
        for (int o = 0; o < 512; ++o)
            for (int c = 0; c < 512; ++c)
                for (int j = 0; j < k; ++j) {
                    const op_t v = f2op(cw[((size_t)o * 512 + c) * k + j]);
                    fw[(size_t)o * (k * 512) + (size_t)j * 512 + c] = v;
                    bw[((size_t)j * 512 + c) * 512 + o] = v;  // dgrad: per tap [cin][cout]
                }
        NB_TRY(upload(h, fw, &w.conv_w[l]));
        NB_TRY(upload(h, bw, &w.conv_wt[l]));
        if (k == 3) {
            std::vector<op_t> ew((size_t)512 * 1024);
            for (int c = 0; c < 512; ++c)
                for (int o = 0; o < 512; ++o) {
                    ew[(size_t)c * 1024 + o] = f2op(cw[((size_t)o * 512 + c) * 3 + 2]);
                    ew[(size_t)c * 1024 + 512 + o] = f2op(cw[((size_t)o * 512 + c) * 3 + 0]);
                }
            NB_TRY(upload(h, ew, &w.conv_wte[l]));
        }
    }
    GET(l0g, P + "layer_norm.weight", 512);
    GET(l0b, P + "layer_norm.bias", 512);
    NB_TRY(upload_f32(h, l0g, 512, &w.ln0_g));
    NB_TRY(upload_f32(h, l0b, 512, &w.ln0_b));
    GET(pw, P + "post_extract_proj.weight", 768LL * 512);
    GET(pb, P + "post_extract_proj.bias", 768);
    {
        std::vector<op_t> v = to_op(pw, 768 * 512);
        NB_TRY(upload(h, v, &w.proj_w));
        std::vector<op_t> vt = transpose_op(v, 768, 512);
        NB_TRY(upload(h, vt, &w.proj_wt));
    }
    NB_TRY(upload_f32(h, pb, 768, &w.proj_b));
    // --- positional conv: fold weight_norm(dim=2): w = g * v / ||v||, norm over (out, in) per tap
    GET(pv, P + "encoder.pos_conv.0.weight_v", 768LL * POS_GC * POS_K);
    GET(pg, P + "encoder.pos_conv.0.weight_g", POS_K);
    GET(pbias, P + "encoder.pos_conv.0.bias", 768);
    {
        std::vector<double> nrm(POS_K, 0.0);
        for (size_t i = 0; i < (size_t)768 * POS_GC; ++i)
            for (int k = 0; k < POS_K; ++k) {
                const double v = pv[i * POS_K + k];
                nrm[k] += v * v;
            }
        for (int k = 0; k < POS_K; ++k) nrm[k] = (double)pg[k] / std::sqrt(nrm[k]);
        // forward: [g][n][tap * 48 + c] = w[g*48+n][c][tap]
        // dgrad:   [g][c][tap' * 48 + n] = w[g*48+n][c][127 - tap']  (correlation with the flipped kernel)
        std::vector<op_t> fw((size_t)POS_G * POS_GC * POS_K * POS_GC), bw(fw.size());
        for (int g = 0; g < POS_G; ++g)
            for (int n = 0; n < POS_GC; ++n)
                for (int c = 0; c < POS_GC; ++c)
                    for (int k = 0; k < POS_K; ++k) {
                        const float val = (float)((double)pv[((size_t)(g * POS_GC + n) * POS_GC + c) * POS_K + k] * nrm[k]);
                        const op_t v = f2op(val);
                        fw[((size_t)(g * POS_GC + n)) * (POS_K * POS_GC) + (size_t)k * POS_GC + c] = v;
                        bw[((size_t)(g * POS_GC + c)) * (POS_K * POS_GC) + (size_t)(POS_K - 1 - k) * POS_GC + n] = v;
                    }
        NB_TRY(upload(h, fw, &w.pos_w));
        NB_TRY(upload(h, bw, &w.pos_wt));
    }
    NB_TRY(upload_f32(h, pbias, 768, &w.pos_b));
    GET(leg, P + "encoder.layer_norm.weight", 768);
    GET(leb, P + "encoder.layer_norm.bias", 768);
    NB_TRY(upload_f32(h, leg, 768, &w.lne_g));
    NB_TRY(upload_f32(h, leb, 768, &w.lne_b));
    // --- transformer layers
    for (int l = 0; l < LAYERS; ++l) {
        LayerWeights& L = w.layer[l];
        const std::string Q = P + "encoder.layers." + std::to_string(l) + ".";
        GET(wq, Q + "self_attn.q_proj.weight", 768LL * 768);
        GET(wk, Q + "self_attn.k_proj.weight", 768LL * 768);
        GET(wv, Q + "self_attn.v_proj.weight", 768LL * 768);
        GET(bq, Q + "self_attn.q_proj.bias", 768);
        GET(bk, Q + "self_attn.k_proj.bias", 768);
        GET(bv, Q + "self_attn.v_proj.bias", 768);
        const float qs = 0.125f;  // head_dim^-0.5, exact in op_t
        {
            std::vector<op_t> v((size_t)2304 * 768);
            for (size_t i = 0; i < (size_t)768 * 768; ++i) {
                v[i] = f2op(wq[i] * qs);
                v[(size_t)768 * 768 + i] = f2op(wk[i]);
                v[(size_t)2 * 768 * 768 + i] = f2op(wv[i]);
            }
            NB_TRY(upload(h, v, &L.w_qkv));
            std::vector<op_t> vt = transpose_op(v, 2304, 768);
            NB_TRY(upload(h, vt, &L.wt_qkv));
            std::vector<float> bb(2304);
            for (int i = 0; i < 768; ++i) { bb[i] = bq[i] * qs; bb[768 + i] = bk[i]; bb[1536 + i] = bv[i]; }
            NB_TRY(upload(h, bb, &L.b_qkv));
        }
        GET(wo, Q + "self_attn.out_proj.weight", 768LL * 768);
        GET(bo, Q + "self_attn.out_proj.bias", 768);
        GET(w1, Q + "fc1.weight", 3072LL * 768);
        GET(b1, Q + "fc1.bias", 3072);
        GET(w2, Q + "fc2.weight", 768LL * 3072);
        GET(b2, Q + "fc2.bias", 768);
        {
            std::vector<op_t> v = to_op(wo, 768 * 768);
            NB_TRY(upload(h, v, &L.w_o));
            std::vector<op_t> vt = transpose_op(v, 768, 768);
            NB_TRY(upload(h, vt, &L.wt_o));
            v = to_op(w1, (size_t)3072 * 768);
            NB_TRY(upload(h, v, &L.w_fc1));
            vt = transpose_op(v, 3072, 768);
            NB_TRY(upload(h, vt, &L.wt_fc1));
            v = to_op(w2, (size_t)768 * 3072);
            NB_TRY(upload(h, v, &L.w_fc2));
            vt = transpose_op(v, 768, 3072);
            NB_TRY(upload(h, vt, &L.wt_fc2));
        }
        NB_TRY(upload_f32(h, bo, 768, &L.b_o));
        NB_TRY(upload_f32(h, b1, 3072, &L.b_fc1));
        NB_TRY(upload_f32(h, b2, 768, &L.b_fc2));
        GET(g1, Q + "self_attn_layer_norm.weight", 768);
        GET(e1, Q + "self_attn_layer_norm.bias", 768);
        GET(g2, Q + "final_layer_norm.weight", 768);
        GET(e2, Q + "final_layer_norm.bias", 768);
        NB_TRY(upload_f32(h, g1, 768, &L.ln1_g));
        NB_TRY(upload_f32(h, e1, 768, &L.ln1_b));
        NB_TRY(upload_f32(h, g2, 768, &L.ln2_g));
        NB_TRY(upload_f32(h, e2, 768, &L.ln2_b));
        {
            const float* wp[1] = {w1};
            const float* bp[1] = {b1};
            NB_TRY(upload_folded(h, wp, bp, 1, 3072, 768, g1, e1, 1.0f, &L.w_fc1_f, &L.s_fc1, &L.c_fc1));
        }
        L.w_qkv_f = nullptr;
        L.s_qkv = L.c_qkv = nullptr;
        if (l > 0) {  // this layer's QKV reads the previous layer's final_layer_norm
            const std::string Qp = P + "encoder.layers." + std::to_string(l - 1) + ".";
            GET(pg2, Qp + "final_layer_norm.weight", 768);
            GET(pe2, Qp + "final_layer_norm.bias", 768);
            const float* wp[3] = {wq, wk, wv};
            const float* bp[3] = {bq, bk, bv};
            NB_TRY(upload_folded(h, wp, bp, 3, 768, 768, pg2, pe2, qs, &L.w_qkv_f, &L.s_qkv, &L.c_qkv));
        }
    }
    // --- scoring head (nomad.py:219-222): Linear(768, 256) stored transposed for coalesced GEMV
    GET(hw, "embedding_layer.1.weight", 256LL * 768);
    GET(hb, "embedding_layer.1.bias", 256);
    {
        std::vector<float> t((size_t)768 * 256);
        for (int o = 0; o < 256; ++o)
            for (int k = 0; k < 768; ++k) t[(size_t)k * 256 + o] = hw[(size_t)o * 768 + k];
        NB_TRY(upload(h, t, &w.head_wt));
    }
    NB_TRY(upload_f32(h, hb, 256, &w.head_b));
    w.loss_head_wt = nullptr;
    w.loss_head_w = nullptr;
    w.loss_head_b = nullptr;
    w.pos_scale_tmp = nullptr;
    return 0;
}

// fp32-class mode: every GEMM weight as hi + lo planes of w * 2^k (see precise.cu)
static int upload_split(Handle* h, const std::vector<float>& w, SplitW* out) {
    float mx = 0.f;
    for (float v : w) mx = std::fmax(mx, std::fabs(v));
    int k = 0;
    if (mx > 0.f) k = (int)std::floor(std::log2(16000.0f / mx));
    k = k < -24 ? -24 : (k > 24 ? 24 : k);
    const float sc = std::ldexp(1.0f, k);
    std::vector<op_t> hi(w.size()), lo(w.size());
    for (size_t i = 0; i < w.size(); ++i) {
        const float v = w[i] * sc;
        hi[i] = f2op(v);
        lo[i] = f2op(v - op2f(hi[i]));
    }
    NB_TRY(upload(h, hi, &out->hi));
    NB_TRY(upload(h, lo, &out->lo));
    out->inv_scale = std::ldexp(1.0f, -k);
    return 0;
}

static std::vector<float> transpose_f32(const float* w, size_t rows, size_t cols) {
    std::vector<float> t(rows * cols);
    for (size_t r = 0; r < rows; ++r)
        for (size_t c = 0; c < cols; ++c) t[c * rows + r] = w[r * cols + c];
    return t;
}

// The transposed planes (the *_t members, for the dgrad GEMMs of the fp32-class waveform backward) take as much device
// memory as the forward planes: ~0.38 GB more per FP32 handle.  Their max |w| and so their power-of-two scale equal the
// forward tensor's, so the hi / lo values are the forward planes' values, transposed.
static int build_weights_precise(Handle* h, TensorTable& tt) {
    PreciseWeights& pw = h->pw;
    const std::string P = "ssl_model.";
    for (int l = 1; l < 7; ++l) {
        const int k = CONV_KERNEL[l];
        GET(cw, P + "feature_extractor.conv_layers." + std::to_string(l) + ".0.weight", 512LL * 512 * k);
        std::vector<float> fw((size_t)512 * 512 * k);  // (cout, cin, tap) -> [cout][tap * 512 + cin]
        for (int o = 0; o < 512; ++o)
            for (int c = 0; c < 512; ++c)
                for (int j = 0; j < k; ++j) fw[(size_t)o * (k * 512) + (size_t)j * 512 + c] = cw[((size_t)o * 512 + c) * k + j];
        NB_TRY(upload_split(h, fw, &pw.conv[l]));
        std::vector<float> bw((size_t)512 * 512 * k);  // dgrad: per tap [cin][cout]
        for (int o = 0; o < 512; ++o)
            for (int c = 0; c < 512; ++c)
                for (int j = 0; j < k; ++j) bw[((size_t)j * 512 + c) * 512 + o] = cw[((size_t)o * 512 + c) * k + j];
        NB_TRY(upload_split(h, bw, &pw.conv_t[l]));
        if (k == 3) {  // even input rows: [cin][tap 2: cout | tap 0: cout]
            std::vector<float> ew((size_t)512 * 1024);
            for (int c = 0; c < 512; ++c)
                for (int o = 0; o < 512; ++o) {
                    ew[(size_t)c * 1024 + o] = cw[((size_t)o * 512 + c) * 3 + 2];
                    ew[(size_t)c * 1024 + 512 + o] = cw[((size_t)o * 512 + c) * 3 + 0];
                }
            NB_TRY(upload_split(h, ew, &pw.conv_te[l]));
        }
    }
    GET(pwt, P + "post_extract_proj.weight", 768LL * 512);
    NB_TRY(upload_split(h, std::vector<float>(pwt, pwt + 768 * 512), &pw.proj));
    NB_TRY(upload_split(h, transpose_f32(pwt, 768, 512), &pw.proj_t));
    GET(pv, P + "encoder.pos_conv.0.weight_v", 768LL * POS_GC * POS_K);
    GET(pg, P + "encoder.pos_conv.0.weight_g", POS_K);
    {
        std::vector<double> nrm(POS_K, 0.0);
        for (size_t i = 0; i < (size_t)768 * POS_GC; ++i)
            for (int k = 0; k < POS_K; ++k) nrm[k] += (double)pv[i * POS_K + k] * pv[i * POS_K + k];
        for (int k = 0; k < POS_K; ++k) nrm[k] = (double)pg[k] / std::sqrt(nrm[k]);
        // forward [g][n][tap * 48 + c]; dgrad [g][c][tap' * 48 + n] with tap' = 127 - tap (as Weights::pos_wt)
        std::vector<float> fw((size_t)POS_G * POS_GC * POS_K * POS_GC), bw(fw.size());
        for (int g = 0; g < POS_G; ++g)
            for (int n = 0; n < POS_GC; ++n)
                for (int c = 0; c < POS_GC; ++c)
                    for (int k = 0; k < POS_K; ++k) {
                        const float v = (float)((double)pv[((size_t)(g * POS_GC + n) * POS_GC + c) * POS_K + k] * nrm[k]);
                        fw[((size_t)(g * POS_GC + n)) * (POS_K * POS_GC) + (size_t)k * POS_GC + c] = v;
                        bw[((size_t)(g * POS_GC + c)) * (POS_K * POS_GC) + (size_t)(POS_K - 1 - k) * POS_GC + n] = v;
                    }
        NB_TRY(upload_split(h, fw, &pw.pos));
        NB_TRY(upload_split(h, bw, &pw.pos_t));
    }
    for (int l = 0; l < LAYERS; ++l) {
        const std::string Q = P + "encoder.layers." + std::to_string(l) + ".";
        GET(wq, Q + "self_attn.q_proj.weight", 768LL * 768);
        GET(wk, Q + "self_attn.k_proj.weight", 768LL * 768);
        GET(wv, Q + "self_attn.v_proj.weight", 768LL * 768);
        std::vector<float> v((size_t)2304 * 768);
        for (size_t i = 0; i < (size_t)768 * 768; ++i) {
            v[i] = wq[i] * 0.125f;  // head_dim^-0.5, exact
            v[(size_t)768 * 768 + i] = wk[i];
            v[(size_t)2 * 768 * 768 + i] = wv[i];
        }
        NB_TRY(upload_split(h, v, &pw.qkv[l]));
        NB_TRY(upload_split(h, transpose_f32(v.data(), 2304, 768), &pw.qkv_t[l]));
        GET(wo, Q + "self_attn.out_proj.weight", 768LL * 768);
        GET(w1, Q + "fc1.weight", 3072LL * 768);
        GET(w2, Q + "fc2.weight", 768LL * 3072);
        NB_TRY(upload_split(h, std::vector<float>(wo, wo + 768 * 768), &pw.o[l]));
        NB_TRY(upload_split(h, std::vector<float>(w1, w1 + (size_t)3072 * 768), &pw.fc1[l]));
        NB_TRY(upload_split(h, std::vector<float>(w2, w2 + (size_t)768 * 3072), &pw.fc2[l]));
        NB_TRY(upload_split(h, transpose_f32(wo, 768, 768), &pw.o_t[l]));
        NB_TRY(upload_split(h, transpose_f32(w1, 3072, 768), &pw.fc1_t[l]));
        NB_TRY(upload_split(h, transpose_f32(w2, 768, 3072), &pw.fc2_t[l]));
    }
    pw.built = true;
    return 0;
}

// ================================================================================================
// Forward pass
static constexpr int META_SLOTS = 4;

int upload_meta(Handle* h, const Plan& p, const Workspace& ws, cudaStream_t st) {
    const size_t meta_bytes = sizeof(UttMeta) * p.B, item_bytes = sizeof(uint32_t) * p.attn_items.size();
    const size_t need = align_up(meta_bytes, 64) + item_bytes;
    if (h->meta_cap < need) {
        if (h->meta_host) {
            NB_CUDA(cudaDeviceSynchronize());
            NB_CUDA(cudaFreeHost(h->meta_host));
        }
        h->meta_cap = need < (64u << 10) ? (64u << 10) : need * 2;
        NB_CUDA(cudaMallocHost((void**)&h->meta_host, h->meta_cap * META_SLOTS));
    }
    if (!h->meta_event) {
        // one event per slot, stored contiguously
        cudaEvent_t* ev = new cudaEvent_t[META_SLOTS];
        for (int i = 0; i < META_SLOTS; ++i) NB_CUDA(cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming));
        h->meta_event = (cudaEvent_t)(void*)ev;
    }
    cudaEvent_t* ev = (cudaEvent_t*)(void*)h->meta_event;
    h->meta_slot = (h->meta_slot + 1) % META_SLOTS;  // per handle (a handle is not thread-safe, see the header)
    const int slot = h->meta_slot;
    NB_CUDA(cudaEventSynchronize(ev[slot]));  // no-op unless this slot's previous copy is still in flight
    char* stage = h->meta_host + (size_t)slot * h->meta_cap;
    memcpy(stage, p.utt.data(), meta_bytes);
    memcpy(stage + align_up(meta_bytes, 64), p.attn_items.data(), item_bytes);
    NB_CUDA(cudaMemcpyAsync(ws.meta, stage, meta_bytes, cudaMemcpyHostToDevice, st));
    if (item_bytes)
        NB_CUDA(cudaMemcpyAsync(ws.attn_items, stage + align_up(meta_bytes, 64), item_bytes, cudaMemcpyHostToDevice, st));
    NB_CUDA(cudaEventRecord(ev[slot], st));
    return 0;
}

GemmEpilogue epi_linear(int flags, const float* bias, const float* resid, float* out_f, op_t* out_h, long long ld) {
    GemmEpilogue e;
    memset(&e, 0, sizeof(e));
    e.flags = flags;
    e.bias = bias;
    e.resid = resid;
    e.ldr = ld;
    e.out_f = out_f;
    e.out_h = out_h;
    e.ldo = ld;
    return e;
}

// wav (device, packed) -> residual stream after the 12th layer (ws.x), optionally the 12 layer outputs.
int forward_encoder(Handle* h, const Plan& p, const Workspace& ws, const float* wav, cudaStream_t st,
                    float* layers_out, int layer_T, const FrontPipe* pipe) {
    const Weights& w = h->w;
    const int impl = h->gemm_impl;
    const long long F = p.frames;
    const bool save = ws.save;
    // The rows just past a level's last utterance are read by the next conv (its last padding output rows): keep
    // them finite.  (Padding rows never mix with valid rows, but a NaN there would survive as 0 * NaN in P V.)
    for (int l = 0; l < 6; ++l)
        NB_CUDA(cudaMemsetAsync(ws.y[l] + (p.rows0 >> l) * CONV_DIM, 0, 2ull * CONV_DIM * 8, st));
    // conv0 + GroupNorm + GELU, then conv1, per utterance group (one group unless the caller pipelines the H2D copy);
    // conv0 of group g + 1 is issued before conv1 of group g because conv1's padding rows read one row ahead
    FrontPipe whole;
    whole.n_groups = 1;
    whole.first[0] = 0;
    whole.first[1] = p.B;
    const FrontPipe& fp = (pipe != nullptr && pipe->n_groups > 0) ? *pipe : whole;
    auto row_of = [&](int b) { return b < p.B ? (long long)p.utt[b].row0 : p.rows0; };
    auto conv_level = [&](int l, long long r0, long long r1) -> int {  // level-l rows of the level-0 row range [r0, r1)
        const long long M = (r1 - r0) >> l;
        if (M <= 0) return 0;
        GemmOperand A{ws.y[l - 1] + (r0 >> (l - 1)) * CONV_DIM, M, 2 * CONV_DIM, 0, 0};
        GemmOperand Bw{w.conv_w[l], CONV_DIM, (long long)CONV_KERNEL[l] * CONV_DIM, 0, 0};
        GemmEpilogue e = epi_linear(EPI_GELU | EPI_OUT_H16, nullptr, nullptr, nullptr, ws.y[l] + (r0 >> l) * CONV_DIM, CONV_DIM);
        if (save) {
            e.flags |= EPI_SAVE_DGELU;
            e.aux_out = ws.aux[l] + (r0 >> l) * CONV_DIM;
        }
        return gemm_h16(st, A, Bw, (int)M, CONV_DIM, CONV_KERNEL[l] * CONV_DIM, 1, e, impl);
    };
    for (int g = 0; g <= fp.n_groups; ++g) {
        if (g < fp.n_groups) {
            const int b0 = fp.first[g], nb = fp.first[g + 1] - fp.first[g];
            if (pipe != nullptr && pipe->n_groups > 0) NB_CUDA(cudaStreamWaitEvent(st, fp.copied[g], 0));
            NB_TRY(launch_wave_stats(st, wav, ws.meta, b0, nb, p.max_chunks, ws.stat_part));
            NB_TRY(launch_gn_fold(st, ws.stat_part, ws.meta, b0, nb, p.max_chunks, w.conv0_w, w.gn_g, w.gn_b, ws.c0_fold,
                                  ws.gn_stat, ws.c0_fold_h));
            if (ws.aux0_raw) NB_TRY(launch_fold_unit_dgelu_gain(st, ws.c0_fold, b0, nb));
            NB_TRY(launch_conv0_apply(st, wav, ws.meta, p.B, row_of(b0), row_of(b0 + nb), ws.c0_fold,
                                      impl == 0 ? ws.c0_fold_h : nullptr, ws.y[0], ws.aux[0]));
        }
        if (g > 0) NB_TRY(conv_level(1, row_of(fp.first[g - 1]), row_of(fp.first[g])));
    }
    if (save) NB_TRY(launch_zero_pad_rows(st, ws.aux[1], ws.meta, p.B, 1));
    // conv 2..6 as overlapping-row GEMMs over the flat channels-last activation
    for (int l = 2; l < 7; ++l) {
        NB_TRY(conv_level(l, 0, p.rows0));
        if (save) NB_TRY(launch_zero_pad_rows(st, ws.aux[l], ws.meta, p.B, l));
    }
    // LayerNorm(512) -> projection -> x0
    NB_TRY(launch_ln512(st, ws.y[6], F, w.ln0_g, w.ln0_b, ws.ln0_out));
    {
        GemmOperand A{ws.ln0_out, F, CONV_DIM, 0, 0};
        GemmOperand Bw{w.proj_w, EMBED, CONV_DIM, 0, 0};
        GemmEpilogue e = epi_linear(EPI_BIAS | EPI_OUT_F32, w.proj_b, nullptr, ws.x0, nullptr, EMBED);
        NB_TRY(gemm_h16(st, A, Bw, (int)F, EMBED, CONV_DIM, 1, e, impl));
    }
    // positional conv (grouped, k = 128) as 16 overlapping-row GEMMs + residual + encoder LayerNorm
    {
        const long long rows_alloc = p.pos_rows + POS_K;
        NB_CUDA(cudaMemsetAsync(ws.pos_g, 0, 2ull * POS_G * POS_GC * rows_alloc, st));
        NB_TRY(launch_pos_scatter(st, ws.x0, ws.meta, p.B, F, rows_alloc, ws.pos_g));
        if (impl == 0) {
            NB_TRY(launch_posconv(st, ws.pos_g, rows_alloc, p.pos_rows, w.pos_w, w.pos_b,
                                  EPI_BIAS | EPI_GELU | (save ? EPI_SAVE_DGELU : 0), ws.pos_y, ws.pos_aux));
        } else {  // cross-check path: the same conv through the generic overlapping-row GEMM
            GemmOperand A{ws.pos_g, p.pos_rows, POS_GC, rows_alloc * POS_GC, 0};
            GemmOperand Bw{w.pos_w, POS_GC, (long long)POS_K * POS_GC, (long long)POS_GC * POS_K * POS_GC, 0};
            GemmEpilogue e = epi_linear(EPI_BIAS | EPI_GELU | EPI_OUT_H16, w.pos_b, nullptr, nullptr, ws.pos_y, EMBED);
            e.bias_bstride = POS_GC;
            e.out_bstride = POS_GC;
            if (save) {
                e.flags |= EPI_SAVE_DGELU;
                e.aux_out = ws.pos_aux;
            }
            NB_TRY(gemm_h16(st, A, Bw, (int)p.pos_rows, POS_GC, POS_K * POS_GC, POS_G, e, impl));
        }
        NB_TRY(launch_pos_finish_ln(st, ws.x0, ws.pos_y, ws.meta, p.B, F, w.lne_g, w.lne_b, ws.x, ws.xh));
    }
    // Scoring path (tensor-core GEMMs, nothing saved, no per-layer outputs wanted): no LayerNorm kernel runs inside
    // the layer stack.  A residual-adding GEMM (out-proj, FC2) stores its fp32 pre-LN rows, a 16-bit copy of them and
    // per-row partial statistics; the next GEMM takes the un-normalised copy as its A operand and applies the
    // LayerNorm algebraically in its epilogue (EPI_LN_FOLD); the next residual is rebuilt from the fp32 rows
    // (EPI_RESID_LN).  Only the last layer's final_layer_norm is materialised, for the pooling kernel.
    const bool fold_ln = impl == 0 && !save && layers_out == nullptr &&
                         !(getenv("NOMAD_B200_LN_FOLD") && atoi(getenv("NOMAD_B200_LN_FOLD")) == 0);
    for (int l = 0; l < LAYERS; ++l) {
        const LayerWeights& L = w.layer[l];
        const LayerBufs& Lb = ws.layer[l];
        if (l == 0 || save) NB_CUDA(cudaMemsetAsync(Lb.attn, 0, 2ull * EMBED * F, st));  // padded rows stay finite
        float* part1 = fold_ln ? ws.ln_part : nullptr;                             // statistics of pre1 (this layer)
        float* part2 = fold_ln ? ws.ln_part + 2ll * LN_PARTS * F : nullptr;        // statistics of pre2
        {
            GemmOperand A{ws.xh, F, EMBED, 0, 0};
            GemmOperand Bw{(fold_ln && l > 0) ? L.w_qkv_f : L.w_qkv, 3 * EMBED, EMBED, 0, 0};
            GemmEpilogue e = epi_linear(EPI_BIAS | EPI_OUT_H16, L.b_qkv, nullptr, nullptr, Lb.qkv, 3 * EMBED);
            if (fold_ln && l > 0) {  // xh holds the un-normalised pre2 of layer l - 1
                e.flags = EPI_LN_FOLD | EPI_OUT_H16;
                e.ln_part = part2;
                e.fold_s = L.s_qkv;
                e.fold_c = L.c_qkv;
            }
            NB_TRY(gemm_h16(st, A, Bw, (int)F, 3 * EMBED, EMBED, 1, e, impl));
        }
        if (impl == 0) {
            NB_TRY(launch_attention_fa(st, Lb.qkv, ws.attn_items, (int)(p.attn_items.size() / 4), F, Lb.attn, Lb.lse));
        } else {
            NB_TRY(launch_attention(st, Lb.qkv, ws.meta, p.B, p.max_T, Lb.attn, Lb.lse, 0));
        }
        // Residual stream bookkeeping: a LayerNorm kernel emits only the 16-bit operand + (mean, rstd) per row;
        // the next residual-adding GEMM epilogue rebuilds LN(pre) from the pre-LN buffer (EPI_RESID_LN).  Only the
        // encoder-LN output (layer 0 input) and the last layer's output exist as fp32 tensors.
        float* st1 = ws.ln_stats;            // stats of this layer's self_attn_layer_norm input
        float* st2 = ws.ln_stats + 2 * F;    // stats of a layer's final_layer_norm input
        {
            GemmOperand A{Lb.attn, F, EMBED, 0, 0};
            GemmOperand Bw{L.w_o, EMBED, EMBED, 0, 0};
            GemmEpilogue e;
            if (l == 0) {
                e = epi_linear(EPI_BIAS | EPI_RESID | EPI_OUT_F32, L.b_o, ws.x, Lb.pre1, nullptr, EMBED);
            } else {
                e = epi_linear(EPI_BIAS | EPI_RESID_LN | EPI_OUT_F32, L.b_o, ws.layer[l - 1].pre2, Lb.pre1, nullptr, EMBED);
                e.ln_stats = st2;
                e.ln_part = part2;
                e.ln_g = w.layer[l - 1].ln2_g;
                e.ln_b = w.layer[l - 1].ln2_b;
            }
            if (fold_ln) {
                e.flags |= EPI_OUT_H16 | EPI_STATS_OUT;
                e.out_h = ws.xh;
                e.part_out = part1;
            }
            NB_TRY(gemm_h16(st, A, Bw, (int)F, EMBED, EMBED, 1, e, impl));
        }
        if (!fold_ln) NB_TRY(launch_ln768(st, Lb.pre1, ws.meta, p.B, F, L.ln1_g, L.ln1_b, nullptr, ws.xh, st1, nullptr, 0));
        {
            GemmOperand A{ws.xh, F, EMBED, 0, 0};
            GemmOperand Bw{fold_ln ? L.w_fc1_f : L.w_fc1, FFN, EMBED, 0, 0};
            GemmEpilogue e = epi_linear(EPI_BIAS | EPI_GELU | EPI_OUT_H16, L.b_fc1, nullptr, nullptr, Lb.ffn_h ? Lb.ffn_h : ws.ffn_h, FFN);
            if (fold_ln) {
                e.flags = EPI_LN_FOLD | EPI_GELU | EPI_OUT_H16;
                e.ln_part = part1;
                e.fold_s = L.s_fc1;
                e.fold_c = L.c_fc1;
            }
            if (save) {
                e.flags |= EPI_SAVE_DGELU;
                e.aux_out = Lb.ffn_aux;
            }
            NB_TRY(gemm_h16(st, A, Bw, (int)F, FFN, EMBED, 1, e, impl));
        }
        {
            GemmOperand A{Lb.ffn_h ? Lb.ffn_h : ws.ffn_h, F, FFN, 0, 0};
            GemmOperand Bw{L.w_fc2, EMBED, FFN, 0, 0};
            GemmEpilogue e = epi_linear(EPI_BIAS | EPI_RESID_LN | EPI_OUT_F32, L.b_fc2, Lb.pre1, Lb.pre2, nullptr, EMBED);
            e.ln_stats = st1;
            e.ln_part = part1;
            e.ln_g = L.ln1_g;
            e.ln_b = L.ln1_b;
            const bool last = l == LAYERS - 1;
            if (fold_ln && !last) {
                e.flags |= EPI_OUT_H16 | EPI_STATS_OUT;
                e.out_h = ws.xh;
                e.part_out = part2;
            }
            NB_TRY(gemm_h16(st, A, Bw, (int)F, EMBED, FFN, 1, e, impl));
            float* lo = layers_out ? layers_out + (size_t)l * p.B * layer_T * EMBED : nullptr;
            if (!fold_ln || last)
                NB_TRY(launch_ln768(st, Lb.pre2, ws.meta, p.B, F, L.ln2_g, L.ln2_b, last ? ws.x : nullptr, ws.xh, st2, lo,
                                    layer_T));
        }
    }
    return 0;
}

static int check_handle(const nomad_b200_handle* hh) {
    NB_CHECK(hh != nullptr, "null nomad_b200 handle");
    return 0;
}

}  // namespace nb

using namespace nb;


extern "C" {

int nomad_b200_create(nomad_b200_handle** out, const nomad_b200_tensor* tensors, int n_tensors, int precision_mode,
                      int device) {
    NB_CHECK(out != nullptr && tensors != nullptr && n_tensors > 0, "create: bad arguments");
    NB_CHECK(precision_mode == NOMAD_B200_PRECISION_FP16 || precision_mode == NOMAD_B200_PRECISION_FP32,
             "create: precision_mode must be 0 (fp16 operands) or 1 (fp32-class split operands)");
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    NB_CHECK(ce == cudaSuccess && ndev > 0,
             "nomad_b200 needs a CUDA device (sm_100a) and has no CPU fallback: %s",
             ce == cudaSuccess ? "no device found" : cudaGetErrorString(ce));
    NB_CHECK(device >= 0 && device < ndev, "create: device %d out of range (%d devices)", device, ndev);
    NB_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    NB_CUDA(cudaGetDeviceProperties(&prop, device));
    NB_CHECK(prop.major == 10, "nomad_b200 is built for sm_100a only; device %d is sm_%d%d", device, prop.major,
             prop.minor);
    nomad_b200_handle* hh = new nomad_b200_handle();
    hh->h.device = device;
    TensorTable tt;
    for (int i = 0; i < n_tensors; ++i)
        if (tensors[i].name && tensors[i].data) tt.map[tensors[i].name] = &tensors[i];
    if (build_weights(&hh->h, tt) || (precision_mode == NOMAD_B200_PRECISION_FP32 && build_weights_precise(&hh->h, tt))) {
        nomad_b200_destroy(hh);
        return 1;
    }
    hh->h.precision = precision_mode;
    *out = hh;
    return 0;
}

int nomad_b200_set_precision(nomad_b200_handle* hh, int precision_mode) {
    NB_TRY(check_handle(hh));
    NB_CHECK(precision_mode == NOMAD_B200_PRECISION_FP16 || precision_mode == NOMAD_B200_PRECISION_FP32,
             "precision_mode must be 0 (fp16 operands) or 1 (fp32-class split operands)");
    NB_CHECK(precision_mode == NOMAD_B200_PRECISION_FP16 || hh->h.pw.built,
             "this handle was created with precision_mode 0: the fp32-class weights were not built");
    hh->h.precision = precision_mode;
    return 0;
}

int nomad_b200_get_precision(nomad_b200_handle* hh) { return hh ? hh->h.precision : -1; }

int nomad_b200_destroy(nomad_b200_handle* hh) {
    if (!hh) return 0;
    cudaSetDevice(hh->h.device);
    cudaDeviceSynchronize();
    for (void* p : hh->h.allocs) cudaFree(p);
    for (auto& e : hh->h.loss_graphs)
        if (e.exec) cudaGraphExecDestroy(e.exec);
    if (hh->h.graph_stream) cudaStreamDestroy(hh->h.graph_stream);
    if (hh->h.meta_host) cudaFreeHost(hh->h.meta_host);
    if (hh->h.copy_stream) {
        cudaStreamDestroy(hh->h.copy_stream);
        cudaEventDestroy(hh->h.fork_event);
        for (int i = 0; i < 8; ++i) cudaEventDestroy(hh->h.copied[i]);
    }
    if (hh->h.meta_event) {
        cudaEvent_t* ev = (cudaEvent_t*)(void*)hh->h.meta_event;
        for (int i = 0; i < META_SLOTS; ++i) cudaEventDestroy(ev[i]);
        delete[] ev;
    }
    delete hh;
    return 0;
}

int nomad_b200_set_gemm_impl(nomad_b200_handle* hh, int gemm_impl) {
    NB_TRY(check_handle(hh));
    NB_CHECK(gemm_impl == 0 || gemm_impl == 1, "gemm_impl must be 0 (tcgen05) or 1 (simt)");
    hh->h.gemm_impl = gemm_impl;
    return 0;
}

int nomad_b200_set_loss_head(nomad_b200_handle* hh, const float* w, const float* b) {
    NB_TRY(check_handle(hh));
    NB_CHECK(w && b, "set_loss_head: null pointer");
    Handle* h = &hh->h;
    NB_CUDA(cudaSetDevice(h->device));
    std::vector<float> t((size_t)768 * 256);
    for (int o = 0; o < 256; ++o)
        for (int k = 0; k < 768; ++k) t[(size_t)k * 256 + o] = w[(size_t)o * 768 + k];
    if (!h->w.loss_head_wt) {
        NB_TRY(upload(h, t, &h->w.loss_head_wt));
        NB_TRY(upload_f32(h, w, 256 * 768, &h->w.loss_head_w));
        NB_TRY(upload_f32(h, b, 256, &h->w.loss_head_b));
    } else {
        // earlier loss steps on the caller's (possibly non-blocking) streams may still read the old head
        NB_CUDA(cudaDeviceSynchronize());
        NB_CUDA(cudaMemcpy(h->w.loss_head_wt, t.data(), t.size() * 4, cudaMemcpyHostToDevice));
        NB_CUDA(cudaMemcpy(h->w.loss_head_w, w, 256 * 768 * 4, cudaMemcpyHostToDevice));
        NB_CUDA(cudaMemcpy(h->w.loss_head_b, b, 256 * 4, cudaMemcpyHostToDevice));
    }
    h->has_loss_head = true;
    return 0;
}

size_t nomad_b200_embed_workspace_bytes(const int64_t* sample_offsets, int B) {
    Plan p;
    if (make_plan(sample_offsets, B, &p)) return 0;
    return carve_workspace(p, nullptr, nullptr, false);
}

size_t nomad_b200_embed_workspace_bytes_mode(const int64_t* sample_offsets, int B, int precision_mode) {
    Plan p;
    if (make_plan(sample_offsets, B, &p)) return 0;
    const size_t a = carve_workspace(p, nullptr, nullptr, false);
    if (precision_mode != NOMAD_B200_PRECISION_FP32) return a;
    const size_t b = precise_workspace_bytes(p);
    return a > b ? a : b;
}

}  // extern "C"

// `pipe`: the caller stages the waveform in groups on a side stream (see FrontPipe); `issue_copies` is called right
// after the small metadata uploads, so that those do not queue behind the bulk copies on the H2D copy engine.
template <typename F>
static int embed_impl(nomad_b200_handle* hh, const float* wav_dev, const int64_t* sample_offsets, int B, float* emb_dev,
                      void* workspace_dev, size_t workspace_bytes, void* stream, const FrontPipe* pipe, F issue_copies) {
    NB_TRY(check_handle(hh));
    Handle* h = &hh->h;
    NB_CHECK(wav_dev && emb_dev && workspace_dev, "embed: null pointer");
    NB_CUDA(cudaSetDevice(h->device));
    Plan p;
    NB_TRY(make_plan(sample_offsets, B, &p));
    // wav_dev points at sample sample_offsets[0]
    for (auto& m : p.utt) m.wav_off -= sample_offsets[0];
    NB_CHECK(((uintptr_t)workspace_dev & 1023) == 0, "embed: workspace must be 1024-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    if (h->precision == NOMAD_B200_PRECISION_FP32) {  // fp32-class mode (precise.cu); host copies are waited for up front
        NB_TRY(issue_copies());
        if (pipe != nullptr)
            for (int g = 0; g < pipe->n_groups; ++g) NB_CUDA(cudaStreamWaitEvent(st, pipe->copied[g], 0));
        return embed_precise(h, p, workspace_dev, workspace_bytes, wav_dev, st, nullptr, 0, h->w.head_wt, h->w.head_b, emb_dev);
    }
    Workspace ws;
    const size_t need = carve_workspace(p, workspace_dev, &ws, false);
    NB_CHECK(workspace_bytes >= need, "embed: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
    NB_TRY(upload_meta(h, p, ws, st));
    NB_TRY(issue_copies());
    NB_TRY(forward_encoder(h, p, ws, wav_dev, st, nullptr, 0, pipe));
    NB_TRY(launch_pool_head(st, ws.x, ws.meta, p.B, h->w.head_wt, h->w.head_b, emb_dev, nullptr));
    return 0;
}

// HOST waveform -> device staging area -> embeddings (device).  H2D in up to 8 utterance groups on a side stream; the
// compute stream picks each group up as it lands (front end of group g overlaps the copy of group g + 1).  The first
// group is half the size of the others so that the GPU starts computing as early as possible.
static int embed_staged(nomad_b200_handle* hh, const float* wav_host, float* wav_dev, const int64_t* sample_offsets, int B,
                        float* emb_dev, void* workspace_dev, size_t core_bytes, void* stream) {
    Handle* h = &hh->h;
    NB_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    const long long total = sample_offsets[B] - sample_offsets[0];
    static const int max_groups = getenv("NOMAD_B200_H2D_GROUPS") ? atoi(getenv("NOMAD_B200_H2D_GROUPS")) : 8;
    FrontPipe pipe;
    if (!h->copy_stream) {
        NB_CUDA(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
        NB_CUDA(cudaEventCreateWithFlags(&h->fork_event, cudaEventDisableTiming));
        for (int i = 0; i < 8; ++i) NB_CUDA(cudaEventCreateWithFlags(&h->copied[i], cudaEventDisableTiming));
    }
    {
        int G = max_groups < 1 ? 1 : (max_groups > 8 ? 8 : max_groups);
        if (G > B) G = B;
        pipe.n_groups = G;
        pipe.first[0] = 0;
        int b = 0;
        for (int g = 1; g < G; ++g) {  // cut where the cumulative sample count passes (2 g - 1) / (2 G) of the total
            const long long cut = sample_offsets[0] + total * (2 * g - 1) / (2 * G);
            while (b < B - (G - g) && sample_offsets[b + 1] <= cut) ++b;
            if (b <= pipe.first[g - 1]) b = pipe.first[g - 1] + 1;
            pipe.first[g] = b;
        }
        pipe.first[G] = B;
        for (int g = 0; g < G; ++g) pipe.copied[g] = h->copied[g];
    }
    auto issue_copies = [&]() -> int {
        NB_CUDA(cudaEventRecord(h->fork_event, st));  // the staging area may still be read by earlier work on st
        NB_CUDA(cudaStreamWaitEvent(h->copy_stream, h->fork_event, 0));
        for (int g = 0; g < pipe.n_groups; ++g) {
            const long long s0 = sample_offsets[pipe.first[g]], s1 = sample_offsets[pipe.first[g + 1]];
            NB_CUDA(cudaMemcpyAsync(wav_dev + (s0 - sample_offsets[0]), wav_host + s0, (size_t)(s1 - s0) * 4,
                                    cudaMemcpyHostToDevice, h->copy_stream));
            NB_CUDA(cudaEventRecord(h->copied[g], h->copy_stream));
        }
        return 0;
    };
    return embed_impl(hh, wav_dev, sample_offsets, B, emb_dev, workspace_dev, core_bytes, stream, &pipe, issue_copies);
}

extern "C" {

int nomad_b200_embed(nomad_b200_handle* hh, const float* wav_dev, const int64_t* sample_offsets, int B, float* emb_dev,
                     void* workspace_dev, size_t workspace_bytes, void* stream) {
    return embed_impl(hh, wav_dev, sample_offsets, B, emb_dev, workspace_dev, workspace_bytes, stream, nullptr,
                      [] { return 0; });
}

int nomad_b200_embed_host(nomad_b200_handle* hh, const float* wav_host, const int64_t* sample_offsets, int B,
                          float* emb_host, void* workspace_dev, size_t workspace_bytes, void* stream) {
    NB_TRY(check_handle(hh));
    NB_CHECK(wav_host && emb_host && sample_offsets && B > 0, "embed_host: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    const long long total = sample_offsets[B] - sample_offsets[0];
    // the tail of the caller's workspace holds the staged waveform and the embeddings
    const size_t core = align_up(nomad_b200_embed_workspace_bytes_mode(sample_offsets, B, hh->h.precision), 1024);
    NB_CHECK(core != 0, "embed_host: %s", nomad_b200_last_error());
    const size_t wav_bytes = align_up((size_t)total * 4 + 64, 1024), emb_bytes = align_up((size_t)B * EMB * 4, 1024);
    NB_CHECK(workspace_bytes >= core + wav_bytes + emb_bytes,
             "embed_host: workspace too small (%zu < %zu bytes; embed_workspace_bytes + 4*samples + 1024*B + 4096)",
             workspace_bytes, core + wav_bytes + emb_bytes);
    float* wav_dev = (float*)((char*)workspace_dev + core);
    float* emb_dev = (float*)((char*)workspace_dev + core + wav_bytes);
    NB_TRY(embed_staged(hh, wav_host, wav_dev, sample_offsets, B, emb_dev, workspace_dev, core, stream));
    NB_CUDA(cudaMemcpyAsync(emb_host, emb_dev, (size_t)B * EMB * 4, cudaMemcpyDeviceToHost, st));
    NB_CUDA(cudaStreamSynchronize(st));
    return 0;
}

int nomad_b200_paired_dist(const float* a_dev, const float* b_dev, int64_t n, double* out_dev, void* stream) {
    NB_CHECK(n >= 0 && (n == 0 || (a_dev && b_dev && out_dev)), "paired_dist: bad arguments");
    return launch_paired_dist((cudaStream_t)stream, a_dev, b_dev, n, out_dev);
}

size_t nomad_b200_attention_workspace_bytes(const int32_t* T, int n_utts) {
    size_t entries = 0;
    for (int u = 0; T != nullptr && u < n_utts; ++u) entries += (size_t)((T[u] + 127) / 128);
    return entries * 16 + 1024;
}

int nomad_b200_attention_f16(const void* qkv_f16, int64_t frames, const int32_t* frame0, const int32_t* T, int n_utts,
                             void* out_f16, float* lse, void* workspace_dev, size_t workspace_bytes, void* stream) {
    NB_CHECK(qkv_f16 && frame0 && T && out_f16 && workspace_dev && n_utts > 0 && frames > 0, "attention: bad arguments");
    Plan p;
    p.B = n_utts;
    p.utt.resize(n_utts);
    for (int u = 0; u < n_utts; ++u) {
        NB_CHECK(T[u] >= 1 && frame0[u] >= 0 && (int64_t)frame0[u] + T[u] <= frames, "attention: utterance %d out of range", u);
        memset(&p.utt[u], 0, sizeof(UttMeta));
        p.utt[u].T = T[u];
        p.utt[u].frame0 = frame0[u];
    }
    std::vector<uint32_t> items;
    build_attention_items(p, &items);
    NB_CHECK(workspace_bytes >= items.size() * 4, "attention: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    NB_CUDA(cudaMemcpyAsync(workspace_dev, items.data(), items.size() * 4, cudaMemcpyHostToDevice, st));
    NB_CUDA(cudaStreamSynchronize(st));  // items is a pageable temporary
    return launch_attention_fa(st, (const op_t*)qkv_f16, (const uint32_t*)workspace_dev, (int)(items.size() / 4), frames,
                               (op_t*)out_f16, lse);
}

int64_t nomad_b200_num_frames(int64_t n) {
    long long t = n;
    for (int l = 0; l < 7; ++l) {
        if (t < CONV_KERNEL[l]) return 0;
        t = (t - CONV_KERNEL[l]) / CONV_STRIDE[l] + 1;
    }
    return t;
}

static int uniform_offsets(int B, int64_t N, std::vector<int64_t>* off) {
    NB_CHECK(B > 0 && N >= NOMAD_B200_MIN_SAMPLES, "need B > 0 and N >= %d samples", NOMAD_B200_MIN_SAMPLES);
    off->resize(B + 1);
    for (int b = 0; b <= B; ++b) (*off)[b] = (int64_t)b * N;
    return 0;
}

size_t nomad_b200_layers_workspace_bytes(int B, int64_t N) {
    std::vector<int64_t> off;
    if (uniform_offsets(B, N, &off)) return 0;
    return nomad_b200_embed_workspace_bytes(off.data(), B);
}

size_t nomad_b200_layers_workspace_bytes_mode(int B, int64_t N, int precision_mode) {
    std::vector<int64_t> off;
    if (uniform_offsets(B, N, &off)) return 0;
    return nomad_b200_embed_workspace_bytes_mode(off.data(), B, precision_mode);
}

int nomad_b200_layers_fwd(nomad_b200_handle* hh, const float* wav_dev, int B, int64_t N, float* layers_dev,
                          float* emb_dev, void* workspace_dev, size_t workspace_bytes, void* stream) {
    NB_TRY(check_handle(hh));
    Handle* h = &hh->h;
    NB_CHECK(wav_dev && workspace_dev, "layers_fwd: null pointer");
    NB_CUDA(cudaSetDevice(h->device));
    std::vector<int64_t> off;
    NB_TRY(uniform_offsets(B, N, &off));
    Plan p;
    NB_TRY(make_plan(off.data(), B, &p));
    cudaStream_t st = (cudaStream_t)stream;
    if (h->precision == NOMAD_B200_PRECISION_FP32) {
        const bool lh = h->has_loss_head;
        return embed_precise(h, p, workspace_dev, workspace_bytes, wav_dev, st, layers_dev, p.max_T,
                             lh ? h->w.loss_head_wt : h->w.head_wt, lh ? h->w.loss_head_b : h->w.head_b, emb_dev);
    }
    Workspace ws;
    const size_t need = carve_workspace(p, workspace_dev, &ws, false);
    NB_CHECK(workspace_bytes >= need, "layers_fwd: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
    NB_TRY(upload_meta(h, p, ws, st));
    NB_TRY(forward_encoder(h, p, ws, wav_dev, st, layers_dev, p.max_T));
    if (emb_dev) {
        const bool lh = h->has_loss_head;
        NB_TRY(launch_pool_head(st, ws.x, ws.meta, p.B, lh ? h->w.loss_head_wt : h->w.head_wt,
                                lh ? h->w.loss_head_b : h->w.head_b, emb_dev, nullptr));
    }
    return 0;
}

// Small problems (and the SIMT cross-check) use the fp32 direct-difference kernel; everything else the
// tensor-core Gram kernel.
static bool cdist_use_tc(int64_t n, int64_t m, int gemm_impl) { return gemm_impl == 0 && n * m >= (1 << 16); }

size_t nomad_b200_cdist_workspace_bytes(int64_t n, int64_t m) {
    if (n < 0 || m < 0) return 0;
    const size_t a = cdist_use_tc(n, m, 0) ? cdist_tc_workspace(n, m) : 0, b = cdist_fp32_workspace(n, m);
    return a > b ? a : b;  // the SIMT cross-check of a large problem takes the fp32 kernel
}

int nomad_b200_cdist_mean(const float* deg_dev, int64_t n, const float* nmr_dev, int64_t m, float* dm_dev,
                          double* row_mean_dev, void* workspace_dev, size_t workspace_bytes, int gemm_impl,
                          void* stream) {
    NB_CHECK(n >= 0 && m >= 0, "cdist: negative size");
    NB_CHECK(n == 0 || (deg_dev && row_mean_dev), "cdist: null pointer");
    NB_CHECK(m == 0 || nmr_dev, "cdist: null pointer");
    if (cdist_use_tc(n, m, gemm_impl))
        return launch_cdist_tc((cudaStream_t)stream, deg_dev, n, nmr_dev, m, dm_dev, row_mean_dev, workspace_dev,
                               workspace_bytes, 0);
    return launch_cdist_fp32((cudaStream_t)stream, deg_dev, n, nmr_dev, m, dm_dev, row_mean_dev, workspace_dev,
                             workspace_bytes);
}

// ---- one batch of Nomad.predict: embed + distance rows against a resident NMR set ---------------------------------
size_t nomad_b200_score_workspace_bytes(const int64_t* sample_offsets, int B, int64_t m) {
    return nomad_b200_score_workspace_bytes_mode(sample_offsets, B, m, NOMAD_B200_PRECISION_FP16);
}

size_t nomad_b200_score_workspace_bytes_mode(const int64_t* sample_offsets, int B, int64_t m, int precision_mode) {
    const size_t e = nomad_b200_embed_workspace_bytes_mode(sample_offsets, B, precision_mode);
    if (e == 0 || m < 0) return 0;
    const long long total = sample_offsets[B] - sample_offsets[0];
    // embed workspace | cdist workspace | staged waveform, embeddings, matrix rows, means (the *_host variant)
    return align_up(e, 1024) + align_up(nomad_b200_cdist_workspace_bytes(B, m), 1024) + align_up((size_t)total * 4 + 64, 1024) +
           align_up((size_t)B * EMB * 4, 1024) + align_up((size_t)B * (size_t)m * 4, 1024) + align_up((size_t)B * 8, 1024);
}

int nomad_b200_score(nomad_b200_handle* hh, const float* wav_dev, const int64_t* sample_offsets, int B,
                     const float* nmr_dev, int64_t m, float* emb_dev, float* dm_dev, double* row_mean_dev,
                     void* workspace_dev, size_t workspace_bytes, void* stream) {
    NB_TRY(check_handle(hh));
    NB_CHECK(sample_offsets && B > 0 && m >= 0 && emb_dev && row_mean_dev, "score: bad arguments");
    const size_t e = align_up(nomad_b200_embed_workspace_bytes_mode(sample_offsets, B, hh->h.precision), 1024);
    NB_CHECK(e != 0, "score: %s", nomad_b200_last_error());
    const size_t c = nomad_b200_cdist_workspace_bytes(B, m);
    NB_CHECK(workspace_dev && workspace_bytes >= e + c, "score: workspace too small (%zu < %zu bytes)", workspace_bytes, e + c);
    NB_TRY(nomad_b200_embed(hh, wav_dev, sample_offsets, B, emb_dev, workspace_dev, e, stream));
    return nomad_b200_cdist_mean(emb_dev, B, nmr_dev, m, dm_dev, row_mean_dev, (char*)workspace_dev + e, c, 0, stream);
}

int nomad_b200_score_host(nomad_b200_handle* hh, const float* wav_host, const int64_t* sample_offsets, int B,
                          const float* nmr_dev, int64_t m, float* emb_host, float* dm_host, double* row_mean_host,
                          void* workspace_dev, size_t workspace_bytes, void* stream) {
    NB_TRY(check_handle(hh));
    NB_CHECK(wav_host && sample_offsets && B > 0 && m >= 0 && row_mean_host, "score_host: bad arguments");
    const size_t need = nomad_b200_score_workspace_bytes_mode(sample_offsets, B, m, hh->h.precision);
    NB_CHECK(need != 0, "score_host: %s", nomad_b200_last_error());
    NB_CHECK(workspace_dev && workspace_bytes >= need, "score_host: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
    const long long total = sample_offsets[B] - sample_offsets[0];
    const size_t e = align_up(nomad_b200_embed_workspace_bytes_mode(sample_offsets, B, hh->h.precision), 1024);
    const size_t c = align_up(nomad_b200_cdist_workspace_bytes(B, m), 1024);
    char* base = (char*)workspace_dev;
    float* wav_dev = (float*)(base + e + c);
    float* emb_dev = (float*)((char*)wav_dev + align_up((size_t)total * 4 + 64, 1024));
    float* dm_dev = (float*)((char*)emb_dev + align_up((size_t)B * EMB * 4, 1024));
    double* rm_dev = (double*)((char*)dm_dev + align_up((size_t)B * (size_t)m * 4, 1024));
    cudaStream_t st = (cudaStream_t)stream;
    // waveform H2D in utterance groups on the side stream, front end of group g overlapping the copy of group g + 1
    NB_TRY(embed_staged(hh, wav_host, wav_dev, sample_offsets, B, emb_dev, workspace_dev, e, stream));
    NB_TRY(nomad_b200_cdist_mean(emb_dev, B, nmr_dev, m, dm_host ? dm_dev : nullptr, rm_dev, base + e, c, 0, stream));
    if (emb_host) NB_CUDA(cudaMemcpyAsync(emb_host, emb_dev, (size_t)B * EMB * 4, cudaMemcpyDeviceToHost, st));
    if (dm_host && m > 0) NB_CUDA(cudaMemcpyAsync(dm_host, dm_dev, (size_t)B * (size_t)m * 4, cudaMemcpyDeviceToHost, st));
    NB_CUDA(cudaMemcpyAsync(row_mean_host, rm_dev, (size_t)B * 8, cudaMemcpyDeviceToHost, st));
    NB_CUDA(cudaStreamSynchronize(st));
    return 0;
}

int nomad_b200_cdist_mean_host(const float* deg_host, int64_t n, const float* nmr_host, int64_t m, float* dm_host,
                               double* row_mean_host, void* workspace_dev, size_t workspace_bytes, void* stream) {
    NB_CHECK(n > 0 && m > 0 && deg_host && nmr_host && row_mean_host, "cdist_host: bad arguments");
    const size_t a_b = align_up((size_t)n * EMB * 4, 1024), b_b = align_up((size_t)m * EMB * 4, 1024);
    const size_t dm_b = dm_host ? align_up((size_t)n * m * 4, 1024) : 0, rm_b = align_up((size_t)n * 8, 1024);
    const size_t core = align_up(nomad_b200_cdist_workspace_bytes(n, m), 1024);
    NB_CHECK(workspace_dev && workspace_bytes >= a_b + b_b + dm_b + rm_b + core,
             "cdist_host: workspace too small (%zu < %zu bytes)", workspace_bytes, a_b + b_b + dm_b + rm_b + core);
    cudaStream_t st = (cudaStream_t)stream;
    char* base = (char*)workspace_dev;
    float* a_d = (float*)base;
    float* b_d = (float*)(base + a_b);
    float* dm_d = dm_host ? (float*)(base + a_b + b_b) : nullptr;
    double* rm_d = (double*)(base + a_b + b_b + dm_b);
    NB_CUDA(cudaMemcpyAsync(a_d, deg_host, (size_t)n * EMB * 4, cudaMemcpyHostToDevice, st));
    NB_CUDA(cudaMemcpyAsync(b_d, nmr_host, (size_t)m * EMB * 4, cudaMemcpyHostToDevice, st));
    NB_TRY(nomad_b200_cdist_mean(a_d, n, b_d, m, dm_d, rm_d, base + a_b + b_b + dm_b + rm_b, core, 0, stream));
    if (dm_host) NB_CUDA(cudaMemcpyAsync(dm_host, dm_d, (size_t)n * m * 4, cudaMemcpyDeviceToHost, st));
    NB_CUDA(cudaMemcpyAsync(row_mean_host, rm_d, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
    NB_CUDA(cudaStreamSynchronize(st));
    return 0;
}

}  // extern "C"
