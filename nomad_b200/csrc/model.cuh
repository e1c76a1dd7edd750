// Host-side model state (device weights in kernel-ready layouts) and the per-call batch plan.
#pragma once
#include <vector>

#include "gemm.cuh"

namespace nb {

static constexpr int CONV_DIM = 512;
static constexpr int EMBED = 768;
static constexpr int FFN = 3072;
static constexpr int HEADS = 12;
static constexpr int HEAD_DIM = 64;
static constexpr int LAYERS = 12;
static constexpr int POS_K = 128;
static constexpr int POS_G = 16;
static constexpr int POS_GC = 48;  // channels per group
// zero rows between consecutive utterances in the padded positional-conv layout: one gap serves as the right context
// (63 rows) of the utterance before it and the left context (64 rows) of the one after it
static constexpr int POS_GAP = 64;
static constexpr int EMB = 256;
static constexpr int NSTAT = 65;   // 10 tap sums + 55 tap cross-products of the waveform
static constexpr int STAT_CHUNK = 4096;  // conv0 frames per wave-stats block
static const int CONV_KERNEL[7] = {10, 3, 3, 3, 3, 2, 2};
static const int CONV_STRIDE[7] = {5, 2, 2, 2, 2, 2, 2};

// Per-utterance geometry, one entry per utterance, resident on the device for the kernels that need
// to know where an utterance starts and how much of it is valid.
struct UttMeta {
    long long wav_off;  // first sample in the packed waveform buffer
    int n;              // samples
    int T0;             // valid conv0 frames
    int row0;           // first row in the flat level-0 activation (multiple of 64)
    int rows0;          // rows reserved at level 0 (T0 rounded up to a multiple of 64)
    int T;              // valid frames after the conv encoder (level 6)
    int frame0;         // first row in the flat frame-level buffers = row0 / 64
    int frames;         // rows reserved at frame level = rows0 / 64
    int pos0;           // first row of this utterance in the zero-padded positional-conv layout
};

struct LayerWeights {
    op_t *w_qkv, *w_o, *w_fc1, *w_fc2;          // [N][K] K-major op_t
    float *b_qkv, *b_o, *b_fc1, *b_fc2;
    float *ln1_g, *ln1_b, *ln2_g, *ln2_b;
    // LayerNorm folded into the consuming GEMM (scoring path, EPI_LN_FOLD): weights times the gamma of the
    // LayerNorm that feeds them (QKV: previous layer's final_layer_norm, null for layer 0; FC1: this layer's
    // self_attn_layer_norm), s = row sums of the rounded folded weights, c = W beta + bias
    op_t *w_qkv_f, *w_fc1_f;
    float *s_qkv, *c_qkv, *s_fc1, *c_fc1;
    // transposed copies for the dgrad GEMMs of the loss path
    op_t *wt_qkv, *wt_o, *wt_fc1, *wt_fc2;      // [K][N] -> used as [N'=K][K'=N]
};

struct Weights {
    float* conv0_w;      // [512][10]
    float *gn_g, *gn_b;  // [512]
    op_t* conv_w[7];     // l = 1..6: [512][k*512], K index = tap*512 + cin
    op_t* conv_wt[7];    // dgrad: [k][cin=512][cout=512] -> per tap [N'=cin][K'=cout]
    op_t* conv_wte[7];   // dgrad of the even input rows of the k=3 layers: [cin][tap2: cout | tap0: cout]
    op_t* conv0_wh;      // conv0 dgrad: [16][512] = w0[c][j] transposed, rows 10..15 zero
    float *ln0_g, *ln0_b;  // LayerNorm(512)
    op_t* proj_w;        // [768][512]
    op_t* proj_wt;       // [512][768]
    float* proj_b;
    op_t* pos_w;         // [16][48][128*48], K index = tap*48 + cin
    op_t* pos_wt;        // dgrad: [16][48 (cin)][128*48], K index = tap'*48 + cout (taps flipped)
    float* pos_b;        // [768]
    float *lne_g, *lne_b;  // encoder LayerNorm(768)
    LayerWeights layer[LAYERS];
    float* head_wt;      // scoring head, transposed [768][256]
    float* head_b;       // [256]
    float* loss_head_wt; // loss head (LossNetLayers.embedding_layer), transposed [768][256]
    float* loss_head_w;  // [256][768] (backward)
    float* loss_head_b;
    double* pos_scale_tmp;  // [128] g / ||v|| per tap, scratch of nomad_b200_refresh_weights (allocated on first use)
};

// fp32-class mode (precise.cu): a GEMM weight as hi + lo fp16 planes of w * 2^k (k per tensor, so that the lo plane
// stays in fp16's normal range); inv_scale = 2^-k goes into the epilogue.
struct SplitW {
    op_t* hi;
    op_t* lo;
    float inv_scale;
};
struct PreciseWeights {
    bool built = false;
    SplitW conv[7]{};   // l = 1..6, same layout as Weights::conv_w
    SplitW proj{}, pos{};
    SplitW qkv[LAYERS]{}, o[LAYERS]{}, fc1[LAYERS]{}, fc2[LAYERS]{};
    // transposed planes for the dgrad GEMMs of the fp32-class waveform backward (precise_bwd.cu), in the layouts of
    // Weights::conv_wt / conv_wte / proj_wt / pos_wt / wt_*: the same hi / lo values, the same inv_scale
    SplitW conv_t[7]{}, conv_te[7]{};
    SplitW proj_t{}, pos_t{};
    SplitW qkv_t[LAYERS]{}, o_t[LAYERS]{}, fc1_t[LAYERS]{}, fc2_t[LAYERS]{};
};

struct Plan {
    int B = 0;
    std::vector<UttMeta> utt;
    long long total_samples = 0;
    long long rows0 = 0;   // flat rows at level 0 (multiple of 64)
    long long frames = 0;  // flat rows at frame level = rows0 / 64
    long long pos_rows = 0;  // rows of the padded positional-conv layout (outputs)
    int max_T = 0;
    int max_chunks = 0;    // wave-stats chunks of the longest utterance
    bool uniform = false;  // all utterances the same length
    std::vector<uint32_t> attn_items;  // 4 words per (utterance, query tile), longest utterances first (attention_fa.cu)
};

// Device pointers carved from the caller's workspace for one forward pass.  In scoring mode the conv
// levels ping-pong between two buffers and the per-layer pointers alias shared scratch; in "save" mode
// (loss path) every tensor the backward needs gets its own storage.
struct LayerBufs {
    op_t* qkv;      // frames x 2304
    op_t* attn;     // frames x 768 (attention output O)
    float* lse;     // frames x 12 log-sum-exp of the attention rows (save mode) or nullptr
    float* pre1;    // frames x 768: x_in + out_proj(attn)        (input of self_attn_layer_norm)
    op_t* ffn_aux;  // frames x 3072: gelu'(fc1 pre-activation)   (save mode) or nullptr
    float* pre2;    // frames x 768: x1 + fc2(h)                   (input of final_layer_norm)
    op_t* ffn_h;    // frames x 3072: GELU(fc1) of THIS layer (train mode: the fc2 weight gradient needs it) or nullptr
};

struct Workspace {
    bool save;
    bool train;          // save mode + what the parameter gradients need (per-layer FFN activations)
    bool aux0_raw;       // save mode, conv encoder training: aux[0] holds gelu' itself (the GroupNorm affine
                         // gradients need dL/du0 without the gamma * rstd factor, and gamma may be 0)
    UttMeta* meta;       // [B]
    uint32_t* attn_items;  // [Plan::attn_items.size()] work list of the attention kernel
    double* stat_part;   // [B][max_chunks][65]
    float* c0_fold;      // [B][512][12]: 10 folded taps, shift, gamma * rstd
    op_t* c0_fold_h;     // [B][512][32]: the folded taps as 16-bit hi | lo halves, K padded to 16 (tensor-core conv0)
    float* gn_stat;      // save mode: [B][512][2] mean and rstd of the raw conv0 output per (utt, channel)
    op_t* y[7];          // conv level outputs, level l: (rows0 >> l) + 8 rows x 512
    op_t* aux[7];        // save mode: gelu'(pre-activation) per level (level 0: times gamma * rstd unless aux0_raw)
    op_t* ln0_out;       // LayerNorm(512) output, frames x 512
    float* x0;           // feature projection output, frames x 768 fp32
    op_t* pos_g;         // [16][pos_rows + 128][48]
    op_t* pos_y;         // [pos_rows][768] GELU(pos conv)
    op_t* pos_aux;       // save mode: gelu' of the pos conv pre-activation, [pos_rows][768]
    float* ln_stats;     // frames x 2: (mean, rstd) of the most recent LayerNorm(768) input rows
    float* ln_part;      // 2 x frames x LN_PARTS x 2: partial (mean, M2) of the pre-LN rows (scoring path)
    float* x;            // residual stream, frames x 768 fp32
    op_t* xh;            // 16-bit copy (GEMM operand)
    op_t* ffn_h;         // frames x 3072
    LayerBufs layer[LAYERS];
    size_t bytes;
};

// one captured loss step (loss.cu): replayed while shape, gradient request and workspace stay the same
struct LossGraphEntry {
    int mode;  // precision_mode the step was recorded in
    int B;
    long long N;
    int with_grad;
    float fgm;
    void* ws;
    cudaGraphExec_t exec;
    long long kernels;  // kernel launches the graph replays (for nomad_b200_launch_count)
    bool failed;        // capture was refused once: this shape stays eager
};

struct Handle {
    int device = 0;
    int gemm_impl = 0;
    int precision = 0;          // 0: fp16 tensor-core operands (default), 1: fp32-class split operands (precise.cu)
    Weights w{};
    PreciseWeights pw{};
    std::vector<void*> allocs;  // everything cudaMalloc'ed for the weights
    bool has_loss_head = false;
    char* meta_host = nullptr;  // pinned staging for the per-call metadata (UttMeta[B] + attention work list)
    size_t meta_cap = 0;        // bytes per staging slot
    int meta_slot = 0;          // staging slot of the most recent call
    cudaEvent_t meta_event = nullptr;  // last use of meta_host by an async copy
    std::vector<LossGraphEntry> loss_graphs;
    cudaStream_t graph_stream = nullptr;  // capture stream of the loss-step graphs (capture is not legal on stream 0)
    cudaStream_t copy_stream = nullptr;  // H2D side stream of the *_host entry points
    cudaEvent_t fork_event = nullptr;
    cudaEvent_t copied[8] = {};
};

int make_plan(const int64_t* sample_offsets, int B, Plan* plan);
size_t carve_workspace(const Plan& p, void* base, Workspace* ws, bool save, bool train = false);
// Host-buffer entry points copy the waveform in utterance groups on a side stream; the front end (statistics, conv0,
// conv1) of group g then runs while group g + 1 is still crossing PCIe.
struct FrontPipe {
    int n_groups = 0;
    int first[9] = {0};          // group g = utterances [first[g], first[g + 1])
    cudaEvent_t copied[8] = {};  // recorded on the copy stream after group g's H2D copy
};
int forward_encoder(Handle* h, const Plan& p, const Workspace& ws, const float* wav, cudaStream_t st, float* layers_out,
                    int layer_T, const FrontPipe* pipe = nullptr);
int upload_meta(Handle* h, const Plan& p, const Workspace& ws, cudaStream_t st);
void build_attention_items(const Plan& p, std::vector<uint32_t>* items);
GemmEpilogue epi_linear(int flags, const float* bias, const float* resid, float* out_f, op_t* out_h, long long ld);
// precise.cu
size_t precise_workspace_bytes(const Plan& p);
int embed_precise(Handle* h, const Plan& p, void* workspace, size_t workspace_bytes, const float* wav, cudaStream_t st,
                  float* layers_out, int layer_T, const float* head_wt, const float* head_b, float* emb_dev);

}  // namespace nb

struct nomad_b200_handle {
    nb::Handle h;
};
