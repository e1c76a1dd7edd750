// Launchers of the non-GEMM kernels of the path (all stream-ordered, no syncs).
#pragma once
#include "model.cuh"

namespace nb {

// ---- frontend.cu: waveform -> conv0 + GroupNorm + GELU, LayerNorm(512)
// utterances [b0, b0 + nb)
int launch_wave_stats(cudaStream_t st, const float* wav, const UttMeta* meta, int b0, int nb, int max_chunks,
                      double* part);
int launch_gn_fold(cudaStream_t st, const double* part, const UttMeta* meta, int b0, int nb, int max_chunks,
                   const float* conv0_w, const float* gn_g, const float* gn_b, float* fold, float* stat_out,
                   op_t* fold_h);
// level-0 rows [row_begin, row_end) (multiples of 64, utterance boundaries)
// fold[b][c][11] := 1 for utterances [b0, b0 + nb): conv0's saved GELU gradient is then gelu' itself
int launch_fold_unit_dgelu_gain(cudaStream_t st, float* fold, int b0, int nb);
int launch_conv0_apply(cudaStream_t st, const float* wav, const UttMeta* meta, int B, long long row_begin,
                       long long row_end, const float* fold, const op_t* fold_h, op_t* out, op_t* aux_out);
// zero rows [T_l, rows_l) of every utterance at conv level l (so masked rows carry no gradient)
int launch_zero_pad_rows(cudaStream_t st, op_t* buf, const UttMeta* meta, int B, int level);
int launch_ln512(cudaStream_t st, const op_t* in, long long rows, const float* g, const float* b, op_t* out);

// ---- encoder.cu
int launch_pos_scatter(cudaStream_t st, const float* x, const UttMeta* meta, int B, long long frames,
                       long long pos_rows_alloc, op_t* pos_g);
// x = LN(x0 + y[pos row]) on valid frames, 0 elsewhere
int launch_pos_finish_ln(cudaStream_t st, const float* x0, const op_t* pos_y, const UttMeta* meta, int B,
                         long long frames, const float* g, const float* b, float* x, op_t* xh);
// LN(pre) on valid frames, 0 elsewhere -> 16-bit xh; optional fp32 x, optional (mean, rstd) per row (so a later
// GEMM epilogue can rebuild the fp32 residual), optional compact copy layer_out[(utt * T + t) * 768 + c]
int launch_ln768(cudaStream_t st, const float* pre, const UttMeta* meta, int B, long long frames, const float* g,
                 const float* b, float* x, op_t* xh, float* stats, float* layer_out, int layer_T);
// streaming mma.sync kernel (any T): the attention of the SIMT cross-check path (gemm_impl = 1); skip_T_le = 0
int launch_attention(cudaStream_t st, const op_t* qkv, const UttMeta* meta, int B, int max_T, op_t* out, float* lse,
                     int skip_T_le);
// attention_fa.cu: persistent tcgen05 flash attention over the plan's work list (any T)
int launch_attention_fa(cudaStream_t st, const op_t* qkv, const uint32_t* items, int n_items,
                        long long frames, op_t* out, float* lse);
int launch_pool_head(cudaStream_t st, const float* x, const UttMeta* meta, int B, const float* head_wt,
                     const float* head_b, float* emb, float* pooled_out);

// ---- posconv.cu: grouped positional conv (and its dgrad with flipped, transposed taps) on tcgen05
int launch_posconv(cudaStream_t st, const op_t* pos_g, long long rows_alloc, long long pos_rows, const op_t* w,
                   const float* bias, int flags, op_t* out, op_t* aux_out);

// ---- distance.cu
size_t cdist_fp32_workspace(long long n, long long m);
int launch_cdist_fp32(cudaStream_t st, const float* a, long long n, const float* b, long long m, float* dm,
                      double* row_mean, void* ws, size_t ws_bytes);
int launch_paired_dist(cudaStream_t st, const float* a, const float* b, long long n, double* out);
size_t cdist_tc_workspace(long long n, long long m);
int launch_cdist_tc(cudaStream_t st, const float* a, long long n, const float* b, long long m, float* dm,
                    double* row_mean, void* ws, size_t ws_bytes, int impl);

__device__ __forceinline__ int find_utt_by_frame(const UttMeta* __restrict__ meta, int B, int f) {
    int lo = 0, hi = B - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (meta[mid].frame0 <= f) lo = mid; else hi = mid - 1;
    }
    return lo;
}

}  // namespace nb
