/* nomad_b200 -- C ABI of the B200-native NOMAD scoring + loss hot path.
 *
 * The reference (alessandroragano/nomad) has no FFI of its own: the seam is the set of Python
 * attribute calls inside ``Nomad`` (reference src/nomad_audio/nomad.py).  Each entry point below
 * replaces one of those calls; the cited lines are the reference interface it stands in for.
 * ``INTEGRATION.md`` shows the ctypes binding a maintainer of the reference would add.
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; ``nomad_b200_last_error()`` then
 *     returns a thread-local, human-readable message.
 *   - "device" pointers are CUDA device pointers into caller-owned memory (e.g. torch tensors'
 *     data_ptr()); ``stream`` is a ``cudaStream_t`` passed as ``void*``.  Work is enqueued on that
 *     stream; no entry point synchronises the device except the ``*_host`` variants, which take HOST
 *     buffers, copy in, run, copy out and synchronise the stream before returning.
 *   - the library owns no activation memory: the caller provides a workspace whose size the
 *     matching ``*_workspace_bytes`` call reports (plain pointers and sizes, no torch types).
 *   - one handle per (process, device); a handle is not thread-safe.
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef NOMAD_B200_H
#define NOMAD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define NOMAD_B200_API __attribute__((visibility("default")))
#else
#define NOMAD_B200_API
#endif

#define NOMAD_B200_EMB_DIM 256   /* nomad.py:55  EMB_DIM     */
#define NOMAD_B200_SSL_DIM 768   /* nomad.py:54  SSL_OUT_DIM */
#define NOMAD_B200_NUM_LAYERS 12
#define NOMAD_B200_MIN_SAMPLES 400 /* shortest waveform the conv encoder accepts (1 frame) */

typedef struct nomad_b200_handle nomad_b200_handle;

/* One named fp32 tensor of the checkpoint, HOST memory, contiguous, fairseq key names exactly as in
 * ``TripletModel.state_dict()`` (reference nomad.py:65, train_triplet.py:177), e.g.
 * "ssl_model.encoder.layers.3.fc1.weight", "embedding_layer.1.bias". */
typedef struct {
    const char* name;
    const float* data;
    int64_t numel;
} nomad_b200_tensor;

/* Arithmetic class of the scoring path (``precision_mode``).  The reference is fp32 everywhere (nomad.py:226-230).
 *   FP16: fp16 tensor-core operands, fp32 accumulation / residual stream / statistics: embeddings within 1e-3 of the
 *         fp32 reference (measured ~3.5e-4) -- the throughput mode.
 *   FP32: every tensor-core operand as hi + lo fp16 planes, three MMA passes per product (~22 significant bits), fp32
 *         attention and libdevice erff GELU: embeddings within 1e-5 of the reference arithmetic. */
#define NOMAD_B200_PRECISION_FP16 0
#define NOMAD_B200_PRECISION_FP32 1

/* GEMM back end selector (``gemm_impl``): the tensor-core kernel is the product; the SIMT kernel
 * exists so the GPU tests can cross-check it on device. */
#define NOMAD_B200_GEMM_TCGEN05 0
#define NOMAD_B200_GEMM_SIMT 1

NOMAD_B200_API const char* nomad_b200_last_error(void);
NOMAD_B200_API const char* nomad_b200_version(void);

/* Replaces model construction + ``load_state_dict`` (nomad.py:53-68).  Folds weight-norm, permutes
 * conv weights to K-major, fuses q/k/v, converts to op_t and uploads to ``device``. */
NOMAD_B200_API int nomad_b200_create(nomad_b200_handle** out, const nomad_b200_tensor* tensors, int n_tensors,
                                     int precision_mode, int device);
/* Switch a handle created with NOMAD_B200_PRECISION_FP32 between the two arithmetic classes (a handle created with
 * NOMAD_B200_PRECISION_FP16 holds the fp16 weights only).  The scoring entry points (embed, score, layers_fwd and
 * their _host variants) honour the mode; the loss path always runs fp16 operands. */
NOMAD_B200_API int nomad_b200_set_precision(nomad_b200_handle* h, int precision_mode);
NOMAD_B200_API int nomad_b200_get_precision(nomad_b200_handle* h);
NOMAD_B200_API int nomad_b200_destroy(nomad_b200_handle* h);
NOMAD_B200_API int nomad_b200_set_gemm_impl(nomad_b200_handle* h, int gemm_impl);

/* Replaces the fresh ``nn.Linear(768, 256)`` of ``LossNetLayers`` (nomad.py:238-241): head used by the
 * 13th loss term.  Host pointers: w [256*768] row-major (out, in), b [256]. */
NOMAD_B200_API int nomad_b200_set_loss_head(nomad_b200_handle* h, const float* w, const float* b);

/* ---- scoring: ``TripletModel.forward`` for a batch of variable-length utterances -----------------
 * Replaces the per-file loop ``model(wave, lengths)`` of nomad.py:166-189 / 224-231.
 * ``wav`` is the concatenation of the B waveforms (fp32 mono 16 kHz); utterance i is
 * wav[sample_offsets[i] .. sample_offsets[i+1]).  ``sample_offsets`` is a HOST array of B+1 entries.
 * Every utterance is embedded exactly as if it were run alone (length-masked GroupNorm, positional
 * conv, attention and pooling).  ``emb`` receives B x 256 unit-norm fp32 rows.
 * Fails if an utterance is shorter than NOMAD_B200_MIN_SAMPLES (the reference raises RuntimeError). */
NOMAD_B200_API size_t nomad_b200_embed_workspace_bytes(const int64_t* sample_offsets, int B);
/* The plain *_workspace_bytes functions size the workspace for NOMAD_B200_PRECISION_FP16; a handle in FP32 mode needs
 * the size the *_mode variants report (hi + lo planes, fp32 QKV rows). */
NOMAD_B200_API size_t nomad_b200_embed_workspace_bytes_mode(const int64_t* sample_offsets, int B, int precision_mode);
NOMAD_B200_API int nomad_b200_embed(nomad_b200_handle* h, const float* wav_dev, const int64_t* sample_offsets, int B,
                     float* emb_dev, void* workspace_dev, size_t workspace_bytes, void* stream);
/* Same, HOST buffers in and out (pinned or pageable); H2D + compute + D2H + stream sync inside. */
NOMAD_B200_API int nomad_b200_embed_host(nomad_b200_handle* h, const float* wav_host, const int64_t* sample_offsets, int B,
                          float* emb_host, void* workspace_dev, size_t workspace_bytes, void* stream);

/* ---- loss: ``Nomad.forward(estimate, clean)`` (nomad.py:142-146, 243-282) + its backward ---------
 * est, clean: B x N fp32 device (the (B,1,N) tensors squeezed).  loss: 1 fp32 device.
 * d_est: B x N fp32 device = d loss / d estimate (already including ``feature_grad_mult``), or NULL
 * for forward only.  Weight gradients are not produced (wheel 0.0.8 semantics, see DESIGN.md). */
NOMAD_B200_API size_t nomad_b200_loss_workspace_bytes(int B, int64_t N, int with_grad);
NOMAD_B200_API int nomad_b200_loss_fwd_bwd(nomad_b200_handle* h, const float* est_dev, const float* clean_dev, int B, int64_t N,
                            float feature_grad_mult, float* loss_dev, float* d_est_dev, void* workspace_dev,
                            size_t workspace_bytes, void* stream);

/* ``LossNetLayers.forward`` (nomad.py:243-258): the 12 layer outputs (12 x B x T x 768 fp32, layer
 * major) and the head output (B x 256) for a fixed-length batch.  Either output may be NULL. */
NOMAD_B200_API size_t nomad_b200_layers_workspace_bytes(int B, int64_t N);
NOMAD_B200_API size_t nomad_b200_layers_workspace_bytes_mode(int B, int64_t N, int precision_mode);
NOMAD_B200_API int64_t nomad_b200_num_frames(int64_t n_samples);
NOMAD_B200_API int nomad_b200_layers_fwd(nomad_b200_handle* h, const float* wav_dev, int B, int64_t N, float* layers_dev,
                          float* emb_dev, void* workspace_dev, size_t workspace_bytes, void* stream);

/* ---- distance: ``cdist(test, nmr)`` + ``np.mean(axis=1)`` (nomad.py:108,111) ---------------------
 * deg: n x 256, nmr: m x 256 fp32 device.  dm (n x m fp32 device, may be NULL when only the means are
 * wanted) and row_mean (n fp64 device; NaN when m == 0, like np.mean of an empty row).  Row means are summed in a
 * fixed order: bit-identical from run to run.  No handle: the kernel has no weights. */
NOMAD_B200_API size_t nomad_b200_cdist_workspace_bytes(int64_t n, int64_t m);
NOMAD_B200_API int nomad_b200_cdist_mean(const float* deg_dev, int64_t n, const float* nmr_dev, int64_t m, float* dm_dev,
                          double* row_mean_dev, void* workspace_dev, size_t workspace_bytes, int gemm_impl,
                          void* stream);
NOMAD_B200_API int nomad_b200_cdist_mean_host(const float* deg_host, int64_t n, const float* nmr_host, int64_t m, float* dm_host,
                               double* row_mean_host, void* workspace_dev, size_t workspace_bytes, void* stream);

/* ---- one batch of ``Nomad.predict``: the per-file ``model(wave)`` calls (nomad.py:166-189) for B utterances followed by
 * ``cdist`` + ``np.mean`` of their embeddings against a resident NMR set (nomad.py:108,111) -- one call, no host round
 * trip in between.  nmr: m x 256 fp32 DEVICE rows (e.g. the all-gathered NMR embeddings of the sharded scoring path).
 * Outputs: emb B x 256, dm B x m fp32 (may be NULL), row_mean B fp64.  The ``_host`` variant takes the waveforms from
 * HOST memory (staged H2D overlapping the front end), writes its outputs to HOST memory (emb_host / dm_host may be
 * NULL) and synchronises the stream. */
NOMAD_B200_API size_t nomad_b200_score_workspace_bytes(const int64_t* sample_offsets, int B, int64_t m);
NOMAD_B200_API size_t nomad_b200_score_workspace_bytes_mode(const int64_t* sample_offsets, int B, int64_t m, int precision_mode);
NOMAD_B200_API int nomad_b200_score(nomad_b200_handle* h, const float* wav_dev, const int64_t* sample_offsets, int B,
                     const float* nmr_dev, int64_t m, float* emb_dev, float* dm_dev, double* row_mean_dev,
                     void* workspace_dev, size_t workspace_bytes, void* stream);
NOMAD_B200_API int nomad_b200_score_host(nomad_b200_handle* h, const float* wav_host, const int64_t* sample_offsets, int B,
                          const float* nmr_dev, int64_t m, float* emb_host, float* dm_host, double* row_mean_host,
                          void* workspace_dev, size_t workspace_bytes, void* stream);

/* ---- result formatting: ``df.round(3)`` + ``to_csv`` (nomad.py:113-120, 138-139) without pandas ------------------
 * Writes ``index_name,col_labels...`` then one line per row: ``row_label,v,v,...`` with every value rounded like
 * numpy (rint(x * 10^decimals) / 10^decimals; decimals < 0 = no rounding) and printed like Python's repr (shortest
 * round-trip digits, "1.0", "1e-05"); NaN -> empty field, labels quoted like csv.QUOTE_MINIMAL.  The bytes equal
 * what the reference's pandas calls write.  HOST pointers, host threads (0 = all cores); no GPU involved. */
NOMAD_B200_API int nomad_b200_write_scores_csv(const char* path, const char* index_name, const char* const* row_labels,
                                int64_t n_rows, const char* const* col_labels, int64_t n_cols, const double* values,
                                int decimals, int threads);

/* Paired distances d[i] = ||a[i] - b[i]|| (fp64 out): the diagonal of ``cdist`` that the reference's full-reference
 * evaluation takes (src/training/train_triplet.py:267-274), without materialising the matrix.  a, b: n x 256 fp32
 * device. */
NOMAD_B200_API int nomad_b200_paired_dist(const float* a_dev, const float* b_dev, int64_t n, double* out_dev, void* stream);

/* ---- triplet fine-tuning step (reference src/training/train_triplet.py:112-133; conv feature encoder frozen as in
 * src/config/train_triplet.yaml `freeze_convnet: True`) ---------------------------------------------------------------
 * wav: 3B x N fp32 device rows: B anchors, then B positives, then B negatives (the zero-padded batches of the
 * reference's collate_fn).  Computes the embeddings of all three, loss = nn.TripletMarginLoss(margin)(A, P, N) and the
 * gradient of the loss wrt EVERY trainable parameter: LayerNorm(512), feature projection, positional conv (as the
 * gradient of the weight-norm-folded weight), encoder LayerNorm, the 12 transformer layers (q/k/v fused, q rows carrying
 * the head_dim^-0.5 scale) and the embedding head.  Activation gradients run the loss path's dgrad chain; every weight
 * gradient dW = dY^T X is a tensor-core GEMM over the token dimension.  grads: nomad_b200_triplet_grad_floats() fp32
 * values laid out as nomad_b200_triplet_grad_segment enumerates, all multiplied by *grad_scale_out (a power of two
 * that keeps 16-bit activation gradients in range; divide it out).  The optimiser step itself (Adam, train_triplet.py:
 * 92-107) is host plumbing: see nomad_b200/triplet.py. */
/* After the optimiser step (train_triplet.py:129-130): rebuild the kernel-ready weights of everything trainable (16-bit
 * copies, fused q|k|v with the q scale, transposes for the dgrad GEMMs, LayerNorm folds, weight-norm fold of the positional
 * conv, head) from fp32 master tensors that live on the DEVICE -- same names as nomad_b200_create, `data` = device pointers.
 * A few bandwidth-bound kernels on `stream`; the frozen conv feature encoder is not touched. */
NOMAD_B200_API int nomad_b200_refresh_weights(nomad_b200_handle* h, const nomad_b200_tensor* tensors_dev, int n_tensors, void* stream);
/* Test hook for the refresh path: copy one kernel-ready weight buffer to the host (see refresh.cu for the names). */
NOMAD_B200_API int nomad_b200_debug_read_weight(nomad_b200_handle* h, const char* which, void* dst_host, size_t bytes);
NOMAD_B200_API int64_t nomad_b200_triplet_grad_floats(void);
NOMAD_B200_API int nomad_b200_triplet_grad_segment(int i, char* name, int name_cap, int64_t* offset, int64_t* numel);
NOMAD_B200_API size_t nomad_b200_triplet_workspace_bytes(int B, int64_t N);
NOMAD_B200_API int nomad_b200_triplet_fwd_bwd(nomad_b200_handle* h, const float* wav_dev, int B, int64_t N, float margin,
                               float* loss_dev, float* grads_dev, float* grad_scale_out, void* workspace_dev,
                               size_t workspace_bytes, void* stream);

/* ---- building block exposed for the parity tests --------------------------------------------------
 * C (m x n, ldc) = epilogue(A (m x k op_t, row stride lda elements, may overlap) * B^T (n x k op_t)).
 * flags: 1 bias, 2 GELU(erf), 4 + residual fp32 (ld = ldc), 8 store fp32 (c_f32), 16 store op_t (c_f16).
 * a_rows = rows addressable in A's buffer; k_wrap as documented in DESIGN.md (0 = plain). */
NOMAD_B200_API int nomad_b200_gemm_f16(const void* a_f16, int64_t a_rows, int64_t lda, int k_wrap, const void* b_f16, int m,
                         int n, int k, int batch, int64_t a_bstride, int64_t b_bstride, int64_t c_bstride,
                         const float* bias, const float* resid, float* c_f32, void* c_f16, int64_t ldc, int flags,
                         int gemm_impl, void* stream);

/* Same building block in fp32-class mode (NOMAD_B200_PRECISION_FP32): A and B as hi + lo fp16 planes, three K segments
 * (A_hi B_hi + A_lo B_hi + A_hi B_lo) into one accumulator, times acc_scale, then flags 1 bias, 2 GELU (libdevice erff),
 * 8 store fp32 (c_f32), 16 store hi + lo planes (c_hi, c_lo).  A: m x k (row stride lda), B: n x k, C: m x n (ldc). */
NOMAD_B200_API int nomad_b200_gemm_split(const void* a_hi, const void* a_lo, int64_t lda, const void* b_hi, const void* b_lo,
                          int m, int n, int k, float acc_scale, const float* bias, float* c_f32, void* c_hi, void* c_lo,
                          int64_t ldc, int flags, void* stream);

/* ---- ingest: ``Nomad.load_processing`` (nomad.py:192-212) after the file has been decoded to PCM ------------
 * pcm: n_frames x channels interleaved int16 DEVICE samples at ``sr`` Hz.  out: mono fp32 at ``target_sr``:
 * sample / 32768, mean of the first two channels when channels > 1 (nomad.py:199-200), torchaudio's default
 * ``Resample(sr, target_sr)`` (sinc-Hann, width 6, rolloff 0.99; nomad.py:203-205) when the rates differ, cut to
 * 10 s when ``trim`` (nomad.py:208-210).  ``nomad_b200_ingest_out_samples`` gives the output length (host only). */
NOMAD_B200_API int64_t nomad_b200_ingest_out_samples(int64_t n_frames, int sr, int target_sr, int trim);
NOMAD_B200_API int nomad_b200_ingest_pcm16(const int16_t* pcm_dev, int64_t n_frames, int channels, int sr, int target_sr, int trim,
                            float* out_dev, void* stream);

/* Sample formats of the wav files the native reader handles (``torchaudio.load`` decode, nomad.py:196), each decoded to
 * fp32 exactly as the host path ``nomad_b200.audio.load_wav`` does: U8 (x - 128) / 128; S16 x / 2^15; S24 (packed
 * 3-byte little-endian) x / 2^23; S32 float32(x) rounded to nearest, then / 2^31; F32 as is; F64 rounded to fp32.  The
 * container width decides the format (WAVE_FORMAT_EXTENSIBLE's valid-bits field is ignored, as ``wave`` ignores it). */
#define NOMAD_B200_WAV_U8 1
#define NOMAD_B200_WAV_S16 2
#define NOMAD_B200_WAV_S24 3
#define NOMAD_B200_WAV_S32 4
#define NOMAD_B200_WAV_F32 5
#define NOMAD_B200_WAV_F64 6

/* One file of a batched ingest (``load_processing`` of nomad.py:192-212 for n files in one call).  Its raw data bytes
 * (n_frames x channels interleaved samples of ``format``, as stored in the file) start at src_dev + byte_offset, which
 * must be aligned to the sample size (1 for U8 and S24).  The first out_samples mono fp32 samples at ``target_sr`` --
 * mean of the first two channels when channels > 1 (nomad.py:199-200), torchaudio's default Resample when the rates
 * differ (nomad.py:203-205) -- go to out_dev + out_offset.  out_samples is at most
 * nomad_b200_ingest_out_samples(n_frames, sample_rate, target_sr, 0); passing
 * nomad_b200_ingest_out_samples(..., 1) gives the 10 s trim (nomad.py:208-210). */
typedef struct {
    int64_t byte_offset;
    int64_t n_frames;
    int64_t out_offset;
    int64_t out_samples;
    int32_t channels;
    int32_t format;       /* NOMAD_B200_WAV_* */
    int32_t sample_rate;
    int32_t reserved;     /* 0 */
} nomad_b200_ingest_item;

/* ``load_processing`` for a batch of wav files, still undecoded: src_dev holds the raw data bytes of all of them, items is a
 * HOST array of n descriptors.  One kernel launch for the items already at target_sr plus one per distinct other
 * sample rate, whatever n is.  The device copy of the descriptor table lives in the caller's workspace (size from
 * ``nomad_b200_ingest_workspace_bytes``, 0 = bad descriptors, see ``nomad_b200_last_error``).  S16 items give the
 * same bits as ``nomad_b200_ingest_pcm16``. */
NOMAD_B200_API size_t nomad_b200_ingest_workspace_bytes(const nomad_b200_ingest_item* items, int64_t n, int target_sr);
NOMAD_B200_API int nomad_b200_ingest_batch(const void* src_dev, const nomad_b200_ingest_item* items, int64_t n, int target_sr,
                                           float* out_dev, void* workspace_dev, size_t workspace_bytes, void* stream);

/* Decode step of ``load_processing`` (``torchaudio.load``, nomad.py:196) for 16-bit PCM RIFF/WAVE files, on `threads` host
 * threads (0 = all cores), no GPU involved.  ``wav_probe`` parses the headers: frames[i] = -1 marks a file that is not
 * plain 16-bit PCM (the caller decodes it some other way).  ``wav_read_pcm16`` then reads n_samples[i] (= frames x channels)
 * interleaved samples of file i, starting at data_offset[i], into dst + dst_offset[i] -- e.g. a pinned staging buffer
 * laid out in batch order, so the whole batch crosses PCIe in one copy. */
NOMAD_B200_API int nomad_b200_wav_probe(const char* const* paths, int64_t n, int32_t* sample_rate, int32_t* channels,
                         int64_t* frames, int64_t* data_offset, int threads);
NOMAD_B200_API int nomad_b200_wav_read_pcm16(const char* const* paths, int64_t n, const int64_t* data_offset,
                              const int64_t* n_samples, const int64_t* dst_offset, int16_t* dst, int threads);
/* The same for every format above (``torchaudio.load``, nomad.py:196; decoded on the device by
 * ``nomad_b200_ingest_batch``).  ``wav_probe_format`` accepts format tag 1 (PCM, 8/16/24/32 bits), tag 3 (IEEE float,
 * 32/64 bits) and WAVE_FORMAT_EXTENSIBLE with the full PCM or IEEE_FLOAT sub-format GUID, with block_align = channels x
 * sample bytes; format[i] = NOMAD_B200_WAV_*, or frames[i] = -1 and format[i] = 0 for anything else (u-law, A-law,
 * ADPCM, RIFX, a ``data`` chunk before ``fmt ``, unreadable files).  frames counts the whole frames present (a truncated
 * ``data`` chunk is cut at the end of the file).  ``wav_probe`` / ``wav_read_pcm16`` above are this parser and reader
 * restricted to S16.  ``wav_read`` reads n_bytes[i] bytes of file i from byte src_offset[i] to (char*)dst +
 * dst_offset[i]. */
NOMAD_B200_API int nomad_b200_wav_probe_format(const char* const* paths, int64_t n, int32_t* sample_rate, int32_t* channels,
                                               int64_t* frames, int64_t* data_offset, int32_t* format, int threads);
NOMAD_B200_API int nomad_b200_wav_read(const char* const* paths, int64_t n, const int64_t* src_offset, const int64_t* n_bytes,
                                       const int64_t* dst_offset, void* dst, int threads);

/* The attention core of one encoder layer, softmax(Q K^T) V per (utterance, head) (fairseq
 * MultiheadAttention inside TransformerSentenceEncoderLayer; mirror torchaudio components.py:237-330).
 * qkv: frames x 2304 op_t device (q | k | v per row, q already scaled by head_dim^-0.5); utterance u owns rows
 * [frame0[u], frame0[u] + T[u]) (HOST arrays).  out: frames x 768 op_t device (rows of valid frames are written);
 * lse: frames x 12 fp32 device (log-sum-exp of each softmax row, used by the loss backward) or NULL.
 * workspace: device scratch for the kernel's work list. */
NOMAD_B200_API size_t nomad_b200_attention_workspace_bytes(const int32_t* T, int n_utts);
NOMAD_B200_API int nomad_b200_attention_f16(const void* qkv_f16, int64_t frames, const int32_t* frame0, const int32_t* T,
                             int n_utts, void* out_f16, float* lse, void* workspace_dev, size_t workspace_bytes,
                             void* stream);

/* In-situ timing of the tensor-core GEMM launches (one CUDA event pair per launch, on the launching
 * stream) for the roofline leg of bench.py: enable, run steps, read the summed device time (ms), the
 * algorithmic FLOPs (2*M*N*K) and the launch count; reading synchronises on the recorded events. */
NOMAD_B200_API int nomad_b200_profile_gemm(int enable);
NOMAD_B200_API int nomad_b200_profile_gemm_read(double* total_ms, double* total_flops, int64_t* launches);

/* Number of kernels this library has launched in this process (bench.py's ``gpu_launches``). */
NOMAD_B200_API int64_t nomad_b200_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* NOMAD_B200_H */
