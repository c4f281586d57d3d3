/* wenet_b200.h — C ABI of libwenet_b200.so: the B200 (sm_100a) Conformer ASR inference hot path
 * (fbank -> ConformerEncoder -> CTC -> ctc_prefix_beam_search -> attention_rescoring) behind WeNet's
 * Python API.  This is the drop-in boundary: plain C, raw device pointers, explicit sizes, a
 * cudaStream_t, int return codes.  No torch types.
 *
 * Conventions (modelled on the reference's own C API, runtime/core/api/wenet_api.h:26-107:
 * opaque handle, init/free, plain scalars, library-owned result strings):
 *   - every function returns 0 (WB_OK) or a negative wb_status; wb_last_error() gives the message
 *     (thread-local, owned by the library — same ownership rule as wenet_get_result,
 *     wenet_api.h:73).  Nothing throws, nothing aborts.
 *   - "dev" pointers are CUDA device pointers on the current device, "host" pointers are CPU.
 *     The caller owns all inputs, outputs and workspaces (PyTorch allocates them so its caching
 *     allocator / stream semantics hold); the library owns only the weights it was given
 *     (wb_model_set_tensor copies) and its TMA descriptors.
 *   - a wb_model is immutable after wb_model_finalize(): concurrent calls from several host
 *     threads on different streams are safe as long as they use different workspaces (mirrors
 *     TorchAsrModel::Copy sharing one module, runtime/core/decoder/torch_asr_model.cc:87-111).
 *   - one model handle per GPU; cudaSetDevice is the caller's job.  No collectives: utterances
 *     shard independently across GPUs (SURVEY.md section 8e).
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails with
 *     WB_ERR_CUDA.
 *
 * Each entry point cites the reference interface it replaces (file:line under the reference repo).
 */
#ifndef WENET_B200_H_
#define WENET_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* wb_stream_t; /* cudaStream_t */

typedef enum {
  WB_OK = 0,
  WB_ERR_BAD_ARG = -1,
  WB_ERR_UNSUPPORTED = -2, /* configuration outside the implemented set (no silent fallback) */
  WB_ERR_CUDA = -3,
  WB_ERR_NOT_LOADED = -4, /* a required weight tensor is missing */
  WB_ERR_WORKSPACE = -5   /* caller workspace too small */
} wb_status;

const char* wb_last_error(void);
const char* wb_version(void);
/* number of CUDA kernels this library has launched in this process (bench.py: gpu_launches) */
unsigned long long wb_launch_count(void);

/* Per-kernel-family profiler: when enabled, every launch is bracketed by CUDA events on the
 * launching stream.  wb_prof_collect synchronises the device and returns, per tag, the summed
 * elapsed ms, the summed algorithmic work (FLOPs for gemm_tcgen05, bytes for the memory-bound
 * kernels, 0 where not tracked) and the number of launches since wb_prof_reset. */
/* the persistent GEMM kernels use (num_SMs - n) CTAs, leaving n SMs for latency-bound kernels (prefix beam
 * search) of other in-flight batches running on other streams; default 0 */
void wb_set_sm_reserve(int n);
void wb_prof_enable(int on);
void wb_prof_reset(void);
int wb_prof_num_tags(void);
const char* wb_prof_tag_name(int tag);
int wb_prof_collect(double* ms, double* work, long long* launches);
/* Stall accounting of the tcgen05 GEMM kernel (cycles, summed over CTAs and launches since the last reset):
 * out8 = {producer waits for a ring slot, MMA waits for operands, MMA waits for a drained accumulator stage,
 * epilogue waits for an accumulator, epilogue waits for its staging buffer, epilogue loop time (one warp),
 * CTA lifetime, tiles, epilogue tcgen05.ld wait, epilogue bias + activation, epilogue staging stores + TMA issue, 0}
 * (12 values).  Tuning aid used by tools/bench_ops.py; out12 may be NULL (reset only).  The accounting is compiled
 * into the kernel only when the library is built with -DWB_GEMM_DIAG (NVCC_EXTRA=-DWB_GEMM_DIAG python -m
 * wenet_b200.build --force); the default build returns WB_ERR_UNSUPPORTED. */
int wb_gemm_diag(uint64_t* out12, int reset);

/* ------------------------------------------------------------------------------------------
 * A. fbank  — replaces wenet/dataset/processor.py:226-256 compute_fbank, i.e.
 *    torchaudio.compliance.kaldi.fbank(waveform*32768, num_mel_bins, 25 ms / 10 ms, dither 0,
 *    energy_floor 0, povey window)  (torchaudio/compliance/kaldi.py:514-645)
 * ------------------------------------------------------------------------------------------ */
typedef struct wb_fbank wb_fbank;
/* window[frame_len] and mel[num_mel][nfft/2+1] are host arrays computed by the caller with the
 * reference formulas (povey window kaldi.py:99-100, mel banks :436-511 incl. the zero last column
 * :627); preemph = 0.97. */
int wb_fbank_create(wb_fbank** out, int num_mel, int frame_len, int frame_shift, float preemph,
                    const float* window_host, const float* mel_host);
void wb_fbank_destroy(wb_fbank* fb);
/* pcm_dev: [batch][pcm_stride] float32 (pcm_is_int16 = 0) or int16 (= 1); num_samples_dev[batch].
 * Each sample is multiplied by `scale` (32768 for [-1,1) float input, processor.py:245; 1 for
 * int16).  feats_dev: [batch][frames_stride][num_mel] float32; frames past an utterance's own count
 * 1 + (n - frame_len) / frame_shift are written as 0 (zero padding of processor.padding,
 * processor.py:562-566). */
int wb_fbank_forward(const wb_fbank* fb, const void* pcm_dev, int pcm_is_int16, int64_t pcm_stride,
                     const int32_t* num_samples_dev, int batch, float scale, float* feats_dev,
                     int64_t frames_stride, int max_frames, wb_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Model handle — the packed weights of one ASRModel (ConformerEncoder + CTC + optional
 * (Bi)TransformerDecoder); replaces load_state_dict on the reference modules
 * (wenet/utils/checkpoint.py:26-43).  Tensor names/layouts are produced by the host-side packer
 * wenet_b200/weights.py from the reference state_dict keys (SURVEY.md section 8a key table).
 * ------------------------------------------------------------------------------------------ */
typedef struct wb_model wb_model;

typedef struct {
  int32_t input_dim;   /* 80 */
  int32_t d_model;     /* encoder_conf.output_size */
  int32_t heads;       /* attention_heads (d_model / heads must be 64) */
  int32_t ffn_dim;     /* linear_units */
  int32_t enc_layers;  /* num_blocks */
  int32_t cnn_kernel;  /* cnn_module_kernel */
  int32_t cnn_causal;  /* causal */
  int32_t cnn_norm;    /* 0 = layer_norm, 1 = batch_norm (folded, eval) */
  int32_t vocab;       /* output_dim; 0 = encoder-only handle (no CTC head, no decoder) */
  int32_t dec_layers;  /* left (l2r) decoder blocks, 0 = no decoder */
  int32_t rdec_layers; /* right (r2l) decoder blocks, 0 = none */
  int32_t dec_heads;
  int32_t dec_ffn_dim;
  int32_t max_pos;     /* positional-encoding table length (5000) */
  int32_t has_cmvn;    /* GlobalCMVN present */
  int32_t precise;     /* 0: bf16 operands (throughput mode).  1: PARITY mode - every encoder / CTC GEMM runs as bf16x3
                          (activations [hi | lo | hi], weights [hi | hi | lo] along K: the packer must deliver the
                          encoder, conv2, embed and CTC weights as [N][3K]), q/k/v, attention and the depthwise conv
                          in fp32 on CUDA cores: encoder_out / CTC log-probs within 1e-3 of the fp32 reference.
                          enc_out_bf16_dev then has 3 * d_model columns ([hi | lo | hi]) everywhere in this API;
                          the rescoring decoder reads its hi block and stays bf16.  Full forward only. */
  float ln_eps;        /* encoder LayerNorm eps (encoder_conf.norm_eps, 1e-5) */
  float dec_ln_eps;    /* decoder LayerNorm eps (decoder_conf.norm_eps, decoder.py:83); <= 0 means "same as ln_eps" */
  int32_t arch;        /* 0: ConformerEncoder (conv2d subsampling, rel-pos attention, conv module) - everything above.
                          1: Whisper = TransformerEncoder with input_layer conv1d2 (Conv1dSubsampling2, subsampling.py:117-171),
                             pos_enc abs_pos_whisper (embedding.py:150-164), gelu FFN, key_bias false, pre-norm
                             (wenet/models/whisper/whisper.py:28-96, encoder.py:365-440, encoder_layer.py:28-135);
                             cnn_* / has_cmvn / precise are ignored (must be 0) */
  int32_t dec_flavor;  /* 0: wenet TransformerDecoder input_layer "embed" (sinusoid PE, x*sqrt(d), relu).
                          1: Whisper decoder: input_layer embed_learnable_pe (embedding.py:167-176, xscale 1), gelu;
                             key_bias false and tie_word_embedding are weight-level properties (the packer delivers a zero
                             key bias and the tied output matrix) */
  int32_t dec_max_len; /* dec_flavor 1: rows of the learnable decoder position table (448) */
} wb_model_config;

enum { WB_F32 = 0, WB_BF16 = 1, WB_I32 = 2 };

int wb_model_create(wb_model** out, const wb_model_config* cfg);
void wb_model_destroy(wb_model* m);
/* copies `host_data` (numel elements of dtype) to the device under `name` */
int wb_model_set_tensor(wb_model* m, const char* name, const void* host_data, int dtype,
                        int64_t numel);
/* checks that every required tensor is present, builds TMA descriptors and the per-layer
 * relative-position projections P_l = linear_pos(pe) (weight-only, attention.py:395-397) */
int wb_model_finalize(wb_model* m, wb_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * B. encoder — replaces ConformerEncoder.forward (wenet/models/transformer/encoder.py:122-181):
 *    GlobalCMVN -> Conv2dSubsampling4 -> RelPositionalEncoding -> N x ConformerEncoderLayer ->
 *    after_norm.  Output is PACKED: rows of all utterances' valid frames back to back
 *    (utterance b occupies rows [seq_start[b], seq_start[b] + T'_b), T'_b = ((T_b-1)/2-1)/2);
 *    wb_unpack_rows scatters into the reference's padded (B, T'max, d) layout.
 *    decoding_chunk_size < 0: full attention; > 0: chunk mask of mask.py:88-123 with
 *    num_left_chunks (mask.py:164-173); 0 (random training chunk) is rejected.
 * ------------------------------------------------------------------------------------------ */
size_t wb_encoder_workspace_bytes(const wb_model* m, int batch, const int32_t* feat_lens_host);
/* total packed rows M = sum_b T'_b (also returned through *out_rows by wb_encoder_forward) */
int64_t wb_encoder_out_rows(int batch, const int32_t* feat_lens_host);
int wb_encoder_forward(const wb_model* m, const float* feats_dev, int64_t feats_stride_b,
                       const int32_t* feat_lens_host, int batch, int decoding_chunk_size,
                       int num_decoding_left_chunks, int pad_to_frames /* T'max of the padded batch (symmetric conv quirk) */,
                       float* enc_out_dev /* [M][d] fp32 */, void* enc_out_bf16_dev /* [M][d] bf16 */,
                       int32_t* seq_start_dev /* [batch] */, int32_t* seq_len_dev /* [batch] */,
                       float* layer_dump_dev /* optional [(layers+1)][M][d]: embed out, then each layer */,
                       void* workspace_dev, size_t workspace_bytes, wb_stream_t stream);

/* streaming step — replaces BaseEncoder.forward_chunk (encoder.py:204-300), batch 1.
 * xs_dev [T][input_dim]; att_cache_dev [layers][heads][cache_t1][128] (K|V halves) or NULL when
 * cache_t1 = 0; cnn_cache_dev [layers][d][cnn_kernel-1] or NULL (first chunk);
 * outputs: y [chunk][d]; r_att_cache [layers][heads][cache_t1+chunk-next_cache_start][128];
 * r_cnn_cache [layers][d][cnn_kernel-1]. */
size_t wb_encoder_chunk_workspace_bytes(const wb_model* m, int T, int cache_t1);
int wb_encoder_forward_chunk(const wb_model* m, const float* xs_dev, int T, int offset,
                             int required_cache_size, const float* att_cache_dev, int cache_t1,
                             const float* cnn_cache_dev, float* y_dev, float* r_att_cache_dev,
                             float* r_cnn_cache_dev, int* out_chunk, int* out_new_cache_t1,
                             void* workspace_dev, size_t workspace_bytes, wb_stream_t stream);
/* Capture-safe form of the same step for CUDA graphs (steady-state streaming: T, cache_t1 and the buffers are
 * fixed, only the position changes): issues no host -> device copy and no synchronisation, reads the position
 * offset from offset_dev (device int32; positions are clamped to the table), and expects the workspace to have been
 * used by a regular wb_encoder_forward_chunk call with the same T / cache_t1 before (that call leaves the small
 * shape block in it).  Capture it once (e.g. torch.cuda.CUDAGraph), then per chunk: write xs / offset, replay. */
int wb_encoder_forward_chunk_static(const wb_model* m, const float* xs_dev, int T, const int32_t* offset_dev,
                                    int required_cache_size, const float* att_cache_dev, int cache_t1,
                                    const float* cnn_cache_dev, float* y_dev, float* r_att_cache_dev,
                                    float* r_cnn_cache_dev, void* workspace_dev, size_t workspace_bytes,
                                    wb_stream_t stream);

/* Batched streaming - `sessions` concurrent forward_chunk streams advanced in lockstep by one encoder pass (SURVEY
 * section 8f-4; the batched-cache design of wenet/bin/export_onnx_gpu.py:83-232 StreamingEncoder).  Per session the
 * arithmetic is that of wb_encoder_forward_chunk (encoder.py:204-300), row for row; the GEMMs see sessions x chunk rows.
 * All sessions share T and cache_t1; each has its own position offset.  bf16 mode only.
 * xs_dev [S][T][input_dim]; att_cache_dev [S][layers][heads][cache_t1][128] (NULL when cache_t1 = 0); cnn_cache_dev
 * [S][layers][d][cnn_kernel-1] (NULL: first chunk); y_dev [S][chunk][d]; r_att_cache_dev [S][layers][heads][new_t1][128];
 * r_cnn_cache_dev like cnn_cache_dev.  The _static form is capture-safe (offsets read from the device, no copy, no
 * synchronisation; the workspace must have been used by a regular call with the same T / cache_t1 / sessions before). */
size_t wb_encoder_chunk_batch_workspace_bytes(const wb_model* m, int T, int cache_t1, int sessions);
int wb_encoder_forward_chunk_batch(const wb_model* m, const float* xs_dev, int T, int sessions,
                                   const int32_t* offsets_host, int required_cache_size, const float* att_cache_dev,
                                   int cache_t1, const float* cnn_cache_dev, float* y_dev, float* r_att_cache_dev,
                                   float* r_cnn_cache_dev, int* out_chunk, int* out_new_cache_t1, void* workspace_dev,
                                   size_t workspace_bytes, wb_stream_t stream);
int wb_encoder_forward_chunk_batch_static(const wb_model* m, const float* xs_dev, int T, int sessions,
                                          const int32_t* offsets_dev, int required_cache_size,
                                          const float* att_cache_dev, int cache_t1, const float* cnn_cache_dev,
                                          float* y_dev, float* r_att_cache_dev, float* r_cnn_cache_dev,
                                          void* workspace_dev, size_t workspace_bytes, wb_stream_t stream);

/* packed [M][d] -> padded [batch][t_stride][d] (rows past seq_len zeroed) and back */
int wb_unpack_rows(const float* packed_dev, const int32_t* seq_start_dev, const int32_t* seq_len_dev,
                   int batch, int max_len, int d, float* padded_dev, int64_t t_stride, wb_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * C. CTC posteriors — replaces ASRModel.ctc_logprobs / CTC.log_softmax
 *    (asr_model.py:254-265, ctc.py:73-81) + the per-frame logp.topk(beam) of search.py:158.
 *    logp_dev [M][ldl] fp32 (ldl >= vocab, multiple of 4) receives the full log-probabilities.
 * ------------------------------------------------------------------------------------------ */
int wb_ctc_logprobs(const wb_model* m, const void* enc_out_bf16_dev, int64_t rows, int blank_id,
                    float blank_penalty, float* logp_dev, int64_t ldl, int topk, float* topk_val_dev,
                    int32_t* topk_idx_dev, wb_stream_t stream);

/* Same posteriors, but only the per-frame top-k leaves the kernel: topk_val_dev [M][topk] holds the log-probabilities
 * (log-softmax normalised, blank penalty applied) of the topk best tokens in (value desc, index asc) order and
 * topk_idx_dev their ids.  logits_scratch_dev [M][ldl] receives the RAW CTC logits (not normalised); it is scratch
 * for the caller.  This is what decode() uses: the [frames, V] matrix is read twice and never rewritten. */
int wb_ctc_topk(const wb_model* m, const void* enc_out_bf16_dev, int64_t rows, int blank_id, float blank_penalty,
                float* logits_scratch_dev, int64_t ldl, int topk, float* topk_val_dev, int32_t* topk_idx_dev,
                wb_stream_t stream);

/* D1. replaces ctc_greedy_search (search.py:109-124) + remove_duplicates_and_blank
 *     (wenet/utils/ctc_utils.py:23-33).  tokens_dev [batch][out_stride], lens_dev [batch]. */
int wb_ctc_greedy_search(const int32_t* topk_idx_dev, int topk, const int32_t* seq_start_dev,
                         const int32_t* seq_len_dev, int batch, int blank_id, int32_t* tokens_dev,
                         int out_stride, int32_t* lens_dev, wb_stream_t stream);

/* D2. replaces ctc_prefix_beam_search (search.py:127-249; scores are IEEE doubles, log_add of
 *     common.py:302-310).  Outputs per utterance up to `beam` hypotheses, best first:
 *     tokens/times [batch][beam][max_len], lens [batch][beam], scores [batch][beam], nhyp [batch]. */
size_t wb_prefix_beam_workspace_bytes(int batch, int beam, int max_len);
int wb_ctc_prefix_beam_search(const float* topk_val_dev, const int32_t* topk_idx_dev, int topk,
                              const int32_t* seq_start_dev, const int32_t* seq_len_dev, int batch,
                              int beam, int blank_id, int max_len, int32_t* tokens_dev,
                              int32_t* times_dev, int32_t* lens_dev, double* scores_dev,
                              int32_t* nhyp_dev, void* workspace_dev, size_t workspace_bytes,
                              wb_stream_t stream);

/* D2 with context biasing - replaces ctc_prefix_beam_search(..., context_graph) (search.py:127-249 incl. :171-173,
 *     :200-203, :229-234) with wenet/utils/context_graph.py:212-265 walked inside the kernel.  The graph is the
 *     reference's Aho-Corasick trie flattened by the host (wenet_b200/context.py): node 0 = root (token -1), children of
 *     node n = entries [child_off[n], child_off[n+1]) of (child_tok, child_node) sorted by token, fail arcs, and the
 *     per-node token / node / output scores as doubles.  All pointers are DEVICE pointers.  cg == NULL or
 *     num_nodes == 0: identical to wb_ctc_prefix_beam_search.  scores_dev then holds total_score() after finalize(). */
typedef struct {
  int32_t num_nodes;
  const int32_t* child_off;   /* [num_nodes + 1] */
  const int32_t* child_tok;   /* [num_edges] */
  const int32_t* child_node;  /* [num_edges] */
  const int32_t* fail;        /* [num_nodes] */
  const int32_t* token;       /* [num_nodes] */
  const double* node_score;   /* [num_nodes] */
  const double* token_score;  /* [num_nodes] */
  const double* output_score; /* [num_nodes] */
} wb_context_graph;
int wb_ctc_prefix_beam_search_ctx(const float* topk_val_dev, const int32_t* topk_idx_dev, int topk,
                                  const int32_t* seq_start_dev, const int32_t* seq_len_dev, int batch, int beam,
                                  int blank_id, int max_len, const wb_context_graph* cg, int32_t* tokens_dev,
                                  int32_t* times_dev, int32_t* lens_dev, double* scores_dev, int32_t* nhyp_dev,
                                  void* workspace_dev, size_t workspace_bytes, wb_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * E. attention rescoring — replaces attention_rescoring (search.py:374-458) and
 *    ASRModel.forward_attention_decoder (asr_model.py:453-547): (Bi)TransformerDecoder over all
 *    hypotheses of all utterances in one batch, cross-attention K/V projected once per utterance; with
 *    host-side tokens (wb_attention_rescoring) decoder rows of an utterance that share an input prefix are
 *    computed once (bit-identical to computing every row, which wb_attention_rescoring_dev does).
 *    Hypotheses are given flattened, utterance-major: hyp h belongs to utterance hyp_utt[h]
 *    (non-decreasing), has hyp_len[h] tokens at hyp_tokens[hyp_tok0[h] ...].
 *    Outputs: tok_logp_l2r/r2l [R] with R = sum_h (len_h + 1): log p of token j of hyp h at row
 *    hyp_row0[h] + j, the <eos> term at + len_h (r2l rows are indexed by decoder position);
 *    hyp_score[h] = (1-rw)*l2r + rw*r2l + ctc_weight*ctc_score (fp32, reference summation order);
 *    best[b] = index (within utterance b) of the first maximum.
 * ------------------------------------------------------------------------------------------ */
size_t wb_rescoring_workspace_bytes(const wb_model* m, int64_t enc_rows, int64_t total_tokens_plus_hyps);
int wb_attention_rescoring(const wb_model* m, const void* enc_out_bf16_dev, int64_t enc_rows,
                           const int32_t* seq_start_host, const int32_t* seq_len_host, int batch,
                           int n_hyp, const int32_t* hyp_utt_host, const int32_t* hyp_len_host,
                           const int32_t* hyp_tok0_host, const int32_t* hyp_tokens_host,
                           const double* ctc_score_host, int sos, int eos, float ctc_weight,
                           float reverse_weight, float* tok_logp_l2r_dev, float* tok_logp_r2l_dev,
                           float* hyp_score_dev, int32_t* best_dev, void* workspace_dev,
                           size_t workspace_bytes, wb_stream_t stream);
/* Same, with the hypothesis tokens still ON THE DEVICE: hyp h reads hyp_len[h] tokens at
 * hyp_tokens_dev[hyp_tok0[h] ...] (e.g. the [batch][beam][max_len] token buffer written by
 * wb_ctc_prefix_beam_search with hyp_tok0 = (b*beam + rank)*max_len).  Only the per-hypothesis lengths and
 * CTC scores cross to the host between the two stages; the reference moves every n-best list to Python
 * and back (search.py:236-248 -> :395-412). */
int wb_attention_rescoring_dev(const wb_model* m, const void* enc_out_bf16_dev, int64_t enc_rows,
                               const int32_t* seq_start_host, const int32_t* seq_len_host, int batch,
                               int n_hyp, const int32_t* hyp_utt_host, const int32_t* hyp_len_host,
                               const int32_t* hyp_tok0_host, const int32_t* hyp_tokens_dev,
                               const double* ctc_score_host, int sos, int eos, float ctc_weight,
                               float reverse_weight, float* tok_logp_l2r_dev, float* tok_logp_r2l_dev,
                               float* hyp_score_dev, int32_t* best_dev, void* workspace_dev,
                               size_t workspace_bytes, wb_stream_t stream);
/* Host-only helper (no CUDA call): the prefix-sharing tables wb_attention_rescoring builds for one decoder direction
 * (dir 0 = left-to-right, 1 = right-to-left).  Rows are hypothesis-major, (len_h + 1) per hypothesis.  Outputs:
 * uniq_of_row [R], rep_row / tok_u / pos_u [<= R], utt_q0_u / utt_qn_u [batch].  Returns the number of unique rows
 * (>= 0) or a negative error code.  Exposed for the CPU unit tests. */
int wb_prefix_share_tables(int dir, int batch, int n_hyp, const int32_t* hyp_utt_host, const int32_t* hyp_len_host,
                           const int32_t* hyp_tok0_host, const int32_t* hyp_tokens_host, int sos,
                           int32_t* uniq_of_row, int32_t* rep_row, int32_t* tok_u, int32_t* pos_u,
                           int32_t* utt_q0_u, int32_t* utt_qn_u);
/* full decoder posteriors for API parity with forward_attention_decoder: logp [R][ldl] (l2r) and
 * r_logp [R][ldl] (r2l, may be NULL) */
int wb_decoder_logprobs(const wb_model* m, const void* enc_out_bf16_dev, int64_t enc_rows,
                        const int32_t* seq_start_host, const int32_t* seq_len_host, int batch, int n_hyp,
                        const int32_t* hyp_utt_host, const int32_t* hyp_len_host,
                        const int32_t* hyp_tok0_host, const int32_t* hyp_tokens_host, int sos, int eos,
                        int use_r2l, float* logp_dev, float* r_logp_dev, int64_t ldl, void* workspace_dev,
                        size_t workspace_bytes, wb_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * F. autoregressive attention decoding — replaces attention_beam_search (wenet/models/transformer/search.py:252-371)
 *    over TransformerDecoder.forward_one_step (decoder.py:226-281) with its self / cross attention caches
 *    (decoder_layer.py:68-153, attention.py:431-520): decode mode "attention" of ASRModel.decode (asr_model.py:315-318)
 *    and the only mode of Whisper (whisper.py:31).  Rows are utterance-major (b * beam + n).  The cross-attention K/V of
 *    every layer are projected once per utterance; the self-attention cache is never re-ordered (a per-row ancestry
 *    table replaces the reference's index_select of every layer's K/V, search.py:315-323).
 *    prefix_host [batch][prefix_len]: the forced start of every hypothesis — {sos} for wenet models, {sot, language, task,
 *    no_timestamps} for Whisper (common.py:159-238 add_whisper_tokens).  max_len = encoder_out.size(1) + 1 of the padded
 *    reference batch = the token capacity incl. the prefix (the loop `for i in range(prefix_len, maxlen + 1)`).
 *    Outputs: tokens_dev [batch][out_stride] = the best hypothesis of every utterance after the prefix with every <eos>
 *    removed (search.py:357-371), lens_dev [batch], scores_dev [batch] (may be NULL) its score / len^length_penalty.
 *    The call polls the "every hypothesis ended" flag (search.py:301-302) on the stream every 8 steps, i.e. it
 *    synchronises the stream; *steps_run_host (may be NULL) receives the number of beam steps taken.
 * ------------------------------------------------------------------------------------------ */
size_t wb_attention_beam_workspace_bytes(const wb_model* m, int64_t enc_rows, int batch, int beam, int max_len);
int wb_attention_beam_search(const wb_model* m, const void* enc_out_bf16_dev, int64_t enc_rows,
                             const int32_t* seq_start_host, const int32_t* seq_len_host, int batch, int beam,
                             const int32_t* prefix_host, int prefix_len, int eos, int max_len, float length_penalty,
                             int32_t* tokens_dev, int out_stride, int32_t* lens_dev, float* scores_dev,
                             int32_t* steps_run_host, void* workspace_dev, size_t workspace_bytes, wb_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * G. Whisper (wb_model_config.arch = 1) — SURVEY section 8f-1, BASELINE configs[4]
 *    log-mel: replaces compute_log_mel_spectrogram (wenet/dataset/processor.py:320-369): torch.stft(n_fft, hop, hann,
 *    center / reflect) -> |.|^2 (last frame dropped) -> mel filterbank -> log10(clamp 1e-10) -> max(., utterance max - 8)
 *    -> (. + 4) / 4.  window_host [n_fft] (torch.hann_window) and mel_host [num_mel][n_fft/2+1]
 *    (librosa.filters.mel: slaney scale + slaney norm) are computed by the caller.  pcm_dev [batch][pcm_stride] float32 in
 *    [-1, 1); feats_dev [batch][frames_stride][num_mel]; utterance b has num_samples[b] / hop frames, the rest of its
 *    max_frames rows are zeroed (processor.padding); scratch_dev: batch int32.
 *    encoder: replaces TransformerEncoder.forward (encoder.py:122-181 with encoder.py:365-440) for input_layer conv1d2
 *    (subsampling.py:117-171), abs_pos_whisper (embedding.py:150-164), gelu.  padded_frames = xs.size(1) of the padded
 *    reference batch (it fixes the sub-sampled mask parity, subsampling.py:171).  Output rows are packed as in section B:
 *    utterance b owns T'_b = len_b / 2 (padded_frames even) or (len_b + 1) / 2 (odd) rows.
 * ------------------------------------------------------------------------------------------ */
typedef struct wb_logmel wb_logmel;
int wb_logmel_create(wb_logmel** out, int n_fft, int hop_length, int num_mel, const float* window_host,
                     const float* mel_host);
void wb_logmel_destroy(wb_logmel* lm);
int wb_logmel_forward(const wb_logmel* lm, const float* pcm_dev, int64_t pcm_stride, const int32_t* num_samples_dev,
                      int batch, float* feats_dev, int64_t frames_stride, int max_frames, int32_t* scratch_dev,
                      wb_stream_t stream);
int64_t wb_whisper_encoder_out_rows(int batch, const int32_t* feat_lens_host, int padded_frames);
size_t wb_whisper_encoder_workspace_bytes(const wb_model* m, int batch, const int32_t* feat_lens_host, int padded_frames);
int wb_whisper_encoder_forward(const wb_model* m, const float* feats_dev, int64_t feats_stride_b,
                               const int32_t* feat_lens_host, int batch, int padded_frames, float* enc_out_dev,
                               void* enc_out_bf16_dev, int32_t* seq_start_dev, int32_t* seq_len_dev, void* workspace_dev,
                               size_t workspace_bytes, wb_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Operator-level entry points (used by the parity tests and micro-benchmarks; same kernels the
 * stage entry points launch).
 * ------------------------------------------------------------------------------------------ */
/* C = epi(A[M,K] * B[N,K]^T + bias); A, B bf16 row-major (lda, K); epi: 0 bf16, 1 bf16+SiLU,
 * 2 bf16+ReLU, 3 fp32 residual add (C += alpha*(.)), 4 GLU->bf16 (weights packed [16 value|16 gate]
 * per 32 rows), 5 fp32, 9 bf16+GELU (erf) */
int wb_op_gemm(const void* a_dev, int64_t lda, const void* b_dev, int M, int N, int K,
               const float* bias_dev, int epi, float alpha, void* c_dev, int64_t ldc, int split3,
               wb_stream_t stream);
/* C (fp32) += alpha * (A B^T + bias) for FEW rows and a long K (the residual projections of autoregressive decoding): the K
 * range is cut into pieces that meet in the TMA reduce-add of C, so that more than ceil(M/128) * N/128 CTAs stream the
 * weights; the fp32 summation order is not reproducible run to run (the encoder paths never use it). */
int wb_op_gemm_resid_splitk(const void* a_dev, int64_t lda, const void* b_dev, int M, int N, int K,
                            const float* bias_dev, float alpha, float* c_dev, int64_t ldc, wb_stream_t stream);
/* x += alpha * (a b^T + bias) and ln_out = LayerNorm(x) * gamma + beta (bf16) in one kernel; N must be 256.  Replaces a
 * residual-update Linear followed by the next module's LayerNorm (wenet/models/transformer/encoder_layer.py:221-263).
 * gamma1_dev / beta1_dev non-null: the layer boundary (:262-263 then the next layer's :221-223) -
 * x = LayerNorm(gamma1, beta1)(x + ...) is stored (fp32) and ln_out = LayerNorm(gamma, beta)(x). */
int wb_op_gemm_resid_ln(const void* a_dev, int64_t lda, const void* b_dev, int M, int N, int K,
                        const float* bias_dev, float alpha, float* x_dev, int64_t ldx, const float* gamma1_dev,
                        const float* beta1_dev, const float* gamma_dev, const float* beta_dev, float eps,
                        void* ln_out_bf16_dev, int64_t ld_ln, wb_stream_t stream);
int wb_op_layernorm(const float* x_dev, int64_t ldx, int M, int d, const float* gamma_dev,
                    const float* beta_dev, float eps, void* out_bf16_dev, int64_t ld_bf16, int split3,
                    float* out_f32_dev, int64_t ld_f32, wb_stream_t stream);
/* fp32 rows -> bf16 rows; split3 != 0 writes [hi | lo | hi] blocks of width d (row pitch ld_bf16 >= 3 d) */
int wb_op_cast_bf16(const float* x_dev, int64_t ldx, int M, int d, void* out_bf16_dev, int64_t ld_bf16, int split3,
                    wb_stream_t stream);
int wb_op_attention(const void* q_dev, int64_t ldq, int64_t q_rows, int q_col0, const void* k_dev,
                    int64_t ldk, int64_t k_rows, int k_col0, const void* v_dev, int64_t ldv,
                    int64_t v_rows, int v_col0, const float* kbias_dev, int ld_kbias,
                    const int32_t* q_start_dev, const int32_t* q_len_dev, const int32_t* k_start_dev,
                    const int32_t* k_len_dev, int batch, int heads, int max_q_len, int chunk_size,
                    int num_left_chunks, float scale, void* out_dev, int64_t ldo, int out_col0,
                    int v_mode, wb_stream_t stream);
/* wb_op_attention with the modes the model paths use internally:
 *   kbias_scaled != 0: kbias_dev already holds bias * scale * log2(e) (as wb_op_relpos_kprep's output times that factor; the
 *     encoder's form), read by cp.async instead of being scaled in the kernel.
 *   part_o_dev != null: split-key mode.  `batch` = blocks x splits items; item b * splits + s is piece s of the keys of query
 *     block b (the same q_start / q_len for every piece of a block, its own k_start / k_len, possibly empty).  Scratch:
 *     part_o_dev batch * heads * max_q_len * 64 floats, part_ml_dev batch * heads * max_q_len * 8 bytes.  A merge kernel
 *     combines the pieces into out; a block whose pieces hold no key gets zero rows. */
int wb_op_attention_ex(const void* q_dev, int64_t ldq, int64_t q_rows, int q_col0, const void* k_dev, int64_t ldk,
                       int64_t k_rows, int k_col0, const void* v_dev, int64_t ldv, int64_t v_rows, int v_col0,
                       const float* kbias_dev, int ld_kbias, const int32_t* q_start_dev, const int32_t* q_len_dev,
                       const int32_t* k_start_dev, const int32_t* k_len_dev, int batch, int heads, int max_q_len,
                       int chunk_size, int num_left_chunks, float scale, void* out_dev, int64_t ldo, int out_col0,
                       int v_mode, int kbias_scaled, int splits, float* part_o_dev, void* part_ml_dev, wb_stream_t stream);
int wb_op_relpos_kprep(const void* k_dev, int64_t ldk, const float* pos_proj_dev,
                       const int32_t* row_pos_dev, const float* bias_u_dev, const float* bias_v_dev,
                       int M, int heads, void* kprime_dev, int64_t ldkp, float* kbias_dev,
                       wb_stream_t stream);
int wb_op_dwconv(const void* g_dev, int64_t ldg, const int32_t* seq_start_dev,
                 const int32_t* seq_len_dev, const int32_t* out_start_dev, int batch, int max_len,
                 int lead, int d, int ksize, int causal, const float* w_dev, const float* bias_dev,
                 int norm_type, const float* gamma_dev, const float* beta_dev, float eps,
                 const float* pad_vec_dev, int pad_until, void* out_dev, int64_t ldo,
                 wb_stream_t stream);
/* one step of attention_beam_search after the decoder call (search.py:309-355 + mask.py:258-310): rows are b * beam + n;
 * topk_* [R][beam] log-softmax top-`beam` of every row; score / end flags [R]; hyp / anc [R][max_len] (tokens, ancestry of
 * the self-attention cache); pos = position of the token just consumed.  Candidates are ranked (score desc, index asc). */
int wb_op_attention_beam_step(const float* topk_val_dev, const int32_t* topk_idx_dev, const float* score_in_dev,
                              const int32_t* end_in_dev, const int32_t* hyp_in_dev, const int32_t* anc_in_dev, int batch,
                              int beam, int max_len, int pos, int eos, float* score_out_dev, int32_t* end_out_dev,
                              int32_t* hyp_out_dev, int32_t* anc_out_dev, int32_t* next_tok_dev, int32_t* next_pos_dev,
                              int32_t* utt_ended_dev, wb_stream_t stream);
int wb_op_logsoftmax_topk(float* logits_dev, int64_t ldl, int M, int V, int blank_id,
                          float blank_penalty, int topk, float* topk_val_dev, int32_t* topk_idx_dev,
                          wb_stream_t stream);
int wb_op_lse_topk(const float* logits_dev, int64_t ldl, int M, int V, int blank_id, float blank_penalty,
                   int topk, float* topk_val_dev, int32_t* topk_idx_dev, wb_stream_t stream);

/* wb_op_lse_topk for few rows over a huge vocabulary (the output layer of attention decoding, logp.topk(beam_size) of
 * search.py:309): every row is cut into `slices` pieces taken by different warps and merged; same (value desc, index asc)
 * order.  scratch_dev: M * slices * (topk * 8 + 8) + 256 bytes. */
int wb_op_lse_topk_sliced(const float* logits_dev, int64_t ldl, int M, int V, int topk, int slices, float* topk_val_dev,
                          int32_t* topk_idx_dev, void* scratch_dev, size_t scratch_bytes, wb_stream_t stream);

/* Decoder output layer of attention rescoring without the [M, N] logits.  wb_op_gemm_lse_partials writes, per row of
 * v = A[M,K] B[N,K]^T + bias, wb_op_lse_parts(N, K) (max, sum) float pairs: one per half of each column tile, max of
 * v * log2(e) over the half's columns and sum of 2^(v log2 e - max); a half with no column < N holds (-inf, 0).
 * part_dev: M * wb_op_lse_parts(N, K) float pairs. */
int wb_op_lse_parts(int N, int K);
int wb_op_gemm_lse_partials(const void* a_dev, int64_t lda, const void* b_dev, int M, int N, int K, const float* bias_dev,
                            float* part_dev, wb_stream_t stream);
/* tok_logp[r] = a[s] . w[t] + bias[t] - logsumexp(row s), s = row_map[r] (identity when null), t = target[r]; the log-sum-exp
 * comes from the partials of row s.  A target outside [0, V) gives 0 (padding positions). */
int wb_op_lse_target_logprob(const float* part_dev, int n_parts, const void* a_dev, int64_t lda, const void* w_dev, int d,
                             const float* bias_dev, const int32_t* target_dev, const int32_t* row_map_dev, int R, int V,
                             float* tok_logp_dev, wb_stream_t stream);
/* x[r] = emb[tokens[r]] * xscale + pe[pos[r]] (fp32 rows of d, d % 4 == 0) */
int wb_op_embed_tokens(const int32_t* tokens_dev, const int32_t* pos_dev, int R, int d, const float* emb_dev,
                       const float* pe_dev, float xscale, float* x_dev, wb_stream_t stream);
/* score combine of attention rescoring (search.py:421-452): hypothesis h has hyp_len[h] tokens and its token log-probs at
 * l2r[hyp_row0[h] ..] (tokens then <eos>; r2l the same for the right-to-left decoder, or null); utterance b owns
 * hypotheses [utt_hyp0[b], + utt_nhyp[b]).  hyp_score[h] = mix of the fp32 sums + ctc_score * ctc_weight, best[b] = first
 * maximum within the utterance (0 without hypotheses). */
int wb_op_rescore_combine(const float* l2r_dev, const float* r2l_dev, const int32_t* hyp_row0_dev, const int32_t* hyp_len_dev,
                          const int32_t* utt_hyp0_dev, const int32_t* utt_nhyp_dev, int batch, const double* ctc_score_dev,
                          float ctc_weight, float reverse_weight, float* hyp_score_dev, int32_t* best_dev, wb_stream_t stream);
/* cached self attention of one new position per decoder row (attention decoding): qkv [R][3d] bf16 of this step, d = 64 H;
 * writes row r's K / V into slot (pos, r) of kv [L][R][2d] bf16 and ctx[r] ([R][d] bf16) = softmax(q k^T * scale) v over
 * positions 0..pos, position j < pos read from slot (j, anc[r * anc_stride + j]). */
int wb_op_dec_self_attn_step(const void* qkv_dev, void* kv_dev, const int32_t* anc_dev, int anc_stride, int pos, int R, int H,
                             int d, float scale, void* ctx_dev, wb_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* WENET_B200_H_ */
