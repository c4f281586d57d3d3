// Internal (C++) interface between the kernel translation units and api.cu.
// Everything here is implementation detail; the public surface is include/wenet_b200.h.
#pragma once
#include <cuda_runtime.h>
#include <cuda.h>
#include <stdint.h>

namespace wb {

// ---- GEMM epilogues (gemm.cu) ----------------------------------------------------------------
enum GemmEpi : int {
    EPI_BF16 = 0,       // out_bf16 = alpha * (acc + bias)
    EPI_BF16_SILU = 1,  // out_bf16 = alpha * silu(acc + bias)
    EPI_BF16_RELU = 2,  // out_bf16 = alpha * relu(acc + bias)
    EPI_RESID_F32 = 3,  // out_f32 += alpha * (acc + bias)      (in-place residual stream update)
    EPI_GLU_BF16 = 4,   // out_bf16[:, N/2] = a * sigmoid(g), weight rows packed [16 a | 16 g] x N/32
    EPI_F32 = 5,        // out_f32  = alpha * (acc + bias)
    EPI_LSE = 6,        // no matrix output: per (row, 128-column half tile) partial log-sum-exp (max2, sum) of acc + bias
    EPI_RESID_LN = 7,   // EPI_RESID_F32 + LayerNorm of the updated rows -> bf16 (gemm_resid_ln only; N == 256)
    EPI_RESID_LN2 = 8,  // x = LayerNorm_1(x + alpha (acc + bias)) (fp32), out_bf16 = LayerNorm(x) (gemm_resid_ln with gamma1)
    EPI_BF16_GELU = 9,  // out_bf16 = alpha * gelu(acc + bias), exact erf form (torch.nn.GELU(); Whisper FFN / Conv1dSubsampling2)
};

int gemm_bn_for(int N, int K, int epi = EPI_BF16);
// tensor maps of a [N, K] bf16 weight (B operand): `one` fetches a whole tile's rows (gemm_bn_for), `pair` half of them
// (CTA-pair tiles: each CTA of the pair holds half of B)
struct WeightMaps {
    CUtensorMap one, pair;
};
void gemm_set_sm_reserve(int n);
// tensor map for a [N, K] bf16 weight (B operand), box rows = gemm_bn_for(N, K)
// (epi: the epilogue the weight will be used with - only EPI_GLU_BF16 changes the tile width)
int make_weight_tmap(WeightMaps* out, const void* w, int N, int K, int epi = EPI_BF16);
// C = epi(A[M,K](lda) * B[N,K]^T + bias). tmap_b_opt may be null (then built from B).
// split3: bf16 outputs are written as [hi | lo | hi] column blocks of width N (N/2 for GLU) so the
// next GEMM can run in "bf16x3" mode against weights packed as [hi | hi | lo].
int gemm_bf16(const void* A, long long lda, const WeightMaps* tmap_b_opt, const void* B, int M, int N,
              int K, const float* bias, int epi, float alpha, void* out, long long ldc, int split3,
              cudaStream_t stream);

// log-softmax denominators without the logits: part[row][2 * n_tiles] = (max of v log2 e, sum 2^(v log2 e - max)) over each
// 128-column half of each n-tile of v = A B^T + bias.  lse_parts() = entries per row for a given N.
int lse_parts(int N, int K);
// x[M,N] (fp32, pitch ldx) += alpha * (A * B^T + bias), then ln_out_bf16 = LayerNorm(x) * gamma + beta, in ONE kernel:
// the residual-update GEMMs of a Conformer layer (positionwise FFN w_2, attention linear_out, pointwise_conv2) are each
// followed by the LayerNorm of the next module (encoder_layer.py:221-263), and with N = d = 256 an output tile holds whole
// rows.  Supported when gemm_resid_ln_supported(N); callers fall back to gemm_bf16(EPI_RESID_F32) + layernorm_rows.
// gamma1 / beta1 != null: the layer boundary - x = LayerNorm(gamma1, beta1)(x + ...) (norm_final, fp32, stored) and
// ln_out_bf16 = LayerNorm(gamma, beta)(x) (the next layer's norm_ff_macaron), as layernorm2_rows.
bool gemm_resid_ln_supported(int N);
int gemm_resid_ln(const void* A, long long lda, const WeightMaps* tmap_b_opt, const void* B, int M, int N, int K,
                  const float* bias, float alpha, float* x, long long ldx, const float* gamma1, const float* beta1,
                  const float* gamma, const float* beta, float eps, void* ln_out_bf16, long long ld_ln,
                  cudaStream_t stream);

// gemm_act16.cu: weight-stationary K <= 256 GEMM + activation with sixteen epilogue warps; returns 1 when the shape is not
// handled (the caller then uses gemm_tcgen05_kernel)
int gemm_act16_try(const void* A, long long lda, const CUtensorMap* tmap_b_one, int M, int N, int K, const float* bias, int epi,
                   void* out, long long ldc, int sm_reserve, cudaStream_t stream);

int gemm_resid_splitk(const void* A, long long lda, const WeightMaps* tmap_b_opt, const void* B, int M, int N, int K,
                      const float* bias, float alpha, float* out, long long ldc, cudaStream_t stream);
int gemm_lse_partials(const void* A, long long lda, const WeightMaps* tmap_b_opt, const void* B, int M, int N, int K,
                      const float* bias, float2* part, cudaStream_t stream);

// stall accounting of gemm_tcgen05_kernel (see gemm.cu); out8 may be null
int gemm_diag(unsigned long long* out8, int reset);

// Conv2d(d->d, 3x3, s2) + ReLU as an implicit GEMM whose A tiles are fetched by 3-D strided TMA boxes (no im2col buffer)
int gemm_conv2_implicit(const void* out1, long long t1_total, int F1, int d, const WeightMaps* tmap_w, const float* bias,
                        const void* tile_tab_dev /*int4 per tile*/, int num_tiles, long long rows_out, void* out2,
                        cudaStream_t stream);

// ---- fbank (fbank.cu) ------------------------------------------------------------------------
struct FbankPlan {  // device-resident constants, built once by fbank_plan_create
    float* window;      // [frame_len]
    float* twiddle;     // [nfft/2] complex (cos, -sin) pairs for the nfft/2-point complex FFT
    float* twiddle_r;   // [nfft/2 + 1] complex for the real-FFT split step
    int* mel_start;     // [num_mel]
    int* mel_len;       // [num_mel]
    int* mel_off;       // [num_mel] offset into mel_w
    float* mel_w;       // flat non-zero weights
    // fbank512_kernel: balanced assignment of mel bins to lanes: tap_km[lane * 4 + j] = j-th bin of the lane or -1
    int* tap_km;
    float* tap_w;       // (unused placeholder)
    int taps_per_lane;  // 4
    int num_mel, frame_len, frame_shift, nfft, mel_nnz;
    float preemph;
};
int fbank_plan_create(FbankPlan** out, int sample_rate, int num_mel, int frame_len, int frame_shift,
                      float low_freq, float preemph, const float* window_host,
                      const float* mel_dense_host /*[num_mel, nfft/2+1]*/);
void fbank_plan_destroy(FbankPlan* p);
// pcm: [B, pcm_stride] (float if !is_int16 else int16), num_samples[B] (device int32)
// out: [B, out_frames_stride, num_mel] fp32; frames beyond the utterance's own count are zeroed.
int fbank_forward(const FbankPlan* plan, const void* pcm, int is_int16, long long pcm_stride,
                  const int* num_samples_dev, int batch, float scale, float* out,
                  long long out_frames_stride, int max_frames, cudaStream_t stream);

// ---- row-wise ops (norm.cu) --------------------------------------------------------------------
// y = (x - mean) / sqrt(var + eps) * gamma + beta over the last dim (d).  out_bf16 / out_f32 are
// optional; out_f32 may alias x.  split3: bf16 output as [hi|lo|hi] blocks (row pitch ld_bf16).
int layernorm_rows(const float* x, long long ldx, int M, int d, const float* gamma, const float* beta,
                   float eps, void* out_bf16, long long ld_bf16, int split3, float* out_f32,
                   long long ld_f32, cudaStream_t stream);
// y = LN1(x) (fp32, optional write-back; may alias x), z = LN2(y) (bf16 and / or fp32): one read of x for two norms
int layernorm2_rows(const float* x, long long ldx, int M, int d, const float* g1, const float* b1, const float* g2,
                    const float* b2, float eps, float* y_f32, long long ld_y, void* z_bf16, long long ld_zb, int split3,
                    float* z_f32, long long ld_zf, cudaStream_t stream);
// f32 -> bf16 row copy with optional split3
int cast_rows_bf16(const float* x, long long ldx, int M, int d, void* out_bf16, long long ld_bf16,
                   int split3, cudaStream_t stream);

// ---- conv2d subsampling front (subsample.cu) ---------------------------------------------------
// feats: [B, feat_stride_t, idim] fp32 padded; writes conv1 output (ReLU) channels-last bf16:
// row (off1[b] + t1 * F1 + f1), d channels.  Only t1 < T1[b] rows are produced.
int subsample_conv1(const float* feats, long long feat_stride_b, int idim, const int* t1_len,
                    const long long* off1, int batch, int max_t1, const float* cmvn_mean,
                    const float* cmvn_istd, const float* w /*[9][d] fp32*/, const float* bias, int d,
                    void* out1_bf16, int split3 /*rows become [hi|lo|hi], 3d wide*/, cudaStream_t stream);
// im2col for conv2 (3x3 stride 2) from channels-last conv1 output.
// out row (off2[b] + t2 * F2 + f2) has K = 9*d entries ordered (kh, kw, c).
int subsample_im2col(const void* out1_bf16, const long long* off1, const int* t2_len,
                     const long long* off2, int batch, int max_t2, int F1, int F2, int d,
                     void* a2_bf16, int split3, cudaStream_t stream);

// ---- attention (attention.cu) ------------------------------------------------------------------
struct AttnArgs {
    const void* q;  long long ldq;  long long q_rows;   // bf16 [q_rows, ldq]; head h at col q_col0 + 64h
    int q_col0;
    const void* k;  long long ldk;  long long k_rows;   int k_col0;
    const void* v;  long long ldv;  long long v_rows;   int v_col0;
    const float* kbias;  int ld_kbias;                  // [k_rows, heads] fp32 or null
    int kbias_scaled = 0;                               // 1: kbias already multiplied by scale * log2(e) (relpos_kprep kbias_scale)
    const int* q_start; const int* q_len;               // [batch] device
    const int* k_start; const int* k_len;               // [batch] device
    int batch, heads, max_q_len;
    int chunk_size;        // 0: no chunk mask.  >0: key j visible to query i iff
    int num_left_chunks;   //   max((i/c - left)*c, 0) <= j < (i/c + 1)*c   (left < 0: from 0)
    float scale;
    void* out; long long ldo;  int out_col0;            // bf16 [q_rows, ldo]
    int split3_out;                                     // write [hi|lo|hi] with block width heads*64
    int v_mode;                                         // 0: MN-major UMMA descriptor, 1: smem transpose
    // split-key mode (flash-decoding): `batch` = blocks x splits items, item b * splits + s holding piece s of the keys of
    // query block b (same q_start / q_len for the pieces of a block, its own k_start / k_len); the kernel leaves
    // unnormalised fp32 partial outputs part_o [batch][heads][max_q_len][64] and (reference point, sum) part_ml
    // [batch][heads][max_q_len] (float2), and a merge kernel writes `out`.  Any max_q_len (blocks of more than 128 queries
    // take several CTAs per piece, each writing its own rows of the part buffers).
    float* part_o = nullptr;
    void* part_ml = nullptr;
    int splits = 1;
};
int attention_forward(const AttnArgs& a, cudaStream_t stream);
// K' = bf16(k + P[pos]) and c[m,h] = sum_i u[h,i]*k[m,h,i] + v[h,i]*P[pos,h,i]
// (rel-pos attention with rel_shift removed, wenet attention.py:395-417, folded into one score GEMM)
int relpos_kprep(const void* k_bf16, long long ldk, const float* P /*[maxlen, d]*/, const int* row_pos,
                 const float* bias_u, const float* bias_v, int M, int heads, void* kprime_bf16,
                 long long ldkp, float* kbias /*[M, heads]*/, cudaStream_t stream, float kbias_scale = 1.0f);

// ---- convolution module tail (convmod.cu) ------------------------------------------------------
struct DwConvArgs {
    const void* g; long long ldg;          // bf16 [rows, ldg] post-GLU activations
    const int* seq_start; const int* seq_len;  // per sequence rows in g (including `lead` context rows)
    int batch, max_len;
    int lead;            // leading rows per sequence that are context only (streaming cnn cache); 0 offline
    int d, ksize, causal;
    const float* w;      // [d, ksize]
    const float* bias;   // [d]
    int norm_type;       // 0: LayerNorm over channels, 1: folded BatchNorm (scale/shift per channel)
    const float* gamma; const float* beta; float eps;
    const float* pad_vec;   // symmetric mode: value of frames in [len, pad_until) (GLU(bias)), or null
    int pad_until;          // padded batch length (reference zero-masks *before* pointwise_conv1)
    void* out; long long ldo; int split3;   // bf16 [rows_out, ldo]; out row = out_start[b] + t
    const int* out_start;
    int in_split3 = 0;   // precise mode: g rows are [hi | lo | hi] blocks of width d (value = hi + lo)
};
int dwconv_norm_silu(const DwConvArgs& a, cudaStream_t stream);
// fp32 CUDA-core version for the precise parity mode (precise.cu); honours in_split3
int dwconv_norm_silu_f32(const DwConvArgs& a, cudaStream_t stream);

// ---- fp32 attention for the precise parity mode (precise.cu) ------------------------------------
struct AttnF32Args {
    const float* q; long long ldq;          // fp32 [q_rows, ldq]; head h at col 64h
    const float* k; long long ldk;
    const float* v; long long ldv;
    const float* pos_proj;                  // [max_pos][heads*64] projected positions or null (plain attention)
    const int* row_pos;                     // [k_rows] position of each key row
    const float* pos_u; const float* pos_v; // [heads*64]
    const int* q_start; const int* q_len; const int* k_start; const int* k_len;
    int batch, heads, max_q_len;
    int chunk_size, num_left_chunks;        // same meaning as AttnArgs
    float scale;
    void* out; long long ldo; int split3_out;   // bf16 [q_rows, ldo], optionally [hi|lo|hi]
};
int attention_f32(const AttnF32Args& a, cudaStream_t stream);

// ---- CTC head + searches (ctc.cu, search.cu) ---------------------------------------------------
// in-place log-softmax over V of logits [M, ldl] (+ optional blank penalty), plus per-row top-k.
int ctc_logsoftmax_topk(float* logits, long long ldl, int M, int V, int blank_id, float blank_penalty,
                        int topk, float* topk_val, int* topk_idx, cudaStream_t stream);
// top-k of the log-softmax (values normalised) without writing the matrix back; logits are left untouched
int ctc_lse_topk(const float* logits, long long ldl, int M, int V, int blank_id, float blank_penalty, int topk,
                 float* topk_val, int* topk_idx, cudaStream_t stream);
// the same top-k of the log-softmax for FEW rows over a HUGE vocabulary (attention decoding): rows cut into `slices` pieces
size_t lse_topk_sliced_scratch_bytes(int M, int slices, int topk);
int lse_topk_sliced(const float* logits, long long ldl, int M, int V, int topk, int slices, float* topk_val, int* topk_idx,
                    void* scratch, cudaStream_t stream);
// greedy collapse: per sequence, frames [start, start+len) of top-1 ids (stride topk)
int ctc_greedy(const int* topk_idx, int topk, const int* seq_start, const int* seq_len, int batch,
               int blank_id, int* out_tokens, int out_stride, int* out_len, cudaStream_t stream);
struct PrefixBeamArgs {
    const float* topk_val; const int* topk_idx; int topk;   // [M, topk] per frame
    const int* seq_start; const int* seq_len; int batch;    // frames of each utterance
    int beam, blank_id, max_len;                            // max_len >= max seq_len
    // outputs
    int* out_tokens;     // [batch, beam, max_len]
    int* out_times;      // [batch, beam, max_len]
    int* out_lens;       // [batch, beam]
    double* out_scores;  // [batch, beam]   log_add(s, ns)
    int* out_nhyp;       // [batch]
    void* workspace; size_t workspace_bytes;
    // optional context graph (cg_nodes == 0: none); see include/wenet_b200.h wb_context_graph
    int cg_nodes = 0;
    const int* cg_child_off = nullptr; const int* cg_child_tok = nullptr; const int* cg_child_node = nullptr;
    const int* cg_fail = nullptr; const int* cg_token = nullptr;
    const double* cg_node_score = nullptr; const double* cg_token_score = nullptr; const double* cg_output_score = nullptr;
};
size_t prefix_beam_workspace_bytes(int batch, int beam, int max_len);
int ctc_prefix_beam_search(const PrefixBeamArgs& a, cudaStream_t stream);

// ---- decoder helpers (decoder.cu) --------------------------------------------------------------
// x[r] = emb[token[r]] * xscale + pe[pos[r]]
int embed_tokens(const int* tokens, const int* pos, int R, int d, const float* emb /*[V,d]*/,
                 const float* pe /*[maxlen,d]*/, float xscale, float* x, cudaStream_t stream);
// tok_logp[r] = (a[r] . W[target[r]] + bias[target[r]]) - logsumexp_r, the latter from gemm_lse_partials (target < 0 -> 0)
int lse_target_logprob(const float2* part, int n_parts, const void* a_bf16, long long lda, const void* w_bf16, int d,
                       const float* bias, const int* target, const int* row_map /*null: identity*/, int R, int V,
                       float* tok_logp, cudaStream_t stream);
// per utterance rescoring combine (wenet search.py:421-452)
struct RescoreArgs {
    const float* l2r;  const float* r2l;  // [R] token log-probs, rows hyp-major, (len+1) per hyp
    const int* hyp_row0;  const int* hyp_len;  // [n_hyp_total]
    const int* utt_hyp0;  const int* utt_nhyp; int batch;  // hyps of utterance b: [utt_hyp0[b], +utt_nhyp[b])
    const double* ctc_score;  // [n_hyp_total]
    float ctc_weight, reverse_weight;
    float* hyp_score;  // [n_hyp_total] final score
    int* best;         // [batch] best hyp index within the utterance
};
int rescore_combine(const RescoreArgs& a, cudaStream_t stream);

// small utility kernels (util.cu)
// row_pos[seq_start[b] + t] = clamp(pos_offset + (pos_offset_dev ? pos_offset_dev[per_seq_offset ? b : 0] : 0) + t)
int fill_row_pos(const int* seq_start, const int* seq_len, int batch, int pos_offset, int* row_pos,
                 int max_len, cudaStream_t stream, const int* pos_offset_dev = nullptr, int max_pos = 0x7fffffff,
                 int per_seq_offset = 0);

}  // namespace wb
