// Internal model representation behind the opaque wb_model handle.
#pragma once
#include "common.cuh"
#include "kernels.h"
#include "../../include/wenet_b200.h"
#include <map>
#include <string>
#include <vector>

namespace wb {

struct DevTensor {
    void* ptr = nullptr;
    int dtype = 0;
    int64_t numel = 0;
};

struct Linear {
    const void* w = nullptr;   // bf16 [N][K]
    const float* b = nullptr;  // [N] or null
    int N = 0, K = 0;
    WeightMaps tmap;
};

struct Norm {
    const float* g = nullptr;
    const float* b = nullptr;
};

struct EncLayer {
    Norm n_ffm, n_mha, n_conv, n_ff, n_final;
    Linear ffm1, ffm2, ff1, ff2, qkv, out, pw1, pw2;
    const float* pos_u = nullptr;
    const float* pos_v = nullptr;
    const void* pos_w3 = nullptr;  // bf16 [d][3d] packed hi|hi|lo
    float* pos_proj = nullptr;     // [max_pos][d] fp32, built by finalize
    const float* dw_w = nullptr;
    const float* dw_b = nullptr;
    Norm n_cnn;                    // LayerNorm gamma/beta or folded BatchNorm scale/shift
    const float* pad_vec = nullptr;
};

struct DecLayer {
    Norm n1, n2, n3;
    Linear sa_qkv, sa_out, ca_q, ca_kv, ca_out, ff1, ff2;
};

struct Decoder {
    const float* emb = nullptr;  // [V][d]
    std::vector<DecLayer> layers;
    Norm after;
    Linear out;
    // input layer flavour: wenet "embed" = emb * sqrt(d) + sinusoid PE (the encoder's table), Whisper
    // "embed_learnable_pe" = emb + learnable PE (xscale 1); FFN activation: EPI_BF16_RELU or EPI_BF16_GELU
    const float* pe = nullptr;
    int pe_len = 0;
    float xscale = 1.0f;
    int act_epi = EPI_BF16_RELU;
};

// TransformerEncoderLayer of the Whisper encoder (encoder_layer.py:28-135, pre-norm)
struct TrLayer {
    Norm n1, n2;
    Linear qkv, out, ff1, ff2;
};
struct WhisperEnc {
    Linear conv1, conv2;          // Conv1d(k=3) as GEMMs over im2col rows: [d][3*idim], [d][3*d] ((tap, channel) order)
    const float* pe = nullptr;    // [max_pos][d] WhisperPositionalEncoding
    std::vector<TrLayer> layers;
    Norm after;
};

struct Model {
    wb_model_config cfg;
    std::map<std::string, DevTensor> tensors;
    bool finalized = false;
    int F1 = 0, F2 = 0;
    // encoder front
    const float* cmvn_mean = nullptr;
    const float* cmvn_istd = nullptr;
    const float* conv1_w = nullptr;
    const float* conv1_b = nullptr;
    Linear conv2, embed_out;
    const float* pe = nullptr;  // [max_pos][d]
    std::vector<EncLayer> layers;
    Norm after;
    Linear ctc;
    Decoder left, right;
    WhisperEnc wenc;            // cfg.arch == 1
    std::vector<void*> owned;  // extra device allocations made by finalize
};

int model_get(const Model* m, const std::string& name, int dtype, int64_t numel, const void** out);

// ---- autoregressive attention decoding (attdecode.cu) ----------------------------------------------------------------
size_t attention_beam_workspace_bytes(const Model* m, long long enc_rows, int batch, int beam, int max_len);
int attention_beam_search(const Model* m, const void* enc_bf16, long long enc_rows, const int32_t* seq_start_host,
                          const int32_t* seq_len_host, int batch, int beam, const int32_t* prefix_host, int prefix_len, int eos,
                          int max_len, float length_penalty, int32_t* out_tokens_dev, int out_stride, int32_t* out_lens_dev,
                          float* out_scores_dev, int32_t* steps_run_host, void* ws, size_t ws_bytes, cudaStream_t st);

// cached self attention of ONE new position per row (R = batch x beam rows, H heads of 64, d = 64 H): qkv [R][3d] bf16 of this
// step; writes K / V of row r into cache slot kv[pos][r] ([L][R][2d] bf16) and ctx[r] (bf16 [R][d]) = softmax attention over
// positions 0..pos of r's history, position j < pos read from slot (j, anc[r * anc_stride + j])
int dec_self_attn_step(const void* qkv, void* kv, const int* anc, int anc_stride, int pos, int R, int H, int d, float scale,
                       void* ctx, cudaStream_t st);

int attention_beam_step_op(const float* topv, const int* topi, const float* score_in, const int* end_in, const int* hyp_in,
                           const int* anc_in, int batch, int beam, int L, int pos, int eos, float* score_out, int* end_out,
                           int* hyp_out, int* anc_out, int* cur_tok, int* cur_pos, int* utt_ended, cudaStream_t st);

// ---- batched streaming (stream_batch.cu) ------------------------------------------------------------------------------
size_t encoder_chunk_batch_workspace_bytes(const Model* m, int T, int cache_t1, int sessions);
int encoder_forward_chunk_batch(const Model* m, const float* xs, int T, int S, const int32_t* offsets_host,
                                const int32_t* offsets_dev, int required_cache_size, const float* att_cache, int cache_t1,
                                const float* cnn_cache, float* y, float* r_att, float* r_cnn, int* out_chunk,
                                int* out_new_cache_t1, void* ws, size_t ws_bytes, cudaStream_t st);

// ---- Whisper front-end + encoder (whisper.cu) ------------------------------------------------------------------------
struct LogMelPlan;
int logmel_plan_create(LogMelPlan** out, int n_fft, int hop, int n_mel, const float* window_host, const float* mel_host);
void logmel_plan_destroy(LogMelPlan* p);
int logmel_forward(const LogMelPlan* p, const float* pcm, long long pcm_stride, const int* num_samples_dev, int batch, float* out,
                   long long frames_stride, int max_frames, int* scratch_dev, cudaStream_t st);
long long whisper_encoder_out_rows(int batch, const int32_t* lens, int time_pad);
size_t whisper_encoder_workspace_bytes(const Model* m, int batch, const int32_t* lens, int time_pad);
int whisper_encoder_forward(const Model* m, const float* feats, long long feats_stride_b, const int32_t* lens_host, int batch,
                            int time_pad, float* enc_out, void* enc_out_bf16, int32_t* seq_start_dev, int32_t* seq_len_dev,
                            void* ws, size_t ws_bytes, cudaStream_t st);

}  // namespace wb
