// C-ABI of libwenet_b200.so (see include/wenet_b200.h): handle management, weight upload,
// operator-level entry points.  Stage orchestration lives in encoder.cu / rescoring.cu.
#include "model.h"
#include <math.h>
#include <string.h>

namespace wb {

static size_t dtype_size(int dt) { return dt == WB_BF16 ? 2 : 4; }

int model_get(const Model* m, const std::string& name, int dtype, int64_t numel, const void** out) {
    auto it = m->tensors.find(name);
    if (it == m->tensors.end()) {
        set_last_error("model: required tensor '%s' was not provided", name.c_str());
        return WB_ERR_NOT_LOADED;
    }
    if (it->second.dtype != dtype || (numel >= 0 && it->second.numel != numel)) {
        set_last_error("model: tensor '%s' has dtype %d numel %lld, expected dtype %d numel %lld", name.c_str(),
                       it->second.dtype, (long long)it->second.numel, dtype, (long long)numel);
        return WB_ERR_BAD_ARG;
    }
    *out = it->second.ptr;
    return WB_OK;
}

static int get_linear(Model* m, const std::string& base, int N, int K, bool bias, Linear* L, int epi = EPI_BF16) {
    const void* p;
    int rc = model_get(m, base + ".w", WB_BF16, (int64_t)N * K, &p);
    if (rc != WB_OK) return rc;
    L->w = p;
    L->N = N;
    L->K = K;
    L->b = nullptr;
    if (bias) {
        rc = model_get(m, base + ".b", WB_F32, N, &p);
        if (rc != WB_OK) return rc;
        L->b = (const float*)p;
    }
    return make_weight_tmap(&L->tmap, L->w, N, K, epi);
}

static int get_norm(Model* m, const std::string& base, int d, Norm* n) {
    const void* p;
    int rc = model_get(m, base + ".g", WB_F32, d, &p);
    if (rc != WB_OK) return rc;
    n->g = (const float*)p;
    rc = model_get(m, base + ".b", WB_F32, d, &p);
    if (rc != WB_OK) return rc;
    n->b = (const float*)p;
    return WB_OK;
}

#define RC(x)                  \
    do {                       \
        int _rc = (x);         \
        if (_rc != WB_OK) return _rc; \
    } while (0)

static int finalize_decoder(Model* m, const std::string& pfx, int nlayers, Decoder* D) {
    const int d = m->cfg.d_model, V = m->cfg.vocab, ff = m->cfg.dec_ffn_dim;
    const void* p;
    RC(model_get(m, pfx + ".emb", WB_F32, (int64_t)V * d, &p));
    D->emb = (const float*)p;
    D->layers.resize(nlayers);
    for (int i = 0; i < nlayers; ++i) {
        const std::string b = pfx + "." + std::to_string(i);
        DecLayer& L = D->layers[i];
        RC(get_norm(m, b + ".norm1", d, &L.n1));
        RC(get_norm(m, b + ".norm2", d, &L.n2));
        RC(get_norm(m, b + ".norm3", d, &L.n3));
        RC(get_linear(m, b + ".sa.qkv", 3 * d, d, true, &L.sa_qkv));
        RC(get_linear(m, b + ".sa.out", d, d, true, &L.sa_out));
        RC(get_linear(m, b + ".ca.q", d, d, true, &L.ca_q));
        RC(get_linear(m, b + ".ca.kv", 2 * d, d, true, &L.ca_kv));
        RC(get_linear(m, b + ".ca.out", d, d, true, &L.ca_out));
        RC(get_linear(m, b + ".ff.w1", ff, d, true, &L.ff1));
        RC(get_linear(m, b + ".ff.w2", d, ff, true, &L.ff2));
    }
    RC(get_norm(m, pfx + ".after_norm", d, &D->after));
    RC(get_linear(m, pfx + ".out", V, d, true, &D->out));
    if (m->cfg.dec_flavor == 1) {
        // Whisper: embed_learnable_pe (embedding.py:167-176: xscale 1, learnable table), gelu FFN
        WB_REQUIRE(m->cfg.dec_max_len > 0, WB_ERR_BAD_ARG, "dec_flavor 1 needs dec_max_len");
        RC(model_get(m, pfx + ".pe", WB_F32, (int64_t)m->cfg.dec_max_len * d, &p));
        D->pe = (const float*)p;
        D->pe_len = m->cfg.dec_max_len;
        D->xscale = 1.0f;
        D->act_epi = EPI_BF16_GELU;
    } else {
        D->pe = nullptr;   // the encoder's sinusoid table (embedding.py:50-59)
        D->pe_len = m->cfg.max_pos;
        D->xscale = sqrtf((float)d);
        D->act_epi = EPI_BF16_RELU;
    }
    return WB_OK;
}

// cfg.arch == 1: TransformerEncoder with Conv1dSubsampling2 / abs_pos_whisper (whisper.cu)
static int finalize_whisper_encoder(Model* m) {
    const wb_model_config& c = m->cfg;
    const int d = c.d_model, ff = c.ffn_dim;
    WB_REQUIRE(c.input_dim % 8 == 0 && c.input_dim > 0, WB_ERR_UNSUPPORTED, "whisper: input_dim %d must be a multiple of 8", c.input_dim);
    WB_REQUIRE(!c.has_cmvn, WB_ERR_UNSUPPORTED, "whisper: global CMVN is not part of this path");
    const int p3 = c.precise ? 3 : 1;   // precise: encoder / CTC weights arrive packed [hi | hi | lo] along K
    WhisperEnc& E = m->wenc;
    const void* p;
    RC(get_linear(m, "wenc.conv1", d, 3 * c.input_dim * p3, true, &E.conv1));
    RC(get_linear(m, "wenc.conv2", d, 3 * d * p3, true, &E.conv2));
    RC(model_get(m, "wenc.pe", WB_F32, (int64_t)c.max_pos * d, &p));
    E.pe = (const float*)p;
    m->pe = E.pe;
    E.layers.resize(c.enc_layers);
    for (int i = 0; i < c.enc_layers; ++i) {
        const std::string b = "wenc." + std::to_string(i);
        TrLayer& L = E.layers[i];
        RC(get_norm(m, b + ".norm1", d, &L.n1));
        RC(get_norm(m, b + ".norm2", d, &L.n2));
        RC(get_linear(m, b + ".att.qkv", 3 * d, d * p3, true, &L.qkv));
        RC(get_linear(m, b + ".att.out", d, d * p3, true, &L.out));
        RC(get_linear(m, b + ".ff.w1", ff, d * p3, true, &L.ff1));
        RC(get_linear(m, b + ".ff.w2", d, ff * p3, true, &L.ff2));
    }
    RC(get_norm(m, "after_norm", d, &E.after));
    m->after = E.after;
    return WB_OK;
}

static int model_finalize(Model* m, cudaStream_t stream) {
    const wb_model_config& c = m->cfg;
    WB_REQUIRE(c.d_model % 128 == 0 && c.d_model == c.heads * 64, WB_ERR_UNSUPPORTED,
               "unsupported attention geometry: d_model=%d heads=%d (d_k must be 64, d_model %% 128 == 0)", c.d_model,
               c.heads);
    WB_REQUIRE(c.input_dim >= 7 && c.ffn_dim % 64 == 0, WB_ERR_UNSUPPORTED, "unsupported input_dim/ffn_dim");
    WB_REQUIRE(c.arch == 0 || c.arch == 1, WB_ERR_UNSUPPORTED, "unknown arch %d", c.arch);
    if (c.arch == 1) {
        if (c.dec_layers > 0)
            WB_REQUIRE(c.dec_heads * 64 == c.d_model && c.dec_ffn_dim % 64 == 0, WB_ERR_UNSUPPORTED,
                       "unsupported decoder geometry (heads=%d)", c.dec_heads);
        RC(finalize_whisper_encoder(m));
        if (c.vocab > 0 && m->tensors.count("ctc.w"))
            RC(get_linear(m, "ctc", c.vocab, c.d_model * (c.precise ? 3 : 1), true, &m->ctc));
        if (m->cfg.dec_ln_eps <= 0.f) m->cfg.dec_ln_eps = m->cfg.ln_eps;
        if (c.dec_layers > 0) RC(finalize_decoder(m, "dec.left", c.dec_layers, &m->left));
        WB_CHECK_CUDA(cudaStreamSynchronize(stream));
        m->finalized = true;
        return WB_OK;
    }
    WB_REQUIRE(c.cnn_kernel >= 1 && c.cnn_kernel <= 31 && (c.cnn_causal || c.cnn_kernel % 2 == 1), WB_ERR_UNSUPPORTED,
               "unsupported cnn_module_kernel %d", c.cnn_kernel);
    WB_REQUIRE(c.vocab > 0 || c.dec_layers == 0, WB_ERR_BAD_ARG, "a decoder needs a vocabulary");
    if (c.dec_layers > 0)
        WB_REQUIRE(c.dec_heads * 64 == c.d_model && c.dec_ffn_dim % 64 == 0, WB_ERR_UNSUPPORTED,
                   "unsupported decoder geometry (heads=%d)", c.dec_heads);
    const int d = c.d_model, ff = c.ffn_dim;
    // precise mode: every encoder / CTC weight arrives packed [hi | hi | lo] along K (weights.py split3), K -> 3K
    const int p3 = c.precise ? 3 : 1;
    m->F1 = (c.input_dim - 3) / 2 + 1;
    m->F2 = (m->F1 - 3) / 2 + 1;
    const void* p;
    if (c.has_cmvn) {
        RC(model_get(m, "cmvn.mean", WB_F32, c.input_dim, &p));
        m->cmvn_mean = (const float*)p;
        RC(model_get(m, "cmvn.istd", WB_F32, c.input_dim, &p));
        m->cmvn_istd = (const float*)p;
    }
    RC(model_get(m, "embed.conv1.w", WB_F32, 9 * d, &p));
    m->conv1_w = (const float*)p;
    RC(model_get(m, "embed.conv1.b", WB_F32, d, &p));
    m->conv1_b = (const float*)p;
    RC(get_linear(m, "embed.conv2", d, 9 * d * p3, true, &m->conv2));
    RC(get_linear(m, "embed.out", d, m->F2 * d * p3, true, &m->embed_out));
    RC(model_get(m, "embed.pe", WB_F32, (int64_t)c.max_pos * d, &p));
    m->pe = (const float*)p;

    // bf16x3 copy of the PE table for the (one-off) position projections
    void* pe3 = nullptr;
    WB_CHECK_CUDA(cudaMalloc(&pe3, (size_t)c.max_pos * 3 * d * 2));
    RC(cast_rows_bf16(m->pe, d, c.max_pos, d, pe3, 3 * d, 1, stream));

    m->layers.resize(c.enc_layers);
    for (int i = 0; i < c.enc_layers; ++i) {
        const std::string b = "enc." + std::to_string(i);
        EncLayer& L = m->layers[i];
        RC(get_norm(m, b + ".norm_ff_macaron", d, &L.n_ffm));
        RC(get_norm(m, b + ".norm_mha", d, &L.n_mha));
        RC(get_norm(m, b + ".norm_conv", d, &L.n_conv));
        RC(get_norm(m, b + ".norm_ff", d, &L.n_ff));
        RC(get_norm(m, b + ".norm_final", d, &L.n_final));
        RC(get_linear(m, b + ".ffm.w1", ff, d * p3, true, &L.ffm1));
        RC(get_linear(m, b + ".ffm.w2", d, ff * p3, true, &L.ffm2));
        RC(get_linear(m, b + ".ff.w1", ff, d * p3, true, &L.ff1));
        RC(get_linear(m, b + ".ff.w2", d, ff * p3, true, &L.ff2));
        RC(get_linear(m, b + ".att.qkv", 3 * d, d * p3, true, &L.qkv));
        RC(get_linear(m, b + ".att.out", d, d * p3, true, &L.out));
        RC(get_linear(m, b + ".conv.pw1", 2 * d, d * p3, true, &L.pw1, EPI_GLU_BF16));
        RC(get_linear(m, b + ".conv.pw2", d, d * p3, true, &L.pw2));
        RC(model_get(m, b + ".att.pos_u", WB_F32, d, &p));
        L.pos_u = (const float*)p;
        RC(model_get(m, b + ".att.pos_v", WB_F32, d, &p));
        L.pos_v = (const float*)p;
        RC(model_get(m, b + ".att.pos.w3", WB_BF16, (int64_t)d * 3 * d, &p));
        L.pos_w3 = p;
        RC(model_get(m, b + ".conv.dw.w", WB_F32, (int64_t)d * c.cnn_kernel, &p));
        L.dw_w = (const float*)p;
        RC(model_get(m, b + ".conv.dw.b", WB_F32, d, &p));
        L.dw_b = (const float*)p;
        RC(get_norm(m, b + ".conv.norm", d, &L.n_cnn));
        RC(model_get(m, b + ".conv.pad_vec", WB_F32, d, &p));
        L.pad_vec = (const float*)p;
        // P_l = pe @ W_pos^T in bf16x3 (fp32-grade): A = [hi|lo|hi], B = [hi|hi|lo]
        WB_CHECK_CUDA(cudaMalloc((void**)&L.pos_proj, (size_t)c.max_pos * d * sizeof(float)));
        m->owned.push_back(L.pos_proj);
        RC(gemm_bf16(pe3, 3 * d, nullptr, L.pos_w3, c.max_pos, d, 3 * d, nullptr, EPI_F32, 1.0f, L.pos_proj, d, 0,
                     stream));
    }
    RC(get_norm(m, "after_norm", d, &m->after));
    if (c.vocab > 0) RC(get_linear(m, "ctc", c.vocab, d * p3, true, &m->ctc));
    if (m->cfg.dec_ln_eps <= 0.f) m->cfg.dec_ln_eps = m->cfg.ln_eps;
    if (c.dec_layers > 0) RC(finalize_decoder(m, "dec.left", c.dec_layers, &m->left));
    if (c.rdec_layers > 0) RC(finalize_decoder(m, "dec.right", c.rdec_layers, &m->right));
    WB_CHECK_CUDA(cudaStreamSynchronize(stream));
    cudaFree(pe3);
    m->finalized = true;
    return WB_OK;
}

}  // namespace wb

using namespace wb;

extern "C" {

const char* wb_last_error(void) { return get_last_error(); }
const char* wb_version(void) { return "wenet_b200 0.1 (sm_100a)"; }
unsigned long long wb_launch_count(void) { return g_launch_count.load(); }

void wb_set_sm_reserve(int n) { gemm_set_sm_reserve(n); }
void wb_prof_enable(int on) { g_prof_on = on; }
void wb_prof_reset(void) { wb::prof_reset(); }
int wb_prof_num_tags(void) { return PT_COUNT; }
const char* wb_prof_tag_name(int tag) {
    static const char* names[PT_COUNT] = {"gemm_tcgen05", "attention", "layernorm", "dwconv_norm_silu", "conv1",
                                          "im2col", "relpos_kprep", "fbank", "logsoftmax_topk", "ctc_greedy",
                                          "ctc_prefix_beam", "embed_tokens", "gather_logprob", "rescore_combine",
                                          "misc", "gemm_tcgen05+layernorm"};
    return (tag >= 0 && tag < PT_COUNT) ? names[tag] : "?";
}
int wb_prof_collect(double* ms, double* work, long long* launches) { return wb::prof_collect(ms, work, launches); }
int wb_gemm_diag(uint64_t* out8, int reset) { return wb::gemm_diag(reinterpret_cast<unsigned long long*>(out8), reset); }

// ---------------------------------------------------------------- fbank
struct wb_fbank {
    FbankPlan* plan;
};

int wb_fbank_create(wb_fbank** out, int num_mel, int frame_len, int frame_shift, float preemph,
                    const float* window_host, const float* mel_host) {
    WB_REQUIRE(out && window_host && mel_host, WB_ERR_BAD_ARG, "fbank_create: null argument");
    FbankPlan* plan = nullptr;
    int rc = fbank_plan_create(&plan, 16000, num_mel, frame_len, frame_shift, 20.f, preemph, window_host, mel_host);
    if (rc != WB_OK) return rc;
    wb_fbank* fb = new wb_fbank();
    fb->plan = plan;
    *out = fb;
    return WB_OK;
}
void wb_fbank_destroy(wb_fbank* fb) {
    if (!fb) return;
    fbank_plan_destroy(fb->plan);
    delete fb;
}
int wb_fbank_forward(const wb_fbank* fb, const void* pcm_dev, int pcm_is_int16, int64_t pcm_stride,
                     const int32_t* num_samples_dev, int batch, float scale, float* feats_dev, int64_t frames_stride,
                     int max_frames, wb_stream_t stream) {
    WB_REQUIRE(fb && pcm_dev && num_samples_dev && feats_dev, WB_ERR_BAD_ARG, "fbank_forward: null argument");
    return fbank_forward(fb->plan, pcm_dev, pcm_is_int16, pcm_stride, num_samples_dev, batch, scale, feats_dev,
                         frames_stride, max_frames, (cudaStream_t)stream);
}

// ---------------------------------------------------------------- model
int wb_model_create(wb_model** out, const wb_model_config* cfg) {
    WB_REQUIRE(out && cfg, WB_ERR_BAD_ARG, "model_create: null argument");
    Model* m = new Model();
    m->cfg = *cfg;
    *out = reinterpret_cast<wb_model*>(m);
    return WB_OK;
}
void wb_model_destroy(wb_model* mm) {
    if (!mm) return;
    Model* m = reinterpret_cast<Model*>(mm);
    for (auto& kv : m->tensors) cudaFree(kv.second.ptr);
    for (void* p : m->owned) cudaFree(p);
    delete m;
}
int wb_model_set_tensor(wb_model* mm, const char* name, const void* host_data, int dtype, int64_t numel) {
    WB_REQUIRE(mm && name && host_data && numel > 0, WB_ERR_BAD_ARG, "set_tensor: bad argument");
    Model* m = reinterpret_cast<Model*>(mm);
    WB_REQUIRE(!m->finalized, WB_ERR_BAD_ARG, "set_tensor: model already finalized");
    DevTensor t;
    t.dtype = dtype;
    t.numel = numel;
    const size_t bytes = (size_t)numel * dtype_size(dtype);
    WB_CHECK_CUDA(cudaMalloc(&t.ptr, (bytes + 255) / 256 * 256));
    WB_CHECK_CUDA(cudaMemcpy(t.ptr, host_data, bytes, cudaMemcpyHostToDevice));
    auto it = m->tensors.find(name);
    if (it != m->tensors.end()) {
        cudaFree(it->second.ptr);
        it->second = t;
    } else {
        m->tensors[name] = t;
    }
    return WB_OK;
}
int wb_model_finalize(wb_model* mm, wb_stream_t stream) {
    WB_REQUIRE(mm, WB_ERR_BAD_ARG, "finalize: null model");
    return model_finalize(reinterpret_cast<Model*>(mm), (cudaStream_t)stream);
}

// ---------------------------------------------------------------- CTC / searches
int wb_ctc_logprobs(const wb_model* mm, const void* enc_out_bf16_dev, int64_t rows, int blank_id, float blank_penalty,
                    float* logp_dev, int64_t ldl, int topk, float* topk_val_dev, int32_t* topk_idx_dev,
                    wb_stream_t stream) {
    const Model* m = reinterpret_cast<const Model*>(mm);
    WB_REQUIRE(m && m->finalized && m->ctc.w, WB_ERR_NOT_LOADED, "ctc_logprobs: model not finalized / no CTC head");
    WB_REQUIRE(ldl >= m->cfg.vocab, WB_ERR_BAD_ARG, "ctc_logprobs: ldl < vocab");
    cudaStream_t st = (cudaStream_t)stream;
    RC(gemm_bf16(enc_out_bf16_dev, m->ctc.K, &m->ctc.tmap, m->ctc.w, (int)rows, m->cfg.vocab, m->ctc.K,
                 m->ctc.b, EPI_F32, 1.0f, logp_dev, ldl, 0, st));
    return ctc_logsoftmax_topk(logp_dev, ldl, (int)rows, m->cfg.vocab, blank_id, blank_penalty, topk, topk_val_dev,
                               topk_idx_dev, st);
}

int wb_ctc_topk(const wb_model* mm, const void* enc_out_bf16_dev, int64_t rows, int blank_id, float blank_penalty,
                float* logits_scratch_dev, int64_t ldl, int topk, float* topk_val_dev, int32_t* topk_idx_dev,
                wb_stream_t stream) {
    const Model* m = reinterpret_cast<const Model*>(mm);
    WB_REQUIRE(m && m->finalized && m->ctc.w, WB_ERR_NOT_LOADED, "ctc_topk: model not finalized / no CTC head");
    WB_REQUIRE(ldl >= m->cfg.vocab && topk_val_dev && topk_idx_dev && logits_scratch_dev, WB_ERR_BAD_ARG,
               "ctc_topk: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    RC(gemm_bf16(enc_out_bf16_dev, m->ctc.K, &m->ctc.tmap, m->ctc.w, (int)rows, m->cfg.vocab, m->ctc.K,
                 m->ctc.b, EPI_F32, 1.0f, logits_scratch_dev, ldl, 0, st));
    return ctc_lse_topk(logits_scratch_dev, ldl, (int)rows, m->cfg.vocab, blank_id, blank_penalty, topk, topk_val_dev,
                        topk_idx_dev, st);
}

int wb_ctc_greedy_search(const int32_t* topk_idx_dev, int topk, const int32_t* seq_start_dev,
                         const int32_t* seq_len_dev, int batch, int blank_id, int32_t* tokens_dev, int out_stride,
                         int32_t* lens_dev, wb_stream_t stream) {
    return ctc_greedy(topk_idx_dev, topk, seq_start_dev, seq_len_dev, batch, blank_id, tokens_dev, out_stride, lens_dev,
                      (cudaStream_t)stream);
}

size_t wb_prefix_beam_workspace_bytes(int batch, int beam, int max_len) {
    return prefix_beam_workspace_bytes(batch, beam, max_len);
}

int wb_ctc_prefix_beam_search(const float* topk_val_dev, const int32_t* topk_idx_dev, int topk,
                              const int32_t* seq_start_dev, const int32_t* seq_len_dev, int batch, int beam,
                              int blank_id, int max_len, int32_t* tokens_dev, int32_t* times_dev, int32_t* lens_dev,
                              double* scores_dev, int32_t* nhyp_dev, void* workspace_dev, size_t workspace_bytes,
                              wb_stream_t stream) {
    return wb_ctc_prefix_beam_search_ctx(topk_val_dev, topk_idx_dev, topk, seq_start_dev, seq_len_dev, batch, beam, blank_id,
                                         max_len, nullptr, tokens_dev, times_dev, lens_dev, scores_dev, nhyp_dev,
                                         workspace_dev, workspace_bytes, stream);
}

int wb_ctc_prefix_beam_search_ctx(const float* topk_val_dev, const int32_t* topk_idx_dev, int topk,
                                  const int32_t* seq_start_dev, const int32_t* seq_len_dev, int batch, int beam,
                                  int blank_id, int max_len, const wb_context_graph* cg, int32_t* tokens_dev,
                                  int32_t* times_dev, int32_t* lens_dev, double* scores_dev, int32_t* nhyp_dev,
                                  void* workspace_dev, size_t workspace_bytes, wb_stream_t stream) {
    PrefixBeamArgs a;
    if (cg != nullptr && cg->num_nodes > 0) {
        a.cg_nodes = cg->num_nodes;
        a.cg_child_off = cg->child_off;
        a.cg_child_tok = cg->child_tok;
        a.cg_child_node = cg->child_node;
        a.cg_fail = cg->fail;
        a.cg_token = cg->token;
        a.cg_node_score = cg->node_score;
        a.cg_token_score = cg->token_score;
        a.cg_output_score = cg->output_score;
    }
    a.topk_val = topk_val_dev;
    a.topk_idx = topk_idx_dev;
    a.topk = topk;
    a.seq_start = seq_start_dev;
    a.seq_len = seq_len_dev;
    a.batch = batch;
    a.beam = beam;
    a.blank_id = blank_id;
    a.max_len = max_len;
    a.out_tokens = tokens_dev;
    a.out_times = times_dev;
    a.out_lens = lens_dev;
    a.out_scores = scores_dev;
    a.out_nhyp = nhyp_dev;
    a.workspace = workspace_dev;
    a.workspace_bytes = workspace_bytes;
    return ctc_prefix_beam_search(a, (cudaStream_t)stream);
}

// ---------------------------------------------------------------- operator-level entry points
int wb_op_gemm(const void* a_dev, int64_t lda, const void* b_dev, int M, int N, int K, const float* bias_dev, int epi,
               float alpha, void* c_dev, int64_t ldc, int split3, wb_stream_t stream) {
    return gemm_bf16(a_dev, lda, nullptr, b_dev, M, N, K, bias_dev, epi, alpha, c_dev, ldc, split3,
                     (cudaStream_t)stream);
}
int wb_op_gemm_resid_splitk(const void* a_dev, int64_t lda, const void* b_dev, int M, int N, int K, const float* bias_dev,
                            float alpha, float* c_dev, int64_t ldc, wb_stream_t stream) {
    return gemm_resid_splitk(a_dev, lda, nullptr, b_dev, M, N, K, bias_dev, alpha, c_dev, ldc, (cudaStream_t)stream);
}
int wb_op_gemm_resid_ln(const void* a_dev, int64_t lda, const void* b_dev, int M, int N, int K, const float* bias_dev,
                        float alpha, float* x_dev, int64_t ldx, const float* gamma1_dev, const float* beta1_dev,
                        const float* gamma_dev, const float* beta_dev, float eps, void* ln_out_bf16_dev, int64_t ld_ln,
                        wb_stream_t stream) {
    return gemm_resid_ln(a_dev, lda, nullptr, b_dev, M, N, K, bias_dev, alpha, x_dev, ldx, gamma1_dev, beta1_dev, gamma_dev,
                         beta_dev, eps, ln_out_bf16_dev, ld_ln, (cudaStream_t)stream);
}
int wb_op_layernorm(const float* x_dev, int64_t ldx, int M, int d, const float* gamma_dev, const float* beta_dev,
                    float eps, void* out_bf16_dev, int64_t ld_bf16, int split3, float* out_f32_dev, int64_t ld_f32,
                    wb_stream_t stream) {
    return layernorm_rows(x_dev, ldx, M, d, gamma_dev, beta_dev, eps, out_bf16_dev, ld_bf16, split3, out_f32_dev,
                          ld_f32, (cudaStream_t)stream);
}
int wb_op_cast_bf16(const float* x_dev, int64_t ldx, int M, int d, void* out_bf16_dev, int64_t ld_bf16, int split3,
                    wb_stream_t stream) {
    return cast_rows_bf16(x_dev, ldx, M, d, out_bf16_dev, ld_bf16, split3, (cudaStream_t)stream);
}
int wb_op_attention(const void* q_dev, int64_t ldq, int64_t q_rows, int q_col0, const void* k_dev, int64_t ldk,
                    int64_t k_rows, int k_col0, const void* v_dev, int64_t ldv, int64_t v_rows, int v_col0,
                    const float* kbias_dev, int ld_kbias, const int32_t* q_start_dev, const int32_t* q_len_dev,
                    const int32_t* k_start_dev, const int32_t* k_len_dev, int batch, int heads, int max_q_len,
                    int chunk_size, int num_left_chunks, float scale, void* out_dev, int64_t ldo, int out_col0,
                    int v_mode, wb_stream_t stream) {
    AttnArgs a;
    a.q = q_dev; a.ldq = ldq; a.q_rows = q_rows; a.q_col0 = q_col0;
    a.k = k_dev; a.ldk = ldk; a.k_rows = k_rows; a.k_col0 = k_col0;
    a.v = v_dev; a.ldv = ldv; a.v_rows = v_rows; a.v_col0 = v_col0;
    a.kbias = kbias_dev; a.ld_kbias = ld_kbias;
    a.q_start = q_start_dev; a.q_len = q_len_dev; a.k_start = k_start_dev; a.k_len = k_len_dev;
    a.batch = batch; a.heads = heads; a.max_q_len = max_q_len;
    a.chunk_size = chunk_size; a.num_left_chunks = num_left_chunks; a.scale = scale;
    a.out = out_dev; a.ldo = ldo; a.out_col0 = out_col0; a.split3_out = 0; a.v_mode = v_mode;
    return attention_forward(a, (cudaStream_t)stream);
}
int wb_op_attention_ex(const void* q_dev, int64_t ldq, int64_t q_rows, int q_col0, const void* k_dev, int64_t ldk,
                       int64_t k_rows, int k_col0, const void* v_dev, int64_t ldv, int64_t v_rows, int v_col0,
                       const float* kbias_dev, int ld_kbias, const int32_t* q_start_dev, const int32_t* q_len_dev,
                       const int32_t* k_start_dev, const int32_t* k_len_dev, int batch, int heads, int max_q_len,
                       int chunk_size, int num_left_chunks, float scale, void* out_dev, int64_t ldo, int out_col0,
                       int v_mode, int kbias_scaled, int splits, float* part_o_dev, void* part_ml_dev, wb_stream_t stream) {
    AttnArgs a;
    a.q = q_dev; a.ldq = ldq; a.q_rows = q_rows; a.q_col0 = q_col0;
    a.k = k_dev; a.ldk = ldk; a.k_rows = k_rows; a.k_col0 = k_col0;
    a.v = v_dev; a.ldv = ldv; a.v_rows = v_rows; a.v_col0 = v_col0;
    a.kbias = kbias_dev; a.ld_kbias = ld_kbias; a.kbias_scaled = kbias_scaled;
    a.q_start = q_start_dev; a.q_len = q_len_dev; a.k_start = k_start_dev; a.k_len = k_len_dev;
    a.batch = batch; a.heads = heads; a.max_q_len = max_q_len;
    a.chunk_size = chunk_size; a.num_left_chunks = num_left_chunks; a.scale = scale;
    a.out = out_dev; a.ldo = ldo; a.out_col0 = out_col0; a.split3_out = 0; a.v_mode = v_mode;
    a.part_o = part_o_dev; a.part_ml = part_ml_dev; a.splits = splits;
    return attention_forward(a, (cudaStream_t)stream);
}
int wb_op_relpos_kprep(const void* k_dev, int64_t ldk, const float* pos_proj_dev, const int32_t* row_pos_dev,
                       const float* bias_u_dev, const float* bias_v_dev, int M, int heads, void* kprime_dev,
                       int64_t ldkp, float* kbias_dev, wb_stream_t stream) {
    return relpos_kprep(k_dev, ldk, pos_proj_dev, row_pos_dev, bias_u_dev, bias_v_dev, M, heads, kprime_dev, ldkp,
                        kbias_dev, (cudaStream_t)stream);
}
int wb_op_dwconv(const void* g_dev, int64_t ldg, const int32_t* seq_start_dev, const int32_t* seq_len_dev,
                 const int32_t* out_start_dev, int batch, int max_len, int lead, int d, int ksize, int causal,
                 const float* w_dev, const float* bias_dev, int norm_type, const float* gamma_dev,
                 const float* beta_dev, float eps, const float* pad_vec_dev, int pad_until, void* out_dev, int64_t ldo,
                 wb_stream_t stream) {
    DwConvArgs a;
    a.g = g_dev; a.ldg = ldg; a.seq_start = seq_start_dev; a.seq_len = seq_len_dev; a.out_start = out_start_dev;
    a.batch = batch; a.max_len = max_len; a.lead = lead; a.d = d; a.ksize = ksize; a.causal = causal;
    a.w = w_dev; a.bias = bias_dev; a.norm_type = norm_type; a.gamma = gamma_dev; a.beta = beta_dev; a.eps = eps;
    a.pad_vec = pad_vec_dev; a.pad_until = pad_until; a.out = out_dev; a.ldo = ldo; a.split3 = 0;
    return dwconv_norm_silu(a, (cudaStream_t)stream);
}
int wb_op_logsoftmax_topk(float* logits_dev, int64_t ldl, int M, int V, int blank_id, float blank_penalty, int topk,
                          float* topk_val_dev, int32_t* topk_idx_dev, wb_stream_t stream) {
    return ctc_logsoftmax_topk(logits_dev, ldl, M, V, blank_id, blank_penalty, topk, topk_val_dev, topk_idx_dev,
                               (cudaStream_t)stream);
}
int wb_op_lse_topk(const float* logits_dev, int64_t ldl, int M, int V, int blank_id, float blank_penalty, int topk,
                   float* topk_val_dev, int32_t* topk_idx_dev, wb_stream_t stream) {
    return ctc_lse_topk(logits_dev, ldl, M, V, blank_id, blank_penalty, topk, topk_val_dev, topk_idx_dev,
                        (cudaStream_t)stream);
}

int wb_op_lse_topk_sliced(const float* logits_dev, int64_t ldl, int M, int V, int topk, int slices, float* topk_val_dev,
                          int32_t* topk_idx_dev, void* scratch_dev, size_t scratch_bytes, wb_stream_t stream) {
    WB_REQUIRE(scratch_bytes >= lse_topk_sliced_scratch_bytes(M, slices, topk), WB_ERR_WORKSPACE, "lse_topk_sliced: scratch %zu < %zu",
               scratch_bytes, lse_topk_sliced_scratch_bytes(M, slices, topk));
    return lse_topk_sliced(logits_dev, ldl, M, V, topk, slices, topk_val_dev, topk_idx_dev, scratch_dev, (cudaStream_t)stream);
}

int wb_op_lse_parts(int N, int K) { return lse_parts(N, K); }
int wb_op_gemm_lse_partials(const void* a_dev, int64_t lda, const void* b_dev, int M, int N, int K, const float* bias_dev,
                            float* part_dev, wb_stream_t stream) {
    return gemm_lse_partials(a_dev, lda, nullptr, b_dev, M, N, K, bias_dev, reinterpret_cast<float2*>(part_dev),
                             (cudaStream_t)stream);
}
int wb_op_lse_target_logprob(const float* part_dev, int n_parts, const void* a_dev, int64_t lda, const void* w_dev, int d,
                             const float* bias_dev, const int32_t* target_dev, const int32_t* row_map_dev, int R, int V,
                             float* tok_logp_dev, wb_stream_t stream) {
    return lse_target_logprob(reinterpret_cast<const float2*>(part_dev), n_parts, a_dev, lda, w_dev, d, bias_dev, target_dev,
                              row_map_dev, R, V, tok_logp_dev, (cudaStream_t)stream);
}
int wb_op_embed_tokens(const int32_t* tokens_dev, const int32_t* pos_dev, int R, int d, const float* emb_dev,
                       const float* pe_dev, float xscale, float* x_dev, wb_stream_t stream) {
    return embed_tokens(tokens_dev, pos_dev, R, d, emb_dev, pe_dev, xscale, x_dev, (cudaStream_t)stream);
}
int wb_op_rescore_combine(const float* l2r_dev, const float* r2l_dev, const int32_t* hyp_row0_dev, const int32_t* hyp_len_dev,
                          const int32_t* utt_hyp0_dev, const int32_t* utt_nhyp_dev, int batch, const double* ctc_score_dev,
                          float ctc_weight, float reverse_weight, float* hyp_score_dev, int32_t* best_dev, wb_stream_t stream) {
    RescoreArgs a;
    a.l2r = l2r_dev; a.r2l = r2l_dev;
    a.hyp_row0 = hyp_row0_dev; a.hyp_len = hyp_len_dev;
    a.utt_hyp0 = utt_hyp0_dev; a.utt_nhyp = utt_nhyp_dev; a.batch = batch;
    a.ctc_score = ctc_score_dev;
    a.ctc_weight = ctc_weight; a.reverse_weight = reverse_weight;
    a.hyp_score = hyp_score_dev; a.best = best_dev;
    return rescore_combine(a, (cudaStream_t)stream);
}
int wb_op_dec_self_attn_step(const void* qkv_dev, void* kv_dev, const int32_t* anc_dev, int anc_stride, int pos, int R, int H,
                             int d, float scale, void* ctx_dev, wb_stream_t stream) {
    return dec_self_attn_step(qkv_dev, kv_dev, anc_dev, anc_stride, pos, R, H, d, scale, ctx_dev, (cudaStream_t)stream);
}

// ---------------------------------------------------------------- Whisper log-mel
struct wb_logmel {
    LogMelPlan* plan;
};
int wb_logmel_create(wb_logmel** out, int n_fft, int hop_length, int num_mel, const float* window_host, const float* mel_host) {
    WB_REQUIRE(out && window_host && mel_host, WB_ERR_BAD_ARG, "logmel_create: null argument");
    LogMelPlan* plan = nullptr;
    int rc = logmel_plan_create(&plan, n_fft, hop_length, num_mel, window_host, mel_host);
    if (rc != WB_OK) return rc;
    wb_logmel* lm = new wb_logmel();
    lm->plan = plan;
    *out = lm;
    return WB_OK;
}
void wb_logmel_destroy(wb_logmel* lm) {
    if (!lm) return;
    logmel_plan_destroy(lm->plan);
    delete lm;
}
int wb_logmel_forward(const wb_logmel* lm, const float* pcm_dev, int64_t pcm_stride, const int32_t* num_samples_dev, int batch,
                      float* feats_dev, int64_t frames_stride, int max_frames, int32_t* scratch_dev, wb_stream_t stream) {
    WB_REQUIRE(lm && pcm_dev && num_samples_dev && feats_dev && scratch_dev, WB_ERR_BAD_ARG, "logmel_forward: null argument");
    return logmel_forward(lm->plan, pcm_dev, pcm_stride, num_samples_dev, batch, feats_dev, frames_stride, max_frames, scratch_dev,
                          (cudaStream_t)stream);
}

// ---------------------------------------------------------------- Whisper encoder, attention decoding
int64_t wb_whisper_encoder_out_rows(int batch, const int32_t* feat_lens_host, int padded_frames) {
    return whisper_encoder_out_rows(batch, feat_lens_host, padded_frames);
}
size_t wb_whisper_encoder_workspace_bytes(const wb_model* mm, int batch, const int32_t* feat_lens_host, int padded_frames) {
    const Model* m = reinterpret_cast<const Model*>(mm);
    if (!m || !feat_lens_host) return 0;
    return whisper_encoder_workspace_bytes(m, batch, feat_lens_host, padded_frames);
}
int wb_whisper_encoder_forward(const wb_model* mm, const float* feats_dev, int64_t feats_stride_b, const int32_t* feat_lens_host,
                               int batch, int padded_frames, float* enc_out_dev, void* enc_out_bf16_dev, int32_t* seq_start_dev,
                               int32_t* seq_len_dev, void* workspace_dev, size_t workspace_bytes, wb_stream_t stream) {
    const Model* m = reinterpret_cast<const Model*>(mm);
    WB_REQUIRE(m && m->finalized, WB_ERR_NOT_LOADED, "whisper_encoder_forward: model not finalized");
    WB_REQUIRE(feats_dev && feat_lens_host && enc_out_dev && enc_out_bf16_dev && seq_start_dev && seq_len_dev && workspace_dev,
               WB_ERR_BAD_ARG, "whisper_encoder_forward: null argument");
    return whisper_encoder_forward(m, feats_dev, feats_stride_b, feat_lens_host, batch, padded_frames, enc_out_dev,
                                   enc_out_bf16_dev, seq_start_dev, seq_len_dev, workspace_dev, workspace_bytes,
                                   (cudaStream_t)stream);
}
size_t wb_attention_beam_workspace_bytes(const wb_model* mm, int64_t enc_rows, int batch, int beam, int max_len) {
    const Model* m = reinterpret_cast<const Model*>(mm);
    if (!m || !m->finalized) return 0;
    return attention_beam_workspace_bytes(m, enc_rows, batch, beam, max_len);
}
int wb_attention_beam_search(const wb_model* mm, const void* enc_out_bf16_dev, int64_t enc_rows, const int32_t* seq_start_host,
                             const int32_t* seq_len_host, int batch, int beam, const int32_t* prefix_host, int prefix_len,
                             int eos, int max_len, float length_penalty, int32_t* tokens_dev, int out_stride, int32_t* lens_dev,
                             float* scores_dev, int32_t* steps_run_host, void* workspace_dev, size_t workspace_bytes,
                             wb_stream_t stream) {
    const Model* m = reinterpret_cast<const Model*>(mm);
    WB_REQUIRE(m && m->finalized, WB_ERR_NOT_LOADED, "attention_beam_search: model not finalized");
    WB_REQUIRE(enc_out_bf16_dev && seq_start_host && seq_len_host && prefix_host && tokens_dev && lens_dev && workspace_dev,
               WB_ERR_BAD_ARG, "attention_beam_search: null argument");
    WB_REQUIRE(out_stride >= max_len - prefix_len, WB_ERR_BAD_ARG, "attention_beam_search: out_stride %d < %d", out_stride,
               max_len - prefix_len);
    return attention_beam_search(m, enc_out_bf16_dev, enc_rows, seq_start_host, seq_len_host, batch, beam, prefix_host, prefix_len,
                                 eos, max_len, length_penalty, tokens_dev, out_stride, lens_dev, scores_dev, steps_run_host,
                                 workspace_dev, workspace_bytes, (cudaStream_t)stream);
}
int wb_op_attention_beam_step(const float* topk_val_dev, const int32_t* topk_idx_dev, const float* score_in_dev,
                              const int32_t* end_in_dev, const int32_t* hyp_in_dev, const int32_t* anc_in_dev, int batch, int beam,
                              int max_len, int pos, int eos, float* score_out_dev, int32_t* end_out_dev, int32_t* hyp_out_dev,
                              int32_t* anc_out_dev, int32_t* next_tok_dev, int32_t* next_pos_dev, int32_t* utt_ended_dev,
                              wb_stream_t stream) {
    return attention_beam_step_op(topk_val_dev, topk_idx_dev, score_in_dev, end_in_dev, hyp_in_dev, anc_in_dev, batch, beam,
                                  max_len, pos, eos, score_out_dev, end_out_dev, hyp_out_dev, anc_out_dev, next_tok_dev,
                                  next_pos_dev, utt_ended_dev, (cudaStream_t)stream);
}

// ---------------------------------------------------------------- batched streaming
size_t wb_encoder_chunk_batch_workspace_bytes(const wb_model* mm, int T, int cache_t1, int sessions) {
    const Model* m = reinterpret_cast<const Model*>(mm);
    if (!m || !m->finalized || sessions < 1) return 0;
    return encoder_chunk_batch_workspace_bytes(m, T, cache_t1, sessions);
}
int wb_encoder_forward_chunk_batch(const wb_model* mm, const float* xs_dev, int T, int sessions, const int32_t* offsets_host,
                                   int required_cache_size, const float* att_cache_dev, int cache_t1, const float* cnn_cache_dev,
                                   float* y_dev, float* r_att_cache_dev, float* r_cnn_cache_dev, int* out_chunk,
                                   int* out_new_cache_t1, void* workspace_dev, size_t workspace_bytes, wb_stream_t stream) {
    const Model* m = reinterpret_cast<const Model*>(mm);
    WB_REQUIRE(m && m->finalized, WB_ERR_NOT_LOADED, "forward_chunk_batch: model not finalized");
    WB_REQUIRE(xs_dev && offsets_host && y_dev && r_att_cache_dev && workspace_dev, WB_ERR_BAD_ARG,
               "forward_chunk_batch: null argument");
    return encoder_forward_chunk_batch(m, xs_dev, T, sessions, offsets_host, nullptr, required_cache_size, att_cache_dev, cache_t1,
                                       cnn_cache_dev, y_dev, r_att_cache_dev, r_cnn_cache_dev, out_chunk, out_new_cache_t1,
                                       workspace_dev, workspace_bytes, (cudaStream_t)stream);
}
int wb_encoder_forward_chunk_batch_static(const wb_model* mm, const float* xs_dev, int T, int sessions,
                                          const int32_t* offsets_dev, int required_cache_size, const float* att_cache_dev,
                                          int cache_t1, const float* cnn_cache_dev, float* y_dev, float* r_att_cache_dev,
                                          float* r_cnn_cache_dev, void* workspace_dev, size_t workspace_bytes,
                                          wb_stream_t stream) {
    const Model* m = reinterpret_cast<const Model*>(mm);
    WB_REQUIRE(m && m->finalized, WB_ERR_NOT_LOADED, "forward_chunk_batch_static: model not finalized");
    WB_REQUIRE(xs_dev && offsets_dev && y_dev && r_att_cache_dev && workspace_dev, WB_ERR_BAD_ARG,
               "forward_chunk_batch_static: null argument");
    return encoder_forward_chunk_batch(m, xs_dev, T, sessions, nullptr, offsets_dev, required_cache_size, att_cache_dev, cache_t1,
                                       cnn_cache_dev, y_dev, r_att_cache_dev, r_cnn_cache_dev, nullptr, nullptr, workspace_dev,
                                       workspace_bytes, (cudaStream_t)stream);
}

}  // extern "C"
