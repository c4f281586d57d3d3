// Autoregressive attention decoding: batched beam search over TransformerDecoder.forward_one_step with self / cross
// KV caches.  Replaces wenet/models/transformer/search.py:252-371 (attention_beam_search),
// decoder.py:226-281 (forward_one_step), decoder_layer.py:68-153 (cache handling), attention.py:245-330, 431-520
// (cached self attention, cross attention with the encoder memory shared by the beams of an utterance),
// wenet/utils/mask.py:258-310 (mask_finished_scores / mask_finished_preds).
//
// Layout.  R = batch x beam decoder rows, utterance-major (row = b * beam + n, as the reference's (B*N, ...) tensors).
//   cross K/V   memkv[layer][enc_rows][2d]            bf16, projected ONCE per utterance before the loop
//                                                     (the reference's cross_att_cache, decoder_layer.py:126-135)
//   self K/V    kv[layer][pos][R][2d]                 bf16; position `pos` of physical row r is written once and never moved.
//   ancestry    anc[r][pos] = physical row whose slot holds position pos of row r's history (double-buffered, int32)
//               -> the beam re-ordering of the self-attention cache (search.py:315-323 index_select of every layer's
//               (B*N, H, L, d_k) K and V) becomes a copy of L ints per row; no cache byte is ever moved.
//   hyps        hyp[r][pos] tokens (double-buffered), scores fp32 (the reference's dtype), end flags
// One decoding step = embed the last token of every row, run the layers on R rows (tcgen05 GEMMs with M = R,
// dec_self_attn_step_kernel for the cached self attention, the varlen tcgen05 attention kernel for the cross attention:
// the `beam` queries of an utterance against its own encoder frames), output layer -> log-softmax top-`beam`
// (lse_topk_kernel) -> beam_step_kernel (second prune + bookkeeping, one CTA per utterance).
// Prefix tokens (1 for wenet models: <sos>; 4 for Whisper: sot, language, task, no_timestamps) are fed one position at a
// time without a beam update: every beam holds the same prefix, so this equals the reference's first step on the
// whole prefix under the causal mask.
// The host only polls the "all hypotheses ended" condition (search.py:301-302) every kPoll steps; steps taken after
// every row has ended append <eos> with score + 0 and cannot change the result.
#include "model.h"
#include <math.h>
#include <vector>

namespace wb {

namespace {

inline size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

constexpr int kPoll = 8;
constexpr int kMaxBeam = 32;
constexpr int kCaMaxSplits = 8;    // workspace bound; the default cap is kCaSplits (WB_CA_SPLITS overrides it, tuning only)
constexpr int kCaSplits = 4;
constexpr int kTopkSlices = 16;   // vocabulary slices of the output top-k when V is large   // key pieces of the cross attention (flash-decoding)

#define RC(x)                         \
    do {                              \
        int _rc = (x);                \
        if (_rc != WB_OK) return _rc; \
    } while (0)

// ---- cached self attention of ONE new position per row -----------------------------------------------------------
// warp = (row r, head h).  Writes this position's K/V into the cache slot (pos, r), then attends over positions 0..pos
// of the row's history (slots given by anc) with an exact fp32 softmax.  Lane-per-key scores, lane-per-dim-pair output.
constexpr int SA_WARPS = 4;
__global__ void __launch_bounds__(SA_WARPS * 32)
dec_self_attn_step_kernel(const __nv_bfloat16* __restrict__ qkv, __nv_bfloat16* __restrict__ kv,
                          const int* __restrict__ anc, int anc_stride, int pos, int R, int H, int d, float scale,
                          __nv_bfloat16* __restrict__ ctx) {
    pdl_launch_dependents();
    pdl_wait();
    extern __shared__ float sa_smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int w = blockIdx.x * SA_WARPS + warp;
    if (w >= R * H) return;
    const int r = w / H, h = w - r * H;
    const int n = pos + 1;
    float* sc = sa_smem + (size_t)warp * 2 * n;          // scores, then probabilities
    int* slot = reinterpret_cast<int*>(sc + n);          // physical row of every position
    const __nv_bfloat16* qrow = qkv + (long long)r * 3 * d + h * 64;
    // own K / V -> cache slot (pos, r)
    {
        const uint32_t kk = reinterpret_cast<const uint32_t*>(qrow + d)[lane];
        const uint32_t vv = reinterpret_cast<const uint32_t*>(qrow + 2 * d)[lane];
        __nv_bfloat16* dst = kv + ((long long)pos * R + r) * 2 * d + h * 64;
        reinterpret_cast<uint32_t*>(dst)[lane] = kk;
        reinterpret_cast<uint32_t*>(dst + d)[lane] = vv;
    }
    // q in registers (every lane holds all 64 dims)
    float q[64];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const uint4 u = reinterpret_cast<const uint4*>(qrow)[i];
        const uint32_t ww[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            q[8 * i + 2 * j] = bf16_lo(ww[j]);
            q[8 * i + 2 * j + 1] = bf16_hi(ww[j]);
        }
    }
    float mx = -INFINITY;
    for (int j = lane; j < n; j += 32) {
        const int pr = (j == pos) ? r : anc[(long long)r * anc_stride + j];
        slot[j] = pr;
        // the row's own key of this step is read from the GEMM output (the cache write above is not yet visible warp-wide)
        const __nv_bfloat16* kp = (j == pos) ? (qrow + d) : (kv + ((long long)j * R + pr) * 2 * d + h * 64);
        float acc = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const uint4 u = reinterpret_cast<const uint4*>(kp)[i];
            const uint32_t ww[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                acc = fmaf(q[8 * i + 2 * t], bf16_lo(ww[t]), acc);
                acc = fmaf(q[8 * i + 2 * t + 1], bf16_hi(ww[t]), acc);
            }
        }
        acc *= scale;
        sc[j] = acc;
        mx = fmaxf(mx, acc);
    }
    mx = warp_max(mx);
    float sum = 0.f;
    for (int j = lane; j < n; j += 32) {
        const float e = __expf(sc[j] - mx);
        sc[j] = e;
        sum += e;
    }
    sum = warp_sum(sum);
    __syncwarp();
    const float inv = 1.0f / sum;
    // eight V rows in flight (a one-row-at-a-time loop is a chain of dependent L2 / DRAM latencies: ~100 of them per warp)
    float o0 = 0.f, o1 = 0.f;
    constexpr int VB = 8;
    for (int j0 = 0; j0 < n; j0 += VB) {
        uint32_t vv[VB];
#pragma unroll
        for (int u = 0; u < VB; ++u) {
            const int j = j0 + u;
            vv[u] = 0u;
            if (j < n) {
                const __nv_bfloat16* vp = (j == pos) ? (qrow + 2 * d) : (kv + ((long long)j * R + slot[j]) * 2 * d + d + h * 64);
                vv[u] = reinterpret_cast<const uint32_t*>(vp)[lane];
            }
        }
#pragma unroll
        for (int u = 0; u < VB; ++u) {
            const float p = (j0 + u < n) ? sc[j0 + u] : 0.f;
            o0 = fmaf(p, bf16_lo(vv[u]), o0);
            o1 = fmaf(p, bf16_hi(vv[u]), o1);
        }
    }
    reinterpret_cast<uint32_t*>(ctx + (long long)r * d + h * 64)[lane] = pack_bf16x2(o0 * inv, o1 * inv);
}

// ---- one beam-search step (search.py:309-355), one CTA per utterance -----------------------------------------------
// topv / topi: [R][N] log-softmax top-N of every row (value desc).  Rows that have ended keep exactly one continuation
// (<eos>, + 0); the N*N candidates of the utterance are ranked by (score desc, candidate index asc) and the best N
// become the new rows: tokens / ancestry of the parent row are copied, the chosen token appended.
struct BeamStepArgs {
    const float* topv; const int* topi;
    const float* score_in; float* score_out;
    const int* end_in; int* end_out;
    const int* hyp_in; int* hyp_out;      // [R][L]
    const int* anc_in; int* anc_out;      // [R][L]
    int* cur_tok; int* cur_pos;           // [R] input of the next step
    int* utt_ended;                       // [batch] rows of the utterance whose last token is <eos>
    int N, L, pos, eos;                   // pos = position of the token just consumed (the new token goes to pos + 1)
};
__global__ void __launch_bounds__(128)
beam_step_kernel(BeamStepArgs a) {
    __shared__ float cs[kMaxBeam * kMaxBeam];
    __shared__ int sel[kMaxBeam];
    const int b = blockIdx.x, N = a.N, r0 = b * N;
    const int nc = N * N;
    for (int c = threadIdx.x; c < nc; c += blockDim.x) {
        const int p = c / N, k = c - p * N;
        float lp = a.topv[(long long)(r0 + p) * N + k];
        if (a.end_in[r0 + p]) lp = (k == 0) ? 0.f : -INFINITY;   // mask_finished_scores
        cs[c] = a.score_in[r0 + p] + lp;
    }
    __syncthreads();
    for (int c = threadIdx.x; c < nc; c += blockDim.x) {
        const float v = cs[c];
        int rank = 0;
        for (int o = 0; o < nc; ++o) {
            const float u = cs[o];
            rank += (u > v || (u == v && o < c)) ? 1 : 0;
        }
        if (v != v) rank = nc;   // NaN never selected (cannot occur with finite logits)
        if (rank < N) sel[rank] = c;
    }
    __syncthreads();
    int ended = 0;
    for (int n = 0; n < N; ++n) {
        const int c = sel[n];
        const int p = c / N, k = c - p * N;
        const int pr = r0 + p, nr = r0 + n;
        const int tok = a.end_in[pr] ? a.eos : a.topi[(long long)pr * N + k];   // mask_finished_preds
        for (int j = threadIdx.x; j <= a.pos; j += blockDim.x) {
            a.hyp_out[(long long)nr * a.L + j] = a.hyp_in[(long long)pr * a.L + j];
            a.anc_out[(long long)nr * a.L + j] = (j == a.pos) ? pr : a.anc_in[(long long)pr * a.L + j];
        }
        if (threadIdx.x == 0) {
            a.hyp_out[(long long)nr * a.L + a.pos + 1] = tok;
            a.score_out[nr] = cs[c];
            a.end_out[nr] = (tok == a.eos) ? 1 : 0;
            a.cur_tok[nr] = tok;
            a.cur_pos[nr] = a.pos + 1;
        }
        ended += (tok == a.eos) ? 1 : 0;
    }
    if (threadIdx.x == 0) a.utt_ended[b] = ended;
}

// prefix positions: every row of the utterance consumes prefix[b][pos + 1] next; ancestry is the identity
__global__ void prefix_step_kernel(const int* __restrict__ prefix, int P, int N, int L, int pos, int R, int* hyp0, int* hyp1,
                                   int* anc0, int* anc1, int* cur_tok, int* cur_pos) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    const int b = r / N;
    // pos = -1: initial fill of position 0
    const int np = pos + 1;
    const int tok = prefix[b * P + np];
    hyp0[(long long)r * L + np] = tok;
    hyp1[(long long)r * L + np] = tok;
    if (pos >= 0) {
        anc0[(long long)r * L + pos] = r;
        anc1[(long long)r * L + pos] = r;
    }
    cur_tok[r] = tok;
    cur_pos[r] = np;
}

// best of best (search.py:357-371): score / (#tokens != eos)^length_penalty, first maximum, tokens after the prefix with
// every <eos> removed
__global__ void final_select_kernel(const float* __restrict__ score, const int* __restrict__ hyp, int N, int L, int n_tok,
                                    int P, int eos, float length_penalty, int* __restrict__ out_tok, int out_stride,
                                    int* __restrict__ out_len, float* __restrict__ out_score) {
    const int b = blockIdx.x;
    if (threadIdx.x == 0) {
        float bs = 0.f;
        int bi = -1;
        for (int n = 0; n < N; ++n) {
            const int* hr = hyp + (long long)(b * N + n) * L;
            int len = 0;
            for (int j = 0; j < n_tok; ++j) len += (hr[j] != eos) ? 1 : 0;
            const float s = score[b * N + n] / powf((float)len, length_penalty);
            if (bi < 0 || s > bs) {
                bs = s;
                bi = n;
            }
        }
        if (out_score) out_score[b] = bs;
        const int* hr = hyp + (long long)(b * N + bi) * L;
        int cnt = 0;
        for (int j = P; j < n_tok; ++j)
            if (hr[j] != eos) out_tok[(long long)b * out_stride + cnt++] = hr[j];
        out_len[b] = cnt;
    }
}

struct AbPlan {
    int R = 0, L = 0;
    size_t o_topk_scr = 0, o_memkv = 0, o_kv = 0, o_x = 0, o_a = 0, o_qkv = 0, o_ctx = 0, o_q = 0, o_h = 0, o_logits = 0, o_topv = 0, o_topi = 0,
           o_int = 0, o_part_o = 0, o_part_ml = 0, total = 0;
    long long ldl = 0;
    size_t n_int = 0;
};

void ab_layout(const Model* m, long long enc_rows, int batch, int beam, int max_len, AbPlan* P) {
    const int d = m->cfg.d_model, ff = m->cfg.dec_ffn_dim, nl = (int)m->left.layers.size();
    const size_t R = (size_t)batch * beam;
    P->R = (int)R;
    P->L = max_len;
    P->ldl = (m->cfg.vocab + 7) / 8 * 8;
    size_t o = 0;
    P->o_memkv = o; o += align_up((size_t)nl * enc_rows * 2 * d * 2);
    P->o_kv = o; o += align_up((size_t)nl * max_len * R * 2 * d * 2);
    P->o_x = o; o += align_up(R * d * 4);
    P->o_a = o; o += align_up(R * d * 2);
    P->o_qkv = o; o += align_up(R * 3 * d * 2);
    P->o_ctx = o; o += align_up(R * d * 2);
    P->o_q = o; o += align_up(R * d * 2);
    P->o_h = o; o += align_up(R * ff * 2);
    P->o_logits = o; o += align_up(R * P->ldl * 4);
    P->o_topv = o; o += align_up(R * beam * 4);
    P->o_topi = o; o += align_up(R * beam * 4);
    P->o_topk_scr = o; o += align_up(lse_topk_sliced_scratch_bytes((int)R, kTopkSlices, beam));
    // ints: hyp x2, anc x2 [R][L]; score x2 (float), end x2, cur_tok, cur_pos [R]; q_start, q_len, enc_start, enc_len,
    // utt_ended [batch]; prefix [batch][L]
    P->n_int = 4 * R * max_len + 6 * R + 5 * (size_t)batch + (size_t)batch * max_len + 64 + 4 * (size_t)batch * kCaMaxSplits;
    P->o_int = o; o += align_up(P->n_int * 4);
    // split-key cross attention (attention.cu, AttnArgs::part_o): pieces x heads x beam rows x (64 fp32 + (m, l))
    P->o_part_o = o; o += align_up(R * kCaMaxSplits * m->cfg.dec_heads * 64 * 4);
    P->o_part_ml = o; o += align_up(R * kCaMaxSplits * m->cfg.dec_heads * 8);
    P->total = o + 256;
}

}  // namespace

// x += A W^T + b, then a = LayerNorm(x): one kernel when the tile holds whole rows (d == 256), else GEMM + LayerNorm
static int resid_then_norm(const void* A, long long lda, const Linear& W, int M, int d, float* x, const Norm& n, float eps,
                           void* a_out, cudaStream_t st) {
    if (W.b != nullptr && gemm_resid_ln_supported(d))
        return gemm_resid_ln(A, lda, &W.tmap, W.w, M, d, W.K, W.b, 1.0f, x, d, nullptr, nullptr, n.g, n.b, eps, a_out, d, st);
    int rc = gemm_resid_splitk(A, lda, &W.tmap, W.w, M, d, W.K, W.b, 1.0f, x, d, st);   // few rows, K up to 5120: split-K
    if (rc != WB_OK) return rc;
    return layernorm_rows(x, d, M, d, n.g, n.b, eps, a_out, d, 0, nullptr, 0, st);
}

// op-level entry (tests): one beam step on caller-provided tables
int attention_beam_step_op(const float* topv, const int* topi, const float* score_in, const int* end_in, const int* hyp_in,
                           const int* anc_in, int batch, int beam, int L, int pos, int eos, float* score_out, int* end_out,
                           int* hyp_out, int* anc_out, int* cur_tok, int* cur_pos, int* utt_ended, cudaStream_t st) {
    WB_REQUIRE(beam >= 1 && beam <= kMaxBeam && batch > 0 && pos >= 0 && pos + 1 < L, WB_ERR_BAD_ARG, "beam_step: bad argument");
    BeamStepArgs B;
    B.topv = topv; B.topi = topi;
    B.score_in = score_in; B.score_out = score_out;
    B.end_in = end_in; B.end_out = end_out;
    B.hyp_in = hyp_in; B.hyp_out = hyp_out;
    B.anc_in = anc_in; B.anc_out = anc_out;
    B.cur_tok = cur_tok; B.cur_pos = cur_pos; B.utt_ended = utt_ended;
    B.N = beam; B.L = L; B.pos = pos; B.eos = eos;
    beam_step_kernel<<<batch, 128, 0, st>>>(B);
    count_launch();
    WB_CHECK_LAUNCH();
    return WB_OK;
}

// the self-attention step kernel keeps one score + one slot per past position and warp in shared memory
constexpr size_t kSaSmemMax = 200 * 1024;

int dec_self_attn_step(const void* qkv, void* kv, const int* anc, int anc_stride, int pos, int R, int H, int d, float scale,
                       void* ctx, cudaStream_t st) {
    if (R <= 0) return WB_OK;
    WB_REQUIRE(pos >= 0 && H >= 1 && d == H * 64 && (pos == 0 || anc_stride >= pos), WB_ERR_BAD_ARG,
               "dec_self_attn_step: bad argument (pos %d, H %d, d %d, anc_stride %d)", pos, H, d, anc_stride);
    const size_t smem = (size_t)SA_WARPS * 2 * (pos + 1) * sizeof(float);
    WB_REQUIRE(smem <= kSaSmemMax, WB_ERR_UNSUPPORTED, "dec_self_attn_step: position %d exceeds the %zu positions the kernel holds",
               pos, kSaSmemMax / (SA_WARPS * 2 * sizeof(float)));
    WB_SET_MAX_DYN_SMEM(dec_self_attn_step_kernel, kSaSmemMax);
    ProfScope _ps(PT_ATTENTION, st, 0.0);
    WB_CHECK_CUDA(launch_maybe_pdl(dec_self_attn_step_kernel, dim3(ceil_div(R * H, SA_WARPS)), dim3(SA_WARPS * 32), smem, st,
                                   reinterpret_cast<const __nv_bfloat16*>(qkv), reinterpret_cast<__nv_bfloat16*>(kv), anc,
                                   anc_stride, pos, R, H, d, scale, reinterpret_cast<__nv_bfloat16*>(ctx)));
    count_launch();
    WB_CHECK_LAUNCH();
    return WB_OK;
}

size_t attention_beam_workspace_bytes(const Model* m, long long enc_rows, int batch, int beam, int max_len) {
    AbPlan P;
    ab_layout(m, enc_rows, batch, beam, max_len, &P);
    return P.total;
}

int attention_beam_search(const Model* m, const void* enc_bf16, long long enc_rows, const int32_t* seq_start_host,
                          const int32_t* seq_len_host, int batch, int beam, const int32_t* prefix_host, int prefix_len, int eos,
                          int max_len, float length_penalty, int32_t* out_tokens_dev, int out_stride, int32_t* out_lens_dev,
                          float* out_scores_dev, int32_t* steps_run_host, void* ws_v, size_t ws_bytes, cudaStream_t st) {
    const wb_model_config& c = m->cfg;
    const Decoder& D = m->left;
    WB_REQUIRE(!D.layers.empty(), WB_ERR_NOT_LOADED, "attention_beam_search: the model has no decoder");
    WB_REQUIRE(batch > 0 && beam >= 1 && beam <= kMaxBeam, WB_ERR_BAD_ARG, "attention_beam_search: beam %d outside [1, %d]", beam,
               kMaxBeam);
    WB_REQUIRE(beam <= c.vocab, WB_ERR_BAD_ARG, "attention_beam_search: beam > vocabulary");
    WB_REQUIRE(max_len <= 1536, WB_ERR_UNSUPPORTED, "attention_beam_search: max_len %d > 1536", max_len);
    WB_REQUIRE(prefix_len >= 1 && max_len >= prefix_len, WB_ERR_BAD_ARG, "attention_beam_search: bad prefix_len %d / max_len %d",
               prefix_len, max_len);
    const int pe_len = D.pe_len > 0 ? D.pe_len : c.max_pos;
    // positions 0 .. max_len - 2 are embedded; the reference would index past its table beyond that (embedding.py:80-101)
    WB_REQUIRE(max_len - 1 <= pe_len, WB_ERR_UNSUPPORTED, "attention_beam_search: %d decoding positions exceed the decoder's %d",
               max_len - 1, pe_len);
    AbPlan P;
    ab_layout(m, enc_rows, batch, beam, max_len, &P);
    WB_REQUIRE(ws_bytes >= P.total, WB_ERR_WORKSPACE, "attention_beam_search: workspace %zu < required %zu", ws_bytes, P.total);
    uint8_t* ws = reinterpret_cast<uint8_t*>(ws_v);
    const int d = c.d_model, ff = c.dec_ffn_dim, H = c.dec_heads, R = P.R, L = P.L, N = beam;
    const int nl = (int)D.layers.size();
    float* x = reinterpret_cast<float*>(ws + P.o_x);
    void* a = ws + P.o_a;
    __nv_bfloat16* qkv = reinterpret_cast<__nv_bfloat16*>(ws + P.o_qkv);
    __nv_bfloat16* ctx = reinterpret_cast<__nv_bfloat16*>(ws + P.o_ctx);
    void* q = ws + P.o_q;
    void* hbuf = ws + P.o_h;
    float* logits = reinterpret_cast<float*>(ws + P.o_logits);
    float* topv = reinterpret_cast<float*>(ws + P.o_topv);
    int* topi = reinterpret_cast<int*>(ws + P.o_topi);
    int* ib = reinterpret_cast<int*>(ws + P.o_int);
    int* hyp[2] = {ib, ib + (size_t)R * L};
    int* anc[2] = {ib + 2 * (size_t)R * L, ib + 3 * (size_t)R * L};
    int* tail = ib + 4 * (size_t)R * L;
    float* score[2] = {reinterpret_cast<float*>(tail), reinterpret_cast<float*>(tail + R)};
    int* endf[2] = {tail + 2 * R, tail + 3 * R};
    int* cur_tok = tail + 4 * R;
    int* cur_pos = tail + 5 * R;
    int* q_start = tail + 6 * R;
    int* q_len = q_start + batch;
    int* enc_start = q_len + batch;
    int* enc_len = enc_start + batch;
    int* utt_ended = enc_len + batch;
    int* prefix_dev = utt_ended + batch;

    // ---- host -> device: the small tables
    std::vector<int> hb((size_t)6 * R + 5 * (size_t)batch + (size_t)batch * prefix_len, 0);
    {
        float* s0 = reinterpret_cast<float*>(hb.data());
        for (int r = 0; r < R; ++r) {
            s0[r] = (r % N == 0) ? 0.f : -INFINITY;   // search.py:286-289
            s0[R + r] = s0[r];
        }
        int* t = hb.data() + 6 * (size_t)R;
        for (int b = 0; b < batch; ++b) {
            t[b] = b * N;
            t[batch + b] = N;
            t[2 * batch + b] = seq_start_host[b];
            t[3 * batch + b] = seq_len_host[b];
        }
        for (int i = 0; i < batch * prefix_len; ++i) t[5 * batch + i] = prefix_host[i];
    }
    WB_CHECK_CUDA(cudaMemcpyAsync(tail, hb.data(), hb.size() * sizeof(int), cudaMemcpyHostToDevice, st));
    // Cross attention runs as `ca_splits` key pieces per utterance (multiples of the 64-key tile): one CTA per (utterance,
    // head) walking all key tiles is two waves of the 4-CTA/SM kernel at Whisper size (32 x 20 = 640 CTAs for 592 slots, the
    // second wave 8 % full) - with pieces the tail wave is short.  Item b * S + s: the beam rows of b, piece s of its keys.
    int max_enc_len = 0;
    for (int b = 0; b < batch; ++b) max_enc_len = seq_len_host[b] > max_enc_len ? seq_len_host[b] : max_enc_len;
    int ca_splits = ceil_div(max_enc_len > 0 ? max_enc_len : 1, 64);   // at least one 64-key tile per piece
    static const int ca_cap = [] {
        const char* e = getenv("WB_CA_SPLITS");
        const int v = e ? atoi(e) : kCaSplits;
        return v < 1 ? 1 : (v > kCaMaxSplits ? kCaMaxSplits : v);
    }();
    ca_splits = ca_splits < 1 ? 1 : (ca_splits > ca_cap ? ca_cap : ca_splits);
    int* ca_tab = prefix_dev + (size_t)batch * max_len;   // q_start, q_len, k_start, k_len of the batch * ca_splits items
    {
        const int items = batch * ca_splits;
        std::vector<int> ct((size_t)4 * items);
        for (int b = 0; b < batch; ++b) {
            const int T = seq_len_host[b];
            const int piece = ceil_div(ceil_div(T > 0 ? T : 1, ca_splits), 64) * 64;
            for (int s2 = 0; s2 < ca_splits; ++s2) {
                const int it = b * ca_splits + s2;
                const int k0 = s2 * piece < T ? s2 * piece : T;
                const int k1 = (s2 + 1) * piece < T ? (s2 + 1) * piece : T;
                ct[it] = b * N;
                ct[items + it] = N;
                ct[2 * items + it] = seq_start_host[b] + k0;
                ct[3 * items + it] = k1 - k0;
            }
        }
        WB_CHECK_CUDA(cudaMemcpyAsync(ca_tab, ct.data(), ct.size() * sizeof(int), cudaMemcpyHostToDevice, st));
    }
    WB_CHECK_CUDA(cudaMemsetAsync(ib, 0, (size_t)4 * R * L * sizeof(int), st));
    // the copy above reads pageable host memory: it has completed (staged) when cudaMemcpyAsync returns

    // ---- cross-attention K/V of every layer, once (decoder_layer.py:126-135: cross_att_cache)
    const long long lda_enc = c.precise ? 3 * d : d;   // precise encoder rows are [hi | lo | hi]; the decoder reads hi
    for (int li = 0; li < nl; ++li) {
        const DecLayer& Ly = D.layers[li];
        void* memkv = ws + P.o_memkv + (size_t)li * enc_rows * 2 * d * 2;
        RC(gemm_bf16(enc_bf16, lda_enc, &Ly.ca_kv.tmap, Ly.ca_kv.w, (int)enc_rows, 2 * d, d, Ly.ca_kv.b, EPI_BF16, 1.0f, memkv,
                     2 * d, 0, st));
    }
    prefix_step_kernel<<<ceil_div(R, 128), 128, 0, st>>>(prefix_dev, prefix_len, N, L, -1, R, hyp[0], hyp[1], anc[0], anc[1],
                                                         cur_tok, cur_pos);
    count_launch();
    WB_CHECK_LAUNCH();

    const float scale = 1.0f / sqrtf(64.0f);
    int cur = 0;   // buffer holding the current hyps / ancestry / scores / flags
    int pos = 0;
    std::vector<int> ended_host(batch, 0);
    int steps = 0;
    WB_REQUIRE((size_t)SA_WARPS * 2 * max_len * sizeof(float) <= kSaSmemMax, WB_ERR_UNSUPPORTED,
               "attention_beam_search: max_len %d exceeds the %zu positions the self-attention step kernel holds", max_len,
               kSaSmemMax / (SA_WARPS * 2 * sizeof(float)));
    PdlScope pdl_scope;   // the step loop is a chain of short dependent launches: GEMMs start ahead of their predecessor's end
    // token positions 0 .. max_len - 2 are consumed; the step at position `pos` produces the token of position pos + 1
    for (pos = 0; pos + 1 < max_len; ++pos) {
        const bool beam_update = pos >= prefix_len - 1;
        RC(embed_tokens(cur_tok, cur_pos, R, d, D.emb, D.pe ? D.pe : m->pe, D.xscale, x, st));
        // every LayerNorm but the first rides in the epilogue of the residual GEMM in front of it when d == 256
        RC(layernorm_rows(x, d, R, d, D.layers[0].n1.g, D.layers[0].n1.b, c.dec_ln_eps, a, d, 0, nullptr, 0, st));
        for (int li = 0; li < nl; ++li) {
            const DecLayer& Ly = D.layers[li];
            __nv_bfloat16* kvl = reinterpret_cast<__nv_bfloat16*>(ws + P.o_kv) + (size_t)li * L * R * 2 * d;
            RC(gemm_bf16(a, d, &Ly.sa_qkv.tmap, Ly.sa_qkv.w, R, 3 * d, d, Ly.sa_qkv.b, EPI_BF16, 1.0f, qkv, 3 * d, 0, st));
            RC(dec_self_attn_step(qkv, kvl, anc[cur], L, pos, R, H, d, scale, ctx, st));
            RC(resid_then_norm(ctx, d, Ly.sa_out, R, d, x, Ly.n2, c.dec_ln_eps, a, st));
            RC(gemm_bf16(a, d, &Ly.ca_q.tmap, Ly.ca_q.w, R, d, d, Ly.ca_q.b, EPI_BF16, 1.0f, q, d, 0, st));
            {
                const void* memkv = ws + P.o_memkv + (size_t)li * enc_rows * 2 * d * 2;
                AttnArgs A;
                A.q = q; A.ldq = d; A.q_rows = R; A.q_col0 = 0;
                A.k = memkv; A.ldk = 2 * d; A.k_rows = enc_rows; A.k_col0 = 0;
                A.v = memkv; A.ldv = 2 * d; A.v_rows = enc_rows; A.v_col0 = d;
                A.kbias = nullptr; A.ld_kbias = 0;
                if (ca_splits > 1) {
                    const int items = batch * ca_splits;
                    A.q_start = ca_tab; A.q_len = ca_tab + items; A.k_start = ca_tab + 2 * items; A.k_len = ca_tab + 3 * items;
                    A.batch = items; A.splits = ca_splits;
                    A.part_o = reinterpret_cast<float*>(ws + P.o_part_o);
                    A.part_ml = ws + P.o_part_ml;
                } else {
                    A.q_start = q_start; A.q_len = q_len; A.k_start = enc_start; A.k_len = enc_len;
                    A.batch = batch;
                }
                A.heads = H; A.max_q_len = N;
                A.chunk_size = 0; A.num_left_chunks = -1; A.scale = scale;
                A.out = ctx; A.ldo = d; A.out_col0 = 0; A.split3_out = 0; A.v_mode = 0;
                RC(attention_forward(A, st));
            }
            RC(resid_then_norm(ctx, d, Ly.ca_out, R, d, x, Ly.n3, c.dec_ln_eps, a, st));
            RC(gemm_bf16(a, d, &Ly.ff1.tmap, Ly.ff1.w, R, ff, d, Ly.ff1.b, D.act_epi, 1.0f, hbuf, ff, 0, st));
            // the next layer's norm1, or after_norm behind the last layer (decoder.py:272-273)
            RC(resid_then_norm(hbuf, ff, Ly.ff2, R, d, x, (li + 1 < nl) ? D.layers[li + 1].n1 : D.after, c.dec_ln_eps, a, st));
        }
        if (!beam_update) {
            prefix_step_kernel<<<ceil_div(R, 128), 128, 0, st>>>(prefix_dev, prefix_len, N, L, pos, R, hyp[0], hyp[1], anc[0],
                                                                 anc[1], cur_tok, cur_pos);
            count_launch();
            WB_CHECK_LAUNCH();
            continue;
        }
        RC(gemm_bf16(a, d, &D.out.tmap, D.out.w, R, c.vocab, d, D.out.b, EPI_F32, 1.0f, logits, P.ldl, 0, st));
        if (c.vocab >= 16384 && N + 3 <= c.vocab / kTopkSlices)   // 320 rows x 51 866 columns: one warp per row takes 260 us
            RC(lse_topk_sliced(logits, P.ldl, R, c.vocab, N, kTopkSlices, topv, topi, ws + P.o_topk_scr, st));
        else
            RC(ctc_lse_topk(logits, P.ldl, R, c.vocab, -1, 0.0f, N, topv, topi, st));
        {
            BeamStepArgs B;
            B.topv = topv; B.topi = topi;
            B.score_in = score[cur]; B.score_out = score[cur ^ 1];
            B.end_in = endf[cur]; B.end_out = endf[cur ^ 1];
            B.hyp_in = hyp[cur]; B.hyp_out = hyp[cur ^ 1];
            B.anc_in = anc[cur]; B.anc_out = anc[cur ^ 1];
            B.cur_tok = cur_tok; B.cur_pos = cur_pos; B.utt_ended = utt_ended;
            B.N = N; B.L = L; B.pos = pos; B.eos = eos;
            ProfScope _ps(PT_MISC, st, 0.0);
            beam_step_kernel<<<batch, 128, 0, st>>>(B);
            count_launch();
            WB_CHECK_LAUNCH();
        }
        cur ^= 1;
        ++steps;
        if (steps % kPoll == 0 && pos + 2 < max_len) {
            WB_CHECK_CUDA(cudaMemcpyAsync(ended_host.data(), utt_ended, batch * sizeof(int), cudaMemcpyDeviceToHost, st));
            WB_CHECK_CUDA(cudaStreamSynchronize(st));
            long long tot = 0;
            for (int b = 0; b < batch; ++b) tot += ended_host[b];
            if (tot == R) {   // every hypothesis of every utterance has ended (search.py:301-302)
                ++pos;
                break;
            }
        }
    }
    // hyps now hold tokens at positions 0 .. pos (pos = number of consumed positions)
    const int n_tok = pos + 1 <= max_len ? pos + 1 : max_len;
    final_select_kernel<<<batch, 32, 0, st>>>(score[cur], hyp[cur], N, L, n_tok, prefix_len, eos, length_penalty, out_tokens_dev,
                                              out_stride, out_lens_dev, out_scores_dev);
    count_launch();
    WB_CHECK_LAUNCH();
    if (steps_run_host) *steps_run_host = steps;
    return WB_OK;
}

}  // namespace wb
