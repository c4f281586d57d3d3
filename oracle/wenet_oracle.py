"""CPU ORACLE — a functional restatement (plain torch-CPU ops, no nn.Module, no CUDA) of the
reference's inference hot path.  TEST INFRASTRUCTURE ONLY: imported by tests/, by
__graft_entry__.smoke() and by bench.py's cpu_baseline / `--impl reference` leg, never by the
product package `wenet_b200/` (which has no CPU path at all).

Pinned (tests/test_oracle_pin.py, run in the build container where /root/reference exists, and
through the committed goldens elsewhere):
  * fbank            == torchaudio.compliance.kaldi.fbank via wenet/dataset/processor.py:226-256, AND the
    reference's own C++ front-end (runtime/core/frontend/fbank.h + fft.cc compiled into oracle/_ref/fbank_ref by
    oracle/Makefile) in the runtime's Kaldi configuration
  * slaney_mel_filters == the reference's C++ slaney filterbank (fbank.h:91-150, 176-218) through the same binary
  * encoder / ctc / decoder == the reference modules loaded with the same state_dict (fp32)
  * ctc_prefix_beam_search  == the reference's Python search (incl. 40 random posterior matrices) AND the C++ known-answer
    test runtime/core/test/ctc_prefix_beam_search_test.cc:29-72; the reference's C++ search itself, compiled into
    oracle/_ref/ctc_search_ref, reproduces that KAT and agrees on the best hypothesis everywhere (its deeper n-best differs
    from the reference's Python search, which is the parity target)
  * attention_rescoring     == reference search.py:374-458

Every function cites the reference lines it restates.  Parameters are a flat dict keyed by the
reference's own state_dict names (SURVEY.md section 8a).

`quant` hook: q(t) -> t rounds a tensor to the operand precision of the GPU path (bf16) at exactly
the points where the CUDA kernels round (GEMM operands); with quant=None the oracle is the fp32
reference arithmetic.
"""
import math
from collections import defaultdict
from typing import Dict, List, Optional

import torch
import torch.nn.functional as F

EPS_F32 = 1.1920928955078125e-07  # torch.finfo(torch.float).eps, kaldi.py:22


def bf16_round(t: torch.Tensor) -> torch.Tensor:
    return t.to(torch.bfloat16).to(torch.float32)


def _q(quant, t):
    return t if quant is None else quant(t)


# =============================================================================================
# A. fbank — wenet/dataset/processor.py:226-256 -> torchaudio/compliance/kaldi.py:514-645
# =============================================================================================
def povey_window(n: int) -> torch.Tensor:
    # kaldi.py:99-100  hann_window(periodic=False) ** 0.85
    return torch.hann_window(n, periodic=False, dtype=torch.float32).pow(0.85)


def mel_banks(num_bins: int, padded: int, sample_freq: float, low_freq: float = 20.0,
              high_freq: float = 0.0) -> torch.Tensor:
    """kaldi.py:436-511 (vtln_warp == 1.0) + the zero last column of :627 -> (num_bins, padded/2+1)."""
    num_fft_bins = padded / 2
    nyquist = 0.5 * sample_freq
    if high_freq <= 0.0:
        high_freq += nyquist
    fft_bin_width = sample_freq / padded
    mel_low = 1127.0 * math.log(1.0 + low_freq / 700.0)
    mel_high = 1127.0 * math.log(1.0 + high_freq / 700.0)
    delta = (mel_high - mel_low) / (num_bins + 1)
    b = torch.arange(num_bins).unsqueeze(1)
    left = mel_low + b * delta
    center = mel_low + (b + 1.0) * delta
    right = mel_low + (b + 2.0) * delta
    mel = (1127.0 * (1.0 + (fft_bin_width * torch.arange(num_fft_bins)) / 700.0).log()).unsqueeze(0)
    up = (mel - left) / (center - left)
    down = (right - mel) / (right - center)
    bins = torch.max(torch.zeros(1), torch.min(up, down))
    return F.pad(bins, (0, 1), mode="constant", value=0).to(torch.float32)


def fbank(waveform: torch.Tensor, num_mel_bins: int = 80, frame_length: float = 25.0,
          frame_shift: float = 10.0, sample_rate: int = 16000, preemph: float = 0.97) -> torch.Tensor:
    """waveform: (n,) float32 already scaled to int16 range (processor.py:245 does wav * 32768).
    dither = 0, energy_floor = 0, snip_edges, remove_dc_offset, povey, round_to_power_of_two."""
    shift = int(sample_rate * frame_shift * 0.001)
    size = int(sample_rate * frame_length * 0.001)
    padded = 1 << (size - 1).bit_length()
    n = waveform.numel()
    if n < size:
        return torch.empty(0, num_mel_bins)
    m = 1 + (n - size) // shift                                    # kaldi.py:68
    frames = waveform.as_strided((m, size), (shift, 1))             # :83
    frames = frames - frames.mean(dim=1, keepdim=True)              # :184-186
    prev = F.pad(frames.unsqueeze(0), (1, 0), mode="replicate").squeeze(0)[:, :-1]
    frames = frames - preemph * prev                                # :194-198
    frames = frames * povey_window(size).unsqueeze(0)               # :200-204
    frames = F.pad(frames, (0, padded - size))                      # :207-211
    spec = torch.fft.rfft(frames).abs().pow(2.0)                    # :616-618
    mel = spec @ mel_banks(num_mel_bins, padded, float(sample_rate)).T   # :620-630
    return torch.max(mel, torch.tensor(EPS_F32)).log()              # :633


# =============================================================================================
# B. encoder — wenet/models/transformer/{encoder,encoder_layer,attention,convolution,subsampling,
#    embedding,positionwise_feed_forward,cmvn}.py, wenet/utils/mask.py
# =============================================================================================
def make_pad_mask(lengths: torch.Tensor, max_len: int) -> torch.Tensor:
    # mask.py:201-227 (True = padded)
    return torch.arange(max_len).unsqueeze(0) >= lengths.unsqueeze(1)


def subsequent_chunk_mask(size: int, chunk_size: int, num_left_chunks: int = -1) -> torch.Tensor:
    # mask.py:88-123, vectorised (same truth table as the Python loop)
    i = torch.arange(size)
    start = torch.zeros(size, dtype=torch.long) if num_left_chunks < 0 else \
        torch.clamp((i // chunk_size - num_left_chunks) * chunk_size, min=0)
    end = torch.clamp((i // chunk_size + 1) * chunk_size, max=size)
    j = torch.arange(size).unsqueeze(0)
    return (j >= start.unsqueeze(1)) & (j < end.unsqueeze(1))


def sinusoid_pe(max_len: int, d: int) -> torch.Tensor:
    # embedding.py:50-59
    pe = torch.zeros(max_len, d)
    pos = torch.arange(0, max_len, dtype=torch.float32).unsqueeze(1)
    div = torch.exp(torch.arange(0, d, 2, dtype=torch.float32) * -(math.log(10000.0) / d))
    pe[:, 0::2] = torch.sin(pos * div)
    pe[:, 1::2] = torch.cos(pos * div)
    return pe


def _ln(x, p, name, eps=1e-5):
    return F.layer_norm(x, (x.shape[-1],), p[name + ".weight"], p[name + ".bias"], eps)


def _linear(x, p, name, quant=None, bias=True):
    w = _q(quant, p[name + ".weight"])
    return F.linear(_q(quant, x), w, p.get(name + ".bias") if bias else None)   # key_bias=False: no bias key


def _ffn(x, p, pre, act, quant):
    # positionwise_feed_forward.py:50-58
    return _linear(act(_linear(x, p, pre + ".w_1", quant)), p, pre + ".w_2", quant)


def _relpos_mha(x, mask, pos_emb, p, pre, heads, quant, cache=None):
    """attention.py:364-438 (+ :109-131 forward_qkv, :133-178 forward_attention, :180-245 cache).
    x (B,T,d); mask (B,T,Tk) or (B,1,Tk) bool (True = keep) or None; pos_emb (1,Tk,d).
    cache: None or (k_cache, v_cache) each (B,h,Tc,dk).  Returns (out, (k, v))."""
    B, T, d = x.shape
    dk = d // heads
    q = _linear(x, p, pre + ".linear_q", quant).view(B, T, heads, dk)
    k = _linear(x, p, pre + ".linear_k", quant).view(B, T, heads, dk).transpose(1, 2)
    v = _linear(x, p, pre + ".linear_v", quant).view(B, T, heads, dk).transpose(1, 2)
    if quant is not None:  # the GPU path stores q/k/v as bf16 GEMM outputs
        q, k, v = quant(q), quant(k), quant(v)
    if cache is not None and cache[0].numel() > 0:
        k = torch.cat([cache[0], k], dim=2)
        v = torch.cat([cache[1], v], dim=2)
    new_cache = (k, v)
    # linear_pos has no bias; P is weight-only -> the GPU path computes it once in bf16x3 (~fp32)
    pp = F.linear(pos_emb, p[pre + ".linear_pos.weight"]).view(1, -1, heads, dk).transpose(1, 2)
    u, vb = p[pre + ".pos_bias_u"], p[pre + ".pos_bias_v"]
    if quant is None:
        q_u = (q + u).transpose(1, 2)
        q_v = (q + vb).transpose(1, 2)
        ac = torch.matmul(q_u, k.transpose(-2, -1))
        bd = torch.matmul(q_v, pp.transpose(-2, -1))     # rel_shift NOT applied (:407-409)
        scores = (ac + bd) / math.sqrt(dk)
    else:
        # GPU formulation: scores = (q.(k+p) + (u.k + v.p)) / sqrt(dk) with K' = bf16(k + p)
        kp = quant(k + pp)
        cb = (k * u.view(1, heads, 1, dk)).sum(-1) + (pp * vb.view(1, heads, 1, dk)).sum(-1)  # (B,h,Tk)
        scores = (torch.matmul(q.transpose(1, 2), kp.transpose(-2, -1)) + cb.unsqueeze(2)) / math.sqrt(dk)
    if mask is not None:
        m = mask.unsqueeze(1).eq(0)[..., :scores.size(-1)]
        scores = scores.masked_fill(m, -float("inf"))
    if quant is None:
        attn = torch.softmax(scores, dim=-1)
        if mask is not None:
            attn = attn.masked_fill(m, 0.0)
        ctx = torch.matmul(attn, v)
    else:
        mx = scores.max(dim=-1, keepdim=True).values
        mx = torch.where(torch.isinf(mx), torch.zeros_like(mx), mx)
        pr = quant(torch.exp(scores - mx))                 # unnormalised probabilities, bf16
        den = pr.sum(-1, keepdim=True)
        ctx = torch.matmul(pr, v) / torch.where(den > 0, den, torch.ones_like(den))
        ctx = quant(ctx)
    ctx = ctx.transpose(1, 2).contiguous().view(B, T, d)
    return _linear(ctx, p, pre + ".linear_out", quant), new_cache


def _conv_module(x, mask_pad, p, pre, kernel, causal, use_ln, quant, cache=None):
    """convolution.py:98-153.  x (B,T,d); mask_pad (B,1,T) bool or None; cache (B,d,K-1) or None."""
    x = x.transpose(1, 2)
    if mask_pad is not None:
        x = x.masked_fill(~mask_pad, 0.0)
    lorder = kernel - 1 if causal else 0
    new_cache = None
    if lorder > 0:
        if cache is None or cache.numel() == 0:
            x = F.pad(x, (lorder, 0), "constant", 0.0)
        else:
            x = torch.cat((cache, x), dim=2)
        new_cache = x[:, :, -lorder:]
    x = F.conv1d(_q(quant, x), _q(quant, p[pre + ".pointwise_conv1.weight"]), p[pre + ".pointwise_conv1.bias"])
    x = F.glu(x, dim=1)
    x = _q(quant, x)                                   # GLU epilogue writes bf16
    d = x.shape[1]
    x = F.conv1d(x, p[pre + ".depthwise_conv.weight"], p[pre + ".depthwise_conv.bias"],
                 padding=0 if causal else (kernel - 1) // 2, groups=d)
    if use_ln:
        x = F.layer_norm(x.transpose(1, 2), (d,), p[pre + ".norm.weight"], p[pre + ".norm.bias"], 1e-5).transpose(1, 2)
    else:
        x = F.batch_norm(x, p[pre + ".norm.running_mean"], p[pre + ".norm.running_var"], p[pre + ".norm.weight"],
                         p[pre + ".norm.bias"], False, 0.0, 1e-5)
    x = F.silu(x)
    x = F.conv1d(_q(quant, x), _q(quant, p[pre + ".pointwise_conv2.weight"]), p[pre + ".pointwise_conv2.bias"])
    if mask_pad is not None:
        x = x.masked_fill(~mask_pad, 0.0)
    return x.transpose(1, 2), new_cache


def _encoder_layer(x, mask, pos_emb, mask_pad, p, pre, cfg, quant, att_cache=None, cnn_cache=None):
    # encoder_layer.py:188-265 (normalize_before=True, macaron, conv module)
    x = x + 0.5 * _ffn(_ln(x, p, pre + ".norm_ff_macaron"), p, pre + ".feed_forward_macaron", F.silu, quant)
    att, new_att = _relpos_mha(_ln(x, p, pre + ".norm_mha"), mask, pos_emb, p, pre + ".self_attn", cfg["heads"],
                               quant, att_cache)
    x = x + att
    cv, new_cnn = _conv_module(_ln(x, p, pre + ".norm_conv"), mask_pad, p, pre + ".conv_module", cfg["cnn_kernel"],
                               cfg["causal"], cfg["cnn_norm"] == "layer_norm", quant, cnn_cache)
    x = x + cv
    x = x + 0.5 * _ffn(_ln(x, p, pre + ".norm_ff"), p, pre + ".feed_forward", F.silu, quant)
    return _ln(x, p, pre + ".norm_final"), new_att, new_cnn


def _embed(xs, p, quant, offset=0):
    # cmvn.py:36-47 + subsampling.py:203-228 + embedding.py:134-147
    if "encoder.global_cmvn.mean" in p:
        xs = (xs - p["encoder.global_cmvn.mean"]) * p["encoder.global_cmvn.istd"]
    x = xs.unsqueeze(1)
    x = F.relu(F.conv2d(x, p["encoder.embed.conv.0.weight"], p["encoder.embed.conv.0.bias"], stride=2))
    x = F.relu(F.conv2d(_q(quant, x), _q(quant, p["encoder.embed.conv.2.weight"]), p["encoder.embed.conv.2.bias"],
                        stride=2))
    b, c, t, f = x.shape
    x = _linear(x.transpose(1, 2).contiguous().view(b, t, c * f), p, "encoder.embed.out.0", quant)
    d = x.shape[-1]
    x = x * math.sqrt(d)
    return x


def encoder_cfg(p: Dict[str, torch.Tensor], heads: int, causal: bool, cnn_norm: str) -> dict:
    d = p["encoder.after_norm.weight"].numel()
    n_layers = 1 + max(int(k.split(".")[2]) for k in p if k.startswith("encoder.encoders."))
    return dict(d=d, heads=heads, layers=n_layers, causal=causal, cnn_norm=cnn_norm,
                cnn_kernel=p["encoder.encoders.0.conv_module.depthwise_conv.weight"].shape[-1])


def encoder_forward(p, cfg, xs, xs_lens, decoding_chunk_size=-1, num_decoding_left_chunks=-1, quant=None,
                    taps: Optional[list] = None):
    """encoder.py:122-181.  xs (B,T,80) padded, xs_lens (B,).  Returns (out (B,T',d), masks (B,1,T'))."""
    assert decoding_chunk_size != 0
    T = xs.size(1)
    masks = ~make_pad_mask(xs_lens, T).unsqueeze(1)
    x = _embed(xs, p, quant)
    masks = masks[:, :, 2::2][:, :, 2::2]
    Tp = x.size(1)
    pos_emb = sinusoid_pe(5000, cfg["d"])[:Tp].unsqueeze(0)
    if taps is not None:
        taps.append(x.clone())
    if decoding_chunk_size > 0:
        chunk_masks = masks & subsequent_chunk_mask(Tp, decoding_chunk_size, num_decoding_left_chunks).unsqueeze(0)
    else:
        chunk_masks = masks     # full context (mask.py:164-166)
    for i in range(cfg["layers"]):
        x, _, _ = _encoder_layer(x, chunk_masks, pos_emb, masks, p, "encoder.encoders.%d" % i, cfg, quant)
        if taps is not None:
            taps.append(x.clone())
    return _ln(x, p, "encoder.after_norm"), masks


def encoder_forward_chunk(p, cfg, xs, offset, required_cache_size, att_cache, cnn_cache, quant=None):
    """encoder.py:204-300 (batch 1).  att_cache (L,h,Tc,2dk) or empty; cnn_cache (L,1,d,K-1) or empty."""
    x = _embed(xs, p, quant)
    cache_t1 = att_cache.size(2) if att_cache.numel() > 0 else 0
    chunk = x.size(1)
    key_size = cache_t1 + chunk
    pe = sinusoid_pe(5000, cfg["d"])
    pos_emb = pe[offset - cache_t1: offset - cache_t1 + key_size].unsqueeze(0)
    if required_cache_size < 0:
        nxt = 0
    elif required_cache_size == 0:
        nxt = key_size
    else:
        nxt = max(key_size - required_cache_size, 0)
    dk = cfg["d"] // cfg["heads"]
    r_att, r_cnn = [], []
    for i in range(cfg["layers"]):
        ac = None
        if att_cache.numel() > 0:
            ac = (att_cache[i:i + 1, :, :, :dk], att_cache[i:i + 1, :, :, dk:])
        cc = cnn_cache[i] if cnn_cache.numel() > 0 else None
        x, new_att, new_cnn = _encoder_layer(x, None, pos_emb, None, p, "encoder.encoders.%d" % i, cfg, quant, ac, cc)
        r_att.append(torch.cat(new_att, dim=-1)[:, :, nxt:, :])
        r_cnn.append(new_cnn.unsqueeze(0))
    return _ln(x, p, "encoder.after_norm"), torch.cat(r_att, dim=0), torch.cat(r_cnn, dim=0)


# =============================================================================================
# C. CTC — ctc.py:73-81, asr_model.py:254-265
# =============================================================================================
def ctc_logprobs(p, enc_out, blank_penalty: float = 0.0, blank_id: int = 0, quant=None):
    logits = _linear(enc_out, p, "ctc.ctc_lo", quant)
    if blank_penalty > 0.0:
        logits[:, :, blank_id] -= blank_penalty
    return logits.log_softmax(dim=2)


# =============================================================================================
# D. searches — search.py:30-249, common.py:302-310, ctc_utils.py:23-33
# =============================================================================================
def log_add(*args) -> float:
    if all(a == -float("inf") for a in args):
        return -float("inf")
    a_max = max(args)
    return a_max + math.log(sum(math.exp(a - a_max) for a in args))


def remove_duplicates_and_blank(hyp: List[int], blank_id: int = 0) -> List[int]:
    out, cur = [], 0
    while cur < len(hyp):
        if hyp[cur] != blank_id:
            out.append(hyp[cur])
        prev = cur
        while cur < len(hyp) and hyp[cur] == hyp[prev]:
            cur += 1
    return out


def ctc_greedy_search(ctc_probs: torch.Tensor, ctc_lens: torch.Tensor, blank_id: int = 0) -> List[List[int]]:
    # search.py:109-124
    B, maxlen = ctc_probs.shape[:2]
    idx = ctc_probs.argmax(dim=2)
    idx = idx.masked_fill(make_pad_mask(ctc_lens, maxlen), blank_id)
    return [remove_duplicates_and_blank(h.tolist(), blank_id) for h in idx]


class _PS:
    """PrefixScore, search.py:64-106 (context fields :76-78, :91-106)."""

    def __init__(self, s=-float("inf"), ns=-float("inf"), v_s=-float("inf"), v_ns=-float("inf"), context_state=0,
                 context_score=0.0):
        self.s, self.ns, self.v_s, self.v_ns = s, ns, v_s, v_ns
        self.cur_token_prob = -float("inf")
        self.times_s, self.times_ns = [], []
        self.context_state, self.context_score, self.has_context = context_state, context_score, False

    def score(self):
        return log_add(self.s, self.ns)

    def viterbi_score(self):
        return self.v_s if self.v_s > self.v_ns else self.v_ns

    def times(self):
        return self.times_s if self.v_s > self.v_ns else self.times_ns

    def total_score(self):
        return self.score() + self.context_score


def context_forward_one_step(cg, state: int, token: int):
    """ContextGraph.forward_one_step (wenet/utils/context_graph.py:212-247) on a flattened graph
    (wenet_b200.context.ContextArrays: children / fail arcs / scores by node index, root = 0)."""
    c = cg.child(state, token)
    if c >= 0:
        node = c
        score = float(cg.token_score[node])
    else:
        node = int(cg.fail[state])
        while cg.child(node, token) < 0:
            node = int(cg.fail[node])
            if int(cg.token[node]) == -1:
                break
        c2 = cg.child(node, token)
        if c2 >= 0:
            node = c2
        score = float(cg.node_score[node]) - float(cg.node_score[state])
    return score + float(cg.output_score[node]), node


def ctc_prefix_beam_search(ctc_probs: torch.Tensor, ctc_lens, beam_size: int, blank_id: int = 0, context=None):
    """search.py:127-249.  `context`: None or a flattened context graph (the reference's ContextGraph restated on
    arrays: update_context / copy_context :97-106, finalize context_graph.py:249-265 - NB the reference REPLACES the
    accumulated context score by finalize()'s score at the end, search.py:229-234).  Returns per utterance a dict with
    nbest, nbest_scores, nbest_times (lists, best first)."""
    results = []
    for i in range(ctc_probs.shape[0]):
        ctc_prob = ctc_probs[i]
        num_t = int(ctc_lens[i])
        cur_hyps = [(tuple(), _PS(s=0.0, ns=-float("inf"), v_s=0.0, v_ns=0.0))]

        def copy_ctx(n, ps):
            if context is not None and not n.has_context:
                n.context_score, n.context_state, n.has_context = ps.context_score, ps.context_state, True

        def update_ctx(n, ps, u):
            if context is not None and not n.has_context:
                sc, st = context_forward_one_step(context, ps.context_state, u)
                n.context_score, n.context_state, n.has_context = ps.context_score + sc, st, True

        for t in range(num_t):
            logp = ctc_prob[t]
            next_hyps = defaultdict(_PS)
            _, top_k_index = logp.topk(beam_size)
            for u in top_k_index.tolist():
                prob = logp[u].item()
                for prefix, ps in cur_hyps:
                    last = prefix[-1] if len(prefix) > 0 else None
                    if u == blank_id:
                        n = next_hyps[prefix]
                        n.s = log_add(n.s, ps.score() + prob)
                        n.v_s = ps.viterbi_score() + prob
                        n.times_s = ps.times().copy()
                        copy_ctx(n, ps)
                    elif u == last:
                        n1 = next_hyps[prefix]
                        n1.ns = log_add(n1.ns, ps.ns + prob)
                        if n1.v_ns < ps.v_ns + prob:
                            n1.v_ns = ps.v_ns + prob
                            if n1.cur_token_prob < prob:
                                n1.cur_token_prob = prob
                                n1.times_ns = ps.times_ns.copy()
                                n1.times_ns[-1] = t
                        copy_ctx(n1, ps)
                        n2 = next_hyps[prefix + (u,)]
                        n2.ns = log_add(n2.ns, ps.s + prob)
                        if n2.v_ns < ps.v_s + prob:
                            n2.v_ns = ps.v_s + prob
                            n2.cur_token_prob = prob
                            n2.times_ns = ps.times_s.copy()
                            n2.times_ns.append(t)
                        update_ctx(n2, ps, u)
                    else:
                        n = next_hyps[prefix + (u,)]
                        n.ns = log_add(n.ns, ps.score() + prob)
                        if n.v_ns < ps.viterbi_score() + prob:
                            n.v_ns = ps.viterbi_score() + prob
                            n.cur_token_prob = prob
                            n.times_ns = ps.times().copy()
                            n.times_ns.append(t)
                        update_ctx(n, ps, u)
            nxt = sorted(next_hyps.items(), key=lambda kv: kv[1].total_score(), reverse=True)
            cur_hyps = nxt[:beam_size]
        if context is not None:
            for _, ps in cur_hyps:
                ps.context_score = -float(context.node_score[ps.context_state])   # finalize(): replaces, not adds
                ps.context_state = 0
        results.append(dict(nbest=[list(y[0]) for y in cur_hyps],
                            nbest_scores=[y[1].total_score() for y in cur_hyps],
                            nbest_times=[list(y[1].times()) for y in cur_hyps]))
    return results


# =============================================================================================
# E. rescoring decoder — decoder.py:146-201,430-463, decoder_layer.py:68-153, attention.py:247-304,
#    :441-520, asr_model.py:453-547, search.py:374-458
# =============================================================================================
def _mha(xq, xkv, mask, p, pre, heads, quant):
    B, Tq, d = xq.shape
    dk = d // heads
    q = _linear(xq, p, pre + ".linear_q", quant).view(B, Tq, heads, dk).transpose(1, 2)
    k = _linear(xkv, p, pre + ".linear_k", quant).view(B, -1, heads, dk).transpose(1, 2)
    v = _linear(xkv, p, pre + ".linear_v", quant).view(B, -1, heads, dk).transpose(1, 2)
    if quant is not None:
        q, k, v = quant(q), quant(k), quant(v)
    scores = torch.matmul(q, k.transpose(-2, -1)) / math.sqrt(dk)
    if mask is not None:
        m = mask.unsqueeze(1).eq(0)
        scores = scores.masked_fill(m, -float("inf"))
    if quant is None:
        attn = torch.softmax(scores, dim=-1)
        if mask is not None:
            attn = attn.masked_fill(m, 0.0)
        ctx = torch.matmul(attn, v)
    else:
        mx = scores.max(dim=-1, keepdim=True).values
        mx = torch.where(torch.isinf(mx), torch.zeros_like(mx), mx)
        pr = quant(torch.exp(scores - mx))
        den = pr.sum(-1, keepdim=True)
        ctx = quant(torch.matmul(pr, v) / torch.where(den > 0, den, torch.ones_like(den)))
    ctx = ctx.transpose(1, 2).contiguous().view(B, Tq, d)
    return _linear(ctx, p, pre + ".linear_out", quant)


def decoder_forward(p, pre, n_layers, heads, memory, ys_in_pad, ys_in_lens, quant=None):
    """TransformerDecoder.forward (decoder.py:146-201): returns logits (B, L, V).  memory (B,T,d)."""
    B, L = ys_in_pad.shape
    d = memory.shape[-1]
    tgt_mask = ~make_pad_mask(ys_in_lens, L).unsqueeze(1)                   # (B,1,L)
    tgt_mask = tgt_mask & torch.tril(torch.ones(L, L, dtype=torch.bool)).unsqueeze(0)
    x = F.embedding(ys_in_pad, p[pre + ".embed.0.weight"]) * math.sqrt(d) + sinusoid_pe(5000, d)[:L].unsqueeze(0)
    for i in range(n_layers):
        lp = "%s.decoders.%d" % (pre, i)
        x = x + _mha(_ln(x, p, lp + ".norm1"), _ln(x, p, lp + ".norm1"), tgt_mask, p, lp + ".self_attn", heads, quant)
        x = x + _mha(_ln(x, p, lp + ".norm2"), memory, None, p, lp + ".src_attn", heads, quant)
        x = x + _ffn(_ln(x, p, lp + ".norm3"), p, lp + ".feed_forward", F.relu, quant)
    x = _ln(x, p, pre + ".after_norm")
    return _linear(x, p, pre + ".output_layer", quant)


def forward_attention_decoder(p, dcfg, hyps, hyps_lens, encoder_out, reverse_weight, eos, quant=None):
    """asr_model.py:453-547.  dcfg: dict(bidirectional, layers, r_layers, heads).  hyps (N, L) with sos."""
    N = hyps.size(0)
    memory = encoder_out.repeat(N, 1, 1)
    r_lens = hyps_lens - 1
    r_hyps = hyps[:, 1:]
    max_len = int(r_lens.max())
    idx_range = torch.arange(0, max_len)
    seq_mask = r_lens.unsqueeze(1) > idx_range
    index = ((r_lens.unsqueeze(1) - 1) - idx_range) * seq_mask
    r_hyps = torch.where(seq_mask, torch.gather(r_hyps, 1, index), torch.tensor(eos))
    r_hyps = torch.cat([hyps[:, 0:1], r_hyps], dim=1)
    left = "decoder.left_decoder" if dcfg["bidirectional"] else "decoder"
    if quant is not None:
        memory = quant(memory)
    out = decoder_forward(p, left, dcfg["layers"], dcfg["heads"], memory, hyps, hyps_lens, quant).log_softmax(-1)
    r_out = torch.tensor(0.0)
    if dcfg["bidirectional"] and reverse_weight > 0:
        r_out = decoder_forward(p, "decoder.right_decoder", dcfg["r_layers"], dcfg["heads"], memory, r_hyps,
                                hyps_lens, quant).log_softmax(-1)
    return out, r_out


def attention_rescoring(p, dcfg, beam_results, encoder_outs, encoder_lens, sos, eos, ctc_weight=0.0,
                        reverse_weight=0.0, quant=None):
    """search.py:374-458.  Returns per utterance dict(best_index, best_score, scores[list])."""
    out = []
    for b in range(encoder_outs.shape[0]):
        enc = encoder_outs[b, :int(encoder_lens[b]), :].unsqueeze(0)
        hyps = beam_results[b]["nbest"]
        ctc_scores = beam_results[b]["nbest_scores"]
        lens = torch.tensor([len(h) for h in hyps], dtype=torch.long)
        L = int(lens.max()) if len(hyps) else 0
        pad = torch.full((len(hyps), L + 1), eos, dtype=torch.long)   # add_sos_eos: pad ys_in with eos
        pad[:, 0] = sos
        for i, h in enumerate(hyps):
            if len(h):
                pad[i, 1:1 + len(h)] = torch.tensor(h, dtype=torch.long)
        dec, r_dec = forward_attention_decoder(p, dcfg, pad, lens + 1, enc, reverse_weight, eos, quant)
        best_score, best_index, scores = -float("inf"), 0, []
        for i, hyp in enumerate(hyps):
            score = 0.0
            for j, w in enumerate(hyp):
                score += dec[i][j][w]
            score += dec[i][len(hyp)][eos]
            if reverse_weight > 0 and r_dec.dim() > 0:
                r_score = 0.0
                for j, w in enumerate(hyp):
                    r_score += r_dec[i][len(hyp) - j - 1][w]
                r_score += r_dec[i][len(hyp)][eos]
                score = score * (1 - reverse_weight) + r_score * reverse_weight
            score += ctc_scores[i] * ctc_weight
            scores.append(float(score))
            if score > best_score:
                best_score = float(score)
                best_index = i
        out.append(dict(best_index=best_index, best_score=best_score, scores=scores,
                        tokens=hyps[best_index] if hyps else []))
    return out


# =============================================================================================
# Whisper (SURVEY section 8f-1): log-mel front-end, TransformerEncoder with Conv1dSubsampling2, and the
# autoregressive attention_beam_search shared with ASRModel.decode(mode "attention")
# =============================================================================================
def slaney_mel_filters(sr: int = 16000, n_fft: int = 400, n_mels: int = 128) -> torch.Tensor:
    """librosa.filters.mel(sr, n_fft, n_mels) (slaney scale, slaney norm) restated from its published algorithm; the
    reference calls it at processor.py:360-361.  librosa is not installed in the build container, so the pin is the
    REFERENCE'S OWN C++ implementation of the same filterbank (runtime/core/frontend/fbank.h:91-150 InitMelFilters with
    MelType::kSlaney, :176-218 MelScale / InverseMelScale), compiled from the reference sources into oracle/_ref/fbank_ref:
    same support and weights to fp32 rounding for 128 and 80 bins on the C++ front-end's 512-point grid
    (tests/test_oracle_pin.py::test_slaney_mel_filters_vs_reference_cxx; n_fft enters this function only through the
    bin-frequency grid `fft`).  The Python call site is pinned with this restatement injected as librosa.filters.mel
    (test_whisper_oracle_matches_reference compares everything around it with compute_log_mel_spectrogram)."""
    def hz_to_mel(f):
        f_sp, min_log_hz = 200.0 / 3, 1000.0
        if f >= min_log_hz:
            return min_log_hz / f_sp + math.log(f / min_log_hz) / (math.log(6.4) / 27.0)
        return f / f_sp

    def mel_to_hz(m):
        f_sp, min_log_hz = 200.0 / 3, 1000.0
        min_log_mel = min_log_hz / f_sp
        if m >= min_log_mel:
            return min_log_hz * math.exp(math.log(6.4) / 27.0 * (m - min_log_mel))
        return f_sp * m

    nb = 1 + n_fft // 2
    fft = [i * (sr / 2.0) / (nb - 1) for i in range(nb)]
    lo, hi = hz_to_mel(0.0), hz_to_mel(sr / 2.0)
    mel_f = [mel_to_hz(lo + (hi - lo) * i / (n_mels + 1)) for i in range(n_mels + 2)]
    w = torch.zeros(n_mels, nb, dtype=torch.float64)
    for i in range(n_mels):
        for k in range(nb):
            lower = (fft[k] - mel_f[i]) / (mel_f[i + 1] - mel_f[i])
            upper = (mel_f[i + 2] - fft[k]) / (mel_f[i + 2] - mel_f[i + 1])
            w[i, k] = max(0.0, min(lower, upper)) * 2.0 / (mel_f[i + 2] - mel_f[i])
    return w.float()


def log_mel_spectrogram(waveform: torch.Tensor, n_fft: int = 400, hop_length: int = 160, num_mel_bins: int = 80,
                        sample_rate: int = 16000) -> torch.Tensor:
    """processor.py:320-369 with padding = 0, pad_or_trim = False.  waveform (n,) float in [-1, 1) -> (n // hop, mel)."""
    window = torch.hann_window(n_fft)
    stft = torch.stft(waveform, n_fft, hop_length, window=window, return_complex=True)
    magnitudes = stft[..., :-1].abs() ** 2
    mel_spec = slaney_mel_filters(sample_rate, n_fft, num_mel_bins) @ magnitudes
    log_spec = torch.clamp(mel_spec, min=1e-10).log10()
    log_spec = torch.maximum(log_spec, log_spec.max() - 8.0)
    log_spec = (log_spec + 4.0) / 4.0
    return log_spec.transpose(0, 1)


def whisper_sinusoids(max_len: int, d: int) -> torch.Tensor:
    # embedding.py:150-164
    inc = math.log(10000) / (d // 2 - 1)
    inv = torch.exp(-inc * torch.arange(d // 2))
    st = torch.arange(max_len)[:, None] * inv[None, :]
    return torch.cat([torch.sin(st), torch.cos(st)], dim=1)


def whisper_encoder_forward(p, heads: int, xs: torch.Tensor, xs_lens: torch.Tensor, quant=None):
    """TransformerEncoder.forward (encoder.py:122-181) for conv1d2 / abs_pos_whisper / gelu / pre-norm:
    Conv1dSubsampling2 (subsampling.py:117-171), layers (encoder_layer.py:28-135), after_norm.
    xs (B, T, idim) zero padded, xs_lens (B,).  Returns (B, T', d), masks (B, 1, T')."""
    B, T, _ = xs.shape
    masks = ~make_pad_mask(xs_lens, T).unsqueeze(1)
    x = xs.transpose(1, 2)
    x = F.gelu(F.conv1d(_q(quant, x), _q(quant, p["encoder.embed.conv.0.weight"]), p["encoder.embed.conv.0.bias"], padding=1))
    x = F.gelu(F.conv1d(_q(quant, x), _q(quant, p["encoder.embed.conv.2.weight"]), p["encoder.embed.conv.2.bias"], stride=2,
                        padding=1))
    x = _q(quant, x.transpose(1, 2))
    d = x.shape[-1]
    pe = p.get("encoder.embed.pos_enc.pe")
    pe = whisper_sinusoids(1500, d) if pe is None else pe.reshape(-1, d)
    x = x + pe[:x.shape[1]].unsqueeze(0)                      # xscale = 1
    masks = masks[:, :, (T + 1) % 2::2]
    n_layers = 0
    while "encoder.encoders.%d.norm1.weight" % n_layers in p:
        n_layers += 1
    for i in range(n_layers):
        lp = "encoder.encoders.%d" % i
        xn = _ln(x, p, lp + ".norm1")
        x = x + _mha(xn, xn, masks, p, lp + ".self_attn", heads, quant)
        x = x + _ffn(_ln(x, p, lp + ".norm2"), p, lp + ".feed_forward", F.gelu, quant)
    return _ln(x, p, "encoder.after_norm"), masks


def decoder_last_logp(p, pre, n_layers, heads, memory, mem_mask, hyps, flavor: str, quant=None):
    """TransformerDecoder.forward_one_step (decoder.py:226-281) WITHOUT the caches: the decoder is re-run on the whole
    prefix and the last position kept - the caches (decoder_layer.py:101-139) only memoise exactly these values.
    memory (Bm, T, d) with Bm == B or B % Bm == 0 (the beams of an utterance share it, attention.py:488-497).
    flavor "wenet": emb * sqrt(d) + sinusoid PE, relu; "whisper": emb + learnable PE, gelu."""
    R, L = hyps.shape
    d = memory.shape[-1]
    if memory.shape[0] != R:
        rep = R // memory.shape[0]
        memory = memory.repeat_interleave(rep, dim=0)
        mem_mask = mem_mask.repeat_interleave(rep, dim=0)
    emb = F.embedding(hyps, p[pre + ".embed.0.weight"])
    if flavor == "whisper":
        x = emb + p[pre + ".embed.1.pe"].reshape(-1, d)[:L].unsqueeze(0)
        act = F.gelu
    else:
        x = emb * math.sqrt(d) + sinusoid_pe(5000, d)[:L].unsqueeze(0)
        act = F.relu
    tgt_mask = torch.tril(torch.ones(L, L, dtype=torch.bool)).unsqueeze(0).expand(R, L, L)
    if quant is not None:
        memory = quant(memory)
    for i in range(n_layers):
        lp = "%s.decoders.%d" % (pre, i)
        xn = _ln(x, p, lp + ".norm1")
        x = x + _mha(xn, xn, tgt_mask, p, lp + ".self_attn", heads, quant)
        x = x + _mha(_ln(x, p, lp + ".norm2"), memory, mem_mask, p, lp + ".src_attn", heads, quant)
        x = x + _ffn(_ln(x, p, lp + ".norm3"), p, lp + ".feed_forward", act, quant)
    y = _ln(x[:, -1], p, pre + ".after_norm")
    return torch.log_softmax(_linear(y, p, pre + ".output_layer", quant), dim=-1)


def beam_step(top_k_logp, top_k_index, scores, end_flag, hyps, beam_size: int, eos: int):
    """One iteration of search.py:309-355 after the decoder call: masks (mask.py:258-310), second prune, hypothesis
    update.  Shapes as the reference: (B*N, N), (B*N, N), (B*N, 1), (B*N, 1) bool, (B*N, i)."""
    running = top_k_logp.shape[0]
    batch = running // beam_size
    top_k_logp = top_k_logp.clone()
    top_k_index = top_k_index.clone()
    for r in range(running):
        if bool(end_flag[r]):
            top_k_logp[r, 0] = 0.0
            top_k_logp[r, 1:] = -float("inf")
            top_k_index[r, :] = eos
    cand = (scores + top_k_logp).view(batch, beam_size * beam_size)
    new_scores = torch.zeros(batch, beam_size)
    new_hyps = torch.zeros(running, hyps.shape[1] + 1, dtype=torch.long)
    parents = torch.zeros(running, dtype=torch.long)
    for b in range(batch):
        order = sorted(range(beam_size * beam_size), key=lambda c: (-float(cand[b, c]), c))[:beam_size]
        for n, c in enumerate(order):
            pr = b * beam_size + c // beam_size
            new_scores[b, n] = cand[b, c]
            new_hyps[b * beam_size + n, :-1] = hyps[pr]
            new_hyps[b * beam_size + n, -1] = top_k_index[pr, c % beam_size]
            parents[b * beam_size + n] = pr
    new_end = new_hyps[:, -1].eq(eos).view(-1, 1)
    return new_scores.view(-1, 1), new_end, new_hyps, parents


def attention_beam_search(p, pre, n_layers, heads, encoder_out, encoder_mask, beam_size: int, prefix, eos: int,
                          length_penalty: float = 0.0, flavor: str = "wenet", quant=None, maxlen: Optional[int] = None,
                          return_beams: bool = False):
    """search.py:252-371.  prefix: (B, P) long - [[sos]] * B for wenet models, add_whisper_tokens' forced start for
    Whisper (common.py:198-226).  Returns the best hypothesis of every utterance (prefix and eos stripped); with
    return_beams also every utterance's final beams as (hypothesis, score) pairs."""
    B = encoder_out.shape[0]
    if maxlen is None:
        maxlen = encoder_out.shape[1]      # the reference's bound (search.py:263); tests may shorten the loop
    running = B * beam_size
    hyps = torch.as_tensor(prefix, dtype=torch.long).repeat_interleave(beam_size, dim=0)
    P = hyps.shape[1]
    scores = torch.tensor([0.0] + [-float("inf")] * (beam_size - 1)).repeat(B).unsqueeze(1)
    end_flag = torch.zeros_like(scores, dtype=torch.bool)
    for i in range(P, maxlen + 1):
        if int(end_flag.sum()) == running:
            break
        logp = decoder_last_logp(p, pre, n_layers, heads, encoder_out, encoder_mask, hyps, flavor, quant)
        top_k_logp, top_k_index = logp.topk(beam_size)
        scores, end_flag, hyps, _ = beam_step(top_k_logp, top_k_index, scores, end_flag, hyps, beam_size, eos)
    scores = scores.view(B, beam_size)
    lengths = hyps.ne(eos).sum(dim=1).view(B, beam_size).float()
    scores = scores / lengths.pow(length_penalty)
    best = scores.argmax(dim=-1)
    strip = lambda h: h[P:][h[P:] != eos].tolist()      # noqa: E731
    out = [strip(hyps[b * beam_size + int(best[b])]) for b in range(B)]
    if return_beams:
        return out, [[(strip(hyps[b * beam_size + n]), float(scores[b, n])) for n in range(beam_size)] for b in range(B)]
    return out
