"""Operator-level parity (GPU) of the kernels that turn encoder output into the final answer: the output layer of
attention rescoring (gemm_lse_partials + lse_target_logprob), the token embedding, the rescoring score combine, the
attention kernel in the modes only the model paths use (split-key pieces + merge, pre-scaled key bias, column offsets
into fused buffers) and the cached self-attention step of attention decoding.

Every reference is plain torch / numpy in fp64 (fp32 where the reference itself computes in fp32) on the SAME
bf16-rounded operands the kernel sees, and every gate is derived from the arithmetic in the test's docstring.  The
observed worst error is printed (run with -s)."""
import math

import numpy as np
import pytest
import torch

from wenet_b200 import _lib
from wenet_b200._lib import check, cur_stream, ptr

pytestmark = pytest.mark.gpu

LOG2E = 1.4426950408889634


def _dev():
    return torch.device("cuda:0")


def _ti(x):
    return torch.tensor(x, dtype=torch.int32, device=_dev())


def _grid_operands(M, N, K, g, lda=None):
    """bf16 operands on a coarse grid: a in {-8..8}/8, w in {-16..16}/64.  Every product is a multiple of 2^-9 and every
    partial sum over K <= 512 stays below 2^8 in magnitude, so the fp32 accumulation of the tensor core (and of any other
    summation order) is EXACT: the logits a w^T differ from the fp64 reference only by the one rounding of + bias.  The
    logits still spread like a decoder's (std ~2)."""
    lda = lda or K
    a_full = torch.zeros(M, lda, dtype=torch.bfloat16)
    a_full[:, :K] = (torch.randint(-8, 9, (M, K), generator=g).float() / 8).to(torch.bfloat16)
    w = (torch.randint(-16, 17, (N, K), generator=g).float() / 64).to(torch.bfloat16)
    return a_full.to(_dev()), w.to(_dev())


# ---------------------------------------------------------------------------------------------------------------- wrappers
def lse_parts(N, K):
    return int(_lib.load().wb_op_lse_parts(N, K))


def gemm_lse_partials(a, w, bias, part):
    M, K = a.shape[0], w.shape[1]
    check(_lib.load().wb_op_gemm_lse_partials(ptr(a), a.stride(0), ptr(w), M, w.shape[0], K, ptr(bias), ptr(part),
                                              cur_stream()), "wb_op_gemm_lse_partials")


def lse_target_logprob(part, n_parts, a, w, bias, target, row_map, V):
    R = target.numel()
    out = torch.full((R,), 12345.0, device=_dev())
    check(_lib.load().wb_op_lse_target_logprob(ptr(part), n_parts, ptr(a), a.stride(0), ptr(w), w.shape[1], ptr(bias),
                                               ptr(target), ptr(row_map), R, V, ptr(out), cur_stream()),
          "wb_op_lse_target_logprob")
    return out


def attention_ex(q, k, v, q_start, q_len, k_start, k_len, heads, max_q_len, out, kbias=None, chunk_size=0,
                 num_left_chunks=-1, scale=0.125, q_col0=0, k_col0=0, v_col0=0, out_col0=0, kbias_scaled=0, splits=1,
                 split_key=False):
    batch = q_start.numel()
    part_o = part_ml = None
    if split_key:
        part_o = torch.full((batch * heads * max_q_len * 64,), float("nan"), device=_dev())
        part_ml = torch.full((batch * heads * max_q_len * 2,), float("nan"), device=_dev())
    check(_lib.load().wb_op_attention_ex(
        ptr(q), q.stride(0), q.shape[0], q_col0, ptr(k), k.stride(0), k.shape[0], k_col0, ptr(v), v.stride(0), v.shape[0],
        v_col0, ptr(kbias), kbias.stride(0) if kbias is not None else 0, ptr(q_start), ptr(q_len), ptr(k_start), ptr(k_len),
        batch, heads, max_q_len, chunk_size, num_left_chunks, float(scale), ptr(out), out.stride(0), out_col0, 0,
        kbias_scaled, splits, ptr(part_o), ptr(part_ml), cur_stream()), "wb_op_attention_ex")
    return out


def _attn_ref64(q, k, v, kbias, q_start, q_len, k_start, k_len, heads, chunk, left, scale, q_col0=0, k_col0=0, v_col0=0):
    """fp64 softmax attention per (query block, head); rows of blocks without keys stay 0 (the kernel's contract)."""
    out = torch.zeros(q.shape[0], heads * 64, dtype=torch.float64)
    for b in range(len(q_start)):
        qs, ql, ks, kl = q_start[b], q_len[b], k_start[b], k_len[b]
        if kl == 0 or ql == 0:
            continue
        for h in range(heads):
            Q = q[qs:qs + ql, q_col0 + h * 64:q_col0 + (h + 1) * 64].double()
            K = k[ks:ks + kl, k_col0 + h * 64:k_col0 + (h + 1) * 64].double()
            V = v[ks:ks + kl, v_col0 + h * 64:v_col0 + (h + 1) * 64].double()
            S = Q @ K.T
            if kbias is not None:
                S = S + kbias[ks:ks + kl, h].double().unsqueeze(0)
            S = S * scale
            if chunk > 0:
                i = torch.arange(ql).unsqueeze(1)
                j = torch.arange(kl).unsqueeze(0)
                start = torch.zeros_like(i) if left < 0 else torch.clamp((i // chunk - left) * chunk, min=0)
                S = S.masked_fill(~((j >= start) & (j < (i // chunk + 1) * chunk)), -float("inf"))
            out[qs:qs + ql, h * 64:(h + 1) * 64] = torch.softmax(S, -1) @ V
    return out


def _attn_gate(got, ref, vmax, what):
    """The gate of test_ops_gpu.py::test_attention: the kernel rounds the probabilities to bf16 (2^-9 relative each,
    relative to a lazily raised running maximum) before P V and rounds the output to bf16 (2^-9 relative): at most
    2^-8 max|v| + 2^-9 |ref| in the worst case, so 2^-7 |ref| + 2^-8 max|v| holds with a factor-2 margin; the typical
    error is an order of magnitude below, hence the mean gate."""
    diff = (got.double() - ref).abs()
    bound = 2 ** -7 * ref.abs() + 2 ** -8 * vmax
    print("%s: max err %.3g (gate at that element %.3g), mean %.3g (gate 1e-3)" % (
        what, diff.max().item(), bound.flatten()[diff.argmax()].item(), diff.mean().item()))
    bad = diff > bound
    assert not bad.any(), "%s: max diff %g at %s" % (what, diff.max().item(), tuple(torch.nonzero(bad)[0].tolist()))
    assert diff.mean().item() < 1e-3, (what, diff.mean().item())


# ---------------------------------------------------------------------------------------------------- 1. LSE partials
def _part_ref(logits64, V, bn):
    """fp64 (max, sum) per half tile, log2 domain, as gemm_lse_partials defines them; empty halves (-inf, 0)."""
    M = logits64.shape[0]
    n_tiles = (V + bn - 1) // bn
    half = bn // 2
    m = torch.full((M, 2 * n_tiles), -math.inf, dtype=torch.float64)
    s = torch.zeros(M, 2 * n_tiles, dtype=torch.float64)
    v2 = logits64 * LOG2E
    for p in range(2 * n_tiles):
        c0, c1 = p * half, min((p + 1) * half, V)
        if c0 >= V:
            continue
        blk = v2[:, c0:c1]
        m[:, p] = blk.max(1).values
        s[:, p] = torch.exp2(blk - m[:, p:p + 1]).sum(1)
    return m, s


def _recombine(m, s):
    """log-sum-exp (natural log) of a row from its (max, sum) pairs, in fp64"""
    M_ = m.max(1, keepdim=True).values
    return (M_.squeeze(1) + torch.log2((s * torch.exp2(m - M_)).sum(1))) * math.log(2.0)


@pytest.mark.parametrize("K", [256, 512])
@pytest.mark.parametrize("V", [128, 300, 1000, 1100, 2048, 4233, 5538])
def test_lse_partials(V, K):
    """gemm_lse_partials (EPI_LSE epilogue) for M in {1, 37, 129, 300, 4000}, with and without bias.  V covers 128-column
    tiles (V < 1024 and V % 256 != 0: halves of 64 columns; 300 leaves the last tile's second half empty, 1000 half-filled)
    and 256-column tiles (1100: the last tile's second half empty, 4233 / 5538: partly filled); K = 512 with M > 128 runs
    CTA pairs (M = 300: an odd number of 128-row tiles, the peer CTA of the last pair has no rows; M = 129: a last tile
    of one row).

    Gate.  The logits are exact before + bias (_grid_operands); the epilogue adds the bias (1 rounding), multiplies by the
    fp32 constant log2 e (1 rounding of the constant, 1 of the product), takes ex2.approx (2^-22 relative) and sums at
    most 128 terms <= 1 in fp32 (<= 127 * 2^-24 relative).  Per half: |max - ref| <= 3 * 2^-24 |max| < 2^-22 |max|; each
    exponent argument carries 3 * 2^-24 of |v| and of |max| in log2 units, i.e. < 2^-21 (|max| + 1) relative on the sum,
    so the sum is within 2^-22 + 2^-17 + 2^-21 (|max| + 1) relative.  The row's log-sum-exp recombined in fp64: the
    error of the max cancels against the sum's, what is left is the per-term error (3 * 2^-24 |v| natural-log units),
    ex2.approx and the fp32 sum: |lse - ref| <= 2^-17 + 2^-21 (1 + |v|max)."""
    g = torch.Generator().manual_seed(V * 10 + K)
    bn = 256 if (V % 256 == 0 or V >= 1024) else 128
    P = lse_parts(V, K)
    assert P == 2 * ((V + bn - 1) // bn)
    worst_lse = worst_m = worst_s = 0.0
    for M in (1, 37, 129, 300, 4000):
        for with_bias in (False, True):
            a, w = _grid_operands(M, V, K, g)
            bias = (torch.randn(V, generator=g) * 2).to(_dev()) if with_bias else None
            sentinel = 777.0
            part = torch.full((M * P + 64, 2), sentinel, device=_dev())
            gemm_lse_partials(a, w, bias, part)
            torch.cuda.synchronize()
            # entries past the M x lse_parts block are never written
            assert (part[M * P:] == sentinel).all(), (M, with_bias)
            got = part[:M * P].view(M, P, 2).double().cpu()
            ref = a.double() @ w.double().T
            if bias is not None:
                ref = ref + bias.double()
            ref = ref.cpu()
            rm, rs = _part_ref(ref, V, bn)
            empty = torch.isinf(rm[0])
            # halves with no valid column: exactly (-inf, 0)
            assert (got[:, empty, 0] == -math.inf).all() and (got[:, empty, 1] == 0).all(), (M, with_bias)
            gm, gs = got[:, ~empty, 0], got[:, ~empty, 1]
            em = (gm - rm[:, ~empty]).abs() / rm[:, ~empty].abs().clamp(min=1.0)
            es = (gs - rs[:, ~empty]).abs() / rs[:, ~empty]
            assert (em <= 2 ** -22).all(), (M, with_bias, em.max().item())
            gate_s = 2 ** -22 + 2 ** -17 + 2 ** -21 * (rm[:, ~empty].abs() + 1)
            assert (es <= gate_s).all(), (M, with_bias, es.max().item())
            lse = _recombine(got[..., 0], got[..., 1])
            ref_lse = torch.logsumexp(ref, 1)
            e = (lse - ref_lse).abs()
            gate = 2 ** -17 + 2 ** -21 * (1 + ref.abs().max(1).values)
            assert (e <= gate).all(), (M, with_bias, e.max().item(), gate.min().item())
            worst_lse, worst_m, worst_s = max(worst_lse, e.max().item()), max(worst_m, em.max().item()), max(worst_s, es.max().item())
    print("lse partials V=%d K=%d: max |lse - ref| %.3g (gate >= %.3g), max rel err of max %.3g (gate %.3g), of sum %.3g "
          "(gate >= %.3g)" % (V, K, worst_lse, 2 ** -17 + 2 ** -21, worst_m, 2 ** -22, worst_s, 2 ** -22 + 2 ** -17 + 2 ** -21))


# ---------------------------------------------------------------------------------------------------- 2. target log-prob
@pytest.mark.parametrize("V,K,lda", [(300, 256, 256), (4233, 256, 320), (5538, 512, 512), (1100, 512, 576)])
def test_lse_target_logprob(V, K, lda):
    """lse_target_logprob against fp64 log_softmax(a w^T + bias)[src, target]: targets 0, V-1, the source row's argmax and
    random ones; -1 and V give exactly 0.  A non-identity row_map with repeated source rows (prefix sharing: several
    decoder positions read the same state row), and A rows with a pitch larger than K.

    Gate.  The target logit is a 1 x K fp32 FMA chain of bf16 products: exact on the grid operands, then + bias (1
    rounding); the log-sum-exp has the error bound of test_lse_partials plus the kernel's own merge (ex2.approx of each
    part, 2^-22 relative; fp32 sum of <= 44 parts, 43 * 2^-24; log2f, 2^-23): |err| <= 2^-16 + 2^-21 (1 + |v|max).
    Cross-check: for the argmax target the value equals lse_topk's top-1 of the same logits (EPI_F32 GEMM, the same
    single rounding of + bias) within the sum of both kernels' bounds, 2^-15 + 2^-20 (1 + |v|max)."""
    import ops
    g = torch.Generator().manual_seed(V + K + lda)
    S = 300                      # decoder state rows (unique prefixes)
    a, w = _grid_operands(S, V, K, g, lda=lda)
    bias = (torch.randn(V, generator=g) * 2).to(_dev())
    P = lse_parts(V, K)
    part = torch.empty(S * P, 2, device=_dev())
    gemm_lse_partials(a, w, bias, part)
    ref = (a[:, :K].double() @ w.double().T + bias.double()).cpu()
    ref_lp = torch.log_softmax(ref, -1)
    amax = ref.argmax(1)
    # scored positions: every state row several times (row_map repeats), with the edge targets mixed in
    R = 4 * S + 5
    row_map = torch.cat([torch.arange(S), torch.randint(0, S, (R - S,), generator=g)]).to(torch.int32)
    row_map = row_map[torch.randperm(R, generator=g)]
    tg = torch.randint(0, V, (R,), generator=g)
    kinds = torch.arange(R) % 6
    tg[kinds == 0] = 0
    tg[kinds == 1] = V - 1
    tg[kinds == 2] = amax[row_map.long()][kinds == 2]
    tg[kinds == 3] = -1
    tg[kinds == 4] = V
    tg = tg.to(torch.int32)
    out = lse_target_logprob(part, P, a, w, bias, tg.to(_dev()), row_map.to(_dev()), V).cpu().double()
    pad = (tg < 0) | (tg >= V)
    assert (out[pad] == 0).all(), "targets outside [0, V) must give exactly 0"
    src, t = row_map.long()[~pad], tg.long()[~pad]
    want = ref_lp[src, t]
    e = (out[~pad] - want).abs()
    gate = 2 ** -16 + 2 ** -21 * (1 + ref.abs().max(1).values[src])
    print("lse target V=%d K=%d lda=%d: max err %.3g (gate >= %.3g)" % (V, K, lda, e.max().item(), gate.min().item()))
    assert (e <= gate).all(), (e.max().item(), int(e.argmax()))
    # identity row_map (null) on the first S rows
    tg0 = amax.to(torch.int32)
    out0 = lse_target_logprob(part, P, a, w, bias, tg0.to(_dev()), None, V).cpu().double()
    assert ((out0 - ref_lp[torch.arange(S), amax]).abs() <= 2 ** -16 + 2 ** -21 * (1 + ref.abs().max(1).values)).all()
    # the same top-1 through the full-logits path
    ldl = (V + 7) // 8 * 8
    logits = torch.zeros(S, ldl, device=_dev())
    ops.gemm(a[:, :K], w, bias, ops.EPI_F32, 1.0, out=logits)
    tv, ti = ops.lse_topk(logits, V, 1, blank_id=0, blank_penalty=0.0)
    assert torch.equal(ti[:, 0].cpu().long(), amax)
    x = (tv[:, 0].cpu().double() - out0).abs()
    print("lse target vs lse_topk top-1: max diff %.3g (gate >= %.3g)" % (x.max().item(), 2 ** -15 + 2 ** -20))
    assert (x <= 2 ** -15 + 2 ** -20 * (1 + ref.abs().max(1).values)).all(), x.max().item()


# ---------------------------------------------------------------------------------------------------- 3. embedding
@pytest.mark.parametrize("d", [256, 512, 1280])
def test_embed_tokens(d):
    """x[r] = fmaf(emb[tok], xscale, pe[pos]) rounds once, so it equals the fp64 value of e * xscale + p rounded to fp32:
    the product of two fp32 numbers is exact in fp64, and the fp64 sum is rounded a second time only when it is inexact
    and lands on an fp32 rounding midpoint (double rounding) - then 1 ulp, which is allowed and counted.  Tokens include
    V - 1 and positions max_len - 1; xscale sqrt(d) (wenet) and 1 (Whisper's learnable PE)."""
    g = torch.Generator().manual_seed(d)
    V, max_len, R = 1000, 448, 777
    emb = torch.randn(V, d, generator=g)
    pe = torch.randn(max_len, d, generator=g)
    tok = torch.randint(0, V, (R,), generator=g, dtype=torch.int32)
    pos = torch.randint(0, max_len, (R,), generator=g, dtype=torch.int32)
    tok[:3] = V - 1
    pos[1:4] = max_len - 1
    pos[5] = 0
    # (device copies held in locals: a temporary's memory could be reused before the kernel runs)
    tok_d, pos_d, emb_d, pe_d = tok.to(_dev()), pos.to(_dev()), emb.to(_dev()), pe.to(_dev())
    for xscale in (float(np.float32(math.sqrt(d))), 1.0):
        x = torch.full((R, d), float("nan"), device=_dev())
        check(_lib.load().wb_op_embed_tokens(ptr(tok_d), ptr(pos_d), R, d, ptr(emb_d), ptr(pe_d), xscale, ptr(x), cur_stream()),
              "wb_op_embed_tokens")
        got = x.cpu().numpy()
        ref = (emb[tok.long()].double() * xscale + pe[pos.long()].double()).float().numpy()
        ulp = np.spacing(np.abs(ref))
        off = np.abs(got.astype(np.float64) - ref.astype(np.float64))
        n_off = int((off > 0).sum())
        print("embed d=%d xscale=%g: %d of %d elements differ from the once-rounded fp64 value (max %.3g ulp)" % (
            d, xscale, n_off, got.size, float((off / ulp).max())))
        assert np.isfinite(got).all()
        assert (off <= ulp).all()
        assert n_off <= got.size // 10000, n_off   # double rounding is rare; anything systematic is a bug


# ---------------------------------------------------------------------------------------------------- 4. rescore combine
def _rescore_ref(l2r, r2l, row0, lens, utt0, nh, ctc, cw, rw):
    """oracle/wenet_oracle.py attention_rescoring (search.py:421-452) in numpy float32, same addition order: token
    log-probs added one by one from 0, then <eos>; r2l reads position len-1-j for token j; mix; + fp32(ctc * cw)."""
    f = np.float32
    scores = np.zeros(len(lens), np.float32)
    best = []
    for b in range(len(nh)):
        bs, bi = -np.inf, 0
        for i in range(nh[b]):
            hy = utt0[b] + i
            r0, n = row0[hy], lens[hy]
            s = f(0.0)
            for j in range(n):
                s = f(s + l2r[r0 + j])
            s = f(s + l2r[r0 + n])
            if rw > 0 and r2l is not None:
                rs = f(0.0)
                for j in range(n):
                    rs = f(rs + r2l[r0 + n - 1 - j])
                rs = f(rs + r2l[r0 + n])
                s = f(f(s * f(1 - rw)) + f(rs * f(rw)))
            s = f(s + f(ctc[hy] * cw))
            scores[hy] = s
            if s > bs:
                bs, bi = s, i
        best.append(bi)
    return scores, np.array(best)


@pytest.mark.parametrize("rw,with_r2l", [(0.0, True), (0.3, True), (0.3, False)])
def test_rescore_combine(rw, with_r2l):
    """rescore_combine against the float32 restatement: utterances with 0, 1, 10, 64, 65 and 130 hypotheses (beyond 64 the
    kernel carries the running best through hyp_score in global memory), zero-length hypotheses, exact ties (the first
    maximum wins, also across the 64-hypothesis rounds), best index exact.  ctc_weight 0.5 is exact in fp32 and fp64.
    reverse_weight 0: bit-identical scores.  reverse_weight 0.3: fp32(1 - 0.3) == 1 - fp32(0.3), but the compiler may
    contract score * (1 - rw) + r_score * rw into one FMA (one rounding fewer): both terms have the same sign, so the
    mix moves by at most 1 ulp, and rounding the final + ctc term adds at most 1 more -> within 2 ulp.  This is a hard
    bound, and it is reached: on these inputs some scores differ by exactly 2 ulp."""
    g = np.random.default_rng(int(rw * 10) + with_r2l)
    nh = [0, 1, 10, 64, 65, 130, 3]
    utt0 = np.concatenate([[0], np.cumsum(nh)[:-1]]).astype(np.int32)
    H = int(sum(nh))
    lens = g.integers(0, 40, H).astype(np.int32)
    lens[::7] = 0                                       # hypotheses without tokens (only <eos> is scored)
    # exact ties (utterance, first, copy): within a round, and from round 0 into round 1 of the > 64 utterances
    ties = [(2, 3, 7), (4, 5, 64), (5, 20, 90)]
    for b, i, j in ties:
        lens[utt0[b] + j] = lens[utt0[b] + i]
    row0 = np.concatenate([[0], np.cumsum(lens + 1)[:-1]]).astype(np.int32)
    total = int(lens.sum()) + H
    l2r = (-g.exponential(1.5, total)).astype(np.float32)
    r2l = (-g.exponential(1.5, total)).astype(np.float32)
    ctc = -g.exponential(10.0, H)
    for b, i, j in ties:   # the first of the pair becomes a clear winner of its utterance, the second an exact copy
        hi, hj, n = utt0[b] + i, utt0[b] + j, lens[utt0[b] + i] + 1
        l2r[row0[hi]:row0[hi] + n] *= np.float32(0.001)
        r2l[row0[hi]:row0[hi] + n] *= np.float32(0.001)
        ctc[hi] = -0.001
        l2r[row0[hj]:row0[hj] + n] = l2r[row0[hi]:row0[hi] + n]
        r2l[row0[hj]:row0[hj] + n] = r2l[row0[hi]:row0[hi] + n]
        ctc[hj] = ctc[hi]

    cw = 0.5
    want, want_best = _rescore_ref(l2r, r2l if with_r2l else None, row0, lens, utt0, nh, ctc, cw, rw)
    batch = len(nh)
    hyp_score = torch.full((H,), float("nan"), device=_dev())
    best = torch.full((batch,), -7, dtype=torch.int32, device=_dev())
    dv = [torch.from_numpy(np.ascontiguousarray(x)).to(_dev()) for x in (l2r, r2l, row0, lens, utt0, np.array(nh, np.int32), ctc)]
    check(_lib.load().wb_op_rescore_combine(ptr(dv[0]), ptr(dv[1]) if with_r2l else None, ptr(dv[2]), ptr(dv[3]), ptr(dv[4]),
                                            ptr(dv[5]), batch, ptr(dv[6]), cw, rw, ptr(hyp_score), ptr(best), cur_stream()),
          "wb_op_rescore_combine")
    got = hyp_score.cpu().numpy()
    got_best = best.cpu().numpy()
    # the constructed ties are real ties, and the restatement picks the first of each
    for b, i, j in ties:
        assert want[utt0[b] + i] == want[utt0[b] + j] and want_best[b] == i, (b, want_best[b])
    assert list(got_best) == list(want_best), (list(got_best), list(want_best))
    ulps = np.abs(got.astype(np.float64) - want) / np.spacing(np.abs(want))
    print("rescore combine rw=%g r2l=%s: max %.3g ulp (gate %s)" % (rw, with_r2l, ulps.max(), "0" if rw == 0 or not with_r2l else "2"))
    if rw == 0 or not with_r2l:
        assert np.array_equal(got, want), ulps.max()
    else:
        assert (ulps <= 2).all(), ulps.max()


# ---------------------------------------------------------------------------------------------------- 5. attention modes
def _pieces(T_list, splits):
    """k_start / k_len of the split-key items, built as attention decoding builds them (attdecode.cu): pieces of a whole
    number of 64-key tiles, the last ones empty when T < splits x piece"""
    ks, kl = [], []
    base = 0
    for T in T_list:
        piece = ((max(T, 1) + splits - 1) // splits + 63) // 64 * 64
        for s in range(splits):
            k0, k1 = min(s * piece, T), min((s + 1) * piece, T)
            ks.append(base + k0)
            kl.append(k1 - k0)
        base += T
    return ks, kl


@pytest.mark.parametrize("q_len", [1, 4, 10, 32, 128, 200])
@pytest.mark.parametrize("splits", [1, 2, 4, 8])
def test_attention_split_key(splits, q_len):
    """Cross attention of attention decoding as key pieces (flash-decoding) + merge: utterances of T = 1, 63, 64, 65, 700
    encoder frames (empty pieces where T < splits x piece) and one of T = 0, whose rows must come out zero.  K / V in one
    [T, 2d] buffer at columns 0 / d, 4 heads.  Against fp64 and against the unsplit launch, both within the gate of
    test_attention (_attn_gate).  q_len 200 > 128: a query block of several CTAs per piece."""
    g = torch.Generator().manual_seed(splits * 1000 + q_len)
    H, d = 4, 256
    T_list = [1, 63, 0, 64, 65, 700]
    B = len(T_list)
    q = torch.randn(B * q_len, d, generator=g).to(torch.bfloat16)
    kv = torch.randn(sum(T_list), 2 * d, generator=g).to(torch.bfloat16)
    q_start = [b * q_len for b in range(B)]
    k_start = list(np.concatenate([[0], np.cumsum(T_list)[:-1]]).astype(int))
    ref = _attn_ref64(q, kv, kv, None, q_start, [q_len] * B, k_start, T_list, H, 0, -1, 0.125, 0, 0, d)
    ks, kl = _pieces(T_list, splits)
    qd, kvd = q.to(_dev()), kv.to(_dev())
    out = torch.full((B * q_len, d), 3.0, dtype=torch.bfloat16, device=_dev())
    attention_ex(qd, kvd, kvd, _ti([s for s in q_start for _ in range(splits)]), _ti([q_len] * (B * splits)), _ti(ks), _ti(kl),
                 H, q_len, out, k_col0=0, v_col0=d, splits=splits, split_key=True)
    plain = torch.full((B * q_len, d), 3.0, dtype=torch.bfloat16, device=_dev())
    attention_ex(qd, kvd, kvd, _ti(q_start), _ti([q_len] * B), _ti(k_start), _ti(T_list), H, q_len, plain, k_col0=0, v_col0=d)
    torch.cuda.synchronize()
    z = T_list.index(0)
    assert (out[z * q_len:(z + 1) * q_len] == 0).all() and (plain[z * q_len:(z + 1) * q_len] == 0).all()
    vmax = float(kv[:, d:].float().abs().max())
    _attn_gate(out.cpu(), ref, vmax, "split-key S=%d q=%d vs fp64" % (splits, q_len))
    _attn_gate(out.cpu(), plain.cpu().double(), vmax, "split-key S=%d q=%d vs unsplit" % (splits, q_len))


@pytest.mark.parametrize("chunk,left", [(16, 3), (1, -1), (0, -1), (16, -1)])
def test_attention_prescaled_bias(chunk, left):
    """Pre-scaled key bias (kbias_scaled = 1, the encoder's form: relpos_kprep writes c * scale * log2 e and the kernel
    fetches it by cp.async): the unscaled path multiplies each bias by the same fp32 factor scale * log2 e inside the
    kernel, so with kbias_scaled = kbias * fp32(scale * log2 e) computed in fp32 the two launches run identical
    arithmetic and must agree BIT FOR BIT; both against fp64 within the gate of test_attention.  Chunk masks 16/3,
    causal, full and 16/-1; 4 heads; sequences of 200, 77, 333, 128, 129, 1, 64 rows."""
    g = torch.Generator().manual_seed(chunk * 10 + left + 5)
    H, d = 4, 256
    lens = [200, 77, 333, 128, 129, 1, 64]
    starts = list(np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(int))
    M = sum(lens)
    qkv = torch.randn(M, 3 * d, generator=g).to(torch.bfloat16)
    kbias = torch.randn(M, H, generator=g) * 4
    scale = 0.125
    ref = _attn_ref64(qkv, qkv, qkv, kbias, starts, lens, starts, lens, H, chunk, left, scale, 0, d, 2 * d)
    f = float(np.float32(np.float32(scale) * np.float32(LOG2E)))
    kbd = kbias.to(_dev())
    kbs = kbd * f
    qd = qkv.to(_dev())
    outs = []
    for kb, flag in ((kbd, 0), (kbs, 1)):
        o = torch.zeros(M, d, dtype=torch.bfloat16, device=_dev())
        attention_ex(qd, qd, qd, _ti(starts), _ti(lens), _ti(starts), _ti(lens), H, max(lens), o, kbias=kb, chunk_size=chunk,
                     num_left_chunks=left, scale=scale, q_col0=0, k_col0=d, v_col0=2 * d, kbias_scaled=flag)
        outs.append(o)
    torch.cuda.synchronize()
    vmax = float(qkv[:, 2 * d:].float().abs().max())
    _attn_gate(outs[1].cpu(), ref, vmax, "pre-scaled bias chunk=%d left=%d vs fp64" % (chunk, left))
    _attn_gate(outs[0].cpu(), ref, vmax, "in-kernel scaled bias chunk=%d left=%d vs fp64" % (chunk, left))
    assert torch.equal(outs[0], outs[1]), float((outs[0].float() - outs[1].float()).abs().max())


@pytest.mark.parametrize("heads", [4, 8, 20])
def test_attention_fused_buffers(heads):
    """Column offsets: the decoder self attention reads Q / K / V at columns 0 / d / 2d of one [R, 3d] buffer (causal),
    the cross attention K / V at 0 / d of one [T, 2d] buffer; the output lands at out_col0 = 64 of a buffer with pitch
    d + 128 whose other columns must keep their sentinel.  Against fp64 within the gate of test_attention."""
    g = torch.Generator().manual_seed(heads)
    d = heads * 64
    hyp = [12, 31, 1, 140, 7]                 # self attention: rows of each hypothesis
    hs = list(np.concatenate([[0], np.cumsum(hyp)[:-1]]).astype(int))
    R = sum(hyp)
    qkv = torch.randn(R, 3 * d, generator=g).to(torch.bfloat16)
    ldo, col0 = d + 128, 64
    sentinel = -5.0
    out = torch.full((R, ldo), sentinel, dtype=torch.bfloat16, device=_dev())
    qd = qkv.to(_dev())
    attention_ex(qd, qd, qd, _ti(hs), _ti(hyp), _ti(hs), _ti(hyp), heads, max(hyp), out, chunk_size=1, num_left_chunks=-1,
                 q_col0=0, k_col0=d, v_col0=2 * d, out_col0=col0)
    # cross attention: 3 utterances, q rows per utterance, keys of the utterance's frames
    ql, T = [10, 4, 130], [300, 65, 129]
    qs = list(np.concatenate([[0], np.cumsum(ql)[:-1]]).astype(int))
    ts = list(np.concatenate([[0], np.cumsum(T)[:-1]]).astype(int))
    q = torch.randn(sum(ql), d, generator=g).to(torch.bfloat16)
    kv = torch.randn(sum(T), 2 * d, generator=g).to(torch.bfloat16)
    out2 = torch.full((sum(ql), ldo), sentinel, dtype=torch.bfloat16, device=_dev())
    kvd = kv.to(_dev())
    attention_ex(q.to(_dev()), kvd, kvd, _ti(qs), _ti(ql), _ti(ts), _ti(T), heads, max(ql), out2, k_col0=0, v_col0=d,
                 out_col0=col0)
    torch.cuda.synchronize()
    for o in (out, out2):
        assert (o[:, :col0] == sentinel).all() and (o[:, col0 + d:] == sentinel).all(), "write outside the output block"
    ref = _attn_ref64(qkv, qkv, qkv, None, hs, hyp, hs, hyp, heads, 1, -1, 0.125, 0, d, 2 * d)
    _attn_gate(out[:, col0:col0 + d].cpu(), ref, float(qkv[:, 2 * d:].float().abs().max()), "fused qkv heads=%d" % heads)
    ref2 = _attn_ref64(q, kv, kv, None, qs, ql, ts, T, heads, 0, -1, 0.125, 0, 0, d)
    _attn_gate(out2[:, col0:col0 + d].cpu(), ref2, float(kv[:, d:].float().abs().max()), "fused kv heads=%d" % heads)


# ---------------------------------------------------------------------------------------------------- 6. self-attn step
@pytest.mark.parametrize("pos", [0, 1, 31, 32, 200])
@pytest.mark.parametrize("B,N,H", [(1, 1, 4), (3, 4, 4), (2, 10, 8), (1, 32, 4)])
def test_dec_self_attn_step(B, N, H, pos):
    """dec_self_attn_step_kernel: R = B x N decoder rows (utterance-major), cache slots of positions < pos filled with
    distinct random K / V as earlier steps would have left them, a random ancestry table anc[r][j] within r's utterance.
    ctx against fp64 softmax attention over the gathered history; the kernel's softmax is fp32 (__expf, 2^-21 relative;
    fp32 sums, ~1e-6 relative) and its output is rounded to bf16 (2^-9 relative): 2^-8 |ref| + 2^-9 max|v| holds with a
    factor-2 margin.  The cache slot (pos, r) must equal row r's K / V columns of qkv exactly, every other slot unchanged."""
    g = torch.Generator().manual_seed(B * 1000 + N * 10 + pos)
    R, d = B * N, H * 64
    L = pos + 2
    qkv = torch.randn(R, 3 * d, generator=g).to(torch.bfloat16)
    kv0 = torch.randn(L, R, 2 * d, generator=g).to(torch.bfloat16)
    anc = torch.zeros(R, L, dtype=torch.int32)
    for r in range(R):
        b = r // N
        anc[r] = b * N + torch.randint(0, N, (L,), generator=g, dtype=torch.int32)
    kv = kv0.to(_dev())
    ctx = torch.full((R, d), float("nan"), dtype=torch.bfloat16, device=_dev())
    qkv_d, anc_d = qkv.to(_dev()), anc.to(_dev())
    check(_lib.load().wb_op_dec_self_attn_step(ptr(qkv_d), ptr(kv), ptr(anc_d), L, pos, R, H, d, 0.125, ptr(ctx), cur_stream()),
          "wb_op_dec_self_attn_step")
    torch.cuda.synchronize()
    kv1 = kv.cpu()
    assert torch.equal(kv1[pos], qkv[:, d:]), "cache slot (pos, r) must hold row r's K / V"
    keep = torch.ones(L, dtype=torch.bool)
    keep[pos] = False
    assert torch.equal(kv1[keep], kv0[keep]), "a cache slot other than (pos, r) changed"
    ref = torch.zeros(R, d, dtype=torch.float64)
    vmax = 0.0
    for r in range(R):
        slots = anc[r, :pos].long()
        Kh = torch.cat([kv0[torch.arange(pos), slots, :d], qkv[r:r + 1, d:2 * d]]).double()
        Vh = torch.cat([kv0[torch.arange(pos), slots, d:], qkv[r:r + 1, 2 * d:]]).double()
        vmax = max(vmax, float(Vh.abs().max()))
        for h in range(H):
            s = (Kh[:, h * 64:(h + 1) * 64] @ qkv[r, h * 64:(h + 1) * 64].double()) * 0.125
            ref[r, h * 64:(h + 1) * 64] = torch.softmax(s, 0) @ Vh[:, h * 64:(h + 1) * 64]
    diff = (ctx.cpu().double() - ref).abs()
    bound = 2 ** -8 * ref.abs() + 2 ** -9 * vmax
    print("self-attn step B=%d N=%d H=%d pos=%d: max err %.3g (gate at that element %.3g)" % (
        B, N, H, pos, diff.max().item(), bound.flatten()[diff.argmax()].item()))
    assert not (diff > bound).any(), diff.max().item()
