"""Operator-level parity (GPU): every hand-written kernel against a plain fp32 reference of the same
op evaluated on the SAME bf16-rounded operands (so the tolerance only has to cover fp32 summation
order and the final bf16 rounding of bf16 outputs), and the integer/search kernels bit-exactly
against the CPU oracle."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import wenet_oracle as O


def _dev():
    return torch.device("cuda:0")


def _rb(t):
    return t.to(torch.bfloat16)


# bf16 output rounding: relative 2^-9; fp32 accumulate order: ~1e-6 relative of the sum of |terms|
def _close(got, ref, rtol, atol):
    diff = (got.float() - ref.float()).abs()
    tol = atol + rtol * ref.float().abs()
    bad = (diff > tol)
    assert not bad.any(), "max diff %g at %s (ref %g)" % (
        diff.max().item(), tuple(torch.nonzero(bad)[0].tolist()), ref.float().flatten()[0].item())


@pytest.mark.parametrize("M,N,K", [(300, 256, 256), (1000, 768, 256), (130, 2048, 256), (257, 256, 2048),
                                   (128, 128, 64), (77, 384, 1152), (4000, 256, 2304)])
@pytest.mark.parametrize("epi", [0, 1, 2, 3, 5])
def test_gemm(M, N, K, epi):
    import ops
    g = torch.Generator(device="cpu").manual_seed(M * 7 + N + K + epi)
    a = _rb(torch.randn(M, K, generator=g)).to(_dev())
    b = _rb(torch.randn(N, K, generator=g) / math.sqrt(K)).to(_dev())
    bias = torch.randn(N, generator=g).to(_dev())
    ref = a.float() @ b.float().T + bias
    alpha = 0.5 if epi == 3 else (1.7 if epi == 5 else 1.0)
    if epi == 1:
        ref = torch.nn.functional.silu(ref)
    elif epi == 2:
        ref = torch.relu(ref)
    if epi == 3:
        c0 = torch.randn(M, N, generator=g).to(_dev())
        out = ops.gemm(a, b, bias, epi, alpha, out=c0.clone())
        _close(out, c0 + alpha * ref, 1e-5, 2e-4)
    elif epi == 5:
        out = ops.gemm(a, b, bias, epi, alpha)
        _close(out, alpha * ref, 1e-5, 2e-4)
    else:
        out = ops.gemm(a, b, bias, epi, alpha)
        assert out.dtype == torch.bfloat16
        _close(out, ref, 2 ** -8, 2e-4)


@pytest.mark.parametrize("M,N,K,epi", [(47872, 2048, 256, 1), (5003, 2048, 256, 1), (2048, 512, 128, 1), (6000, 256, 192, 9),
                                       (2100, 768, 64, 1)])
def test_gemm_sixteen_epilogue_warps(M, N, K, epi):
    """gemm_act16.cu (weight-stationary K <= 256, SiLU / GELU, sixteen epilogue warps alternating tiles, SWIZZLE_64B output
    staging): the shapes gemm_bf16 routes to it (M >= 2048, N % 256 == 0), incl. ragged last row tiles, one tile per CTA
    and several weight panels per CTA - against torch, and bit for bit against the eight-warp kernel (WB_GEMM_ACT16=0 is
    read once per process, so the reference here is the same epilogue arithmetic through a narrower call: M < 2048 rows
    at a time)."""
    import ops
    g = torch.Generator(device="cpu").manual_seed(M + N + K)
    a = _rb(torch.randn(M, K, generator=g)).to(_dev())
    b = _rb(torch.randn(N, K, generator=g) / math.sqrt(K)).to(_dev())
    bias = torch.randn(N, generator=g).to(_dev())
    ref = a.float() @ b.float().T + bias
    ref = torch.nn.functional.silu(ref) if epi == 1 else torch.nn.functional.gelu(ref)
    out = ops.gemm(a, b, bias, epi, 1.0)
    torch.cuda.synchronize()
    assert out.dtype == torch.bfloat16 and out.shape == (M, N)
    _close(out, ref, 2 ** -8, 2e-4)
    # the same rows through the eight-warp kernel (slices below the routing threshold)
    for r0 in range(0, M, 1920):
        r1 = min(M, r0 + 1920)
        part = ops.gemm(a[r0:r1].contiguous(), b, bias, epi, 1.0)
        assert torch.equal(part, out[r0:r1]), (r0, float((part.float() - out[r0:r1].float()).abs().max()))


@pytest.mark.parametrize("M,K", [(300, 256), (47872, 256), (257, 2048), (5000, 2048), (67, 256), (128, 2048)])
def test_gemm_resid_layernorm(M, K):
    """Residual-update GEMM with the next module's LayerNorm fused into its epilogue (N = d = 256): x in place and
    the bf16 normalised rows against x + alpha (a b^T + bias) and torch's layer_norm of that."""
    import ops
    g = torch.Generator(device="cpu").manual_seed(M + K)
    N = 256
    a = _rb(torch.randn(M, K, generator=g)).to(_dev())
    b = _rb(torch.randn(N, K, generator=g) / math.sqrt(K)).to(_dev())
    bias = torch.randn(N, generator=g).to(_dev())
    gamma = (1.0 + 0.2 * torch.randn(N, generator=g)).to(_dev())
    beta = (0.3 * torch.randn(N, generator=g)).to(_dev())
    # rows with a large common offset exercise the variance formula (mean >> spread)
    x0 = (torch.randn(M, N, generator=g) * 2.0 + 3.0 * torch.randn(M, 1, generator=g)).to(_dev())
    alpha = 0.5
    ref_x = x0 + alpha * (a.float() @ b.float().T + bias)
    ref_ln = torch.nn.functional.layer_norm(ref_x, (N,), gamma, beta, 1e-5)
    x = x0.clone()
    out = ops.gemm_resid_ln(a, b, bias, x, gamma, beta, alpha=alpha, eps=1e-5)
    torch.cuda.synchronize()
    _close(x, ref_x, 1e-5, 2e-4)
    assert out.dtype == torch.bfloat16
    _close(out, ref_ln, 2 ** -8, 1e-3)
    # and the same rows as the unfused pair of kernels produces them (bf16 rounding of nearly equal fp32 values)
    x2 = ops.gemm(a, b, bias, 3, alpha, out=x0.clone())
    ln2 = ops.layernorm(x2, gamma, beta, 1e-5)[0]
    assert ((out.float() - ln2.float()).abs() <= 2 ** -7 * ln2.float().abs() + 1e-3).all()


@pytest.mark.parametrize("M,K", [(300, 2048), (47872, 2048), (67, 2048), (1000, 256)])
def test_gemm_resid_two_layernorms(M, K):
    """Layer boundary: x = norm_final(x + alpha (a b^T + bias)) stored in fp32 and the next layer's norm_ff_macaron of
    it in bf16, both inside the GEMM epilogue."""
    import ops
    g = torch.Generator(device="cpu").manual_seed(M * 3 + K)
    N = 256
    a = _rb(torch.randn(M, K, generator=g)).to(_dev())
    b = _rb(torch.randn(N, K, generator=g) / math.sqrt(K)).to(_dev())
    bias = torch.randn(N, generator=g).to(_dev())
    g1 = (1.0 + 0.2 * torch.randn(N, generator=g)).to(_dev())
    b1 = (0.3 * torch.randn(N, generator=g)).to(_dev())
    g2 = (1.0 + 0.2 * torch.randn(N, generator=g)).to(_dev())
    b2 = (0.3 * torch.randn(N, generator=g)).to(_dev())
    x0 = (torch.randn(M, N, generator=g) * 2.0 + 3.0 * torch.randn(M, 1, generator=g)).to(_dev())
    ref_y = x0 + 0.5 * (a.float() @ b.float().T + bias)
    ref_x = torch.nn.functional.layer_norm(ref_y, (N,), g1, b1, 1e-5)
    ref_z = torch.nn.functional.layer_norm(ref_x, (N,), g2, b2, 1e-5)
    x = x0.clone()
    out = ops.gemm_resid_ln(a, b, bias, x, g2, b2, alpha=0.5, eps=1e-5, gamma1=g1, beta1=b1)
    torch.cuda.synchronize()
    _close(x, ref_x, 1e-5, 3e-4)
    _close(out, ref_z, 2 ** -8, 1e-3)


def test_gemm_glu_and_tail():
    import ops
    g = torch.Generator().manual_seed(5)
    M, d, K = 500, 256, 256
    a = _rb(torch.randn(M, K, generator=g)).to(_dev())
    w = _rb(torch.randn(2 * d, K, generator=g) / 16).to(_dev())      # reference layout: [value rows | gate rows]
    bias = torch.randn(2 * d, generator=g).to(_dev())
    from wenet_b200.weights import interleave_glu
    wp, bp = interleave_glu(w, bias)
    out = ops.gemm(a, wp.contiguous(), bp.contiguous(), ops.EPI_GLU_BF16)
    y = a.float() @ w.float().T + bias
    ref = y[:, :d] * torch.sigmoid(y[:, d:])
    _close(out, ref, 2 ** -8, 2e-4)
    # ragged N (vocabulary-sized) fp32 output with padded leading dimension
    N = 4233
    b = _rb(torch.randn(N, K, generator=g) / 16).to(_dev())
    bb = torch.randn(N, generator=g).to(_dev())
    outf = torch.full((M, 4240), -7.0, device=_dev())
    ops.gemm(a, b, bb, ops.EPI_F32, 1.0, out=outf)
    _close(outf[:, :N], a.float() @ b.float().T + bb, 1e-5, 2e-4)
    # the TMA store clips at 16-byte granularity: columns [N, round_up(N, 4)) are zero-filled, the rest of
    # the padded leading dimension is untouched
    assert (outf[:, (N + 3) // 4 * 4:] == -7.0).all()


def test_gemm_split3_fp32_grade():
    """bf16x3: A=[hi|lo|hi], B=[hi|hi|lo] reproduces an fp32 GEMM to ~1e-5 relative."""
    import ops
    from wenet_b200.weights import split3_weight
    g = torch.Generator().manual_seed(11)
    M, N, K = 300, 256, 256
    x = torch.randn(M, K, generator=g).to(_dev())
    w = (torch.randn(N, K, generator=g) / 16).to(_dev())
    gam = torch.ones(K, device=_dev())
    bet = torch.zeros(K, device=_dev())
    a3, _ = ops.layernorm(x, gam, bet, split3=True)
    xn = torch.nn.functional.layer_norm(x, (K,))
    out = ops.gemm(a3, split3_weight(w), None, ops.EPI_F32)
    ref = xn @ w.T
    assert (out - ref).abs().max().item() < 2e-4


@pytest.mark.parametrize("d", [128, 256, 512])
def test_layernorm(d):
    import ops
    g = torch.Generator().manual_seed(d)
    x = (torch.randn(777, d, generator=g) * 3 + 1).to(_dev())
    gam = torch.randn(d, generator=g).to(_dev())
    bet = torch.randn(d, generator=g).to(_dev())
    ob, of = ops.layernorm(x, gam, bet, want_f32=True)
    ref = torch.nn.functional.layer_norm(x, (d,), gam, bet, 1e-5)
    _close(of, ref, 1e-5, 1e-5)
    _close(ob, ref, 2 ** -8, 1e-5)


def _attn_ref(q, k, v, kbias, q_start, q_len, k_start, k_len, heads, chunk, left, scale, round_p=False):
    out = torch.zeros(q.shape[0], heads * 64)
    for b in range(len(q_start)):
        qs, ql, ks, kl = q_start[b], q_len[b], k_start[b], k_len[b]
        for h in range(heads):
            Q = q[qs:qs + ql, h * 64:(h + 1) * 64].float()
            K = k[ks:ks + kl, h * 64:(h + 1) * 64].float()
            V = v[ks:ks + kl, h * 64:(h + 1) * 64].float()
            S = Q @ K.T
            if kbias is not None:
                S = S + kbias[ks:ks + kl, h].unsqueeze(0)
            S = S * scale
            if chunk > 0:
                i = torch.arange(ql).unsqueeze(1)
                j = torch.arange(kl).unsqueeze(0)
                start = torch.zeros_like(i) if left < 0 else torch.clamp((i // chunk - left) * chunk, min=0)
                end = (i // chunk + 1) * chunk
                S = S.masked_fill(~((j >= start) & (j < end)), -float("inf"))
            mx = S.max(dim=-1, keepdim=True).values
            P = torch.exp(S - mx)
            if round_p:
                P = P.to(torch.bfloat16).float()
            out[qs:qs + ql, h * 64:(h + 1) * 64] = (P @ V) / P.sum(-1, keepdim=True)
    return out


@pytest.mark.parametrize("v_mode", [0, 1])
@pytest.mark.parametrize("case", ["self_full", "self_chunk", "causal", "cross"])
def test_attention(case, v_mode):
    import ops
    g = torch.Generator().manual_seed({"self_full": 11, "self_chunk": 12, "causal": 13, "cross": 14}[case])
    heads = 2
    if case == "cross":
        q_len, k_len = [37, 260, 5], [200, 333, 129]
    else:
        q_len = k_len = [200, 77, 333, 128, 129]
    q_start = [0]
    for n in q_len[:-1]:
        q_start.append(q_start[-1] + n)
    k_start = [0]
    for n in k_len[:-1]:
        k_start.append(k_start[-1] + n)
    Mq, Mk = sum(q_len), sum(k_len)
    q = _rb(torch.randn(Mq, heads * 64, generator=g))
    k = _rb(torch.randn(Mk, heads * 64, generator=g))
    v = _rb(torch.randn(Mk, heads * 64, generator=g))
    kbias = torch.randn(Mk, heads, generator=g) if case.startswith("self") else None
    chunk, left = {"self_full": (0, -1), "self_chunk": (16, 3), "causal": (1, -1), "cross": (0, -1)}[case]
    scale = 0.125
    ref = _attn_ref(q, k, v, kbias, q_start, q_len, k_start, k_len, heads, chunk, left, scale)
    ti = lambda x: torch.tensor(x, dtype=torch.int32, device=_dev())
    out = ops.attention(q.to(_dev()), k.to(_dev()), v.to(_dev()), ti(q_start), ti(q_len), ti(k_start), ti(k_len),
                        heads, kbias.to(_dev()) if kbias is not None else None, chunk, left, scale,
                        v_mode=v_mode, max_q_len=max(q_len))
    torch.cuda.synchronize()
    # exact fp32 softmax reference.  The kernel rounds the probabilities to bf16 (2^-9 relative each, relative to a
    # lazily updated running maximum, so the rounding pattern cannot be replayed on the host): the worst case is
    # 2^-8 max|v| per output, the typical error is an order of magnitude below that.
    diff = (out.cpu().float() - ref).abs()
    bound = 2 ** -7 * ref.abs() + 2 ** -8 * float(v.float().abs().max())
    assert not (diff > bound).any(), "max diff %g" % diff.max().item()
    assert diff.mean().item() < 1e-3, diff.mean().item()


def test_relpos_kprep():
    import ops
    g = torch.Generator().manual_seed(2)
    M, heads = 333, 4
    d = heads * 64
    k = _rb(torch.randn(M, 3 * d, generator=g))
    P = torch.randn(500, d, generator=g)
    pos = torch.randint(0, 500, (M,), generator=g, dtype=torch.int32)
    u = torch.randn(d, generator=g)
    v = torch.randn(d, generator=g)
    kp, kb = ops.relpos_kprep(k.to(_dev())[:, d:2 * d], P.to(_dev()), pos.to(_dev()), u.to(_dev()), v.to(_dev()), heads)
    kk = k[:, d:2 * d].float()
    pp = P[pos.long()]
    _close(kp.cpu(), kk + pp, 2 ** -8, 1e-6)
    ref_c = ((kk * u).view(M, heads, 64).sum(-1) + (pp * v).view(M, heads, 64).sum(-1))
    _close(kb.cpu(), ref_c, 1e-5, 1e-4)


@pytest.mark.parametrize("causal,ksize,norm", [(True, 8, 0), (True, 15, 0), (False, 15, 1), (False, 15, 0)])
def test_dwconv(causal, ksize, norm):
    import ops
    g = torch.Generator().manual_seed(ksize + norm)
    d = 256
    lens = [100, 33, 7, 64]
    starts = [0, 100, 133, 140]
    M = sum(lens)
    x = _rb(torch.randn(M, d, generator=g))
    w = torch.randn(d, ksize, generator=g) / 3
    b = torch.randn(d, generator=g)
    gam = torch.randn(d, generator=g)
    bet = torch.randn(d, generator=g)
    pad_vec = torch.randn(d, generator=g)
    pad_until = 100
    ti = lambda t: torch.tensor(t, dtype=torch.int32, device=_dev())
    out = ops.dwconv(x.to(_dev()), ti(starts), ti(lens), ti(starts), w.to(_dev()), b.to(_dev()), gam.to(_dev()),
                     bet.to(_dev()), ksize, causal, norm, pad_vec=pad_vec.to(_dev()), pad_until=pad_until)
    pv = pad_vec.to(torch.bfloat16).float()
    for s, n in zip(starts, lens):
        xi = x[s:s + n].float()
        if causal:
            xin = torch.cat([pv.unsqueeze(0).expand(ksize - 1, d), xi], 0)
        else:
            h = (ksize - 1) // 2
            right = torch.zeros(h, d)
            npad = min(h, pad_until - n)
            if npad > 0:
                right[:npad] = pv
            xin = torch.cat([torch.zeros(h, d), xi, right], 0)
        y = torch.nn.functional.conv1d(xin.T.unsqueeze(0), w.unsqueeze(1), b, groups=d)[0].T
        if norm == 0:
            y = torch.nn.functional.layer_norm(y, (d,), gam, bet, 1e-5)
        else:
            y = y * gam + bet
        ref = torch.nn.functional.silu(y)
        _close(out[s:s + n].cpu(), ref, 2 ** -8, 2e-4)


def _peaky_logits(T, V, g, blank_boost=12.0, spike=20.0, frac=0.15):
    x = torch.randn(T, V, generator=g)
    x[:, 0] += blank_boost
    n = int(T * frac)
    rows = torch.randperm(T, generator=g)[:n]
    cols = torch.randint(1, V, (n,), generator=g)
    x[rows, cols] += spike
    return x


def test_logsoftmax_topk_greedy_and_prefix_beam():
    import ops
    g = torch.Generator().manual_seed(777)
    V, beam = 4233, 10
    lens = [248, 100, 1, 77]
    starts = [0, 248, 348, 349]
    M = sum(lens)
    logits = torch.cat([_peaky_logits(n, V, g) for n in lens], 0)
    ld = 4240
    buf = torch.zeros(M, ld)
    buf[:, :V] = logits
    dbuf = buf.to(_dev())
    tv, ti = ops.logsoftmax_topk(dbuf, V, beam, blank_id=0, blank_penalty=0.0)
    ref_lp = logits.log_softmax(-1)
    got_lp = dbuf[:, :V].cpu()
    assert (got_lp - ref_lp).abs().max().item() < 2e-5
    # top-k of the kernel's own log-probs (identical input => identical order)
    rv, ri = got_lp.topk(beam, dim=-1)
    assert torch.equal(ti.cpu().long(), ri)
    assert torch.equal(tv.cpu(), rv)
    tI = lambda t: torch.tensor(t, dtype=torch.int32, device=_dev())
    toks, tl = ops.ctc_greedy_search(ti, tI(starts), tI(lens))
    # oracle on identical log-probs, padded layout
    T = max(lens)
    padded = torch.zeros(len(lens), T, V)
    for b, (s, n) in enumerate(zip(starts, lens)):
        padded[b, :n] = got_lp[s:s + n]
    ref_g = O.ctc_greedy_search(padded, torch.tensor(lens))
    for b in range(len(lens)):
        assert toks[b, :int(tl[b])].cpu().tolist() == ref_g[b]
    # prefix beam search: ids, times exact; scores to 1e-9 (device libm vs glibc last-ulp differences)
    ptoks, ptimes, plens, pscores, nhyp = ops.ctc_prefix_beam_search(tv, ti, tI(starts), tI(lens), beam)
    ref_b = O.ctc_prefix_beam_search(padded, torch.tensor(lens), beam)
    for b in range(len(lens)):
        n = int(nhyp[b])
        assert n == len(ref_b[b]["nbest"])
        for r in range(n):
            ln = int(plens[b, r])
            assert ptoks[b, r, :ln].cpu().tolist() == ref_b[b]["nbest"][r], (b, r)
            assert ptimes[b, r, :ln].cpu().tolist() == ref_b[b]["nbest_times"][r], (b, r)
            assert abs(float(pscores[b, r]) - ref_b[b]["nbest_scores"][r]) < 1e-9 * max(1.0, abs(ref_b[b]["nbest_scores"][r]))


def test_prefix_beam_random_posteriors_gpu():
    """The 40 random posterior matrices on which the oracle is pinned to the reference (tests/test_oracle_pin.py:
    peaky / flat / blank-heavy / repeated frames, ragged lengths, beams up to the vocabulary size) through the CUDA
    kernels: greedy ids, n-best ids and times exact, scores to 1e-9."""
    import ops
    g = torch.Generator().manual_seed(2024)
    tI = lambda t: torch.tensor(t, dtype=torch.int32, device=_dev())
    for case in range(40):
        B = 1 + case % 3
        T = int(torch.randint(1, 48, (1,), generator=g))
        V = int(torch.randint(3, 14, (1,), generator=g))
        beam = min(int(torch.randint(1, 8, (1,), generator=g)), V)
        sharp = [0.5, 2.0, 6.0][case % 3]
        logits = torch.randn(B, T, V, generator=g) * sharp
        logits[..., 0] += [0.0, 1.5, 3.0][(case // 3) % 3]
        if case % 4 == 0:
            logits = logits.repeat_interleave(2, dim=1)[:, :T]
        lp = logits.log_softmax(-1)
        lens = torch.randint(1, T + 1, (B,), generator=g)
        lens[0] = T
        ref_b = O.ctc_prefix_beam_search(lp, lens, beam)
        ref_g = O.ctc_greedy_search(lp, lens)
        # packed rows, as the library takes them
        starts = [0]
        for n in lens.tolist()[:-1]:
            starts.append(starts[-1] + n)
        rows = torch.cat([lp[b, :int(lens[b])] for b in range(B)], 0)
        tv, ti = rows.topk(beam, dim=-1)
        tvd, tid = tv.to(_dev()).contiguous(), ti.to(torch.int32).to(_dev()).contiguous()
        gt, gl = ops.ctc_greedy_search(tid, tI(starts), tI(lens.tolist()))
        toks, times, plens, scores, nhyp = ops.ctc_prefix_beam_search(tvd, tid, tI(starts), tI(lens.tolist()), beam)
        for b in range(B):
            assert gt[b, :int(gl[b])].cpu().tolist() == ref_g[b], case
            n = int(nhyp[b])
            assert n == len(ref_b[b]["nbest"]), case
            for r in range(n):
                ln = int(plens[b, r])
                assert toks[b, r, :ln].cpu().tolist() == ref_b[b]["nbest"][r], (case, b, r)
                assert times[b, r, :ln].cpu().tolist() == ref_b[b]["nbest_times"][r], (case, b, r)
                want = ref_b[b]["nbest_scores"][r]
                assert abs(float(scores[b, r]) - want) < 1e-9 * max(1.0, abs(want)), (case, b, r)


def test_prefix_beam_kat_gpu():
    """runtime/core/test/ctc_prefix_beam_search_test.cc:29-72 through the CUDA kernel."""
    import ops
    probs = torch.tensor([[0.25, 0.40, 0.35], [0.40, 0.35, 0.25], [0.10, 0.50, 0.40]]).log()
    tv, ti = probs.topk(3, dim=-1)
    tI = lambda t: torch.tensor(t, dtype=torch.int32, device=_dev())
    toks, times, lens, scores, nhyp = ops.ctc_prefix_beam_search(tv.to(_dev()).contiguous(),
                                                                 ti.to(torch.int32).to(_dev()).contiguous(),
                                                                 tI([0]), tI([3]), 3)
    assert int(nhyp[0]) == 3
    got = [toks[0, r, :int(lens[0, r])].cpu().tolist() for r in range(3)]
    assert got == [[2, 1], [1, 2], [1]]
    for r, want in enumerate([0.2185, 0.1550, 0.1525]):
        assert abs(math.exp(float(scores[0, r])) - want) < 1e-4
    assert [times[0, r, :int(lens[0, r])].cpu().tolist() for r in range(3)] == [[0, 2], [0, 2], [2]]


def test_fbank():
    from wenet_b200.fbank import FbankExtractor
    g = torch.Generator().manual_seed(3)
    ns = [16000 * 3 + 123, 16000, 400, 399, 16000 * 2]
    N = max(ns) + 5
    N = (N + 3) // 4 * 4
    pcm_i = torch.zeros(len(ns), N, dtype=torch.int16)
    for b, n in enumerate(ns):
        t = torch.arange(n) / 16000.0
        sig = 2000 * torch.sin(2 * math.pi * (200 + 50 * b) * t) + torch.randn(n, generator=g) * 1500
        pcm_i[b, :n] = sig.clamp(-32767, 32767).round().to(torch.int16)
    ex = FbankExtractor(80)
    nsd = torch.tensor(ns, dtype=torch.int32, device=_dev())
    out_i = ex(pcm_i.to(_dev()), nsd)
    out_f = ex((pcm_i.float() / 32768.0).to(_dev()), nsd)
    torch.cuda.synchronize()
    for b, n in enumerate(ns):
        ref = O.fbank(pcm_i[b, :n].float())
        m = ref.shape[0]
        assert ex.num_frames(n) == m
        if m:
            assert (out_i[b, :m].cpu() - ref).abs().max().item() < 1e-3
            assert (out_f[b, :m].cpu() - ref).abs().max().item() < 1e-3
        assert (out_i[b, m:] == 0).all()


def test_fbank_kernel_vs_reference_cxx():
    """The CUDA fbank against the REFERENCE'S OWN compiled C++ front-end (runtime/core/frontend/fbank.h + fft.cc built by
    oracle/Makefile; Kaldi configuration of feature_pipeline.h:55-63; its output on these 2 s of noise is stored in
    tests/golden/oracle_pin.npz) - the product against the real reference, not only against the restatement.  Gate as
    for torchaudio (two fp32 FFT front-ends): 2e-3."""
    from test_oracle_pin import gold, noise_2s
    from wenet_b200.fbank import FbankExtractor
    wav = noise_2s()
    n = wav.numel()
    ref = gold("fbank_kaldi80")
    ex = FbankExtractor(80)
    N = (n + 3) // 4 * 4
    pcm = torch.zeros(1, N, dtype=torch.int16)
    pcm[0, :n] = wav.to(torch.int16)
    out = ex(pcm.to(_dev()), torch.tensor([n], dtype=torch.int32, device=_dev()))
    torch.cuda.synchronize()
    m = ref.shape[0]
    assert ex.num_frames(n) == m
    d = (out[0, :m].cpu() - ref).abs()
    print("fbank kernel vs reference C++ front-end: max %.3g mean %.3g" % (d.max().item(), d.mean().item()))
    assert d.max().item() < 2e-3 and d.mean().item() < 1e-4


def test_fbank_edge_inputs():
    """Digital silence (the log floor), a large DC offset under a small signal (remove_dc_offset), full-scale int16 and an
    all-maximum row, in one ragged batch: against the oracle, which tests/test_oracle_pin.py pins to torchaudio on the same
    kinds of input."""
    from wenet_b200.fbank import FbankExtractor
    g = torch.Generator().manual_seed(11)
    n = 8000
    rows = [torch.zeros(n),
            torch.randn(n, generator=g) * 50 + 12000,
            torch.where(torch.rand(n, generator=g) > 0.5, 32767.0, -32768.0),
            torch.full((n,), 32767.0)]
    ns = [n, n - 1, n - 160, 4000]
    pcm_i = torch.zeros(len(rows), n, dtype=torch.int16)
    for b, (r, k) in enumerate(zip(rows, ns)):
        pcm_i[b, :k] = r[:k].round().clamp(-32768, 32767).to(torch.int16)
    ex = FbankExtractor(80)
    nsd = torch.tensor(ns, dtype=torch.int32, device=_dev())
    out = ex(pcm_i.to(_dev()), nsd)
    torch.cuda.synchronize()
    assert torch.isfinite(out).all()
    worst = []
    for b, k in enumerate(ns):
        ref = O.fbank(pcm_i[b, :k].float())
        m = ref.shape[0]
        assert ex.num_frames(k) == m
        worst.append((out[b, :m].cpu() - ref).abs().max().item())
        assert (out[b, m:] == 0).all()
    print("fbank edge inputs, max |gpu - oracle| per row (silence, dc, full scale, constant):", worst)
    assert worst[0] == 0.0                      # silence: every bin is log(FLT_EPSILON) on both sides
    assert worst[1] < 1e-2 and worst[2] < 1e-3
    # row 3 is pure DC: after remove_dc_offset what is left is the rounding of the frame mean (exactly zero in the oracle),
    # so only the floor and finiteness are pinned there
    floor = math.log(torch.finfo(torch.float32).eps)
    assert (out[3, :ex.num_frames(ns[3])] >= floor - 1e-3).all() and (out[3, :ex.num_frames(ns[3])] < 0).all()


@pytest.mark.parametrize("V,k", [(4233, 10), (37, 5), (5538, 1), (300, 64)])
def test_lse_topk_without_writeback(V, k):
    """wb_ctc_topk's kernel mode (no normalised matrix written): same top-k as the write-back mode and as torch,
    logits untouched; flat / tied rows (more candidates than the per-warp list holds) take the ordered re-scan path."""
    import ops
    g = torch.Generator().manual_seed(V + k)
    M = 257
    ld = (V + 7) // 8 * 8
    logits = _peaky_logits(M, V, g)
    logits[3] = 0.25                                  # completely flat row: every element ties
    logits[4, : V // 2] = 1.5                         # half the row tied at the maximum
    logits[5] = torch.arange(V, dtype=torch.float32) * 1e-3   # slowly increasing: many near-candidates
    buf = torch.zeros(M, ld)
    buf[:, :V] = logits
    dbuf = buf.to(_dev())
    tv, ti = ops.lse_topk(dbuf, V, k, blank_id=0, blank_penalty=0.5)
    assert torch.equal(dbuf.cpu(), buf)               # input left as it was
    pen = logits.clone()
    pen[:, 0] -= 0.5
    ref = pen.log_softmax(-1)
    # reference order: value descending, index ascending (ties are common in rows 3 and 4)
    order = torch.argsort(-ref.double() + torch.arange(V, dtype=torch.float64) * 0, dim=-1, stable=True)[:, :k]
    got_i = ti.cpu().long()
    got_v = tv.cpu()
    assert (got_v - torch.gather(ref, 1, got_i)).abs().max().item() < 2e-5
    for r in range(M):
        rv = ref[r, order[r]]
        assert (got_v[r] - rv).abs().max().item() < 2e-5, r
        if r in (3, 4, 5) or torch.unique(pen[r]).numel() == V:
            assert torch.equal(got_i[r], order[r]), (r, got_i[r], order[r])
    # the write-back mode agrees bit for bit on the top-k and produces the full normalised matrix
    tv2, ti2 = ops.logsoftmax_topk(dbuf, V, k, blank_id=0, blank_penalty=0.5)
    assert torch.equal(ti2, ti) and torch.equal(tv2, tv)
    assert (dbuf[:, :V].cpu() - ref).abs().max().item() < 2e-5


@pytest.mark.parametrize("M,N,K", [(320, 1280, 5120), (40, 1280, 1280), (257, 256, 2048), (500, 640, 4096)])
def test_gemm_resid_splitk(M, N, K):
    """Few-row residual GEMM with the K range cut into pieces (decoding projections): C += alpha (A B^T + bias), the bias added
    exactly once, against torch in fp32 (the reduce-add order of the pieces is free: tolerance, not bit equality)."""
    from wenet_b200 import _lib
    from wenet_b200._lib import check, cur_stream, ptr
    g = torch.Generator(device="cpu").manual_seed(M + N + K)
    a = _rb(torch.randn(M, K, generator=g)).to(_dev())
    b = _rb(torch.randn(N, K, generator=g) / math.sqrt(K)).to(_dev())
    bias = (torch.randn(N, generator=g) * 3).to(_dev())
    c0 = torch.randn(M, N, generator=g).to(_dev())
    c = c0.clone()
    check(_lib.load().wb_op_gemm_resid_splitk(ptr(a), a.stride(0), ptr(b), M, N, K, ptr(bias), 0.5, ptr(c), c.stride(0),
                                              cur_stream()), "wb_op_gemm_resid_splitk")
    torch.cuda.synchronize()
    _close(c, c0 + 0.5 * (a.float() @ b.float().T + bias), 1e-5, 3e-4)
