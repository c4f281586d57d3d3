"""Whisper path and decode mode "attention" on the GPU (through the C ABI) against the committed goldens produced by the
UNMODIFIED reference (oracle/make_goldens.py: tiny_attention, tiny_bn_attention, whisper_tiny) and the CPU oracle.

Tolerances:
  * log-mel: |GPU - reference| <= 2e-3 in the normalised (x + 4) / 4 domain (two fp32 DFTs; values floor at max - 8 decades)
  * Whisper encoder_out (bf16 GEMM operands) vs the fp32 reference: max <= 6e-2, mean <= 8.2e-3 (the reference's own bf16
    autocast yard-stick used for the Conformer path, BASELINE.md section 4) AND within 3x of the bf16-emulating oracle's
    own distance from fp32
  * attention decoding: best-hypothesis token ids identical to the reference's (the bf16-emulating oracle reproduces the
    goldens, i.e. the margins of these fixtures exceed the operand-rounding noise)
  * one beam step on given inputs (op-level): exact
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from helpers import SEED, err, load_golden
from oracle import wenet_oracle as O
from wenet_b200 import synth


def _whisper_model():
    from wenet_b200.whisper import B200Whisper
    cfg = synth.recipe("whisper_tiny")
    sd = synth.synth_state_dict(cfg, seed=SEED)
    return cfg, sd, B200Whisper(cfg, sd)


def test_logmel_golden():
    from wenet_b200.whisper import LogMelExtractor
    g = load_golden("whisper_tiny")
    ns = g["num_samples"].tolist()
    pcm = synth.synth_pcm(len(ns), ns, seed=SEED)
    ex = LogMelExtractor(32, 400, 160)
    x = (pcm.float() / 32768.0).cuda()
    feats = ex(x, torch.tensor(ns, dtype=torch.int32, device="cuda"), max_frames=g["feats"].shape[1]).cpu()
    ref = torch.from_numpy(g["feats"])
    for b, n in enumerate(ns):
        m = int(g["feat_lens"][b])
        assert m == ex.num_frames(n)
        mx, mean = err(feats[b, :m], ref[b, :m])
        print("log-mel utt %d: max %.2e mean %.2e" % (b, mx, mean))
        assert mx <= 2e-3 and mean <= 5e-5
        assert float(feats[b, m:].abs().max()) == 0.0 if m < feats.shape[1] else True
    # the oracle restatement on the same audio (runs everywhere, no reference needed)
    o = O.log_mel_spectrogram(pcm[0, :ns[0]].float() / 32768.0, 400, 160, 32)
    assert err(feats[0, :o.shape[0]], o)[0] <= 2e-3


@pytest.mark.parametrize("parity", ["even", "odd"])
def test_whisper_encoder_golden(parity):
    g = load_golden("whisper_tiny")
    cfg, sd, model = _whisper_model()
    xs = torch.from_numpy(g["feats"])
    lens = torch.from_numpy(g["feat_lens"]).long()
    key_o, key_l = "enc_out", "enc_lens"
    if parity == "odd":
        xs = xs[:, :xs.shape[1] - 1]
        lens = torch.minimum(lens, torch.tensor(xs.shape[1]))
        key_o, key_l = "enc_out_odd", "enc_lens_odd"
    out, masks = model.encoder(xs.cuda(), lens.cuda())
    ref = torch.from_numpy(g[key_o])
    assert out.shape == ref.shape
    assert masks.squeeze(1).sum(1).cpu().tolist() == g[key_l].tolist()
    with torch.no_grad():
        emu, _ = O.whisper_encoder_forward(sd, 2, xs, lens, O.bf16_round)
    for b in range(xs.shape[0]):
        n = int(g[key_l][b])
        mx, mean = err(out[b, :n].cpu(), ref[b, :n])
        emx, emean = err(emu[b, :n], ref[b, :n])
        print("whisper enc (%s) utt %d: GPU vs fp32 reference max %.2e mean %.2e | bf16-emulating oracle max %.2e mean %.2e"
              % (parity, b, mx, mean, emx, emean))
        assert mx <= 6e-2 and mean <= 8.2e-3
        assert mean <= 3.0 * emean + 1e-4
        assert float(out[b, n:].abs().max()) == 0.0 if n < out.shape[1] else True


def test_whisper_encoder_precise_mode():
    """precise mode (bf16x3 GEMMs, fp32 attention): Whisper encoder_out within 1e-3 of the fp32 reference goldens, both length
    parities; attention decoding on top of it returns the reference's token ids."""
    from wenet_b200.whisper import B200Whisper
    g = load_golden("whisper_tiny")
    cfg = synth.recipe("whisper_tiny")
    sd = synth.synth_state_dict(cfg, seed=SEED)
    model = B200Whisper(cfg, sd, precise=True)
    for key_o, key_l, cut in (("enc_out", "enc_lens", 0), ("enc_out_odd", "enc_lens_odd", 1)):
        xs = torch.from_numpy(g["feats"])
        xs = xs[:, :xs.shape[1] - cut]
        lens = torch.minimum(torch.from_numpy(g["feat_lens"]).long(), torch.tensor(xs.shape[1]))
        out, _ = model.encoder(xs.cuda(), lens.cuda())
        ref = torch.from_numpy(g[key_o])
        for b in range(xs.shape[0]):
            n = int(g[key_l][b])
            mx, mean = err(out[b, :n].cpu(), ref[b, :n])
            print("whisper enc precise (%s) utt %d: max %.2e mean %.2e" % (key_o, b, mx, mean))
            assert mx <= 1e-3
    xs = torch.from_numpy(g["feats"]).cuda()
    lens = torch.from_numpy(g["feat_lens"]).cuda()
    infos = {"tasks": [str(t) for t in g["tasks"]], "langs": [str(t) for t in g["langs"]]}
    res = model.decode(["attention"], xs, lens, beam_size=int(g["beam"]), infos=infos)["attention"]
    assert [list(r.tokens) for r in res] == [g["att%d" % b].tolist() for b in range(len(res))]


def test_whisper_attention_decode_golden():
    g = load_golden("whisper_tiny")
    cfg, sd, model = _whisper_model()
    xs = torch.from_numpy(g["feats"]).cuda()
    lens = torch.from_numpy(g["feat_lens"]).cuda()
    infos = {"tasks": [str(t) for t in g["tasks"]], "langs": [str(t) for t in g["langs"]]}
    res = model.decode(["attention"], xs, lens, beam_size=int(g["beam"]), infos=infos)["attention"]
    got = [list(r.tokens) for r in res]
    want = [g["att%d" % b].tolist() for b in range(len(got))]
    print("whisper attention decode: steps", model.last_attention_steps, "lens", [len(t) for t in got], "reference",
          [len(t) for t in want])
    assert got == want
    # default infos (search.py:270-275) and beam 1 run through
    r1 = model.decode(["attention"], xs, lens, beam_size=1)["attention"]
    assert len(r1) == len(got)


def test_whisper_ctc_modes_and_api():
    g = load_golden("whisper_tiny")
    cfg, sd, model = _whisper_model()
    xs = torch.from_numpy(g["feats"]).cuda()
    lens = torch.from_numpy(g["feat_lens"]).cuda()
    blank = cfg["ctc_conf"]["ctc_blank_id"]
    res = model.decode(["ctc_greedy_search", "ctc_prefix_beam_search"], xs, lens, beam_size=3, blank_id=blank)
    out, masks = model.encoder(xs, lens)
    lp = model.ctc_logprobs(out).cpu()
    el = masks.squeeze(1).sum(1).cpu()
    assert [list(r.tokens) for r in res["ctc_greedy_search"]] == O.ctc_greedy_search(lp, el, blank)
    ob = O.ctc_prefix_beam_search(lp, el, 3, blank)
    for b in range(xs.shape[0]):
        assert [list(h) for h in res["ctc_prefix_beam_search"][b].nbest] == ob[b]["nbest"]
    with pytest.raises(NotImplementedError):
        model.decode(["attention_rescoring"], xs, lens, beam_size=3)
    assert model.sos_symbol() == 100 and model.eos_symbol() == 99 and model.default_decode_method == "attention"


@pytest.mark.parametrize("name,recipe", [("tiny_attention", "tiny"), ("tiny_bn_attention", "tiny_bn")])
def test_attention_mode_conformer_golden(name, recipe):
    """ASRModel.decode(["attention"]) (asr_model.py:315-318) on the U2++ / non-streaming test recipes."""
    from wenet_b200.asr_model import B200ASRModel
    from wenet_b200.fbank import FbankExtractor
    g = load_golden(name)
    ns = g["num_samples"].tolist()
    cfg = synth.recipe(recipe)
    sd = synth.synth_state_dict(cfg, seed=SEED)
    model = B200ASRModel(cfg, sd)
    pcm = synth.synth_pcm(len(ns), ns, seed=SEED)
    ex = FbankExtractor(80)
    feats = ex(pcm.cuda(), torch.tensor(ns, dtype=torch.int32, device="cuda"))
    lens = torch.tensor([ex.num_frames(n) for n in ns], dtype=torch.int64)
    feats = feats[:, :int(lens.max())].contiguous()
    res = model.decode(["attention", "ctc_greedy_search"], feats, lens.cuda(), beam_size=int(g["beam"]),
                       length_penalty=float(g["length_penalty"]))
    got = [list(r.tokens) for r in res["attention"]]
    want = [g["att%d" % b].tolist() for b in range(len(ns))]
    print(name, "steps", model.last_attention_steps, "lens", [len(t) for t in got])
    assert got == want
    assert len(res["ctc_greedy_search"]) == len(ns)


def test_beam_step_exact():
    """beam_step_kernel against the oracle's restatement of search.py:309-355 on random tables (finished rows, -inf scores,
    the first step's [0, -inf, ...] initial scores): scores, tokens, end flags and ancestry exact."""
    from wenet_b200 import _lib
    from wenet_b200._lib import check, cur_stream, ptr
    lib = _lib.load()
    g = torch.Generator().manual_seed(11)
    for B, N, pos in ((3, 4, 5), (2, 10, 0), (5, 1, 2), (1, 7, 9)):
        R, L, eos, V = B * N, 16, 7, 50
        logp = torch.randn(R, V, generator=g).log_softmax(-1)
        topv, topi = logp.topk(N)
        scores = torch.randn(R, 1, generator=g) * 3
        if pos == 0:
            scores = torch.tensor([0.0] + [-float("inf")] * (N - 1)).repeat(B).unsqueeze(1)
        end = (torch.rand(R, 1, generator=g) < 0.3) if pos > 0 else torch.zeros(R, 1, dtype=torch.bool)
        hyps = torch.randint(0, V, (R, pos + 1), generator=g)
        hyps[end.squeeze(1), -1] = eos
        anc = torch.randint(0, N, (R, L), generator=g) + (torch.arange(R) // N * N).unsqueeze(1)
        ns, ne, nh, par = O.beam_step(topv, topi, scores, end, hyps, N, eos)
        d = lambda t, dt: t.to(dt).contiguous().cuda()
        hyp_in = torch.zeros(R, L, dtype=torch.int32)
        hyp_in[:, :pos + 1] = hyps.int()
        so, eo = torch.zeros(R, device="cuda"), torch.zeros(R, dtype=torch.int32, device="cuda")
        ho, ao = torch.zeros(R, L, dtype=torch.int32, device="cuda"), torch.zeros(R, L, dtype=torch.int32, device="cuda")
        nt, npz = torch.zeros(R, dtype=torch.int32, device="cuda"), torch.zeros(R, dtype=torch.int32, device="cuda")
        ue = torch.zeros(B, dtype=torch.int32, device="cuda")
        a = [d(topv, torch.float32), d(topi, torch.int32), d(scores.view(-1), torch.float32), d(end.view(-1), torch.int32),
             hyp_in.cuda(), d(anc, torch.int32)]
        check(lib.wb_op_attention_beam_step(ptr(a[0]), ptr(a[1]), ptr(a[2]), ptr(a[3]), ptr(a[4]), ptr(a[5]), B, N, L, pos, eos,
                                            ptr(so), ptr(eo), ptr(ho), ptr(ao), ptr(nt), ptr(npz), ptr(ue), cur_stream()),
              "wb_op_attention_beam_step")
        torch.cuda.synchronize()
        assert torch.equal(so.cpu(), ns.view(-1))
        assert eo.cpu().bool().tolist() == ne.view(-1).tolist()
        assert torch.equal(ho.cpu()[:, :pos + 2].long(), nh)
        assert nt.cpu().long().tolist() == nh[:, -1].tolist() and npz.cpu().tolist() == [pos + 1] * R
        want_anc = torch.cat([anc[par][:, :pos], par.view(-1, 1)], dim=1)
        assert torch.equal(ao.cpu()[:, :pos + 1].long(), want_anc)
        assert ue.cpu().tolist() == ne.view(B, N).sum(1).tolist()


def test_whisper_through_install():
    """The reference's own init_model / Whisper.decode / processor.compute_log_mel_spectrogram after wenet_b200.install()
    (the `wenet.cli` path: cli/model.py loads the model through init_model and features through processor): same tokens as
    the CPU reference's goldens.  Needs a reference tree (baseline/_ref on the GPU box)."""
    from oracle import shim
    if not shim.have_reference():
        pytest.skip("no reference tree (baseline/_ref or /root/reference)")
    import types
    shim.install()
    from wenet_b200 import plugin
    plugin.install()
    try:
        import wenet.dataset.processor as processor
        from wenet.utils import init_model as im
        g = load_golden("whisper_tiny")
        cfg = synth.recipe("whisper_tiny")
        model = shim.init_reference_model(dict(cfg))
        assert type(model).__name__ == "B200WhisperPlugin" and isinstance(model, im.Whisper)
        model.load_state_dict(synth.synth_state_dict(cfg, seed=SEED), strict=True)
        model = model.cuda().eval()
        # features through the rebound processor function
        ns = g["num_samples"].tolist()
        pcm = synth.synth_pcm(len(ns), ns, seed=SEED)
        feats = []
        for b, n in enumerate(ns):
            s = processor.compute_log_mel_spectrogram(dict(key="k", wav=(pcm[b, :n].float() / 32768.0).unsqueeze(0),
                                                           sample_rate=16000), n_fft=400, hop_length=160, num_mel_bins=32)
            feats.append(s["feat"])
            assert err(s["feat"], torch.from_numpy(g["feats"][b, :s["feat"].shape[0]]))[0] <= 2e-3
        lens = torch.tensor([f.shape[0] for f in feats])
        xs = torch.nn.utils.rnn.pad_sequence(feats, batch_first=True, padding_value=0)
        infos = {"tasks": [str(t) for t in g["tasks"]], "langs": [str(t) for t in g["langs"]]}
        with torch.no_grad():
            res = model.decode(["attention"], xs.cuda(), lens.cuda(), beam_size=int(g["beam"]), infos=infos)["attention"]
        assert [list(r.tokens) for r in res] == [g["att%d" % b].tolist() for b in range(len(ns))]
        assert type(res[0]).__module__.startswith("wenet.")        # the reference's DecodeResult type
    finally:
        plugin.uninstall()


@pytest.mark.parametrize("M,V,k,slices", [(37, 51866, 10, 16), (320, 20001, 4, 16), (3, 70000, 32, 8)])
def test_lse_topk_sliced(M, V, k, slices):
    """Sliced top-k of the log-softmax (few rows, huge vocabulary): values within 1e-5 of torch.log_softmax(...).topk, indices
    identical, incl. exact ties broken by index."""
    from wenet_b200 import _lib
    from wenet_b200._lib import check, cur_stream, ptr
    lib = _lib.load()
    g = torch.Generator().manual_seed(M + V)
    x = torch.randn(M, V, generator=g) * 3
    x[0, 5] = x[0, 40000 % V] = x[0].max() + 1.0          # an exact tie across two slices: lower index first
    ldl = (V + 7) // 8 * 8
    buf = torch.full((M, ldl), float("nan"))
    buf[:, :V] = x
    xd = buf.cuda()
    tv = torch.empty(M, k, device="cuda")
    ti = torch.empty(M, k, dtype=torch.int32, device="cuda")
    scr = torch.empty(M * slices * (k * 8 + 8) + 256, dtype=torch.uint8, device="cuda")
    check(lib.wb_op_lse_topk_sliced(ptr(xd), ldl, M, V, k, slices, ptr(tv), ptr(ti), ptr(scr), scr.numel(), cur_stream()),
          "wb_op_lse_topk_sliced")
    rv, ri = torch.log_softmax(x.double(), -1).topk(k)
    assert (tv.cpu().double() - rv).abs().max().item() < 1e-5
    got = ti.cpu().long()
    assert got[0, 0].item() == 5 and got[0, 1].item() == 40000 % V
    same = got == ri
    assert bool(same[1:].all()) and bool(same[0, 2:].all())


NEAR_TIE = 0.15


def test_whisper_large_widths_against_oracle():
    """The code paths only the large geometry takes - LayerNorm d = 1280, 20 heads, K = 1280 / 5120 GEMMs (128-column tiles for
    few rows, split-K residual projections), cross attention in key pieces, the sliced top-k over V = 51 866 - on a 2 + 2
    layer model of the large-v3 widths, against the CPU oracle: encoder_out vs the fp32 oracle inside the bf16 budget and
    within 3x of the bf16-emulating oracle's own distance; attention decoding (12 tokens per hypothesis, beam 4) token for
    token against the bf16-emulating oracle run on the GPU's encoder output.  Where the oracle's final beams end within
    NEAR_TIE of each other they are not ordered by the arithmetic, and the bf16 path may end on either one: the emulation's
    own 12-step score of one hypothesis moves by 0.06 between decoding utterance 1 alone and in this batch of three, where
    its two best beams end 0.10 apart."""
    from wenet_b200.whisper import B200Whisper, whisper_prefix
    cfg = synth.recipe("whisper_wide")
    sd = synth.synth_whisper_state_dict_fast(cfg, seed=SEED, eos_beta=3.0)
    sd["decoder.output_layer.weight"] = sd["decoder.output_layer.weight"] * 3.0     # peaky posteriors: clear beam margins
    model = B200Whisper(cfg, sd)
    g = torch.Generator().manual_seed(3)
    T, lens = 300, [300, 212, 97]
    xs = torch.randn(len(lens), T, 128, generator=g) * 0.5
    for b, n in enumerate(lens):
        xs[b, n:] = 0.0
    xl = torch.tensor(lens)
    out, masks = model.encoder(xs.cuda(), xl.cuda())
    with torch.no_grad():
        o32, m32 = O.whisper_encoder_forward(sd, 20, xs, xl, None)
        oq, _ = O.whisper_encoder_forward(sd, 20, xs, xl, O.bf16_round)
    assert torch.equal(masks.cpu(), m32)
    for b in range(len(lens)):
        n = int(m32[b].sum())
        mx, mean = err(out[b, :n].cpu(), o32[b, :n])
        emx, emean = err(oq[b, :n], o32[b, :n])
        print("whisper wide enc utt %d: GPU vs fp32 oracle max %.2e mean %.2e | bf16-emulating oracle max %.2e mean %.2e"
              % (b, mx, mean, emx, emean))
        assert mx <= 6e-2 and mean <= 8.2e-3 and mean <= 3.0 * emean + 1e-4
    steps = 12
    model.max_decode_len = steps + 4
    infos = {"tasks": ["transcribe"] * 3, "langs": ["en", "zh", "de"]}
    res = model.decode(["attention"], xs.cuda(), xl.cuda(), beam_size=4, infos=infos)["attention"]
    prefix = whisper_prefix(cfg["tokenizer_conf"]["special_tokens"], infos["tasks"], infos["langs"])
    with torch.no_grad():
        ref, beams = O.attention_beam_search(sd, "decoder", 2, 20, out.cpu(), masks.cpu(), 4, prefix.tolist(), model.eos, 0.0,
                                             "whisper", O.bf16_round, maxlen=steps + 4, return_beams=True)
    got = [list(r.tokens) for r in res]
    agree = [sum(int(a == b2) for a, b2 in zip(x, y)) / max(len(y), 1) for x, y in zip(got, ref)]
    best = [max(s for _, s in bs) for bs in beams]
    near_tie = [any(h == g and best[b] - s <= NEAR_TIE for h, s in beams[b]) for b, g in enumerate(got)]
    print("whisper wide decode: GPU", got, "oracle", ref, "agreement", agree, "oracle beams", beams)
    assert sum(int(x == y) for x, y in zip(got, ref)) >= 2
    assert all(a >= 0.5 or t for a, t in zip(agree, near_tie)), (agree, near_tie)
