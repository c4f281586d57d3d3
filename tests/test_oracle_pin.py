"""Pin the CPU oracle (oracle/wenet_oracle.py) against the reference: its Python modules and its C++ front-end and CTC
prefix beam search.  What the reference computed on the inputs below is stored in tests/golden/oracle_pin.npz
(oracle/make_goldens.py regenerates it from a reference tree, using the input functions of this module); the tests
recompute the oracle side and compare.  The reference's own known-answer test is checked everywhere."""
import json
import math

import pytest
import torch

from helpers import load_golden
from oracle import shim
from oracle import wenet_oracle as O
from wenet_b200 import synth

needs_ref = pytest.mark.skipif(not shim.have_reference(), reason="needs a reference tree (WENET_REFERENCE_ROOT)")

MELSCALE_HZ = [0.0, 20.0, 333.3, 999.9, 1000.0, 1000.1, 2500.0, 7999.0, 8000.0]
_G = {}


def gold(key):
    """the reference's output stored under `key`; ragged results are JSON strings"""
    if not _G:
        _G.update(load_golden("oracle_pin"))
    v = _G[key]
    return json.loads(str(v)) if v.dtype.kind == "U" else torch.from_numpy(v.copy())


def noise_2s():
    """2 s + 123 samples of int16-range noise (the C++ front-end pins, and tests/test_ops_gpu.py)"""
    g = torch.Generator().manual_seed(3)
    return (torch.randn(16000 * 2 + 123, generator=g) * 3000).clamp(-32767, 32767).round()


def random_posteriors():
    """40 random CTC posterior matrices (peaky and flat, blank-heavy, repeated frames, beams up to the vocabulary size):
    per case (log-probs [B, T, V], lengths [B], beam)"""
    g = torch.Generator().manual_seed(2024)
    cases = []
    for case in range(40):
        B = 1 + case % 3
        T = int(torch.randint(1, 48, (1,), generator=g))
        V = int(torch.randint(3, 14, (1,), generator=g))
        beam = min(int(torch.randint(1, 8, (1,), generator=g)), V)   # the reference's topk(beam) needs beam <= V
        logits = torch.randn(B, T, V, generator=g) * [0.5, 2.0, 6.0][case % 3]
        logits[..., 0] += [0.0, 1.5, 3.0][(case // 3) % 3]          # blank-heavy cases
        if case % 4 == 0:                                            # runs of the same token
            logits = logits.repeat_interleave(2, dim=1)[:, :T]
        lp = logits.log_softmax(-1)
        lens = torch.randint(1, T + 1, (B,), generator=g)
        lens[0] = T
        cases.append((lp, lens, beam))
    return cases


@pytest.mark.parametrize("bins", [128, 80])
def test_slaney_mel_filters_vs_reference_cxx(bins):
    """The slaney filterbank (the one function the Python reference takes from librosa, which is not installed): the
    oracle's restatement against the REFERENCE'S OWN C++ implementation, runtime/core/frontend/fbank.h:91-150 (InitMelFilters,
    MelType::kSlaney) with :176-218 (MelScale / InverseMelScale), compiled from the reference sources (oracle/Makefile).
    The C++ front-end works on a 512-point FFT grid (UpperPowerOfTwo(400)); the frequency grid is the only place n_fft
    enters the restatement, so it is evaluated at n_fft = 512: same support, weights equal to fp32 rounding."""
    W = gold("slaney_filters%d" % bins)
    mine = O.slaney_mel_filters(16000, 512, bins)[:, :256]
    assert torch.equal(W > 0, mine > 0)
    assert (W - mine).abs().max().item() < 1e-5 * mine.max().item()
    # the scale functions themselves, below and above the 1 kHz knee: the reference's (Hz, mel, inverse) triples
    f_sp, knee, step = 200.0 / 3, 1000.0, math.log(6.4) / 27.0
    ref = gold("slaney_melscale").tolist()
    assert [r[0] for r in ref] == pytest.approx(MELSCALE_HZ, rel=1e-6)
    for (_, mel, inv), f in zip(ref, MELSCALE_HZ):
        want = knee / f_sp + math.log(f / knee) / step if f >= knee else f / f_sp
        assert abs(mel - want) < 1e-5 * max(1.0, want) and abs(inv - f) < 1e-5 * max(1.0, f)


def test_fbank_vs_reference_cxx():
    """Kaldi fbank: the oracle (pinned to torchaudio below) against the reference's own C++ front-end in the runtime's
    configuration (feature_pipeline.h:55-63 -> fbank.h:247-326: povey window, HTK mel from 20 Hz, pre-emphasis, DC removal,
    natural log with an FLT_EPSILON floor) on 2 s of noise; and the C++ Whisper configuration (feature_pipeline.h:64-73:
    hanning, slaney, log10, max - 8 clamp, (x + 4) / 4) against a per-frame restatement that uses the oracle's slaney
    filterbank.  (The Python Whisper front-end frames differently - centred STFT of size 400 - and is pinned separately.)"""
    wav = noise_2s()
    ref = gold("fbank_kaldi80")
    got = O.fbank(wav)
    assert got.shape == ref.shape
    assert (got - ref).abs().max().item() < 1e-3 and (got - ref).abs().mean().item() < 5e-5
    refw = gold("fbank_whisper128")
    m = 1 + (wav.numel() - 400) // 160
    frames = (wav / 32768.0).as_strided((m, 400), (160, 1)).clone()
    frames = frames - frames.mean(1, keepdim=True)                     # fbank.h:281-286 (remove_dc_offset stays on)
    x = torch.zeros(m, 512, dtype=torch.float64)
    x[:, :400] = (frames * torch.hann_window(400, periodic=True)).double()
    power = torch.fft.rfft(x, dim=1).abs() ** 2
    mel = power[:, :256].float() @ O.slaney_mel_filters(16000, 512, 128)[:, :256].T
    lg = torch.clamp(mel, min=1e-10).log10()
    lg = (torch.maximum(lg, lg.max() - 8.0) + 4.0) / 4.0
    assert refw.shape == lg.shape and (refw - lg).abs().max().item() < 1e-4


KAT_PROBS = [[0.25, 0.40, 0.35], [0.40, 0.35, 0.25], [0.10, 0.50, 0.40]]


def test_reference_cxx_search_kat_and_best_path():
    """The reference has TWO implementations of the CTC prefix beam search: wenet/models/transformer/search.py:127-249 (the
    Python API this build drops in under; the oracle equals it exactly, below) and runtime/core/decoder/ctc_prefix_beam_search.cc
    (the C++ runtime, float32, its own merge / time rules).  The C++ one, compiled from the reference sources,
    (a) reproduces the reference's known-answer test - the vectors test_prefix_beam_search_kat holds were transcribed from
    ctc_prefix_beam_search_test.cc:29-72 - and (b) picks the same BEST hypothesis as the oracle on all utterances of the 40
    random posterior matrices.  Deeper n-best entries, scores and times differ between the reference's own two
    implementations (full list equal on 74 of 79 utterances, best-path scores up to 0.09 apart), which is why the parity
    target is the Python search.  Each C++ hypothesis is stored as [score, tokens, times]."""
    kat = gold("cxx_search_kat")
    assert [h[1] for h in kat] == [[2, 1], [1, 2], [1]]
    for (score, _, _), want in zip(kat, [0.2185, 0.1550, 0.1525]):
        assert abs(math.exp(score) - want) < 1e-4
    assert [h[2] for h in kat] == [[0, 2], [0, 2], [2]]
    want = []
    for lp, lens, beam in random_posteriors():
        want += O.ctc_prefix_beam_search(lp, lens, beam)
    ref = gold("cxx_search_random")
    assert len(ref) == len(want) == 79
    same_list = 0
    for r, o in zip(ref, want):
        assert r[0][1] == o["nbest"][0]
        same_list += [h[1] for h in r] == o["nbest"]
    assert same_list >= 0.9 * len(want)


def test_prefix_beam_search_kat():
    """runtime/core/test/ctc_prefix_beam_search_test.cc:29-72 (the reference's only golden vector on this path)."""
    probs = torch.tensor(KAT_PROBS).log().unsqueeze(0)
    r = O.ctc_prefix_beam_search(probs, torch.tensor([3]), 3)[0]
    assert r["nbest"] == [[2, 1], [1, 2], [1]]
    for got, want in zip(r["nbest_scores"], [0.2185, 0.1550, 0.1525]):
        assert abs(math.exp(got) - want) < 1e-4
    assert r["nbest_times"] == [[0, 2], [0, 2], [2]]
    # frame argmaxes are 1, 0(blank), 1 -> "1 1"
    assert O.ctc_greedy_search(probs, torch.tensor([3])) == [[1, 1]]


def test_prefix_beam_search_random_posteriors_vs_reference():
    """search.py:127-249 on the 40 random posterior matrices: n-best token lists, fp64 scores and times of the oracle equal
    the reference's, element for element; ctc_greedy_search too."""
    ref = gold("py_search_random")
    for case, (lp, lens, beam) in enumerate(random_posteriors()):
        got = O.ctc_prefix_beam_search(lp, lens, beam)
        assert len(ref[case]["nbest"]) == len(got), case
        for b, o in enumerate(got):
            assert ref[case]["nbest"][b] == o["nbest"], case
            assert ref[case]["nbest_scores"][b] == o["nbest_scores"], case
            assert ref[case]["nbest_times"][b] == o["nbest_times"], case
        assert ref[case]["greedy"] == O.ctc_greedy_search(lp, lens), case


def test_fbank_vs_torchaudio():
    import torchaudio.compliance.kaldi as kaldi
    g = torch.Generator().manual_seed(3)
    wav = (torch.randn(1, 16000 * 2 + 123, generator=g) * 3000).clamp(-32767, 32767).round()
    ref = kaldi.fbank(wav, num_mel_bins=80, frame_length=25, frame_shift=10, dither=0.0, energy_floor=0.0,
                      sample_frequency=16000)
    got = O.fbank(wav[0])
    assert got.shape == ref.shape
    assert (got - ref).abs().max().item() < 1e-4


@pytest.mark.parametrize("kind", ["one_frame", "just_short_of_two", "silence", "dc_offset", "full_scale", "mel23"])
def test_fbank_edge_cases_vs_torchaudio(kind):
    """kaldi.py:514-645 on the inputs where a restatement goes wrong first: exactly one frame, one sample short of the
    second frame (snip_edges), digital silence (the log floor), a DC offset (remove_dc_offset), full-scale int16, and a
    different filterbank size."""
    import torchaudio.compliance.kaldi as kaldi
    g = torch.Generator().manual_seed(11)
    mel = 23 if kind == "mel23" else 80
    if kind == "one_frame":
        wav = torch.randn(1, 400, generator=g) * 2000
    elif kind == "just_short_of_two":
        wav = torch.randn(1, 559, generator=g) * 2000
    elif kind == "silence":
        wav = torch.zeros(1, 4000)
    elif kind == "dc_offset":
        wav = torch.randn(1, 8000, generator=g) * 50 + 12000
    elif kind == "full_scale":
        wav = torch.where(torch.rand(1, 8000, generator=g) > 0.5, 32767.0, -32768.0)
    else:
        wav = torch.randn(1, 16000, generator=g) * 3000
    wav = wav.round()
    ref = kaldi.fbank(wav, num_mel_bins=mel, frame_length=25, frame_shift=10, dither=0.0, energy_floor=0.0,
                      sample_frequency=16000)
    got = O.fbank(wav[0], num_mel_bins=mel)
    assert got.shape == ref.shape and ref.shape[0] == 1 + (wav.shape[1] - 400) // 160
    assert torch.isfinite(got).all()
    assert (got - ref).abs().max().item() < 2e-4, (got - ref).abs().max().item()
    # shorter than one window: torchaudio refuses the input (kaldi.py:142 assert); the restatement yields zero frames
    assert O.fbank(wav[0, :399], num_mel_bins=mel).shape[0] == 0
    with pytest.raises(AssertionError):
        kaldi.fbank(wav[:, :399], num_mel_bins=mel, dither=0.0, energy_floor=0.0)


def _tiny_cfg(bidir=True, causal=True, norm="layer_norm", kernel=8):
    return {
        "input_dim": 80, "output_dim": 37, "cmvn": None,
        "encoder": "conformer",
        "encoder_conf": dict(output_size=128, attention_heads=2, linear_units=256, num_blocks=2, dropout_rate=0.0,
                             positional_dropout_rate=0.0, attention_dropout_rate=0.0, input_layer="conv2d",
                             normalize_before=True, cnn_module_kernel=kernel, use_cnn_module=True,
                             activation_type="swish", pos_enc_layer_type="rel_pos",
                             selfattention_layer_type="rel_selfattn", causal=causal, use_dynamic_chunk=causal,
                             cnn_module_norm=norm, use_dynamic_left_chunk=False),
        "decoder": "bitransformer" if bidir else "transformer",
        "decoder_conf": dict(attention_heads=2, linear_units=256, num_blocks=2, dropout_rate=0.0,
                             positional_dropout_rate=0.0, self_attention_dropout_rate=0.0,
                             src_attention_dropout_rate=0.0, **({"r_num_blocks": 1} if bidir else {})),
        "tokenizer": "char", "tokenizer_conf": {},
        "ctc": "ctc", "ctc_conf": {"ctc_blank_id": 0},
        "model": "asr_model",
        "model_conf": dict(ctc_weight=0.3, lsm_weight=0.1, length_normalized_loss=False,
                           **({"reverse_weight": 0.3} if bidir else {})),
    }




def randn(seed, *shape):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed))


def pin_model(variant):
    """config and weights of the model pins: seeded synthetic weights (wenet_b200/synth.py, CTC head not sharpened), which
    the reference model loads for the goldens"""
    cfg = {"u2pp": _tiny_cfg(bidir=True),
           "nonstream_bn": _tiny_cfg(bidir=False, causal=False, norm="batch_norm", kernel=15)}[variant]
    return cfg, synth.synth_state_dict(cfg, seed=777, ctc_alpha=1.0)


STREAM_STARTS = range(0, 131 - 18, 16)      # forward_chunk steps of 19 input frames (chunk 4 after subsampling)


@pytest.mark.parametrize("variant", ["u2pp", "nonstream_bn"])
def test_oracle_matches_reference(variant):
    cfg, p = pin_model(variant)
    ecfg = O.encoder_cfg(p, heads=2, causal=cfg["encoder_conf"]["causal"], cnn_norm=cfg["encoder_conf"]["cnn_module_norm"])
    xs = randn(777, 2, 131, 80)
    lens = torch.tensor([131, 90])
    k = "match_%s_" % variant
    ref_out, ref_mask = gold(k + "enc_out"), gold(k + "enc_mask")
    with torch.no_grad():
        got_out, got_mask = O.encoder_forward(p, ecfg, xs, lens)
        assert torch.equal(ref_mask, got_mask)
        for b in range(2):
            n = int(ref_mask[b].sum())
            assert (ref_out[b, :n] - got_out[b, :n]).abs().max().item() < 2e-5
        if variant == "u2pp":
            r2 = gold(k + "enc_out_chunk4_left2")
            g2, _ = O.encoder_forward(p, ecfg, xs, lens, 4, 2)
            n = int(ref_mask[1].sum())
            assert (r2[1, :n] - g2[1, :n]).abs().max().item() < 2e-5
            # streaming chunk step (encoder.py:204-300): output and both caches after every chunk
            att_o = cnn_o = torch.zeros(0, 0, 0, 0)
            off = 0
            for j, s in enumerate(STREAM_STARTS):
                yo, att_o, cnn_o = O.encoder_forward_chunk(p, ecfg, xs[0:1, s:s + 19], off, 8, att_o, cnn_o)
                y, att, cnn = (gold(k + "stream_%s%d" % (w, j)) for w in ("y", "att", "cnn"))
                off += y.size(1)
                assert (y - yo).abs().max().item() < 2e-5
                assert (att - att_o).abs().max().item() < 2e-5 and (cnn - cnn_o).abs().max().item() < 2e-5
        # CTC + searches (the reference's searches ran on its own log-probs, as the oracle's do here)
        ref_lp = gold(k + "ctc_logp")
        got_lp = O.ctc_logprobs(p, got_out)
        assert (ref_lp - got_lp).abs().max().item() < 5e-5
        enc_lens = ref_mask.squeeze(1).sum(1)
        assert gold(k + "greedy") == O.ctc_greedy_search(ref_lp, enc_lens)
        rb = gold(k + "beam")
        gb = O.ctc_prefix_beam_search(ref_lp, enc_lens, 4)
        for r, g in zip(rb, gb):
            assert r["nbest"] == g["nbest"]
            assert r["nbest_scores"] == g["nbest_scores"]
            assert r["nbest_times"] == g["nbest_times"]
        rw = 0.3 if variant == "u2pp" else 0.0
        dcfg = dict(bidirectional=(variant == "u2pp"), layers=2, r_layers=1, heads=2)
        sos = eos = cfg["output_dim"] - 1
        gr = O.attention_rescoring(p, dcfg, gb, ref_out, enc_lens, sos, eos, 0.5, rw)
        for (tokens, score), g in zip(gold(k + "rescoring"), gr):
            assert tokens == g["tokens"]
            assert abs(score - g["best_score"]) < 1e-4


CHUNK_SETTINGS = [(1, 0), (1, -1), (3, 1), (8, -1), (16, 4), (32, 0)]


@pytest.mark.parametrize("chunk,left", CHUNK_SETTINGS)
def test_oracle_chunk_masks_and_streaming_vs_reference(chunk, left):
    """add_optional_chunk_mask (mask.py:162-227) and forward_chunk_by_chunk (encoder.py:302-362) for chunk / left-chunk
    settings from the degenerate (1 frame, no history) to wider than the utterance: the masked full forward and the chunk
    loop of the oracle equal the reference's, and (with limited history only when left >= 0) each other's cache semantics."""
    cfg, p = pin_model("u2pp")
    ecfg = O.encoder_cfg(p, heads=2, causal=True, cnn_norm="layer_norm")
    xs = randn(777, 2, 99, 80)
    lens = torch.tensor([99, 58])
    k = "chunk%d_left%d_" % (chunk, left)
    r, rm, rs = gold(k + "enc_out"), gold(k + "enc_mask"), gold(k + "stream")
    with torch.no_grad():
        o, om = O.encoder_forward(p, ecfg, xs, lens, chunk, left)
        assert torch.equal(rm, om)
        for b in range(2):
            n = int(rm[b].sum())
            assert (r[b, :n] - o[b, :n]).abs().max().item() < 2e-5, (chunk, left, b)
        # the streaming loop over one utterance (batch 1 by construction, encoder.py:330-333)
        win, stride = (chunk - 1) * 4 + 7, 4 * chunk
        att = cnn = torch.zeros(0, 0, 0, 0)
        off, outs = 0, []
        req = chunk * left if left >= 0 else -1
        for cur in range(0, 99 - 7 + 1, stride):
            y, att, cnn = O.encoder_forward_chunk(p, ecfg, xs[:1, cur:min(cur + win, 99)], off, req, att, cnn)
            outs.append(y)
            off += y.size(1)
        os_ = torch.cat(outs, 1)
        assert os_.shape == rs.shape
        assert (os_ - rs).abs().max().item() < 2e-5, (chunk, left)
        # and the chunk loop reproduces the chunk-masked full forward (same attention context by construction)
        assert (rs[0] - r[0, :rs.size(1)]).abs().max().item() < 1e-4


RESCORING_NBEST = [[[5, 7, 7, 30], [5, 7], [], [36]], [[2, 3, 4], [4, 3, 2]], [[11]]]
RESCORING_SCORES = [[-1.5, -2.25, -9.0, -3.0], [-0.5, -0.5], [-0.1]]
RESCORING_WEIGHTS = [(0.0, 0.0), (0.5, 0.0), (0.3, 0.3), (1.0, 0.5), (0.0, 1.0)]


@pytest.mark.parametrize("ctc_weight,reverse_weight", RESCORING_WEIGHTS)
def test_oracle_rescoring_weights_vs_reference(ctc_weight, reverse_weight):
    """attention_rescoring (search.py:374-458) over the weight settings that change which terms count: decoder only,
    CTC-weighted, bidirectional mix, right-to-left only; n-best lists with empty, single-token and equal-length hypotheses."""
    cfg, p = pin_model("u2pp")
    enc = randn(3, 3, 17, 128)
    lens = torch.tensor([17, 9, 4])
    got_in = [dict(nbest=n, nbest_scores=sc) for n, sc in zip(RESCORING_NBEST, RESCORING_SCORES)]
    sos = eos = cfg["output_dim"] - 1
    with torch.no_grad():
        dcfg = dict(bidirectional=True, layers=2, r_layers=1, heads=2)
        got = O.attention_rescoring(p, dcfg, got_in, enc, lens, sos, eos, ctc_weight, reverse_weight)
    for (tokens, score), g in zip(gold("rescoring_ctc%g_rev%g" % (ctc_weight, reverse_weight)), got):
        assert tokens == g["tokens"]
        assert abs(score - g["best_score"]) < 1e-4


@needs_ref
def test_plugin_config_reconstruction_and_registry():
    """wenet_b200.plugin: the train.yaml subset is recovered from a constructed reference model, and
    install() rebinds the reference's registries (SURVEY.md section 8b)."""
    from wenet_b200 import plugin, synth
    from wenet_b200.weights import ModelSpec
    cfg = synth.recipe("tiny")
    ref_cfg = dict(cfg, cmvn=None)
    ref_cfg.pop("cmvn_conf", None)
    model = shim.init_reference_model(ref_cfg)
    got = plugin.configs_from_reference_model(model)
    a, b = ModelSpec(got), ModelSpec(dict(cfg, cmvn=None))
    for k in ("input_dim", "vocab", "d_model", "heads", "ffn_dim", "enc_layers", "cnn_kernel", "cnn_causal", "cnn_norm",
              "use_dynamic_chunk", "bidirectional", "dec_layers", "rdec_layers", "dec_heads", "dec_ffn_dim", "has_cmvn"):
        assert getattr(a, k) == getattr(b, k), k
    cls = plugin.install()
    try:
        from wenet.utils import init_model as im
        import wenet.dataset.processor as processor
        assert im.WENET_MODEL_CLASSES["asr_model"] is cls and processor.compute_fbank is plugin._fbank_dropin
        assert plugin.install() is cls                      # idempotent
        m2 = shim.init_reference_model(dict(ref_cfg))
        assert type(m2).__name__ == "B200ASRModelPlugin"
        assert type(m2.encoder).__name__ == "B200ConformerEncoderPlugin" and type(m2.ctc).__name__ == "B200CTCPlugin"
        assert set(m2.state_dict().keys()) == set(model.state_dict().keys())
        import wenet_b200._lib as L
        x, n = torch.zeros(1, 50, 80), torch.tensor([50])
        for call in (lambda: m2.decode(["ctc_greedy_search"], x, n), lambda: m2.encoder(x, n),
                     lambda: m2.forward_encoder_chunk(x, 0, -1), lambda: m2.ctc_activation(torch.zeros(1, 4, 128))):
            with pytest.raises(L.WbError):      # CPU model -> loud failure, never a fallback
                call()
        # training mode keeps the reference's autograd path
        m2.train()
        y, _ = m2.encoder(x, n)
        assert y.requires_grad
        m2.eval()
        # dither / DataLoader-worker cases of compute_fbank keep the reference function
        s = processor.compute_fbank(dict(key="k", wav=torch.zeros(1, 1600), sample_rate=16000), num_mel_bins=80, dither=1.0)
        assert s["feat"].shape == (8, 80)
        # configurations outside the implemented set fail at construction
        bad = dict(ref_cfg, encoder_conf=dict(ref_cfg["encoder_conf"], pos_enc_layer_type="abs_pos",
                                              selfattention_layer_type="selfattn"))
        with pytest.raises(NotImplementedError):
            shim.init_reference_model(bad)
    finally:
        plugin.uninstall()      # restore the registries for other tests in this process
    from wenet.models.transformer.asr_model import ASRModel
    assert im.WENET_MODEL_CLASSES["asr_model"] is ASRModel




CONTEXT_WORDS = ["abc", "bcd", "ab", "cdeab", "xyz", "qrs q"]
CONTEXT_FIELDS = ("child_off", "child_tok", "child_node", "fail", "token", "node_score", "token_score", "output_score")


def context_symbols(V=30):
    sym = {"<blank>": 0, "<unk>": 1}
    for i in range(2, V):
        sym[chr(ord("a") + i - 2) if i < 28 else "z%d" % i] = i
    return sym


def context_posteriors(V=30, T=60):
    logits = randn(1, 3, T, V) * 2
    logits[:, :, 0] += 2.0
    return logits.log_softmax(-1), torch.tensor([T, 41, 7])


def test_context_graph_restated_vs_reference():
    """Context biasing (SURVEY.md section 8f-3): wenet_b200.context.build reproduces the arrays wenet_b200.context.flatten
    makes of the reference's ContextGraph (context_graph.py:103-200) for the same phrases, and the oracle's prefix beam
    search with that graph equals the reference's ctc_prefix_beam_search(..., context_graph) - prefixes, float64 scores
    (incl. the finalize() rule) and times - while differing from the un-biased search."""
    import numpy as np
    from wenet_b200 import context as CX
    sym = context_symbols()
    arr = CX.build([[sym.get(c if c != " " else "\u2581", sym["<unk>"]) for c in w] for w in CONTEXT_WORDS], 3.0)
    for n in CONTEXT_FIELDS:
        assert np.array_equal(getattr(arr, n), gold("context_" + n).numpy()), n
    lp, lens = context_posteriors()
    ref = gold("context_search")
    got = O.ctc_prefix_beam_search(lp, lens, 6, 0, arr)
    plain = O.ctc_prefix_beam_search(lp, lens, 6, 0)
    for a, b in zip(ref, got):
        assert a["nbest"] == b["nbest"]
        assert a["nbest_scores"] == b["nbest_scores"]
        assert a["nbest_times"] == b["nbest_times"]
    assert any(g["nbest"] != p["nbest"] for g, p in zip(got, plain))


ATTENTION_SETTINGS = [(4, 0.0), (3, 0.6)]


def test_attention_beam_search_oracle_matches_reference_conformer():
    """decode mode "attention" of a U2++ model (asr_model.py:315-318 -> search.py:252-371, left decoder,
    decoder.py:466-488): the cache-free restatement equals the reference's cached forward_one_step loop."""
    cfg = synth.recipe("tiny")
    p = synth.synth_state_dict(cfg, seed=777)
    enc = randn(5, 2, 21, 128)
    lens = torch.tensor([21, 13])
    mask = ~O.make_pad_mask(lens, 21).unsqueeze(1)
    sos = eos = cfg["output_dim"] - 1
    for (beam, lp), ref in zip(ATTENTION_SETTINGS, gold("attention_conformer")):
        with torch.no_grad():
            got = O.attention_beam_search(p, "decoder.left_decoder", 2, 2, enc, mask, beam, [[sos]] * 2, eos, lp, "wenet")
        assert ref == got, (beam, lp)


WHISPER_SETTINGS = [(4, 0.0), (1, 0.0), (6, 0.8)]     # beam 1 = greedy over the beam machinery; a length penalty
WHISPER_INFOS = {"tasks": ["transcribe", "transcribe", "translate"], "langs": ["en", "zh", "en"]}
WHISPER_LENS = ((150, [150, 111, 64]), (151, [151, 100, 37]))       # odd and even padded lengths (subsampling.py:171)


def whisper_pin_inputs():
    """the Whisper pin's audio (2 s + 77 samples) and its encoder inputs, one zero-padded batch per entry of WHISPER_LENS"""
    pcm = synth.synth_pcm(1, [16000 * 2 + 77], seed=3)[0, :16000 * 2 + 77].float() / 32768.0
    g = torch.Generator().manual_seed(1)
    batches = []
    for T, lens in WHISPER_LENS:
        xs = torch.randn(3, T, 32, generator=g) * 0.5
        for b in range(3):
            xs[b, lens[b]:] = 0.0
        batches.append((xs, torch.tensor(lens)))
    return pcm, batches


def test_whisper_oracle_matches_reference():
    """Whisper (wenet/models/whisper/whisper.py): log-mel call site (the reference's own function with the restated slaney
    filterbank injected as librosa.filters.mel), TransformerEncoder (conv1d2 / abs_pos_whisper / gelu),
    attention_beam_search with the forced Whisper prefix."""
    from wenet_b200.whisper import whisper_prefix
    cfg = synth.recipe("whisper_tiny")
    p = synth.synth_state_dict(cfg, seed=777)
    pcm, batches = whisper_pin_inputs()
    ref = gold("whisper_logmel")
    got = O.log_mel_spectrogram(pcm, 400, 160, 32)
    assert got.shape == ref.shape and (got - ref).abs().max().item() < 1e-5
    # slaney filterbank sanity: every filter is a non-negative triangle of area ~ 1 Hz^-1 * df (slaney norm), rows overlap
    fb = O.slaney_mel_filters(16000, 400, 128)
    assert fb.shape == (128, 201) and float(fb.min()) >= 0.0 and int((fb.sum(1) > 0).sum()) == 128
    assert abs(float((fb.sum(1) * 40.0)[100:].mean()) - 1.0) < 0.05        # bin spacing 40 Hz: area normalised filters
    for (T, lens), (xs, xl) in zip(WHISPER_LENS, batches):
        r_out, r_mask = gold("whisper_enc_out%d" % T), gold("whisper_enc_mask%d" % T)
        with torch.no_grad():
            g_out, g_mask = O.whisper_encoder_forward(p, 2, xs, xl)
        assert torch.equal(r_mask, g_mask)
        for b in range(3):
            n = int(r_mask[b].sum())
            assert (r_out[b, :n] - g_out[b, :n]).abs().max().item() < 2e-5
    # attention decoding on the reference's encoder output of the last batch
    prefix = whisper_prefix(cfg["tokenizer_conf"]["special_tokens"], WHISPER_INFOS["tasks"], WHISPER_INFOS["langs"])
    eos = cfg["tokenizer_conf"]["special_tokens"]["eot"]
    for (beam, lp), ref in zip(WHISPER_SETTINGS, gold("whisper_attention")):
        with torch.no_grad():
            got = O.attention_beam_search(p, "decoder", 2, 2, r_out, r_mask, beam, prefix.tolist(), eos, lp, "whisper")
        assert ref == got, (beam, lp)
        assert sum(len(g) for g in got) > 0
