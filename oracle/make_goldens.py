"""Generate tests/golden/*.npz by running the UNMODIFIED reference (/root/reference, through
oracle/shim.py) on deterministic synthetic weights (wenet_b200/synth.py) and inputs.

Run in the build container only:   python oracle/make_goldens.py
The fixtures hold OUTPUTS only (inputs and weights are regenerated from seeds at test time), so they
stay small.  TEST INFRASTRUCTURE — nothing in wenet_b200/ imports this.
"""
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import shim  # noqa: E402
from wenet_b200 import synth  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
SEED = 777


def ref_fbank(pcm_i16: torch.Tensor, n: int) -> torch.Tensor:
    shim.install()
    from wenet.dataset import processor
    wav = (pcm_i16[:n].float() / 32768.0).unsqueeze(0)
    s = processor.compute_fbank(dict(key="k", wav=wav, sample_rate=16000), num_mel_bins=80, frame_length=25,
                                frame_shift=10, dither=0.0)
    return s["feat"]


def fbank_goldens():
    ns = [32000 + 123, 20800, 400, 16000 * 5]
    pcm = synth.synth_pcm(len(ns), ns, seed=SEED)
    out = {"num_samples": np.array(ns)}
    for b, n in enumerate(ns):
        out["feat%d" % b] = ref_fbank(pcm[b], n).numpy()
    np.savez_compressed(os.path.join(GOLD, "fbank.npz"), **out)
    print("fbank:", {k: v.shape for k, v in out.items()})


def model_goldens(name, recipe, ns, beam=4, ctc_weight=0.5, store_logp=True, chunk=(4, 2), stream=True):
    torch.manual_seed(0)
    cfg = synth.recipe(recipe)
    sd = synth.synth_state_dict(cfg, seed=SEED)
    ref_cfg = dict(cfg, cmvn=None)      # the CMVN statistics come with the state_dict (buffers), not a file
    ref_cfg.pop("cmvn_conf", None)
    model = shim.init_reference_model(ref_cfg)
    if cfg.get("cmvn") is not None:
        from wenet.models.transformer.cmvn import GlobalCMVN
        model.encoder.global_cmvn = GlobalCMVN(torch.zeros(80), torch.ones(80))
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected, unexpected
    assert all(k.endswith("num_batches_tracked") for k in missing), missing
    model.eval()
    pcm = synth.synth_pcm(len(ns), ns, seed=SEED)
    feats = [ref_fbank(pcm[b], n) for b, n in enumerate(ns)]
    lens = torch.tensor([f.shape[0] for f in feats])
    T = int(lens.max())
    xs = torch.zeros(len(ns), T, 80)
    for b, f in enumerate(feats):
        xs[b, :f.shape[0]] = f
    out = {"num_samples": np.array(ns), "beam": np.array(beam), "ctc_weight": np.array(ctc_weight)}
    from wenet.models.transformer.search import (attention_rescoring, ctc_greedy_search, ctc_prefix_beam_search)
    with torch.no_grad():
        enc, mask = model.encoder(xs, lens, decoding_chunk_size=-1, num_decoding_left_chunks=-1)
        enc_lens = mask.squeeze(1).sum(1)
        out["enc_lens"] = enc_lens.numpy()
        out["enc_out"] = enc.numpy()
        logp = model.ctc_logprobs(enc)
        if store_logp:
            out["ctc_logp"] = logp.numpy()
        tv, ti = logp.topk(max(beam, 10), dim=-1)
        out["ctc_topk_val"], out["ctc_topk_idx"] = tv.numpy(), ti.numpy().astype(np.int32)
        g = ctc_greedy_search(logp, enc_lens)
        for b, r in enumerate(g):
            out["greedy%d" % b] = np.array(r.tokens, dtype=np.int32)
        pb = ctc_prefix_beam_search(logp, enc_lens, beam)
        for b, r in enumerate(pb):
            out["nbest_n%d" % b] = np.array(len(r.nbest))
            for i, (h, s, t) in enumerate(zip(r.nbest, r.nbest_scores, r.nbest_times)):
                out["nbest%d_%d" % (b, i)] = np.array(h, dtype=np.int32)
                out["nbest_time%d_%d" % (b, i)] = np.array(t, dtype=np.int32)
            out["nbest_scores%d" % b] = np.array(r.nbest_scores, dtype=np.float64)
        rw = cfg["model_conf"].get("reverse_weight", 0.0)
        rs = attention_rescoring(model, pb, enc, enc_lens, ctc_weight, rw)
        for b, r in enumerate(rs):
            out["resc_tokens%d" % b] = np.array(r.tokens, dtype=np.int32)
            out["resc_score%d" % b] = np.array(r.score, dtype=np.float64)
            out["resc_conf%d" % b] = np.array(r.confidence, dtype=np.float64)
        if cfg["encoder_conf"]["use_dynamic_chunk"]:
            enc_c, _ = model.encoder(xs, lens, decoding_chunk_size=chunk[0], num_decoding_left_chunks=chunk[1])
            out["enc_out_chunk"] = enc_c.numpy()
            out["chunk"] = np.array(chunk)
            if stream:
                # streaming: forward_chunk over utterance 0 (encoder.py:302-362), chunk 4 / 2 left chunks
                ys, _ = model.encoder.forward_chunk_by_chunk(xs[0:1, :lens[0]], chunk[0], chunk[1])
                out["stream_out"] = ys.numpy()
                att = torch.zeros(0, 0, 0, 0)
                cnn = torch.zeros(0, 0, 0, 0)
                win = (chunk[0] - 1) * 4 + 7
                y, att, cnn = model.encoder.forward_chunk(xs[0:1, :win], 0, chunk[0] * chunk[1], att, cnn)
                y2, att2, cnn2 = model.encoder.forward_chunk(xs[0:1, 4 * chunk[0]:4 * chunk[0] + win], y.size(1),
                                                             chunk[0] * chunk[1], att, cnn)
                out["stream_y1"], out["stream_att1"], out["stream_cnn1"] = y.numpy(), att.numpy(), cnn.numpy()
                out["stream_y2"], out["stream_att2"], out["stream_cnn2"] = y2.numpy(), att2.numpy(), cnn2.numpy()
    np.savez_compressed(os.path.join(GOLD, name + ".npz"), **out)
    toks = [len(out["greedy%d" % b]) for b in range(len(ns))]
    blank = float((logp.argmax(-1) == 0).float().mean())
    print(name, "enc", tuple(enc.shape), "greedy tokens", toks, "blank frac %.2f" % blank,
          "nbest0", out["nbest0_0"].tolist()[:12], "size %.0f KB" % (os.path.getsize(os.path.join(GOLD, name + ".npz")) / 1024))


def _ref_model(recipe):
    cfg = synth.recipe(recipe)
    sd = synth.synth_state_dict(cfg, seed=SEED)
    ref_cfg = dict(cfg, cmvn=None)
    ref_cfg.pop("cmvn_conf", None)
    model = shim.init_reference_model(ref_cfg)
    from wenet.models.transformer.cmvn import GlobalCMVN
    model.encoder.global_cmvn = GlobalCMVN(torch.zeros(80), torch.ones(80))
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected and all(k.endswith("num_batches_tracked") for k in missing)
    model.eval()
    return cfg, model


def _ref_batch(ns):
    pcm = synth.synth_pcm(len(ns), ns, seed=SEED)
    feats = [ref_fbank(pcm[b], n) for b, n in enumerate(ns)]
    lens = torch.tensor([f.shape[0] for f in feats])
    xs = torch.zeros(len(ns), int(lens.max()), 80)
    for b, f in enumerate(feats):
        xs[b, :f.shape[0]] = f
    return xs, lens


def long_goldens(name, recipe, ns, beam=10, ctc_weight=0.5, row_stride=4):
    """BASELINE-sized utterances (30 s / 17 s on the 12L/256d recipe, 10 s on 24L/512d): encoder_out rows
    [::row_stride] of the valid frames, CTC top-k (values + ids), greedy / n-best / rescoring results.  No [T', V]
    log-prob matrix (12.7 MB per 30 s utterance)."""
    torch.manual_seed(0)
    cfg, model = _ref_model(recipe)
    xs, lens = _ref_batch(ns)
    out = {"num_samples": np.array(ns), "beam": np.array(beam), "ctc_weight": np.array(ctc_weight),
           "row_stride": np.array(row_stride)}
    from wenet.models.transformer.search import (attention_rescoring, ctc_greedy_search, ctc_prefix_beam_search)
    with torch.no_grad():
        enc, mask = model.encoder(xs, lens, decoding_chunk_size=-1, num_decoding_left_chunks=-1)
        enc_lens = mask.squeeze(1).sum(1)
        out["enc_lens"] = enc_lens.numpy()
        logp = model.ctc_logprobs(enc)
        tv, ti = logp.topk(beam, dim=-1)
        g = ctc_greedy_search(logp, enc_lens)
        pb = ctc_prefix_beam_search(logp, enc_lens, beam)
        rw = cfg["model_conf"].get("reverse_weight", 0.0)
        rs = attention_rescoring(model, pb, enc, enc_lens, ctc_weight, rw)
        for b in range(len(ns)):
            n = int(enc_lens[b])
            out["enc_rows%d" % b] = enc[b, :n:row_stride].numpy()
            out["topk_val%d" % b] = tv[b, :n].numpy()
            out["topk_idx%d" % b] = ti[b, :n].numpy().astype(np.int32)
            out["greedy%d" % b] = np.array(g[b].tokens, dtype=np.int32)
            r = pb[b]
            out["nbest_n%d" % b] = np.array(len(r.nbest))
            for i, (h, t) in enumerate(zip(r.nbest, r.nbest_times)):
                out["nbest%d_%d" % (b, i)] = np.array(h, dtype=np.int32)
                out["nbest_time%d_%d" % (b, i)] = np.array(t, dtype=np.int32)
            out["nbest_scores%d" % b] = np.array(r.nbest_scores, dtype=np.float64)
            out["resc_tokens%d" % b] = np.array(rs[b].tokens, dtype=np.int32)
            out["resc_score%d" % b] = np.array(rs[b].score, dtype=np.float64)
            out["resc_conf%d" % b] = np.array(rs[b].confidence, dtype=np.float64)
    path = os.path.join(GOLD, name + ".npz")
    np.savez_compressed(path, **out)
    print(name, "enc_lens", enc_lens.tolist(), "greedy tokens", [len(out["greedy%d" % b]) for b in range(len(ns))],
          "blank frac %.2f" % float((ti[..., 0] == 0).float().mean()), "size %.0f KB" % (os.path.getsize(path) / 1024))


def stream_goldens(name, recipe, n_samples, chunk=16, left=4, row_stride=2, cache_layers=(0, -1)):
    """BASELINE configs[3]: encoder.forward_chunk with chunk_size 16 / num_left_chunks 4 over a whole utterance
    (>= 20 chunks) by the reference's own forward_chunk_by_chunk loop (encoder.py:302-362), plus the caches after
    the last chunk (attention cache of the first / last layer only, to keep the fixture small)."""
    torch.manual_seed(0)
    cfg, model = _ref_model(recipe)
    xs, lens = _ref_batch([n_samples])
    with torch.no_grad():
        ys, _ = model.encoder.forward_chunk_by_chunk(xs[0:1, :lens[0]], chunk, left)
        # the same loop by hand, to capture the final caches
        win, stride = (chunk - 1) * 4 + 7, 4 * chunk
        att = torch.zeros(0, 0, 0, 0)
        cnn = torch.zeros(0, 0, 0, 0)
        off, outs = 0, []
        for cur in range(0, int(lens[0]) - 7 + 1, stride):
            y, att, cnn = model.encoder.forward_chunk(xs[0:1, cur:min(cur + win, int(lens[0]))], off, chunk * left, att, cnn)
            outs.append(y)
            off += y.size(1)
        assert torch.equal(torch.cat(outs, 1), ys)
    out = {"num_samples": np.array(n_samples), "chunk": np.array([chunk, left]), "row_stride": np.array(row_stride),
           "n_chunks": np.array(len(outs)), "n_out": np.array(ys.size(1)),
           "stream_rows": ys[0, ::row_stride].numpy(), "att_last": att[list(cache_layers)].numpy(),
           "att_layers": np.array([c % att.size(0) for c in cache_layers]), "cnn_last": cnn.numpy()}
    path = os.path.join(GOLD, name + ".npz")
    np.savez_compressed(path, **out)
    print(name, "chunks", len(outs), "frames", ys.size(1), "size %.0f KB" % (os.path.getsize(path) / 1024))


def attention_goldens(name, recipe, ns, beam=4, length_penalty=0.0):
    """decode mode "attention" (asr_model.py:315-318 -> search.py:252-371) of a Conformer recipe: the reference's best
    hypothesis per utterance on the reference's own encoder output."""
    cfg, model = _ref_model(recipe)
    xs, lens = _ref_batch(ns)
    out = {"num_samples": np.array(ns), "beam": np.array(beam), "length_penalty": np.array(length_penalty)}
    with torch.no_grad():
        res = model.decode(["attention"], xs, lens, beam_size=beam, length_penalty=length_penalty)["attention"]
    for b, r in enumerate(res):
        out["att%d" % b] = np.array(r.tokens, dtype=np.int32)
    path = os.path.join(GOLD, name + ".npz")
    np.savez_compressed(path, **out)
    print(name, "attention tokens", [len(r.tokens) for r in res], res[0].tokens[:10])


def whisper_goldens(name="whisper_tiny", recipe="whisper_tiny", ns=(32000 + 77, 24000, 11200), beam=4):
    """Whisper (wenet/models/whisper/whisper.py) at test size: the reference's compute_log_mel_spectrogram (with the
    restated slaney filterbank injected as librosa.filters.mel - librosa is not installed), encoder output on the zero
    padded batch, and attention decoding with the forced [sot, language, task, no_timestamps] prefix."""
    import types
    from oracle import wenet_oracle as O
    cfg = synth.recipe(recipe)
    sd = synth.synth_state_dict(cfg, seed=SEED)
    model = shim.init_reference_model(dict(cfg))
    model.load_state_dict(sd, strict=True)
    import wenet.dataset.processor as processor
    sys.modules["librosa"].filters = types.SimpleNamespace(
        mel=lambda sr, n_fft, n_mels: O.slaney_mel_filters(sr, n_fft, n_mels).numpy())
    mel = cfg["input_dim"]
    pcm = synth.synth_pcm(len(ns), list(ns), seed=SEED)
    feats = []
    for b, n in enumerate(ns):
        wav = (pcm[b, :n].float() / 32768.0).unsqueeze(0)
        feats.append(processor.compute_log_mel_spectrogram(dict(key="k", wav=wav, sample_rate=16000), n_fft=400, hop_length=160,
                                                           num_mel_bins=mel)["feat"])
    lens = torch.tensor([f.shape[0] for f in feats])
    xs = torch.zeros(len(ns), int(lens.max()), mel)
    for b, f in enumerate(feats):
        xs[b, :f.shape[0]] = f
    infos = {"tasks": ["transcribe", "translate", "transcribe"][:len(ns)], "langs": ["en", "zh", "zh"][:len(ns)]}
    out = {"num_samples": np.array(ns), "beam": np.array(beam), "feats": xs.numpy(), "feat_lens": lens.numpy(),
           "tasks": np.array(infos["tasks"]), "langs": np.array(infos["langs"])}
    with torch.no_grad():
        enc, mask = model.encoder(xs, lens)
        out["enc_out"] = enc.numpy()
        out["enc_lens"] = mask.squeeze(1).sum(1).numpy()
        res = model.decode(["attention"], xs, lens, beam_size=beam, infos=infos)["attention"]
        for b, r in enumerate(res):
            out["att%d" % b] = np.array(r.tokens, dtype=np.int32)
        # odd padded length: the other parity of subsampling.py:171
        xs_odd = xs[:, :xs.shape[1] - 1]
        lens_odd = torch.minimum(lens, torch.tensor(xs_odd.shape[1]))
        enc_o, mask_o = model.encoder(xs_odd, lens_odd)
        out["enc_out_odd"] = enc_o.numpy()
        out["enc_lens_odd"] = mask_o.squeeze(1).sum(1).numpy()
    path = os.path.join(GOLD, name + ".npz")
    np.savez_compressed(path, **out)
    print(name, "feats", tuple(xs.shape), "enc", tuple(enc.shape), "attention tokens", [len(r.tokens) for r in res],
          "size %.0f KB" % (os.path.getsize(path) / 1024))


def _ref_exe(name):
    """oracle/_ref/<name>, built from the reference's C++ sources by oracle/Makefile"""
    r = subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), "REF=" + shim.REFERENCE_ROOT], capture_output=True,
                       text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    return os.path.join(ROOT, "oracle", "_ref", name)


def _run(exe, *args, stdin=None):
    r = subprocess.run([exe] + [str(a) for a in args], input=stdin, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    return r.stdout


def _cxx_search(blocks):
    """the reference's C++ CtcPrefixBeamSearch (oracle/cxx/ctc_search_ref_main.cc) on a list of (logp [T, V], beam):
    per block the n-best as [score, tokens, times]"""
    text = ""
    for lp, beam in blocks:
        text += "%d %d %d\n" % (lp.shape[0], lp.shape[1], beam)
        text += "\n".join(" ".join("%.9g" % x for x in row) for row in lp.tolist()) + "\n"
    lines, out, i = _run(_ref_exe("ctc_search_ref"), stdin=text).splitlines(), [], 0
    for _ in blocks:
        n = int(lines[i])
        i += 1
        hyps = []
        for _k in range(n):
            a, b, c = lines[i].split("|")
            i += 1
            hyps.append([float(a.split()[0]), [int(x) for x in b.split()], [int(x) for x in c.split()]])
        out.append(hyps)
    return out


def _search_json(res):
    return [dict(nbest=[list(x) for x in r.nbest], nbest_scores=list(r.nbest_scores), nbest_times=[list(x) for x in r.nbest_times])
            for r in res]


def pin_goldens(name="oracle_pin"):
    """What tests/test_oracle_pin.py (and two checks in test_cpu.py / test_ops_gpu.py) compare the oracle with: the
    reference's outputs - its Python modules, and its C++ front-end / CTC prefix beam search compiled into oracle/_ref -
    on the inputs that test module builds from seeds.  Ragged results are stored as JSON strings."""
    import json
    import tempfile
    import types
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import test_oracle_pin as T
    from oracle import wenet_oracle as O
    js = lambda x: np.array(json.dumps(x))     # noqa: E731
    out = {}
    # C++ front-end: slaney filterbank and mel scale, Kaldi and Whisper fbank of 2 s of noise
    fb = _ref_exe("fbank_ref")
    for bins in (128, 80):
        W = np.zeros((bins, 256), dtype=np.float32)
        for line in _run(fb, "filters", "slaney", bins, 16000, 400, 0).splitlines():
            p = line.split()
            b, first, n = int(p[0]), int(p[1]), int(p[2])
            W[b, first:first + n] = [float(x) for x in p[3:3 + n]]
        out["slaney_filters%d" % bins] = W
    out["slaney_melscale"] = np.array([[float(f)] + [float(x) for x in line.split()[1:]] for f, line in
                                       zip(T.MELSCALE_HZ, _run(fb, "melscale", "slaney", *T.MELSCALE_HZ).splitlines())])
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "pcm.f32")
        with open(path, "wb") as f:
            f.write(T.noise_2s().numpy().astype("<f4").tobytes())
        for key, conf, bins in (("fbank_kaldi80", "kaldi", 80), ("fbank_whisper128", "whisper", 128)):
            out[key] = np.array([[float(x) for x in l.split()] for l in _run(fb, "fbank", conf, bins, path).splitlines()],
                                dtype=np.float32)
    # C++ and Python CTC prefix beam search: the known-answer test and the 40 random posterior matrices
    out["cxx_search_kat"] = js(_cxx_search([(torch.tensor(T.KAT_PROBS).log(), 3)])[0])
    shim.install()
    from wenet.models.transformer.search import (DecodeResult, attention_beam_search, attention_rescoring,
                                                 ctc_greedy_search, ctc_prefix_beam_search)
    blocks, py = [], []
    for lp, lens, beam in T.random_posteriors():
        blocks += [(lp[b, :int(lens[b])], beam) for b in range(lp.shape[0])]
        s = _search_json(ctc_prefix_beam_search(lp, lens, beam))
        py.append(dict(nbest=[r["nbest"] for r in s], nbest_scores=[r["nbest_scores"] for r in s],
                       nbest_times=[r["nbest_times"] for r in s], greedy=[r.tokens for r in ctc_greedy_search(lp, lens)]))
    out["cxx_search_random"] = js(_cxx_search(blocks))
    out["py_search_random"] = js(py)

    def model_of(cfg, sd):
        model = shim.init_reference_model(dict(cfg))
        missing, unexpected = model.load_state_dict(sd, strict=False)
        assert not unexpected and all(k.endswith("num_batches_tracked") for k in missing), (missing, unexpected)
        return model.eval()

    # encoder / CTC / searches / rescoring / streaming of the two tiny Conformer variants
    for variant in ("u2pp", "nonstream_bn"):
        cfg, p = T.pin_model(variant)
        model = model_of(cfg, p)
        assert model.sos_symbol() == model.eos_symbol() == cfg["output_dim"] - 1
        k = "match_%s_" % variant
        xs, lens = T.randn(777, 2, 131, 80), torch.tensor([131, 90])
        with torch.no_grad():
            enc, mask = model.encoder(xs, lens, decoding_chunk_size=-1, num_decoding_left_chunks=-1)
            out[k + "enc_out"], out[k + "enc_mask"] = enc.numpy(), mask.numpy()
            if variant == "u2pp":
                out[k + "enc_out_chunk4_left2"] = model.encoder(xs, lens, decoding_chunk_size=4, num_decoding_left_chunks=2)[0].numpy()
                att = cnn = torch.zeros(0, 0, 0, 0)
                off = 0
                for j, s in enumerate(T.STREAM_STARTS):
                    y, att, cnn = model.encoder.forward_chunk(xs[0:1, s:s + 19], off, 8, att, cnn)
                    off += y.size(1)
                    out[k + "stream_y%d" % j], out[k + "stream_att%d" % j], out[k + "stream_cnn%d" % j] = \
                        y.numpy(), att.numpy(), cnn.numpy()
            lp = model.ctc_logprobs(enc)
            out[k + "ctc_logp"] = lp.numpy()
            el = mask.squeeze(1).sum(1)
            out[k + "greedy"] = js([r.tokens for r in ctc_greedy_search(lp, el)])
            rb = ctc_prefix_beam_search(lp, el, 4)
            out[k + "beam"] = js(_search_json(rb))
            rs = attention_rescoring(model, rb, enc, el, 0.5, 0.3 if variant == "u2pp" else 0.0)
            out[k + "rescoring"] = js([[list(r.tokens), float(r.score)] for r in rs])
    cfg, p = T.pin_model("u2pp")
    model = model_of(cfg, p)
    for chunk, left in T.CHUNK_SETTINGS:
        k = "chunk%d_left%d_" % (chunk, left)
        xs, lens = T.randn(777, 2, 99, 80), torch.tensor([99, 58])
        with torch.no_grad():
            r, rm = model.encoder(xs, lens, decoding_chunk_size=chunk, num_decoding_left_chunks=left)
            out[k + "enc_out"], out[k + "enc_mask"] = r.numpy(), rm.numpy()
            out[k + "stream"] = model.encoder.forward_chunk_by_chunk(xs[:1], chunk, left)[0].numpy()
    enc, lens = T.randn(3, 3, 17, 128), torch.tensor([17, 9, 4])
    for cw, rw in T.RESCORING_WEIGHTS:
        ref_in = [DecodeResult(tokens=n[0], nbest=[tuple(h) for h in n], nbest_scores=sc, nbest_times=[[0] * len(h) for h in n])
                  for n, sc in zip(T.RESCORING_NBEST, T.RESCORING_SCORES)]
        with torch.no_grad():
            rs = attention_rescoring(model, ref_in, enc, lens, cw, rw)
        out["rescoring_ctc%g_rev%g" % (cw, rw)] = js([[list(r.tokens), float(r.score)] for r in rs])
    # context biasing: the reference's ContextGraph, flattened, and its biased search
    from wenet.utils.context_graph import ContextGraph
    from wenet_b200 import context as CX
    with tempfile.TemporaryDirectory() as td:
        f = os.path.join(td, "ctx.txt")
        with open(f, "w") as fh:
            fh.write("\n".join(T.CONTEXT_WORDS) + "\n")
        cg = ContextGraph(f, T.context_symbols(), None, 3.0)
    arr = CX.flatten(cg)
    for n in T.CONTEXT_FIELDS:
        out["context_" + n] = np.asarray(getattr(arr, n))
    lp, lens = T.context_posteriors()
    out["context_search"] = js(_search_json(ctc_prefix_beam_search(lp, lens, 6, cg, 0)))
    # decode mode "attention" of the tiny U2++ recipe
    cfg = synth.recipe("tiny")
    sd = synth.synth_state_dict(cfg, seed=SEED)
    model = model_of(dict(cfg, cmvn=None), {k: v for k, v in sd.items() if not k.startswith("encoder.global_cmvn")})
    enc, lens = T.randn(5, 2, 21, 128), torch.tensor([21, 13])
    mask = ~O.make_pad_mask(lens, 21).unsqueeze(1)
    with torch.no_grad():
        out["attention_conformer"] = js([[list(r.tokens) for r in attention_beam_search(model, enc, mask, beam, lpen)]
                                         for beam, lpen in T.ATTENTION_SETTINGS])
    # Whisper: log-mel (restated slaney filterbank injected as librosa.filters.mel), encoder, attention decoding
    cfg = synth.recipe("whisper_tiny")
    model = shim.init_reference_model(dict(cfg))
    model.load_state_dict(synth.synth_state_dict(cfg, seed=SEED), strict=True)
    model.eval()
    assert model.eos == cfg["tokenizer_conf"]["special_tokens"]["eot"]
    import wenet.dataset.processor as processor
    sys.modules["librosa"].filters = types.SimpleNamespace(
        mel=lambda sr, n_fft, n_mels: O.slaney_mel_filters(sr, n_fft, n_mels).numpy())
    pcm, batches = T.whisper_pin_inputs()
    out["whisper_logmel"] = processor.compute_log_mel_spectrogram(dict(key="k", wav=pcm.unsqueeze(0), sample_rate=16000),
                                                                  n_fft=400, hop_length=160, num_mel_bins=32)["feat"].numpy()
    with torch.no_grad():
        for (Tn, _), (xs, xl) in zip(T.WHISPER_LENS, batches):
            r_out, r_mask = model.encoder(xs, xl)
            out["whisper_enc_out%d" % Tn], out["whisper_enc_mask%d" % Tn] = r_out.numpy(), r_mask.numpy()
        out["whisper_attention"] = js([[list(r.tokens) for r in attention_beam_search(model, r_out, r_mask, beam, lpen, T.WHISPER_INFOS)]
                                       for beam, lpen in T.WHISPER_SETTINGS])
    # the reference's forced Whisper prefix (add_whisper_tokens) for tests/test_cpu.py
    from wenet.utils.common import add_whisper_tokens
    ys_in, _ = add_whisper_tokens(cfg["tokenizer_conf"]["special_tokens"], torch.ones(2, 0, dtype=torch.long), -1,
                                  tasks=["transcribe", "translate"], no_timestamp=True, langs=["zh", "en"], use_prev=False)
    out["whisper_prefix"] = ys_in.numpy()
    path = os.path.join(GOLD, name + ".npz")
    np.savez_compressed(path, **out)
    print(name, len(out), "arrays, size %.0f KB" % (os.path.getsize(path) / 1024))


if __name__ == "__main__":
    os.makedirs(GOLD, exist_ok=True)
    which = sys.argv[1:] or ["fbank", "tiny", "tiny_bn", "u2pp_small", "u2pp_small_long", "u2pp_large_10s",
                             "u2pp_small_stream", "tiny_attention", "whisper_tiny", "oracle_pin"]
    if "oracle_pin" in which:
        pin_goldens()
    if "fbank" in which:
        fbank_goldens()
    if "tiny" in which:
        model_goldens("tiny", "tiny", [32000 + 123, 20800, 48000])
    if "tiny_bn" in which:
        model_goldens("tiny_bn", "tiny_bn", [32000 + 123, 20800, 48000], stream=False)
    if "u2pp_small" in which:
        model_goldens("u2pp_small", "u2pp_small", [48000, 30000], beam=10, store_logp=False, chunk=(16, 4), stream=False)
    if "u2pp_small_long" in which:      # BASELINE configs[1] utterance size: 30 s + a ragged 17 s companion
        long_goldens("u2pp_small_long", "u2pp_small", [480000, 272000], beam=10, row_stride=4)
    if "u2pp_large_10s" in which:       # BASELINE configs[2] model (24L/512d/8h) at depth
        long_goldens("u2pp_large_10s", "u2pp_large", [160000], beam=10, row_stride=2)
    if "tiny_attention" in which:       # decode mode "attention" on the test-sized recipes
        attention_goldens("tiny_attention", "tiny", [32000 + 123, 20800, 48000], beam=4)
        attention_goldens("tiny_bn_attention", "tiny_bn", [32000 + 123, 20800, 48000], beam=3, length_penalty=0.5)
    if "whisper_tiny" in which:         # SURVEY section 8f-1 at test size
        whisper_goldens()
    if "u2pp_small_stream" in which:    # BASELINE configs[3]: chunk 16 / left 4, 21 chunks on the 12-layer model
        stream_goldens("u2pp_small_stream", "u2pp_small", 224000)
