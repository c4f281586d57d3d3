"""CPU-only suite (no GPU, no reference tree needed): oracle vs committed golden vectors, host logic,
C-ABI surface, multi-process sharding over gloo.  Runs in a few minutes."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from helpers import SEED, batch_inputs, decoder_cfg, err, load_golden, oracle_cfg
from oracle import wenet_oracle as O
from wenet_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------ C ABI surface
def test_library_exports_every_declared_symbol():
    from wenet_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "wenet_b200.h")).read()
    declared = set(re.findall(r"\b(wb_[a-z0-9_]+)\s*\(", hdr))
    declared -= {"wb_stream_t"}
    assert declared, "no declarations parsed"
    assert declared == set(_lib.EXPORTED_SYMBOLS), declared ^ set(_lib.EXPORTED_SYMBOLS)
    lib = _lib.load()  # raises if the .so is missing or lacks a symbol (getattr on each prototype)
    for name in declared:
        assert getattr(lib, name) is not None
    assert b"sm_100a" in lib.wb_version()


def test_c_abi_rejects_bad_arguments_with_status_and_message():
    """Every compute entry point validates its handle / pointers before touching CUDA: a negative wb_status and a
    wb_last_error() message, never a crash (include/wenet_b200.h: error convention).  No GPU is needed for this."""
    import ctypes as C
    from wenet_b200 import _lib
    lib = _lib.load()
    NOT_LOADED, BAD_ARG = -4, -1
    null = None
    steps = C.c_int32(0)
    calls = {
        "wb_attention_beam_search": (NOT_LOADED, [null, null, 0, null, null, 1, 10, null, 1, 0, 8, 0.0, null, 8, null, null,
                                                  C.byref(steps), null, 0, null]),
        "wb_whisper_encoder_forward": (NOT_LOADED, [null, null, 0, null, 1, 3000, null, null, null, null, null, 0, null]),
        "wb_encoder_forward_chunk_batch": (NOT_LOADED, [null, null, 67, 2, null, 64, null, 0, null, null, null, null, None, None,
                                                        null, 0, null]),
        "wb_encoder_forward_chunk_batch_static": (NOT_LOADED, [null, null, 67, 2, null, 64, null, 0, null, null, null, null, null,
                                                               0, null]),
        "wb_logmel_forward": (BAD_ARG, [null, null, 0, null, 1, null, 0, 0, null, null]),
    }
    for name, (want, args) in calls.items():
        rc = getattr(lib, name)(*args)
        assert rc == want, (name, rc)
        msg = lib.wb_last_error().decode()
        assert msg and name.replace("wb_", "").replace("encoder_forward_chunk", "forward_chunk").split(":")[0] in msg, (name, msg)
    out = C.c_void_p()
    assert lib.wb_logmel_create(C.byref(out), 400, 160, 128, null, null) == BAD_ARG
    # the size queries answer 0 for a null handle instead of dereferencing it
    assert lib.wb_attention_beam_workspace_bytes(null, 100, 1, 10, 8) == 0
    assert lib.wb_encoder_chunk_batch_workspace_bytes(null, 67, 0, 2) == 0
    assert lib.wb_whisper_encoder_workspace_bytes(null, 1, null, 3000) == 0


def test_bench_reference_arm_prints_one_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside the GPU arm): exactly one JSON line on stdout with
    the contract's keys, the reference (or, without it, the pinned port) timed on host cores, no GPU involved."""
    import json
    import subprocess
    import sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout[-2000:]
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["gpu_launches"] == 0 and d["value"] > 0 and d["unit"] == "audio-s/s"
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    with open(os.path.join(ROOT, "BASELINE.json")) as f:
        assert d["metric"] == json.load(f)["metric"]


def test_bench_dump_outputs_layout(tmp_path):
    """`bench.py --dump-outputs DIR`: the decode results of one step as float64 .npy arrays (ragged rows padded with -1,
    lengths alongside, n-best lists flattened over hypotheses), fields a mode leaves empty omitted, and a fixed seeded
    sample of the utterances when the arrays would exceed the size limit."""
    sys.path.insert(0, ROOT)
    import bench
    from wenet_b200.search import DecodeResult
    res = [DecodeResult([3, 4, 5], score=-1.5, confidence=0.5, times=[0, 2, 4], nbest=[(3, 4, 5), (3,)],
                        nbest_scores=[-1.5, -2.0], nbest_times=[[0, 2, 4], [0]]),
           DecodeResult([], score=-0.25, times=[], nbest=[()], nbest_scores=[-0.25], nbest_times=[[]])]
    bench.dump_outputs(res, str(tmp_path / "a"))
    a = {f[:-4]: np.load(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")}
    assert sorted(a) == ["confidence", "nbest", "nbest_count", "nbest_lengths", "nbest_scores", "nbest_times", "score",
                         "times", "times_lengths", "tokens", "tokens_lengths", "utterance"]
    assert all(v.dtype == np.float64 for v in a.values())
    assert a["tokens"].tolist() == [[3, 4, 5], [-1, -1, -1]] and a["tokens_lengths"].tolist() == [3, 0]
    assert a["nbest"].tolist() == [[3, 4, 5], [3, -1, -1], [-1, -1, -1]] and a["nbest_count"].tolist() == [2, 1]
    assert a["nbest_scores"].tolist() == [-1.5, -2.0, -0.25] and a["score"].tolist() == [-1.5, -0.25]
    for d in ("b", "c"):
        bench.dump_outputs(res * 8, str(tmp_path / d), limit=600)
    b = {f[:-4]: np.load(tmp_path / "b" / f) for f in os.listdir(tmp_path / "b")}
    assert np.array_equal(b["utterance"], np.load(tmp_path / "c" / "utterance.npy")) and 1 <= len(b["utterance"]) < 16
    assert sum(v.nbytes for k, v in b.items() if k != "utterance") <= 600
    assert b["score"].tolist() == [res[int(i) % 2].score for i in b["utterance"]]


def test_bench_reference_arm_under_torchrun_two_ranks():
    """The driver launches the reference arm exactly like the GPU arm: under torchrun for N > 1.  Rank 0 alone runs and
    prints the line, the other rank exits 0 without work."""
    import json
    import subprocess
    import sys
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29531", os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                        "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip().startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 2 and d["value"] > 0


def test_no_cpu_fallback():
    """Without a CUDA device the product path must fail loudly, never route to the oracle."""
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from wenet_b200 import _lib
    from wenet_b200.asr_model import B200ASRModel
    cfg = synth.recipe("tiny")
    with pytest.raises(_lib.WbError):
        B200ASRModel(cfg, synth.synth_state_dict(cfg))
    import wenet_b200
    src = ""
    for f in os.listdir(os.path.dirname(wenet_b200.__file__)):
        if f.endswith(".py"):
            src += open(os.path.join(os.path.dirname(wenet_b200.__file__), f)).read()
    assert "import oracle" not in src and "from oracle" not in src


# ------------------------------------------------------------------ oracle vs golden fixtures
def test_oracle_fbank_vs_golden():
    g = load_golden("fbank")
    ns = g["num_samples"].tolist()
    pcm = synth.synth_pcm(len(ns), ns, seed=SEED)
    for b, n in enumerate(ns):
        got = O.fbank(pcm[b, :n].float())
        ref = torch.from_numpy(g["feat%d" % b])
        assert got.shape == ref.shape
        assert err(got, ref)[0] < 1e-4


@pytest.mark.parametrize("name", ["tiny", "tiny_bn"])
def test_oracle_model_vs_golden(name):
    """The oracle restatement on regenerated synthetic weights reproduces what the unmodified reference
    produced in the build container (also proves synth.py is deterministic across boxes)."""
    g = load_golden(name)
    cfg = synth.recipe(name)
    sd = synth.synth_state_dict(cfg, seed=SEED)
    ns = g["num_samples"].tolist()
    _, xs, lens = batch_inputs(ns, lambda p: O.fbank(p.float()))
    el = g["enc_lens"].tolist()
    with torch.no_grad():
        enc, mask = O.encoder_forward(sd, oracle_cfg(cfg, sd), xs, lens)
        assert mask.squeeze(1).sum(1).tolist() == el
        for b, n in enumerate(el):
            assert err(enc[b, :n], torch.from_numpy(g["enc_out"][b, :n]))[0] < 5e-4
        lp = O.ctc_logprobs(sd, enc)
        for b, n in enumerate(el):
            assert err(lp[b, :n], torch.from_numpy(g["ctc_logp"][b, :n]))[0] < 2e-3
        ref_lp = torch.from_numpy(g["ctc_logp"])
        assert [list(x) for x in O.ctc_greedy_search(ref_lp, torch.tensor(el))] == \
            [g["greedy%d" % b].tolist() for b in range(len(el))]
        beam = int(g["beam"])
        pb = O.ctc_prefix_beam_search(ref_lp, torch.tensor(el), beam)
        for b, r in enumerate(pb):
            n = int(g["nbest_n%d" % b])
            assert r["nbest"] == [g["nbest%d_%d" % (b, i)].tolist() for i in range(n)]
            assert r["nbest_times"] == [g["nbest_time%d_%d" % (b, i)].tolist() for i in range(n)]
            assert np.allclose(r["nbest_scores"], g["nbest_scores%d" % b], rtol=0, atol=1e-12)
        rw = cfg["model_conf"].get("reverse_weight", 0.0)
        rs = O.attention_rescoring(sd, decoder_cfg(cfg), pb, torch.from_numpy(g["enc_out"]), torch.tensor(el),
                                   cfg["output_dim"] - 1, cfg["output_dim"] - 1, float(g["ctc_weight"]), rw)
        for b, r in enumerate(rs):
            assert r["tokens"] == g["resc_tokens%d" % b].tolist()
            assert abs(r["best_score"] - float(g["resc_score%d" % b])) < 1e-3
        if "stream_y1" in g:
            c, l = [int(v) for v in g["chunk"]]
            win = (c - 1) * 4 + 7
            e = oracle_cfg(cfg, sd)
            y, att, cnn = O.encoder_forward_chunk(sd, e, xs[0:1, :win], 0, c * l, torch.zeros(0, 0, 0, 0),
                                                  torch.zeros(0, 0, 0, 0))
            assert err(y, torch.from_numpy(g["stream_y1"]))[0] < 5e-4
            y2, att2, cnn2 = O.encoder_forward_chunk(sd, e, xs[0:1, 4 * c:4 * c + win], y.size(1), c * l, att, cnn)
            assert err(y2, torch.from_numpy(g["stream_y2"]))[0] < 5e-4
            assert err(att2, torch.from_numpy(g["stream_att2"]))[0] < 5e-4
            assert err(cnn2, torch.from_numpy(g["stream_cnn2"]))[0] < 5e-4


def test_oracle_bf16_emulation_is_within_reference_bf16_yardstick():
    """The operand-rounding model of the GPU path stays inside the reference's own bf16 error budget."""
    cfg = synth.recipe("tiny")
    sd = synth.synth_state_dict(cfg, seed=SEED)
    _, xs, lens = batch_inputs([32000, 20000], lambda p: O.fbank(p.float()))
    with torch.no_grad():
        a, m = O.encoder_forward(sd, oracle_cfg(cfg, sd), xs, lens)
        b, _ = O.encoder_forward(sd, oracle_cfg(cfg, sd), xs, lens, quant=O.bf16_round)
    n = int(m[1].sum())
    mx, mn = err(a[1, :n], b[1, :n])
    assert mx < 5.9e-2 and mn < 8.2e-3


# ------------------------------------------------------------------ host logic
def test_packer_layouts():
    from wenet_b200.weights import ModelSpec, interleave_glu, pack_state_dict, split3_weight
    cfg = synth.recipe("tiny")
    sd = synth.synth_state_dict(cfg, seed=SEED)
    spec = ModelSpec(cfg)
    p = pack_state_dict(spec, sd)
    d, F2 = 128, 19
    # embed.out column permutation: reference flattens (c, f), this build (f, c)
    x = torch.randn(3, d, F2)                       # (row, c, f)
    ref = torch.nn.functional.linear(x.reshape(3, d * F2), sd["encoder.embed.out.0.weight"].to(torch.bfloat16).float())
    got = torch.nn.functional.linear(x.permute(0, 2, 1).reshape(3, F2 * d), p["embed.out.w"].float())
    assert torch.allclose(ref, got, atol=1e-5)
    # conv2 im2col order (kh, kw, c_in)
    w = sd["encoder.embed.conv.2.weight"]
    assert torch.equal(p["embed.conv2.w"].float().view(d, 3, 3, d)[5, 1, 2, 7], w[5, 7, 1, 2].to(torch.bfloat16).float())
    # GLU interleave: value/gate pairs stay aligned
    wi, bi = interleave_glu(torch.arange(2 * d).float().unsqueeze(1), torch.arange(2 * d).float())
    assert bi[:16].tolist() == list(range(16)) and bi[16:32].tolist() == list(range(d, d + 16))
    # bf16x3 split reconstructs fp32 weights to ~2^-17
    w32 = torch.randn(8, 16)
    s3 = split3_weight(w32).float()
    assert (s3[:, :16] + s3[:, 32:] - w32).abs().max() < 2e-5 * w32.abs().max() + 1e-6
    assert torch.equal(s3[:, :16], s3[:, 16:32])
    # pad_vec = GLU(pointwise_conv1(0))
    b1 = sd["encoder.encoders.0.conv_module.pointwise_conv1.bias"]
    assert torch.allclose(p["enc.0.conv.pad_vec"], b1[:d] * torch.sigmoid(b1[d:]))


@pytest.mark.parametrize("key,val", [("input_layer", "conv2d6"), ("pos_enc_layer_type", "abs_pos"),
                                     ("selfattention_layer_type", "selfattn"), ("activation_type", "relu")])
def test_unsupported_configs_raise(key, val):
    from wenet_b200.weights import ModelSpec
    cfg = synth.recipe("tiny")
    cfg["encoder_conf"][key] = val
    with pytest.raises(NotImplementedError):
        ModelSpec(cfg)


def test_shard_partition_properties():
    from wenet_b200.shard import shard_utterances
    lens = [2998, 500, 1200, 2998, 800, 1999, 300, 2500, 999, 1500, 2998]
    for ws in (1, 2, 4, 8):
        parts = [shard_utterances(lens, ws, r) for r in range(ws)]
        assert sorted(i for p in parts for i in p) == list(range(len(lens)))
    two = [shard_utterances(lens, 2, r) for r in range(2)]
    load = [sum(lens[i] for i in p) for p in two]
    assert abs(load[0] - load[1]) < 0.2 * sum(lens)


def test_shard_over_gloo_world_size_2(tmp_path):
    """N>1 host path: two processes (gloo), each owns its shard, host-side gather of results only."""
    script = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, %r)
from wenet_b200.shard import shard_utterances
dist.init_process_group("gloo")
rank, ws = dist.get_rank(), dist.get_world_size()
lens = [2998, 500, 1200, 2998, 800, 1999, 300, 2500]
mine = shard_utterances(lens, ws, rank)
res = [None] * ws
dist.all_gather_object(res, {i: [i, lens[i] %% 7] for i in mine})      # token lists stand-in
merged = {}
for r in res: merged.update(r)
assert sorted(merged) == list(range(len(lens))), merged
secs = torch.tensor([sum(lens[i] for i in mine)], dtype=torch.float64)
dist.all_reduce(secs)
assert int(secs.item()) == sum(lens)
dist.barrier()
print("rank", rank, "ok", mine)
''' % ROOT
    f = tmp_path / "shard_gloo.py"
    f.write_text(script)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29611")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29611", str(f)],
                       capture_output=True, text=True, env=env, timeout=240)
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.count("ok") == 2


def test_prefix_share_tables_host_logic():
    """wb_prefix_share_tables (host-only part of wb_attention_rescoring): every decoder row maps to the first row of its
    utterance with the same input prefix (direction-aware), unique rows are numbered hypothesis-major, and the unique
    rows carry the right (token, position) inputs."""
    import numpy as np
    from wenet_b200 import _lib
    from wenet_b200._lib import ptr
    lib = _lib.load()
    rng = np.random.default_rng(7)
    sos = 99
    hyps_per_utt = []
    for b in range(5):
        base = rng.integers(1, 9, size=int(rng.integers(3, 12))).tolist()
        hs = [base]
        for _ in range(int(rng.integers(0, 6))):
            h = list(base)
            for _ in range(int(rng.integers(1, 3))):       # substitute / delete / insert somewhere
                p = int(rng.integers(0, len(h) + 1))
                op = int(rng.integers(0, 3))
                if op == 0 and p < len(h):
                    h[p] = int(rng.integers(1, 9))
                elif op == 1 and len(h) > 1 and p < len(h):
                    del h[p]
                else:
                    h.insert(p, int(rng.integers(1, 9)))
            hs.append(h)
        hyps_per_utt.append(hs)
    hyps_per_utt.append([[]])                               # an utterance whose only hypothesis is empty
    hyp_utt, hyp_len, hyp_tok0, toks = [], [], [], []
    for b, hs in enumerate(hyps_per_utt):
        for h in hs:
            hyp_utt.append(b)
            hyp_len.append(len(h))
            hyp_tok0.append(len(toks))
            toks.extend(h)
    i32 = lambda x: np.ascontiguousarray(np.array(x if len(x) else [0], dtype=np.int32))
    hyp_utt_a, hyp_len_a, hyp_tok0_a, toks_a = i32(hyp_utt), i32(hyp_len), i32(hyp_tok0), i32(toks)
    B, n_hyp = len(hyps_per_utt), len(hyp_utt)
    R = sum(hyp_len) + n_hyp
    flat = [h for hs in hyps_per_utt for h in hs]
    for direction in (0, 1):
        uniq = np.full(R, -1, np.int32)
        rep, tok_u, pos_u = np.full(R, -1, np.int32), np.full(R, -1, np.int32), np.full(R, -1, np.int32)
        q0, qn = np.zeros(B, np.int32), np.zeros(B, np.int32)
        U = lib.wb_prefix_share_tables(direction, B, n_hyp, ptr(hyp_utt_a), ptr(hyp_len_a), ptr(hyp_tok0_a), ptr(toks_a), sos,
                                       ptr(uniq), ptr(rep), ptr(tok_u), ptr(pos_u), ptr(q0), ptr(qn))
        assert U > 0
        # reference: dictionary from (utterance, input prefix) to unique id, in row order
        seen, want, rows = {}, [], []
        for h, (b, y) in enumerate(zip(hyp_utt, flat)):
            s = y if direction == 0 else y[::-1]
            for j in range(len(s) + 1):
                key = (b, tuple(s[:j]))
                if key not in seen:
                    seen[key] = len(seen)
                    rows.append((sos if j == 0 else s[j - 1], j))
                want.append(seen[key])
        assert U == len(seen)
        assert uniq.tolist() == want
        assert tok_u[:U].tolist() == [t for t, _ in rows] and pos_u[:U].tolist() == [j for _, j in rows]
        assert (uniq[rep[:U]] == np.arange(U)).all()
        # unique rows of an utterance are contiguous and cover [q0, q0 + qn)
        r = 0
        for b, hs in enumerate(hyps_per_utt):
            ids = set()
            for h in hs:
                ids.update(uniq[r:r + len(h) + 1].tolist())
                r += len(h) + 1
            assert ids == set(range(int(q0[b]), int(q0[b]) + int(qn[b])))
        assert int(qn.sum()) == U


def test_lazy_decode_result_matches_eager_fields():
    """LazyDecodeResult (what decode() returns) exposes the reference DecodeResult fields with the same Python types,
    materialised from the packed rows on first access; copies and pickles behave like plain objects."""
    import copy
    import pickle

    import numpy as np
    from wenet_b200.search import DecodeResult, LazyDecodeResult
    toks = np.array([[5, 6, 7, 0], [5, 9, 0, 0], [8, 8, 8, 8]], dtype=np.int32)
    times = np.array([[1, 4, 9, 0], [1, 5, 0, 0], [2, 3, 4, 6]], dtype=np.int32)
    lens = np.array([3, 2, 4], dtype=np.int32)
    r = LazyDecodeResult(-1.5, [-1.5, -2.0, -3.25], toks, times, lens, best=1, conf_fn=lambda: (0.75, [0.5, 0.25]))
    assert isinstance(r, DecodeResult)
    assert "tokens" not in r.__dict__ and "nbest" not in r.__dict__
    assert r.tokens == (5, 9) and isinstance(r.tokens, tuple) and all(isinstance(t, int) for t in r.tokens)
    assert r.times == [1, 5]
    assert r.nbest == [(5, 6, 7), (5, 9), (8, 8, 8, 8)]
    assert r.nbest_times == [[1, 4, 9], [1, 5], [2, 3, 4, 6]]
    assert r.nbest_scores == [-1.5, -2.0, -3.25] and r.score == -1.5 and r.text == ''
    assert r.confidence == 0.75 and r.tokens_confidence == [0.5, 0.25]
    assert "tokens" in r.__dict__                      # cached after the first read
    with pytest.raises(AttributeError):
        r.no_such_field
    r2 = LazyDecodeResult(0.0, [0.0], toks[:1], times[:1], lens[:1])
    assert r2.confidence == 0.0 and r2.tokens_confidence is None and r2.tokens == (5, 6, 7)
    c = copy.deepcopy(LazyDecodeResult(-1.0, [-1.0], toks, times, lens))
    assert c.nbest[2] == (8, 8, 8, 8)
    p = pickle.loads(pickle.dumps(LazyDecodeResult(-1.0, [-1.0], toks, times, lens, best=2)))
    assert p.tokens == (8, 8, 8, 8)


def test_ingest_batch_plan_and_wav_reader(tmp_path):
    """wenet_b200.ingest host logic: every utterance lands in exactly one batch, batches respect the padded-seconds
    budget and the size limit, longest first; the wav reader returns the file's int16 samples."""
    import wave
    from wenet_b200 import ingest
    rs = np.random.default_rng(3)
    ns = [int(x) for x in rs.integers(16000 * 2, 16000 * 30, size=300)]
    bs = ingest.plan_batches(ns, max_batch_seconds=600.0, max_batch_size=64)
    flat = [i for b in bs for i in b]
    assert sorted(flat) == list(range(len(ns)))
    prev_longest = None
    for b in bs:
        longest = max(ns[i] for i in b)
        assert len(b) <= 64 and (len(b) == 1 or len(b) * longest <= 600 * 16000)
        assert longest == ns[b[0]]                      # sorted by length inside and across batches
        assert prev_longest is None or longest <= prev_longest
        prev_longest = longest
    assert ingest.plan_batches([5, 5, 5], max_batch_seconds=1e9, max_batch_size=2) == [[0, 1], [2]]
    pcm = synth.synth_pcm(1, 12345, seed=SEED)[0, :12345].numpy()
    path = str(tmp_path / "a.wav")
    with wave.open(path, "wb") as w:
        w.setnchannels(1)
        w.setsampwidth(2)
        w.setframerate(16000)
        w.writeframes(pcm.astype("<i2").tobytes())
    assert ingest.wav_num_samples(path) == 12345
    assert np.array_equal(ingest.read_wav_int16(path), pcm)
    with pytest.raises(ValueError):
        ingest.read_wav_int16(path, sample_rate=8000)


def test_export_model_file_layout(tmp_path):
    """wenet_b200.export writes what runtime/b200_asr_model.cc::Read parses: magic, the wb_model_config struct, sos / eos /
    bidirectional / tensor count, then (name, dtype, numel, data) records."""
    import ctypes as C
    import struct
    from wenet_b200._lib import WbModelConfig
    from wenet_b200.export import MAGIC, export_model
    cfg = synth.recipe("tiny")
    sd = synth.synth_state_dict(cfg, seed=SEED)
    path = str(tmp_path / "m.wbm")
    n = export_model(cfg, sd, path)
    raw = open(path, "rb").read()
    assert raw[:8] == MAGIC
    c = WbModelConfig.from_buffer_copy(raw[8:8 + C.sizeof(WbModelConfig)])
    assert (c.d_model, c.heads, c.enc_layers, c.vocab, c.precise) == (128, 2, 2, 37, 0)
    off = 8 + C.sizeof(WbModelConfig)
    sos, eos, bi, cnt = struct.unpack_from("<4i", raw, off)
    assert (sos, eos, bi, cnt) == (36, 36, 1, n)
    off += 16
    seen = 0
    while off < len(raw):
        ln, = struct.unpack_from("<i", raw, off)
        name = raw[off + 4:off + 4 + ln].decode()
        dt, numel = struct.unpack_from("<iq", raw, off + 4 + ln)
        off += 4 + ln + 12 + numel * (2 if dt == 1 else 4)
        seen += 1
        assert name and numel > 0
    assert seen == n and off == len(raw)


def test_whisper_spec_and_packer_shapes():
    """Whisper configuration parsing and weight packing (host logic, no GPU): conv weights in (tap, channel) order, zero key
    bias slices, learnable decoder positions, precise mode = [hi | hi | lo] per K block."""
    import torch
    from wenet_b200 import synth
    from wenet_b200.weights import ModelSpec, pack_state_dict
    cfg = synth.recipe("whisper_tiny")
    spec = ModelSpec(cfg)
    assert (spec.arch, spec.dec_flavor, spec.dec_max_len, spec.max_pos, spec.sos, spec.eos) == (1, 1, 448, 1500, 100, 99)
    sd = synth.synth_state_dict(cfg, seed=777)
    assert "encoder.encoders.0.self_attn.linear_k.bias" not in sd          # key_bias: false
    pk = pack_state_dict(spec, sd)
    d, idim = spec.d_model, spec.input_dim
    w1 = sd["encoder.embed.conv.0.weight"]                                  # (d, idim, 3)
    assert torch.equal(pk["wenc.conv1.w"].float().view(d, 3, idim)[:, 2, :], w1[:, :, 2].to(torch.bfloat16).float())
    qb = pk["wenc.0.att.qkv.b"]
    assert qb.shape == (3 * d,) and float(qb[d:2 * d].abs().max()) == 0.0 and float(qb[:d].abs().max()) > 0.0
    assert pk["dec.left.pe"].shape == (448, d) and pk["wenc.pe"].shape == (1500, d)
    pp = pack_state_dict(spec, sd, precise=True)
    assert pp["wenc.conv1.w"].shape == (d, 9 * idim) and pp["wenc.0.ff.w1.w"].shape == (spec.ffn_dim, 3 * d)
    hi, hi2, lo = pp["wenc.0.att.out.w"].float().view(d, 3, d).unbind(1)
    w = sd["encoder.encoders.0.self_attn.linear_out.weight"]
    assert torch.equal(hi, hi2) and float((hi + lo - w).abs().max()) < 1e-5   # bf16x3: hi + lo carries 16 mantissa bits
    assert pp["dec.left.0.ff.w1.w"].shape == pk["dec.left.0.ff.w1.w"].shape   # the decoder stays bf16
    with pytest.raises(NotImplementedError):
        ModelSpec(dict(cfg, encoder_conf=dict(cfg["encoder_conf"], input_layer="conv2d")))


def test_whisper_prefix_and_mel_filters():
    """whisper_prefix == the forced start of add_whisper_tokens (common.py:198-226); slaney filterbank restatements of the
    product (numpy) and the oracle (pure Python) agree."""
    import numpy as np
    from oracle import wenet_oracle as O
    from wenet_b200 import synth
    from wenet_b200.whisper import WHISPER_LANGS, slaney_mel_filters, whisper_prefix
    st = synth.recipe("whisper_large_v3")["tokenizer_conf"]["special_tokens"]
    p = whisper_prefix(st, ["transcribe", "translate", "vad"], ["en", "zh", "yue"])
    assert p.tolist() == [[50258, 50259, 50360, 50364], [50258, 50260, 50359, 50364], [50258, 50258 + 100, 50363, 50363]]
    assert len(WHISPER_LANGS) == 100 and len(set(WHISPER_LANGS)) == 100
    a = slaney_mel_filters(16000, 400, 128)
    b = O.slaney_mel_filters(16000, 400, 128).numpy()
    assert a.shape == (128, 201) and float(np.abs(a - b).max()) < 1e-7
    # the reference's add_whisper_tokens (common.py:198-226) on the whisper_tiny tokens (oracle/make_goldens.py)
    st2 = synth.recipe("whisper_tiny")["tokenizer_conf"]["special_tokens"]
    ys_in = load_golden("oracle_pin")["whisper_prefix"]
    assert ys_in.tolist() == whisper_prefix(st2, ["transcribe", "translate"], ["zh", "en"]).tolist()
