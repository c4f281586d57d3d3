#!/usr/bin/env python
"""bench.py — RTFx (audio-seconds decoded per wall-second) of the B200 hot path.

    python bench.py --gpus N --steps K --warmup W            (torchrun launches N ranks for N > 1)
    python bench.py --impl reference --gpus N --steps K --warmup W
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR     (+ what the last timed step decoded, as .npy)

A "step" = one pass of the whole hot path over one batch of synthetic 16 kHz utterances:
fbank -> ConformerEncoder -> CTC log-softmax/top-k -> ctc_prefix_beam_search -> attention_rescoring,
ending with the token ids on the host.  Workload at N=1 (BASELINE.json configs[1] model, decoded in the
mode BASELINE.json's `metric` names): U2++ Conformer 12L/256d/4h (AISHELL-1 recipe), batch 64 x 30 s per
GPU, beam 10, attention_rescoring (which contains ctc_prefix_beam_search).  Weak scaling: every rank
decodes its own 64 x 30 s (utterances shard independently; no data-path collective).

`value`   : inputs (int16 PCM) already resident in HBM when the timed region starts.
`e2e`     : same metric through the public API with HOST (pinned) PCM: H2D copy of the batch and D2H
            of the results inside the timed region.
`roofline`: the dominant kernel family (tcgen05 GEMM) — algorithmic FLOPs / CUDA-event time measured
            live around every launch in the timed steps (wb_prof_*), against MEASURED_PEAKS.json.
`cpu_baseline`: the CPU oracle port of the reference path (oracle/wenet_oracle.py, torch-CPU ops with
            all host threads + the reference's Python search loops) on a bounded sample.
"""
import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "RTFx (audio-s/s) U2++ Conformer attention_rescoring at 1/2/4/8 B200"


def host_cores():
    """CPU cores this process may actually use: the scheduler affinity mask capped by the cgroup CPU quota
    (os.cpu_count() reports the machine, not the container)."""
    try:
        n = len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            with open(path) as f:
                parts = f.read().split()
            if path.endswith("cpu.max"):
                if parts[0] != "max":
                    n = min(n, max(1, int(float(parts[0]) / float(parts[1]) + 0.5)))
            else:
                q = int(parts[0])
                if q > 0:
                    with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f2:
                        n = min(n, max(1, int(q / float(f2.read().split()[0]) + 0.5)))
            break
        except (OSError, ValueError, IndexError):
            continue
    return max(1, n)


def _edit_distance(a, b):
    prev = list(range(len(b) + 1))
    for i, x in enumerate(a, 1):
        cur = [i]
        for j, y in enumerate(b, 1):
            cur.append(min(prev[j] + 1, cur[j - 1] + 1, prev[j - 1] + (x != y)))
        prev = cur
    return prev[-1]


def _padded(rows):
    """ragged rows -> (len(rows), longest) float64 padded with -1, and the row lengths"""
    a = np.full((len(rows), max([len(r) for r in rows] + [0])), -1.0)
    for i, r in enumerate(rows):
        a[i, :len(r)] = r
    return a, np.array([len(r) for r in rows], dtype=np.float64)


def decode_arrays(results):
    """What decode() hands its caller for one batch, as float64 arrays (token ids and frame indices are exact): per
    utterance the best hypothesis (tokens, times, per-token confidence: rows padded with -1, lengths in <name>_lengths),
    its score and confidence, and the n-best lists flattened over hypotheses in utterance order (nbest_count per
    utterance).  Fields a decoding mode leaves empty are omitted."""
    out = {"score": np.array([r.score for r in results], dtype=np.float64),
           "confidence": np.array([r.confidence for r in results], dtype=np.float64)}
    for name in ("tokens", "times", "tokens_confidence"):
        rows = [getattr(r, name) for r in results]
        if all(x is not None for x in rows):
            out[name], out[name + "_lengths"] = _padded(rows)
    if all(r.nbest is not None for r in results):
        out["nbest_count"] = np.array([len(r.nbest) for r in results], dtype=np.float64)
        out["nbest"], out["nbest_lengths"] = _padded([h for r in results for h in r.nbest])
        out["nbest_times"], _ = _padded([t for r in results for t in r.nbest_times])
        out["nbest_scores"] = np.array([s for r in results for s in r.nbest_scores], dtype=np.float64)
    return out


def dump_outputs(results, out_dir, limit=64 << 20):
    """DIR/<name>.npy for every array of decode_arrays(results), at most `limit` bytes in all: a larger batch is
    replaced by a fixed, seeded sample of its utterances (their batch indices in utterance.npy)."""
    idx = np.arange(len(results))
    arrays = decode_arrays(results)
    while sum(a.nbytes for a in arrays.values()) > limit and len(idx) > 1:
        keep = len(idx) // 2
        idx = np.sort(np.random.default_rng(0).choice(len(results), keep, replace=False))
        arrays = decode_arrays([results[i] for i in idx])
    arrays["utterance"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    print("bench.py: %d arrays (%d utterances, %d bytes) written to %s"
          % (len(arrays), len(idx), sum(a.nbytes for a in arrays.values()), out_dir), file=sys.stderr)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons every 200 ms during the timed region (pynvml, else nvidia-smi)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.stop_flag = False
        self.sm, self.reasons, self.sm_max = [], set(), None
        self.power_w, self.power_limit_w = [], None

    def run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.sm_max = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
                     0x80: "hw_power_brake_slowdown"}
            while not self.stop_flag:
                self.sm.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                try:
                    self.power_w.append(pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0)
                    if self.power_limit_w is None:
                        self.power_limit_w = pynvml.nvmlDeviceGetEnforcedPowerLimit(h) / 1000.0
                except Exception:
                    pass
                try:
                    r = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, n in names.items():
                    if r & bit:
                        self.reasons.add(n)
                time.sleep(0.2)
        except Exception:
            import subprocess
            while not self.stop_flag:
                try:
                    o = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=clocks.sm,clocks.max.sm",
                                        "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                    a, b = [float(x) for x in o.strip().split(",")]
                    self.sm.append(a)
                    self.sm_max = b
                except Exception:
                    pass
                time.sleep(0.2)

    def summary(self):
        out = {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.sm_max,
               "reasons": sorted(self.reasons), "samples": len(self.sm)}
        if self.power_w:    # board power next to the clocks: with several batches in flight the step runs AT the power limit
            out["power_w"] = float(np.median(self.power_w))
            out["power_limit_w"] = self.power_limit_w
        return out


def workload(name):
    from wenet_b200 import synth
    if name == "small":
        return dict(recipe="u2pp_small", batch=64, seconds=30.0, beam=10, ctc_weight=0.5, reverse_weight=0.3,
                    label="U2++ Conformer (AISHELL-1 12L/256d/4h), batch 64x30s per GPU, attention_rescoring "
                          "(incl. ctc_prefix_beam_search), beam 10")
    if name == "large":
        return dict(recipe="u2pp_large", batch=32, seconds=30.0, beam=10, ctc_weight=0.5, reverse_weight=0.3,
                    label="U2++ Conformer-large (WenetSpeech 24L/512d/8h), batch 32x30s per GPU, attention_rescoring")
    raise KeyError(name)


# ----------------------------------------------------------------------------------------------
# CPU oracle leg (cpu_baseline and --impl reference)
# ----------------------------------------------------------------------------------------------
def cpu_oracle_step(sd, cfg, pcm_rows, wl, want_enc=False):
    """One pass of the reference path on the CPU (oracle port): fbank -> encoder -> ctc -> prefix beam
    search -> attention rescoring, as wenet/bin/recognize.py:282-303 does per batch."""
    import torch
    from oracle import wenet_oracle as O
    e = cfg["encoder_conf"]
    ecfg = O.encoder_cfg(sd, e["attention_heads"], e["causal"], e["cnn_module_norm"])
    d = cfg["decoder_conf"]
    dcfg = dict(bidirectional=cfg["decoder"] == "bitransformer", layers=d["num_blocks"],
                r_layers=d.get("r_num_blocks", 0), heads=d["attention_heads"])
    with torch.no_grad():
        feats = [O.fbank(r.float()) for r in pcm_rows]
        lens = torch.tensor([f.shape[0] for f in feats])
        xs = torch.zeros(len(feats), int(lens.max()), 80)
        for b, f in enumerate(feats):
            xs[b, :f.shape[0]] = f
        enc, mask = O.encoder_forward(sd, ecfg, xs, lens)
        el = mask.squeeze(1).sum(1)
        lp = O.ctc_logprobs(sd, enc)
        pb = O.ctc_prefix_beam_search(lp, el, wl["beam"])
        V = cfg["output_dim"]
        rs = O.attention_rescoring(sd, dcfg, pb, enc, el, V - 1, V - 1, wl["ctc_weight"], wl["reverse_weight"])
    if want_enc:
        return [r["tokens"] for r in rs], [enc[b, :int(el[b])] for b in range(len(feats))]
    return [r["tokens"] for r in rs]


def cpu_sample(wl, n_utts, seed=777):
    import torch
    from wenet_b200 import synth
    cfg = synth.recipe(wl["recipe"])
    sd = synth.synth_state_dict(cfg, seed=seed)
    n = int(wl["seconds"] * 16000)
    pcm = synth.synth_pcm(n_utts, n, seed=seed)
    return cfg, sd, [pcm[b, :n] for b in range(n_utts)]


# The reference decodes in ONE process with torch intra-op threads (wenet/bin/recognize.py); on a many-core host
# that leaves most cores idle (and 100+ intra-op threads on these small ops is slower than 8), so the CPU arm
# runs P worker processes x T threads, one utterance per task - the way a CPU deployment would be scaled out.
_W = {}


def reference_available():
    """the UNMODIFIED reference (wenet-e2e/wenet) importable on this box: /root/reference in the build container, or its
    pip --target install under baseline/_ref, which travels with the repo snapshot"""
    from oracle import shim
    return shim.have_reference()


def _cpu_worker_init(wl_name, threads):
    import torch
    torch.set_num_threads(threads)
    wl = workload(wl_name)
    cfg, sd, rows = cpu_sample(wl, 4)
    _W.update(wl=wl, cfg=cfg, sd=sd, rows=rows, ref=None)
    if reference_available():
        # the reference's own modules and search code (wenet/bin/recognize.py:289-303 calls exactly model.decode)
        from oracle import shim
        ref_cfg = dict(cfg, cmvn=None)
        ref_cfg.pop("cmvn_conf", None)
        model = shim.init_reference_model(ref_cfg)
        from wenet.models.transformer.cmvn import GlobalCMVN
        model.encoder.global_cmvn = GlobalCMVN(torch.zeros(80), torch.ones(80))
        model.load_state_dict(sd, strict=False)
        model.eval()
        _W["ref"] = model


def reference_step(model, pcm_rows, wl):
    """the reference path itself on the CPU: processor.compute_fbank -> ASRModel.decode(attention_rescoring)"""
    import torch
    from wenet.dataset import processor
    feats = [processor.compute_fbank(dict(key="k", wav=(r.float() / 32768.0).unsqueeze(0), sample_rate=16000),
                                     num_mel_bins=80, frame_length=25, frame_shift=10, dither=0.0)["feat"] for r in pcm_rows]
    lens = torch.tensor([f.shape[0] for f in feats])
    xs = torch.zeros(len(feats), int(lens.max()), 80)
    for b, f in enumerate(feats):
        xs[b, :f.shape[0]] = f
    with torch.no_grad():
        res = model.decode(["attention_rescoring"], xs, lens, wl["beam"], ctc_weight=wl["ctc_weight"],
                           reverse_weight=wl["reverse_weight"])
    return [r.tokens for r in res["attention_rescoring"]]


def _cpu_worker_ready(i):
    return os.getpid()


def _cpu_worker_step(i):
    rows = [_W["rows"][i % len(_W["rows"])]]
    if _W["ref"] is not None:
        toks = reference_step(_W["ref"], rows, _W["wl"])
    else:
        toks = cpu_oracle_step(_W["sd"], _W["cfg"], rows, _W["wl"])
    return len(toks[0])


class CpuArm:
    """P processes x T threads running the oracle port of the reference path, one utterance per task."""

    def __init__(self, wl_name):
        import multiprocessing as mp
        ncpu = host_cores()
        self.threads = min(8, ncpu)
        self.procs = max(1, min(16, ncpu // self.threads))
        self.wl = workload(wl_name)
        self.kind = "reference" if reference_available() else "port"
        self.pool = mp.get_context("spawn").Pool(self.procs, initializer=_cpu_worker_init,
                                                 initargs=(wl_name, self.threads))
        # worker start-up (interpreter, torch import, weight synthesis) is not part of any timed step
        self.pool.map(_cpu_worker_ready, range(4 * self.procs), chunksize=1)

    def step(self, utts_per_proc=1):
        """one pass over procs x utts_per_proc utterances; returns (audio seconds, wall seconds)"""
        n = self.procs * utts_per_proc
        t0 = time.perf_counter()
        self.pool.map(_cpu_worker_step, range(n), chunksize=1)
        return n * self.wl["seconds"], time.perf_counter() - t0

    def describe(self, utts_per_proc=1):
        impl = ("the UNMODIFIED reference (wenet processor.compute_fbank + ASRModel.decode, fp32; /root/reference or its pip --target copy baseline/_ref)"
                if self.kind == "reference" else
                "oracle port of the reference path: torch-CPU ops + the reference's Python search loops")
        return ("%d x %.0f s utterance(s) per step (%d worker processes x %d threads, one utterance each), same "
                "model/mode/beam; %s; %d usable host cores (affinity / cgroup quota), os.cpu_count() = %d"
                % (self.procs * utts_per_proc, self.wl["seconds"], self.procs, self.threads, impl, host_cores(),
                   os.cpu_count() or 0))

    def close(self):
        self.pool.close()
        self.pool.join()


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    arm = CpuArm(args.workload)
    for _ in range(args.warmup):
        arm.step()
    audio = dt = 0.0
    for _ in range(args.steps):
        a, t = arm.step()
        audio += a
        dt += t
    val = audio / max(dt, 1e-9)
    sample = arm.describe()
    wl = arm.wl
    line = {"metric": METRIC, "value": val, "unit": "audio-s/s", "impl": "reference", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(args.steps, 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["label"], "recipe": wl["recipe"], "sample": sample},
            "cpu_baseline": {"value": val, "unit": "audio-s/s", "cores": host_cores(),
                             "threads_used": arm.procs * arm.threads, "kind": arm.kind, "sample": sample},
            "e2e": {"value": val, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    arm.close()
    args.emit(line)
    return 0


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="small", choices=["small", "large"])
    ap.add_argument("--batch", type=int, default=0, help="override utterances per GPU")
    ap.add_argument("--seconds", type=float, default=0.0, help="override utterance length")
    ap.add_argument("--mode", default="attention_rescoring",
                    choices=["attention_rescoring", "ctc_prefix_beam_search", "ctc_greedy_search"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-verify", action="store_true", help="skip the token / encoder_out check against the CPU oracle")
    ap.add_argument("--no-extra", action="store_true",
                    help="skip the extra block (ragged global list, configs[2] large model, configs[3] streaming latency)")
    ap.add_argument("--no-whisper", action="store_true", help="skip the Whisper-large-v3 extra (BASELINE configs[4] geometry)")
    ap.add_argument("--no-profile", action="store_true", help="skip the per-kernel CUDA-event profiler")
    ap.add_argument("--sm-reserve", type=int, default=-1, help="SMs the GEMM / FFN kernels leave free (-1: 8 when in flight > 1)")
    ap.add_argument("--inflight", type=int, default=4,
                    help="batches in flight per GPU (host threads x CUDA streams sharing one weight replica); "
                         "1 = strictly sequential steps")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the decode results of the last timed step to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    # stdout carries exactly ONE line, the JSON result: everything else that lands on fd 1 while the benchmark runs
    # (NCCL prints its version banner there from native code) is sent to stderr instead
    sys.stdout.flush()
    _json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        sys.stdout.flush()
        os.write(_json_fd, (json.dumps(line) + "\n").encode())

    args.emit = emit
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference_arm(args)

    import torch
    import torch.distributed as dist
    from wenet_b200 import _lib, synth
    from wenet_b200.asr_model import B200ASRModel
    from wenet_b200.fbank import FbankExtractor
    from wenet_b200.shard import shard_utterances

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    wl = workload(args.workload)
    if args.batch:
        wl["batch"] = args.batch
    if args.seconds:
        wl["seconds"] = args.seconds
    B, n = wl["batch"], int(wl["seconds"] * 16000)
    cfg = synth.recipe(wl["recipe"])
    sd = synth.synth_state_dict(cfg, seed=777)
    model = B200ASRModel(cfg, sd, device=dev)
    fb = FbankExtractor(80)
    lib = _lib.load()

    # global utterance list (world * B utterances of equal length) sharded without any collective
    mine = shard_utterances([int(wl["seconds"] * 100)] * (world * B), world, rank)
    assert len(mine) == B
    NROT = 3  # rotate over 3 distinct PCM batches: 3 x B x n x 2 B (184 MB at 64 x 30 s) > the 126 MB L2
    host_pcm = [synth.synth_pcm(4, n, seed=1000 * rank + r).repeat((B + 3) // 4, 1)[:B].contiguous().pin_memory()
                for r in range(NROT)]
    for r in range(NROT):   # make the rows of a batch distinct without generating 64 x 30 s three times
        host_pcm[r] += (torch.arange(B, dtype=torch.int16).unsqueeze(1) % 7)
    dev_pcm = [h.to(dev) for h in host_pcm]
    ns = torch.full((B,), n, dtype=torch.int32, device=dev)
    nframes = fb.num_frames(n)
    flens = torch.full((B,), nframes, dtype=torch.int64, device=dev)
    methods = [args.mode]

    def step(pcm_dev, mdl=None):
        feats = fb(pcm_dev, ns)
        return (mdl or model).decode(methods, feats, flens, beam_size=wl["beam"], ctc_weight=wl["ctc_weight"],
                                     reverse_weight=wl["reverse_weight"])

    # several batches in flight: one host thread + one CUDA stream + one workspace set per slot, all on the
    # same (immutable) device weights.  Hides the host-side result handling and the latency-bound search
    # kernel of one batch behind the GEMMs of the next.  A step is still one full pass over one batch.
    import threading
    n_slots = max(1, args.inflight)
    if n_slots > 1:
        sys.setswitchinterval(5e-4)   # the slot threads hand the GIL over between (GIL-releasing) C-ABI calls
    lib.wb_set_sm_reserve(args.sm_reserve if args.sm_reserve >= 0 else (8 if n_slots > 1 else 0))   # room for the other batch's search kernel (batch/8 CTAs)
    slot_models = [model] + [model.clone_shared() for _ in range(n_slots - 1)]
    slot_streams = [torch.cuda.Stream(device=dev) for _ in range(n_slots)]

    def run_steps(fn, steps, slot_models=slot_models):
        """fn(i, mdl) for i in range(steps), distributed over the slots."""
        if n_slots == 1:
            for i in range(steps):
                fn(i, slot_models[0])
            return
        nxt = [0]
        lock = threading.Lock()
        errs = []

        def worker(w):
            try:
                torch.cuda.set_device(dev)
                with torch.cuda.stream(slot_streams[w]):
                    while True:
                        with lock:
                            i = nxt[0]
                            nxt[0] += 1
                        if i >= steps:
                            break
                        fn(i, slot_models[w])
                    slot_streams[w].synchronize()
            except Exception as e:  # noqa: BLE001
                errs.append(e)

        ths = [threading.Thread(target=worker, args=(w,)) for w in range(n_slots)]
        for t in ths:
            t.start()
        for t in ths:
            t.join()
        if errs:
            raise errs[0]

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, slot_models=slot_models):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run_steps(fn, steps, slot_models)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        barrier()
        return ms

    # ---- warm-up ----
    for i in range(args.warmup):
        res = step(dev_pcm[i % NROT])
    run_steps(lambda i, mdl: step(dev_pcm[i % NROT], mdl), 2 * n_slots if n_slots > 1 else 0)   # warm every slot
    torch.cuda.synchronize()
    n_tok = sum(len(r.tokens) for r in res[args.mode])

    # ---- device-resident timing (headline `value`): profiler off, all slots in flight ----
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = lib.wb_launch_count()
    last = {}

    def timed_step(i, mdl):
        res = step(dev_pcm[i % NROT], mdl)
        if i == args.steps - 1:
            last["res"] = res

    ms = timed(timed_step, args.steps)
    launches = lib.wb_launch_count() - launches0

    # ---- per-kernel pass (roofline / kernel table): CUDA events around every launch, ONE batch in flight so that the
    #      durations are not stretched by kernels of other batches sharing the SMs ----
    def profile_pass(step_fn, mdl, steps):
        """per-kernel-family CUDA-event times over `steps` extra steps with ONE batch in flight"""
        lib.wb_set_sm_reserve(0)
        lib.wb_prof_reset()
        lib.wb_prof_enable(1)
        torch.cuda.synchronize()
        t_p0 = time.perf_counter()
        for i in range(steps):
            step_fn(i, mdl)
        torch.cuda.synchronize()
        wall_ms = 1e3 * (time.perf_counter() - t_p0)
        lib.wb_prof_enable(0)
        nt = lib.wb_prof_num_tags()
        pms, pwork, pl = (C.c_double * nt)(), (C.c_double * nt)(), (C.c_longlong * nt)()
        lib.wb_prof_collect(pms, pwork, pl)
        out = {lib.wb_prof_tag_name(t).decode(): {"ms": pms[t], "work": pwork[t], "launches": int(pl[t])}
               for t in range(nt) if pl[t] > 0}
        lib.wb_prof_reset()
        lib.wb_set_sm_reserve(args.sm_reserve if args.sm_reserve >= 0 else (8 if n_slots > 1 else 0))
        return out, wall_ms

    prof = None
    prof_steps = 0
    if not args.no_profile:
        prof_steps = max(2, min(args.steps, 4))
        prof, prof_ms = profile_pass(lambda i, mdl: step(dev_pcm[i % NROT], mdl), model, prof_steps)

    # ---- end to end: pinned host PCM -> H2D -> decode -> results on host ----
    def e2e_step(i, mdl):
        pcm = host_pcm[i % NROT].to(dev, non_blocking=True)
        res = step(pcm, mdl)
        # what recognize.py:296-311 reads of every result: the token list (and the cli the confidence) as Python objects
        n = 0
        for r in res[args.mode]:
            n += len(r.tokens)
            if r.confidence < 0.0:
                raise RuntimeError("negative confidence")
        return n

    if n_slots == 1:
        for i in range(2):
            e2e_step(i, model)
    else:
        run_steps(e2e_step, 2 * n_slots)   # every slot allocates its H2D staging on its own stream before timing
    torch.cuda.synchronize()
    for m_ in slot_models:
        m_.d2h_bytes = 0
    ms_e2e = timed(e2e_step, args.steps)
    d2h = int(sum(m_.d2h_bytes for m_ in slot_models) / max(args.steps, 1))
    sampler.stop_flag = True
    sampler.join(timeout=2)

    audio_per_step = world * B * wl["seconds"]
    value = audio_per_step * args.steps / (ms / 1e3)
    e2e_val = audio_per_step * args.steps / (ms_e2e / 1e3)
    peaks = load_peaks()
    line = {
        "metric": METRIC, "value": value, "unit": "audio-s/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": wl["label"], "recipe": wl["recipe"], "batch_per_gpu": B, "seconds": wl["seconds"],
                   "mode": args.mode, "beam": wl["beam"], "ctc_weight": wl["ctc_weight"],
                   "reverse_weight": wl["reverse_weight"], "parallelism": "dp%d (utterance shards, no collective)" % world,
                   "l2": "inputs rotate over %d distinct PCM batches (%.0f MB > L2) and every step streams GBs of "
                         "activations" % (NROT, NROT * B * n * 2 / 1e6),
                   "weights": "random init, seed 777, CTC head sharpened (synth.py)",
                   "tokens_per_batch": n_tok, "inflight_batches": n_slots},
        "clocks": sampler.summary(),
        "e2e": {"value": e2e_val, "unit": "audio-s/s", "h2d_bytes_per_step": B * n * 2, "d2h_bytes_per_step": d2h,
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": int(launches),
    }
    if prof is not None and "gemm_tcgen05" in prof:
        # dominant kernel family = the tcgen05 GEMMs
        # (both profile tags are gemm_tcgen05_kernel: the second one is its launches whose epilogue also carries the next
        #  module's LayerNorm - same FLOPs, more epilogue work, so fusing lowers this fraction while shortening the step)
        fam = [prof[k] for k in ("gemm_tcgen05", "gemm_tcgen05+layernorm") if k in prof]
        g = {"ms": sum(v["ms"] for v in fam), "work": sum(v["work"] for v in fam),
             "launches": sum(v["launches"] for v in fam)}
        ach = g["work"] / (g["ms"] * 1e-3) / 1e12 if g["ms"] > 0 else 0.0
        traffic, traffic_of = None, None
        try:   # DRAM bytes per launch of the family's largest member, from the committed `ncu --set full` capture
            pdir = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles")
            tfile = os.path.join(pdir, "r2_gemm_traffic.json")
            with open(tfile if os.path.exists(tfile) else os.path.join(pdir, "r1_gemm_traffic.json")) as f:
                tj = json.load(f)
            traffic, traffic_of = tj["traffic_bytes_per_launch"], tj["kernel"]
        except (OSError, KeyError, ValueError):
            pass
        line["roofline"] = {"kernel": "tcgen05 GEMM family: gemm_tcgen05_kernel + gemm_act16_kernel (Linear / pointwise-conv / implicit-GEMM conv2)",
                            "bound": "tensor", "achieved": ach, "peak": peaks["tf_sust"], "unit": "TFLOP/s",
                            "frac": ach / peaks["tf_sust"], "traffic": traffic, "traffic_of": traffic_of,
                            "peak_source": peaks["src"] + " (sustained bf16)",
                            "launches": g["launches"], "avg_launch_us": 1e3 * g["ms"] / max(g["launches"], 1),
                            "share_of_step": g["ms"] / prof_ms,
                            "fused_layernorm_launches": prof.get("gemm_tcgen05+layernorm", {}).get("launches", 0),
                            # the same fraction per profile tag: launches with a plain epilogue / launches whose epilogue also
                            # normalises the rows (same FLOPs counted, extra HBM-bound epilogue work)
                            "frac_plain_epilogue": (prof["gemm_tcgen05"]["work"] / (prof["gemm_tcgen05"]["ms"] * 1e-3) / 1e12
                                                    / peaks["tf_sust"]) if prof["gemm_tcgen05"]["ms"] > 0 else None,
                            "frac_layernorm_epilogue": (prof["gemm_tcgen05+layernorm"]["work"]
                                                        / (prof["gemm_tcgen05+layernorm"]["ms"] * 1e-3) / 1e12 / peaks["tf_sust"])
                            if prof.get("gemm_tcgen05+layernorm", {}).get("ms", 0) > 0 else None,
                            "measured": "CUDA events around every launch of the family, %d extra steps with one batch in "
                                        "flight right after the timed region (%.2f ms/step in that pass)"
                                        % (prof_steps, prof_ms / prof_steps)}
        tot = sum(v["ms"] for v in prof.values())
        line["kernels"] = {k: {"ms_per_step": v["ms"] / prof_steps, "launches_per_step": v["launches"] / prof_steps,
                               "share": v["ms"] / tot,
                               **({"GBps": v["work"] / (v["ms"] * 1e-3) / 1e9} if (v["work"] > 0 and "tcgen05" not in k) else {}),
                               **({"TFLOPs": v["work"] / (v["ms"] * 1e-3) / 1e12} if (v["work"] > 0 and "tcgen05" in k) else {})}
                           for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"])}
    # ---- extra block: ragged global list (all N); BASELINE configs[2] and configs[3] (N = 1) ----
    if not args.no_extra:
        extra = {}
        # (iii) a fixed GLOBAL list of world x B utterances with lengths U[5 s, 30 s], sharded by shard_utterances
        #       (LPT on the attention-aware cost): scaling efficiency on it measures the partition balance
        rs = np.random.Generator(np.random.PCG64(20260923))
        g_secs = np.round(rs.uniform(5.0, 30.0, size=world * B), 2)
        g_frames = [fb.num_frames(int(sec * 16000)) for sec in g_secs]
        mine_r = shard_utterances(g_frames, world, rank, d_model=cfg["encoder_conf"]["output_size"])
        my_n = [int(g_secs[i] * 16000) for i in mine_r]
        order = sorted(range(len(my_n)), key=lambda k: -my_n[k])           # processor.padding sorts by length
        my_n = [my_n[k] for k in order]
        Br = len(my_n)
        nmax = max(my_n)
        rag_pcm = []
        for r in range(NROT):
            t = dev_pcm[r][torch.arange(Br, device=dev) % B, :nmax].clone()
            for b, nb in enumerate(my_n):
                t[b, nb:] = 0
            rag_pcm.append(t)
        ns_r = torch.tensor(my_n, dtype=torch.int32, device=dev)
        flens_r = torch.tensor([fb.num_frames(x) for x in my_n], dtype=torch.int64, device=dev)

        def step_r(i, mdl):
            feats = fb(rag_pcm[i % NROT], ns_r)
            return mdl.decode(methods, feats, flens_r, beam_size=wl["beam"], ctc_weight=wl["ctc_weight"],
                              reverse_weight=wl["reverse_weight"])

        run_steps(step_r, 2 * n_slots)
        ms_r = timed(step_r, args.steps)
        my_audio = float(sum(my_n)) / 16000.0
        aud = torch.tensor([my_audio], device=dev, dtype=torch.float64)
        if world > 1:
            allaud = [torch.zeros_like(aud) for _ in range(world)]
            dist.all_gather(allaud, aud)
            per_rank = [float(a.item()) for a in allaud]
        else:
            per_rank = [my_audio]
        extra["ragged"] = {"value": sum(per_rank) * args.steps / (ms_r / 1e3), "unit": "audio-s/s",
                           "ms_per_step": ms_r / args.steps, "utterances": world * B,
                           "lengths": "U[5 s, 30 s], seed 20260923, fixed global list sharded by shard_utterances (LPT)",
                           "audio_s_per_rank": per_rank, "utts_on_rank0": Br}
        if world == 1 and args.workload == "small":
            # (ii) BASELINE configs[3]: forward_chunk chunk 16 / 4 left chunks, batch 1, steady state as a CUDA graph
            from wenet_b200.asr_model import StreamingSession
            chunk, left, n_chunks, n_warm = 16, 4, 200, 20
            window, hop = (chunk - 1) * 4 + 7, 4 * chunk
            gen = torch.Generator().manual_seed(777)
            sfeats = torch.randn(1, hop * (n_chunks + n_warm) + window, 80, generator=gen).to(dev)
            sess = StreamingSession(model, chunk, left)
            evs = []
            for i in range(n_chunks + n_warm):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                sess.step(sfeats[:, i * hop:i * hop + window])
                e1.record()
                torch.cuda.synchronize()      # one chunk in flight: a latency measurement
                evs.append((e0, e1))
            lat = np.array([a.elapsed_time(b) for a, b in evs[n_warm:]])
            extra["streaming"] = {"config": "S U2++ 12L/256d forward_chunk, chunk 16, num_left_chunks 4, batch 1, CUDA graph",
                                  "p50_ms": float(np.percentile(lat, 50)), "p99_ms": float(np.percentile(lat, 99)),
                                  "chunks": n_chunks, "audio_s_per_chunk": chunk * 0.04,
                                  "chunk_rtf": float(np.percentile(lat, 50)) / 1e3 / (chunk * 0.04)}
            # (ii-b) SURVEY 8f-4: the same streaming step for 64 concurrent sessions in lockstep (batched caches), CUDA graph
            from wenet_b200.asr_model import BatchedStreamingSessions
            S_b, n_b, n_bw = 64, 60, 12
            bfeats = torch.randn(S_b, hop * (n_b + n_bw) + window, 80, generator=gen).to(dev)
            bs = BatchedStreamingSessions(model, S_b, chunk, left)
            evb = []
            for i in range(n_b + n_bw):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                bs.step(bfeats[:, i * hop:i * hop + window])
                e1.record()
                torch.cuda.synchronize()
                evb.append((e0, e1))
            latb = np.array([a.elapsed_time(b) for a, b in evb[n_bw:]])
            extra["streaming_batched"] = {"config": "S U2++ 12L/256d, %d concurrent forward_chunk sessions in lockstep "
                                                    "(wb_encoder_forward_chunk_batch), chunk 16, num_left_chunks 4, CUDA graph" % S_b,
                                          "p50_ms": float(np.percentile(latb, 50)), "p99_ms": float(np.percentile(latb, 99)),
                                          "steps": n_b, "sessions": S_b,
                                          "value": S_b * chunk * 0.04 / (float(np.percentile(latb, 50)) / 1e3),
                                          "unit": "audio-s/s (all sessions)"}
            del bs, bfeats
            # (i) BASELINE configs[2] model: U2++ large 24L/512d/8h, 32 x 30 s, attention_rescoring
            wl_l = workload("large")
            cfg_l = synth.recipe(wl_l["recipe"])
            model_l = B200ASRModel(cfg_l, synth.synth_state_dict(cfg_l, seed=777), device=dev)
            Bl = wl_l["batch"]
            slots_l = [model_l] + [model_l.clone_shared() for _ in range(n_slots - 1)]
            ns_l, flens_l = ns[:Bl], flens[:Bl]

            def step_l(i, mdl):
                feats = fb(dev_pcm[i % NROT][:Bl], ns_l)
                return mdl.decode(methods, feats, flens_l, beam_size=wl_l["beam"], ctc_weight=wl_l["ctc_weight"],
                                  reverse_weight=wl_l["reverse_weight"])

            for i in range(3):
                step_l(i, model_l)
            run_steps(step_l, 2 * n_slots, slots_l)
            steps_l = max(4, args.steps // 2)
            ms_l = timed(step_l, steps_l, slots_l)
            pl_, plw = profile_pass(step_l, model_l, 2)
            gl = pl_.get("gemm_tcgen05", {"ms": 0.0, "work": 0.0})
            ach_l = gl["work"] / (gl["ms"] * 1e-3) / 1e12 if gl["ms"] > 0 else 0.0
            extra["large"] = {"workload": wl_l["label"], "value": Bl * wl_l["seconds"] * steps_l / (ms_l / 1e3),
                              "unit": "audio-s/s", "ms_per_step": ms_l / steps_l, "steps": steps_l,
                              "gemm_tflops": ach_l, "gemm_frac": ach_l / peaks["tf_sust"],
                              "kernels_ms_per_step": {k: v["ms"] / 2 for k, v in sorted(pl_.items(), key=lambda kv: -kv[1]["ms"])}}
            del slots_l, model_l
            torch.cuda.empty_cache()
        if world == 1 and args.workload == "small" and not args.no_whisper:
            # (iv) BASELINE configs[4] / SURVEY 8f-1: Whisper-large-v3 geometry (32 + 32 layers, d 1280, 20 heads, ff 5120,
            #      V 51866, 128 mel), 32 x 30 s, log-mel -> encoder -> attention decoding (beam 10) through B200Whisper.decode.
            #      Random-init weights with <eot> suppressed: exactly `dec_steps` beam steps per batch (~3.2 tokens per audio s).
            from wenet_b200.whisper import B200Whisper, LogMelExtractor
            t_w0 = time.perf_counter()
            cfg_w = synth.recipe("whisper_large_v3")
            model_w = B200Whisper(cfg_w, synth.synth_whisper_state_dict_fast(cfg_w, seed=777), device=dev)
            t_build = time.perf_counter() - t_w0
            Bw, beam_w, dec_steps = 32, 10, 96
            model_w.max_decode_len = dec_steps + 4          # 4 forced prefix tokens
            lm = LogMelExtractor(128, 400, 160)
            pcm_w = [(dev_pcm[r][:Bw].float() / 32768.0).contiguous() for r in range(NROT)]
            ns_w = ns[:Bw]
            flens_w = torch.tensor([lm.num_frames(int(x)) for x in ns_w.tolist()], dtype=torch.int64, device=dev)

            def step_w(i, mdl):
                feats = lm(pcm_w[i % NROT], ns_w)
                return mdl.decode(["attention"], feats, flens_w, beam_size=beam_w)

            for i in range(2):
                step_w(i, model_w)
            torch.cuda.synchronize()
            steps_w = 3
            evw0, evw1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            evw0.record()
            for i in range(steps_w):
                out_w = step_w(i, model_w)
            evw1.record()
            torch.cuda.synchronize()
            ms_w = evw0.elapsed_time(evw1)
            pw_, _ = profile_pass(step_w, model_w, 1)
            gw = pw_.get("gemm_tcgen05", {"ms": 0.0, "work": 0.0})
            ach_w = gw["work"] / (gw["ms"] * 1e-3) / 1e12 if gw["ms"] > 0 else 0.0
            secs_w = float(ns_w.sum().item()) / 16000.0
            extra["whisper"] = {"workload": "Whisper-large-v3 geometry (32+32L, d 1280, 20 heads, ff 5120, V 51866, 128 mel), "
                                            "%d x 30 s, log-mel + encoder + attention decoding beam %d, %d decoding steps" % (Bw, beam_w, dec_steps),
                                "value": secs_w * steps_w / (ms_w / 1e3), "unit": "audio-s/s", "ms_per_step": ms_w / steps_w,
                                "steps": steps_w, "decode_steps": int(model_w.last_attention_steps),
                                "tokens_out": int(sum(len(r.tokens) for r in out_w["attention"])),
                                "gemm_tflops": ach_w, "gemm_frac": ach_w / peaks["tf_sust"], "model_build_s": t_build,
                                "kernels_ms_per_step": {k: v["ms"] for k, v in sorted(pw_.items(), key=lambda kv: -kv[1]["ms"])}}
            del model_w
            torch.cuda.empty_cache()
        line["extra"] = extra

    # ---- verification against the CPU oracle (rank 0, N = 1): tokens of two utterances of batch 0 ----
    if rank == 0 and world == 1 and not args.no_verify and args.mode == "attention_rescoring":
        from wenet_b200.asr_model import B200ASRModel as _M
        n_v = 2
        rows = [host_pcm[0][b, :n] for b in range(n_v)]
        t_v0 = time.perf_counter()
        ref_tok, ref_enc = cpu_oracle_step(sd, cfg, rows, wl, want_enc=True)
        t_oracle = time.perf_counter() - t_v0
        ver = {"utterances": n_v, "checker": "oracle/wenet_oracle.py (fp32, pinned to the reference), %.1f s" % t_oracle}
        for tag, mdl in (("bf16", model), ("precise", _M(cfg, sd, device=dev, precise=True))):
            feats_v = fb(dev_pcm[0][:n_v], ns[:n_v])
            out_v = mdl.decode(methods, feats_v, flens[:n_v], beam_size=wl["beam"], ctc_weight=wl["ctc_weight"],
                               reverse_weight=wl["reverse_weight"])[args.mode]
            enc_v, _ = mdl.encoder(feats_v, flens[:n_v], -1, -1)
            dmax = max(float((enc_v[b, :ref_enc[b].shape[0]].cpu() - ref_enc[b]).abs().max()) for b in range(n_v))
            dmean = float(np.mean([float((enc_v[b, :ref_enc[b].shape[0]].cpu() - ref_enc[b]).abs().mean()) for b in range(n_v)]))
            same = [list(out_v[b].tokens) == list(ref_tok[b]) for b in range(n_v)]
            agree = [1.0 - _edit_distance(list(out_v[b].tokens), list(ref_tok[b])) / max(len(ref_tok[b]), 1) for b in range(n_v)]
            ver[tag] = {"tokens_identical": int(sum(same)), "token_agreement": float(np.mean(agree)),
                        "encoder_out_max_abs": dmax, "encoder_out_mean_abs": dmean}
        line["parity"] = {"mode": "precise", "max": ver["precise"]["encoder_out_max_abs"],
                          "mean": ver["precise"]["encoder_out_mean_abs"],
                          "bf16_mode": {"max": ver["bf16"]["encoder_out_max_abs"], "mean": ver["bf16"]["encoder_out_mean_abs"]},
                          "what": "encoder_out of %d x %.0f s utterances vs the fp32 CPU oracle" % (n_v, wl["seconds"])}
        line["verify"] = ver
        # precise mode: identical token ids and encoder_out within 1e-3; bf16 mode (the one timed above): encoder_out inside
        # the reference's own bf16-autocast budget and >= 90 % token agreement (near-tie frames may flip)
        line["verified"] = bool(ver["precise"]["tokens_identical"] == n_v and ver["precise"]["encoder_out_max_abs"] <= 1e-3
                                and ver["bf16"]["encoder_out_max_abs"] < 5.9e-2 and ver["bf16"]["token_agreement"] >= 0.9)

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        arm = CpuArm(args.workload)
        arm.step()                      # warm-up pass (worker start-up, lazy torch init)
        audio, dt = arm.step()
        line["cpu_baseline"] = {"value": audio / dt, "unit": "audio-s/s", "cores": host_cores(),
                                "threads_used": arm.procs * arm.threads, "kind": arm.kind, "sample": arm.describe()}
        arm.close()
    if rank == 0 and args.dump_outputs:
        dump_outputs(last["res"][args.mode], args.dump_outputs)
    if rank == 0:
        args.emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
