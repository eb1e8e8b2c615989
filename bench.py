#!/usr/bin/env python
"""bench.py - openWakeWord's streaming hot path on B200, measured on BASELINE.json's configs.

  python bench.py [--gpus N] [--steps K] [--warmup W]        # own arm (CUDA, libowwb200)
  python bench.py --impl reference [...]                    # reference arm (CPU, host cores)
  torchrun --nproc-per-node N ... bench.py --gpus N ...      # one rank per GPU, weak scaling
  python bench.py ... --dump-outputs DIR                    # also write the last timed step's outputs as DIR/*.npy

The library is loaded as __graft_entry__.build() left it; the benchmark compiles and writes nothing in the tree.

Headline workload = configs[2]: 8192 concurrent synthetic 16 kHz streams per GPU, 80 ms frames, all six pre-trained
wake-word head shapes (alexa, hey_mycroft, hey_jarvis [two networks + verifier gate], hey_rhasspy, weather:
1536-64-64-1; timer: 3264-128-128-7 -> 11 labels).  The same per-GPU workload at every N (weak scaling: configs[3]'s
65 536 streams on 8 GPUs with configs[2]'s head set).  configs[1] (1024 streams, 1 head) is measured too and reported
under "secondary".  A step = every stream consumes one 1280-sample chunk: log-mel -> embedding CNN -> ring append ->
heads (+ one score gather when N > 1).  Prints ONE JSON line (rank 0).

  value      frames/s with the PCM already resident in HBM (CUDA events on the launching stream, max over ranks)
  e2e        frames/s through the host-buffer C-ABI calls oww_step_host_submit/collect: every step's PCM goes
             pinned host -> H2D and every step's scores come back D2H inside the timed region (wall clock, max over ranks)
  e2e_model  the same through the drop-in surface Model(n_streams=B).predict (synchronous, label dicts, history)
  parity     after the timed regions the SAME engine (same kernels, group size, mode) is reset and driven for 12 steps;
             16 sampled streams (first / last ragged group included) are compared with the NumPy oracle: max |delta|,
             asserted <= 1e-3
  roofline   the step's dominant kernel (tc_inc_kernel): executed and reference-algorithmic FLOP/s against both
             measured bf16 peaks (MEASURED_PEAKS.json)
  cpu_baseline / --impl reference : the NumPy oracle (a port - onnxruntime and the .onnx files do not exist in this
             image) driven as the reference is: one single-stream model per process, one process per usable host core,
             predict() per 80 ms frame, same head set.
Weights are synthetic (seeded, exact reference shapes); PCM is synthetic (SURVEY.md 8d mixes).
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the tree may be read-only: no __pycache__ next to the sources

FLOPS_PER_WINDOW = 2 * 41955840          # SURVEY.md Appendix B (reference-algorithmic, per 76x32 window)
EXEC_FLOPS_PER_FRAME = 2 * 5612544       # what the incremental path computes per frame with one MMA term per K step (SURVEY.md F10)
# multiply-accumulates per frame of the incremental conv layers 0..19 (8 new mel rows; SURVEY.md Appendix B shapes)
INC_MACS = [55296, 442368, 442368, 221184, 442368, 442368, 442368, 331776, 497664, 497664, 497664,
            165888, 221184, 221184, 221184, 110592, 110592, 110592, 110592, 27648]


def exec_flops_per_frame(split_from):
    """FLOPs the tensor pipe issues per frame in cnn_mode 3: layers >= split_from take fp16 hi/lo split operands, i.e.
    three MMA terms per K step (hi*hi + lo*hi + hi*lo)."""
    s = 11 if not split_from else split_from
    return 2 * (sum(INC_MACS[:s]) + 3 * sum(INC_MACS[s:]))
CHUNK = 1280
METRIC = "80ms audio-frames/sec (concurrent streams)"
UNIT = "frames/s"
WORKLOADS = {
    "c3": dict(streams=8192, label="configs[2]: 8192 concurrent synthetic 16 kHz streams per GPU, 80 ms frames, all six "
                                    "pre-trained wake-word head shapes (7 networks incl. hey_jarvis' verifier, 11 labels)"),
    "c2": dict(streams=1024, label="configs[1]: 1024 concurrent synthetic 16 kHz streams per GPU, 80 ms frames, 1 wake-word head"),
}


def synth_pcm(n_streams, n_steps, seed):
    """SURVEY.md 8d input mixes: 50 % +-1000 noise, 25 % full-scale, 25 % gated 0.5 s bursts."""
    rng = np.random.default_rng(seed)
    n = n_steps * CHUNK
    out = np.empty((n_streams, n), np.int16)
    for b in range(n_streams):
        k = b % 4
        if k < 2:
            out[b] = rng.integers(-1000, 1000, n)
        elif k == 2:
            out[b] = (rng.uniform(-1, 1, n) * 32767).astype(np.int16)
        else:
            x = rng.normal(0, 8000, n)
            gate = (np.arange(n) // 8000) % 2 == 1
            out[b] = np.clip(x * gate, -32768, 32767).astype(np.int16)
    return out


def synth_pcm_fast(n_streams, n_steps, seed):
    """Same mixes for large batches: 64 distinct signals tiled over the streams (generation time, not content, differs)."""
    base = synth_pcm(64, n_steps, seed)
    idx = np.random.default_rng(seed + 1).integers(0, 16, n_streams) * 4 + (np.arange(n_streams) % 4)
    return np.ascontiguousarray(base[idx])


def bench_heads(workload):
    """-> ordered {model name: head dict}; names follow the reference registry (openwakeword/__init__.py:8-51)."""
    from openwakeword_b200 import weights as W
    if workload == "c2":
        return {"alexa": W.synthetic_head(n_in=16, hidden=64, n_blocks=1, n_out=1, layernorm=True, final="sigmoid", seed=1)}
    hs = {}
    for i, nm in enumerate(["alexa", "hey_mycroft", "hey_jarvis", "hey_rhasspy", "weather"]):
        if nm == "hey_jarvis":
            hs[nm] = W.synthetic_gated_head(seed_main=10 + i, seed_verifier=40 + i, threshold=0.5)
        else:
            hs[nm] = W.synthetic_head(seed=10 + i)
    hs["timer"] = W.synthetic_head(n_in=34, hidden=128, n_out=7, layernorm=False, final="relu_softmax", seed=20)
    return hs


TIMER_MAP = {"1": "1_minute_timer", "2": "5_minute_timer", "3": "10_minute_timer",
             "4": "20_minute_timer", "5": "30_minute_timer", "6": "1_hour_timer"}


# ---------------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock + throttle reasons sampled through NVML every ~1 ms by a host thread while the timed regions run
    (nvidia-smi's own loop cannot sample a region of a few milliseconds)."""

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.rows = []
        self._stop = threading.Event()
        self.ok = False
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[gpu_index]) if vis and vis.split(",")[gpu_index].isdigit() else gpu_index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.smax = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception as e:                       # noqa: BLE001
            self.err = repr(e)

    def _loop(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                self.rows.append((time.perf_counter(), float(sm), int(rs)))
            except Exception:                        # noqa: BLE001
                pass
            time.sleep(0.001)

    def start(self):
        if self.ok:
            self.t = threading.Thread(target=self._loop, daemon=True)
            self.t.start()

    def stop(self, windows=None):
        """windows: list of (t0, t1) perf_counter intervals of the timed regions; samples outside are dropped."""
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + getattr(self, "err", "?")], "samples": 0}
        self._stop.set()
        self.t.join(timeout=2)
        nv = self.nv
        names = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap}
        rows = self.rows
        if windows:
            rows = [r for r in rows if any(a <= r[0] <= b for a, b in windows)]
        sm = [r[1] for r in rows]
        reasons = sorted({k for r in rows for k, bit in names.items() if r[2] & bit})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.smax, "reasons": reasons,
                "samples": len(sm), "how": "NVML polled every ~1 ms inside the timed regions"}


# ---------------------------------------------------------------------------------- CPU arm
def _cpu_worker(conn, stream_id, seed, workload):
    """One reference-shaped consumer: a single-stream model, predict() per 80 ms frame."""
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(1)                                  # the reference pins ORT to 1 thread/session (model.py:149-151)
    except Exception:
        pass
    from openwakeword_b200 import weights as W
    from oracle import streaming, probe
    om = None
    ok, where = probe.ort_reference_available()
    if ok:
        # the genuine reference: unmodified openwakeword.Model on onnxruntime CPU with the released models (never the case
        # in this image - SURVEY.md F2 - but the arm upgrades itself when the assets exist)
        try:
            import glob
            extra = os.path.join(ROOT, "baseline", "_ref")
            if os.path.isdir(extra) and extra not in sys.path:
                sys.path.insert(0, extra)
            import openwakeword
            hp = sorted(p for p in glob.glob(os.path.join(where, "*.onnx"))
                        if os.path.basename(p) not in ("melspectrogram.onnx", "embedding_model.onnx", "silero_vad.onnx"))
            if workload == "c2":
                hp = [p for p in hp if "alexa" in os.path.basename(p)][:1] or hp[:1]
            om = openwakeword.Model(wakeword_models=hp, inference_framework="onnx",
                                    melspec_model_path=os.path.join(where, "melspectrogram.onnx"),
                                    embedding_model_path=os.path.join(where, "embedding_model.onnx"))
        except Exception:          # noqa: BLE001
            om = None
    kind = "reference" if om is not None else "port"
    if om is None:
        emb = W.synthetic_embedding(0)
        heads = bench_heads(workload)
        cm = {"timer": dict(TIMER_MAP)} if "timer" in heads else None
        om = streaming.OracleModel(emb, heads, cm, feature_init=np.zeros((41, 96), np.float32))
    pcm = synth_pcm(stream_id % 4 + 1, 64, seed + stream_id // 4)[stream_id % 4]
    pos = 0
    conn.send("ready:" + kind)
    while True:
        n = conn.recv()
        if n <= 0:
            break
        t0 = time.perf_counter()
        for _ in range(n):
            om.predict(pcm[pos:pos + CHUNK])
            pos = (pos + CHUNK) % (pcm.shape[0] - CHUNK)
        conn.send(time.perf_counter() - t0)


def usable_cores():
    """Host cores this process may actually run on: the scheduler affinity mask, capped by a cgroup CPU quota when the
    container has one (os.cpu_count() reports the machine's logical CPUs even under a quota, and one busy worker per
    *reported* CPU then measures time-slicing, not the cores)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]            # cgroup v2
        if q != "max":
            quota = int(q) / int(per)
    except Exception:
        try:                                                                  # cgroup v1
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    if quota is not None:
        n = max(1, min(n, int(quota + 0.5)))
    return n


class CpuArm:
    """P persistent worker processes (P = usable host cores); step(n) = every worker runs n frames."""

    def __init__(self, workload, procs=None):
        import multiprocessing as mp
        ctx = mp.get_context("fork")
        self.P = procs or usable_cores()
        self.workers = []
        for i in range(self.P):
            a, b = ctx.Pipe()
            p = ctx.Process(target=_cpu_worker, args=(b, i, 1234, workload), daemon=True)
            p.start()
            self.workers.append((p, a))
        kinds = set()
        for _, a in self.workers:
            msg = a.recv()
            assert msg.startswith("ready:")
            kinds.add(msg.split(":")[1])
        self.kind = "reference" if kinds == {"reference"} else "port"

    def step(self, frames_each):
        t0 = time.perf_counter()
        for _, a in self.workers:
            a.send(frames_each)
        for _, a in self.workers:
            a.recv()
        return time.perf_counter() - t0

    def close(self):
        for p, a in self.workers:
            try:
                a.send(0)
            except Exception:
                pass
        for p, _ in self.workers:
            p.join(timeout=5)


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    wl = args.workload
    arm = CpuArm(wl)
    frames_each = max(1, min(4, 400 // max(args.steps, 1)))      # bounded sample: the whole run stays within minutes
    for _ in range(min(max(args.warmup, 3), 5)):
        arm.step(frames_each)
    t = 0.0
    for _ in range(args.steps):
        t += arm.step(frames_each)
    arm.close()
    frames = arm.P * frames_each * args.steps
    v = frames / t
    n_heads = len(bench_heads(wl))
    sample = (f"{arm.P} single-stream oracle models (one per usable core; os.cpu_count()={os.cpu_count()}), {n_heads} head(s) each, x "
              f"{frames_each} frames per step x {args.steps} steps")
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOADS[wl]["label"] + " - sampled: one single-stream model per host core (the reference's "
                               "own deployment shape); onnxruntime + .onnx files are absent in this image, so the NumPy oracle port is timed",
                   "streams": arm.P, "heads": n_heads},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": arm.P, "kind": arm.kind, "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ---------------------------------------------------------------------------------- own arm
def parity_check(eng, heads, B, rng_seed=4242, steps=12, n_sample=16):
    """Reset the engine that was just timed and compare a fresh run with the oracle on sampled streams (checker only)."""
    from oracle import streaming, heads as oheads
    from openwakeword_b200 import weights as W
    rng = np.random.default_rng(rng_seed)
    fi = rng.normal(0, 1, (41, 96)).astype(np.float32)
    eng.reset(fi)
    pcm = synth_pcm_fast(B, steps, rng_seed)
    sample = sorted(set([0, 1, 6, B - 1, B - 2, B // 2] + list(rng.integers(0, B, n_sample))))[:max(n_sample, 6)]
    emb = W.synthetic_embedding(0)
    orc = {b: streaming.OracleAudioFeatures(emb, feature_init=fi) for b in sample}
    hl = list(heads.values())
    worst = 0.0
    for s in range(steps):
        x = np.ascontiguousarray(pcm[:, s * CHUNK:(s + 1) * CHUNK])
        got = eng.step_host(x, 1)
        for b in sample:
            orc[b](x[b])
            for (col, n_out), h in zip(eng.columns, hl):
                ref = oheads.forward(h, orc[b].get_features(h["n_in"]))[0]
                worst = max(worst, float(np.abs(ref - got[b, col:col + n_out]).max()))
    return {"max_abs_delta": worst, "gate": 1e-3, "streams_checked": len(sample), "steps": steps,
            "ok": bool(worst <= 1e-3)}


def measure(args, wl, rank, world, local, dev, sampler_windows, do_model=True):
    """One workload on this rank's GPU -> dict of raw timings (max over ranks is taken by the caller)."""
    import torch
    import torch.distributed as dist
    from openwakeword_b200 import distributed as owd
    from openwakeword_b200.engine import StreamEngine
    B = WORKLOADS[wl]["streams"]
    n_total = B * world
    K, Wm = args.steps, max(args.warmup, 3)
    heads = bench_heads(wl)
    pool_bytes = 168e6                                           # distinct PCM cycled through: larger than the 126 MB L2
    POOL = max(4, int(np.ceil(pool_bytes / (B * CHUNK * 2))))

    def factory(n_local, lo, hi):
        return StreamEngine(list(heads.values()), n_local, embedding="synthetic:0", device_index=local, max_chunks=1,
                            cnn_mode=args.cnn_mode, fuse_step=not args.no_fuse, tc_heads=not args.no_tc_heads,
                            tc_heads_terms=args.tc_heads_terms, split_from=args.split_from)
    sh = owd.ShardedStreams(n_total, factory, rank=rank, world=world, gather=args.gather)
    eng = sh.engine
    host_pcm = synth_pcm_fast(B, POOL, 1234 + rank)
    pinned = [torch.from_numpy(np.ascontiguousarray(host_pcm[:, i * CHUNK:(i + 1) * CHUNK])).pin_memory() for i in range(POOL)]
    host_steps = [p.numpy() for p in pinned]
    dev_steps = [p.to(dev) for p in pinned]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for k in range(Wm):
        sh.step(dev_steps[k % POOL], 1)
    sh.flush()
    barrier()
    # ---- timed region 1: device-resident inputs, CUDA events, stage events inside the library ----
    l0 = eng.ctx.launch_count
    eng.ctx.enable_stage_timing(min(K, 4096))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_a = time.perf_counter()
    e0.record()
    for k in range(K):
        scores = sh.step(dev_steps[(Wm + k) % POOL], 1)
    sh.flush()
    e1.record()
    barrier()
    sampler_windows.append((t_a, time.perf_counter()))
    ms_dev = e0.elapsed_time(e1)
    stage = eng.ctx.stage_ms()
    eng.ctx.enable_stage_timing(0)
    launches = eng.ctx.launch_count - l0
    dump = {}                                   # name -> what the caller of a timed path received in its last step
    if args.dump_outputs and rank == 0:
        if isinstance(scores, owd.GatheredScores):
            scores = scores.wait()
        dump[f"{wl}_step"] = scores.cpu().numpy()
    # ---- timed region 2: end to end through the host-buffer C-ABI call (two tickets in flight) ----
    h_scores = np.empty((B, eng.n_cols), np.float32)
    for k in range(Wm):
        eng.step_host(host_steps[k % POOL], 1, h_scores)
    barrier()
    t0 = time.perf_counter()
    ticket = eng.submit(host_steps[Wm % POOL], 1)
    for k in range(1, K + 1):
        nxt = eng.submit(host_steps[(Wm + k) % POOL], 1) if k < K else None
        eng.collect(ticket, h_scores)
        gathered = h_scores
        if world > 1:
            gathered = owd.gather_scores(torch.from_numpy(h_scores).to(dev), n_total)
        ticket = nxt
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    sampler_windows.append((t0, t1))
    ms_e2e = 1e3 * (t1 - t0)
    if args.dump_outputs and rank == 0:
        dump[f"{wl}_step_host"] = gathered.cpu().numpy() if world > 1 else gathered.copy()
    out = {"B": B, "ms_dev": ms_dev, "ms_e2e": ms_e2e, "cnn_ms": stage["cnn"], "heads_ms": stage["heads"], "mel_ms": stage["mel"],
           "launches": int(launches), "n_cols": eng.n_cols, "heads": len(heads), "G": None, "gather": sh.gather_kind,
           "h2d": B * CHUNK * 2, "d2h": B * eng.n_cols * 4, "dump": dump}
    # ---- parity of the configuration that was just timed (rank 0, checker only) ----
    if rank == 0:
        out["parity"] = parity_check(eng, heads, B)
    # ---- timed region 3: the drop-in surface, Model(n_streams=B).predict ----
    if do_model and world == 1:
        from openwakeword_b200 import Model
        specs = [{"name": n, "head": h, "class_mapping": (dict(TIMER_MAP) if n == "timer" else None)} for n, h in heads.items()]
        m = Model(wakeword_models=specs, embedding_model_path="synthetic:0", n_streams=B, feature_init=np.zeros((41, 96), np.float32),
                  max_chunks=1, device_index=local, cnn_mode=args.cnn_mode, split_from=args.split_from)
        for k in range(max(Wm, 6)):
            m.predict(host_steps[k % POOL])
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for k in range(K):
            r = m.predict(host_steps[(Wm + k) % POOL])
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        sampler_windows.append((t0, t1))
        out["ms_model"] = 1e3 * (t1 - t0)
        out["n_labels"] = len(r)
        if args.dump_outputs:
            dump.update({f"{wl}_predict_{label}": v for label, v in r.items()})
        del m
    del sh, eng
    torch.cuda.empty_cache()
    return out


def measure_variant(args, wl, local, dev, split_from, sampler_windows):
    """Device-resident step time and oracle parity of the same workload with another split_from."""
    import torch
    from openwakeword_b200.engine import StreamEngine
    B = WORKLOADS[wl]["streams"]
    K = args.steps
    heads = bench_heads(wl)
    POOL = max(4, int(np.ceil(168e6 / (B * CHUNK * 2))))
    eng = StreamEngine(list(heads.values()), B, embedding="synthetic:0", device_index=local, max_chunks=1, cnn_mode=3, split_from=split_from)
    host_pcm = synth_pcm_fast(B, POOL, 1234)
    dev_steps = [torch.from_numpy(np.ascontiguousarray(host_pcm[:, i * CHUNK:(i + 1) * CHUNK])).to(dev) for i in range(POOL)]
    out = torch.empty((B, eng.n_cols), dtype=torch.float32, device=dev)
    for k in range(4):
        eng.step(dev_steps[k % POOL], 1, out)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_a = time.perf_counter()
    e0.record()
    for k in range(K):
        eng.step(dev_steps[(4 + k) % POOL], 1, out)
    e1.record()
    torch.cuda.synchronize()
    sampler_windows.append((t_a, time.perf_counter()))
    ms = e0.elapsed_time(e1) / K
    dump = {f"{wl}_split{split_from}_step": out.cpu().numpy()} if args.dump_outputs else {}
    par = parity_check(eng, heads, B)
    del eng
    torch.cuda.empty_cache()
    return {"split_from": split_from, "value": B / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": K,
            "parity_max_abs_delta": par["max_abs_delta"], "parity_ok": par["ok"],
            "what": ("conv layers >= %d on fp16 hi/lo split operands" % split_from) if split_from < 20 else
                    "plain fp16 operands in every conv layer: the whole step in one launch"}, dump


def run_own_arm(args):
    import torch
    import torch.distributed as dist
    from openwakeword_b200 import distributed as owd
    from openwakeword_b200 import _native
    _native.load_library()                     # as build() left it: a missing library is an error, not a rebuild
    from oracle.probe import parity_label      # labelling only (which oracle the 1e-3 gate was checked against)

    rank, world, local = owd.init_process_group("nccl" if int(os.environ.get("WORLD_SIZE", "1")) > 1 else None)
    if world != args.gpus:
        if rank == 0:
            print(f"[bench] WORLD_SIZE={world} but --gpus {args.gpus}; launch under torchrun for N>1", file=sys.stderr)
        if world == 1 and args.gpus > 1:
            return 2
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    K, Wm = args.steps, max(args.warmup, 3)
    sampler = ClockSampler(local)
    windows = []
    if rank == 0:
        sampler.start()
    res = {}
    order = [args.workload] + ([w for w in ("c2",) if w != args.workload] if args.secondary else [])
    for wl in order:
        res[wl] = measure(args, wl, rank, world, local, dev, windows, do_model=(wl == args.workload))
    # other points of the precision / speed curve of cnn_mode 3 (device-resident timing + the same parity gate), 1 GPU only
    variants = []
    dump = {k: a for wl in order for k, a in res[wl]["dump"].items()}
    if args.variants and world == 1 and args.cnn_mode == 3 and not args.split_from:
        for sf in (15, 20):
            v, d = measure_variant(args, args.workload, local, dev, sf, windows)
            variants.append(v)
            dump.update(d)
    clocks = sampler.stop(windows) if rank == 0 else None
    if dump:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dump.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), np.ascontiguousarray(a, np.float32))

    keys = ["ms_dev", "ms_e2e", "cnn_ms", "heads_ms", "mel_ms"]
    flat = [res[wl][k] for wl in order for k in keys]
    t = torch.tensor(flat, dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    vals = [float(x) for x in t.cpu()]
    for i, wl in enumerate(order):
        for j, k in enumerate(keys):
            res[wl][k] = vals[i * len(keys) + j]
    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return 0

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    pk_sus = peaks.get("bf16_tflops_sustained", 1400.0)
    pk_burst = peaks.get("bf16_tflops", 1590.0)
    peak_src = ("MEASURED_PEAKS.json bf16_tflops_sustained / bf16_tflops (of measured)" if peaks
                else "fallback 1.4 / 1.59 PFLOP/s (of fallback)")
    main = res[args.workload]
    B = main["B"]
    n_total = B * world
    exec_flops = exec_flops_per_frame(args.split_from) if args.cnn_mode == 3 else FLOPS_PER_WINDOW
    cnn_ms = main["cnn_ms"]
    executed_tf = B * exec_flops / (cnn_ms * 1e-3) / 1e12
    achieved_tf = B * FLOPS_PER_WINDOW / (cnn_ms * 1e-3) / 1e12
    timed_s = main["ms_dev"] * 1e-3
    peak_used = pk_burst if timed_s < 1.0 else pk_sus         # burst figure for a short region at full clocks, sustained for a long one
    fused = args.cnn_mode == 3 and not args.no_fuse
    sf = args.split_from or 11
    kernel_name = ((f"tc_inc_kernel<{sf}> (cnn_tc_inc.cu): log-mel frontend + conv layers 0..{sf - 1} of every stream on tcgen05 in ONE persistent launch"
                    + (f"; layers {sf}..19 follow as tc_conv_blk_kernel launches on fp16 hi/lo split operands (3 MMA terms), then heads_grp_kernel"
                       if sf < 20 else " + ring append" + (" + heads" if main["heads_ms"] == 0.0 else "; heads_grp_kernel follows")))
                   if fused else "embedding CNN stage (separate launches)")

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        arm = CpuArm(args.workload)
        arm.step(2)
        tt, fr = 0.0, 0
        while tt < 10.0:
            tt += arm.step(4)
            fr += arm.P * 4
        arm.close()
        cpu = {"value": fr / tt, "unit": UNIT, "cores": arm.P, "kind": arm.kind,
               "sample": f"{arm.P} single-stream NumPy-oracle models (1 BLAS thread each, one per usable core; "
                         f"os.cpu_count()={os.cpu_count()}), {main['heads']} heads, x {fr // arm.P} frames, {tt:.1f} s; "
                         "onnxruntime CPU unavailable in this image"}

    def summary(r, w):
        d = {"workload": WORKLOADS[w]["label"], "value": r["B"] * world * K / (r["ms_dev"] * 1e-3), "ms_per_step": r["ms_dev"] / K,
             "e2e": r["B"] * world * K / (r["ms_e2e"] * 1e-3), "stage_ms": {"mel": r["mel_ms"], "cnn": r["cnn_ms"], "heads": r["heads_ms"]},
             "gpu_launches": r["launches"], "parity": r.get("parity")}
        return d

    par = main.get("parity") or {}
    line = {
        "metric": METRIC, "value": n_total * K / (main["ms_dev"] * 1e-3), "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm,
        "ms_per_step": main["ms_dev"] / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32" if args.cnn_mode == 0 else "f16 operands / f32 accumulate (mel, BN, LayerNorm, sigmoid in f32; heads' first layer as fp16 hi/lo split = f32-grade)",
        "data": "synthetic",
        "config": {"workload": WORKLOADS[args.workload]["label"],
                   "streams_per_gpu": B, "heads": main["heads"], "score_columns": main["n_cols"], "cnn_mode": args.cnn_mode,
                   "split_from": args.split_from or 11,
                   "fused_step": bool(fused),
                   "l2": "inputs larger than L2: distinct PCM batches totalling >= 168 MB cycled",
                   "weights": "synthetic seed 0 (reference shapes); released .onnx weights absent",
                   "parity": parity_label(),
                   "parallelism": f"dp{world} (streams sharded, weights replicated, 1 score gather/step: {main['gather']})"},
        "clocks": clocks,
        "e2e": {"value": n_total * K / (main["ms_e2e"] * 1e-3), "unit": UNIT, "ms_per_step": main["ms_e2e"] / K,
                "h2d_bytes_per_step": main["h2d"] * world, "d2h_bytes_per_step": main["d2h"] * world,
                "api": "oww_step_host_submit/collect (StreamEngine.submit/collect), pinned host PCM in, host scores out, two tickets in flight"},
        "gpu_launches": int(main["launches"]),
        "parity": dict(par, against=parity_label()),
        "roofline": {"bound": "tensor", "kernel": kernel_name,
                     "executed_tflops": executed_tf, "executed_frac": executed_tf / peak_used,
                     "executed_frac_of_sustained": executed_tf / pk_sus, "executed_frac_of_burst": executed_tf / pk_burst,
                     "achieved": achieved_tf, "peak": peak_used, "unit": "TFLOP/s", "frac": achieved_tf / peak_used,
                     "frac_of_sustained": achieved_tf / pk_sus, "frac_of_burst": achieved_tf / pk_burst,
                     "peak_source": peak_src + f"; 'peak' = the {'burst' if peak_used == pk_burst else 'sustained'} figure for a {timed_s * 1e3:.0f} ms timed region",
                     "traffic": None,
                     "flops_per_unit": FLOPS_PER_WINDOW, "executed_flops_per_unit": exec_flops, "units_per_launch": B,
                     "kernel_ms": cnn_ms, "stage_ms": {"mel": main["mel_ms"], "cnn": main["cnn_ms"], "heads": main["heads_ms"]},
                     "note": "executed_* = FLOPs the tensor pipe actually issued (the incremental path computes only the 8 new mel rows "
                             "per frame: 11.2 MFLOP with one MMA term per K step, 16.4 MFLOP with the default three-term split operands "
                             "from layer 11 on; SURVEY.md F10/8d); achieved/frac = reference-algorithmic 83.9 MFLOP per frame delivered per "
                             "second.  kernel_ms is the CNN stage (frontend + conv layers + ring append), CUDA events inside the timed region. "
                             "Why the fraction is low by construction: N = Cout is 24..96 and an M128 x N x K16 tcgen05.mma costs ~60-75 cycles "
                             "for every N <= 128 (scripts/micro/mma_layout.cu, profiles/r2_mma_layout.txt) - at N = 96 the pipe's ceiling is "
                             "~40 % of its N = 256 rate, and layers 0-2 (N = 24) ~10 %; ncu summaries of the same command: profiles/"},
        "cpu_baseline": cpu,
    }
    if "ms_model" in main:
        line["e2e_model"] = {"value": B * K / (main["ms_model"] * 1e-3), "unit": UNIT, "ms_per_step": main["ms_model"] / K,
                             "labels": main["n_labels"],
                             "api": "Model(n_streams=B).predict(int16[B,1280] pinned host array) -> {label: float32[B]} (synchronous: H2D, step, "
                                    "D2H, label mapping, first-5 zeroing, history)"}
    if len(order) > 1:
        line["secondary"] = {w: summary(res[w], w) for w in order[1:]}
    if variants:
        line["variants"] = variants
    ok = par.get("ok", True) and all((res[w].get("parity") or {}).get("ok", True) for w in order)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if not ok:
        print("[bench] PARITY GATE FAILED: max |score - oracle| > 1e-3 on the benchmarked configuration", file=sys.stderr)
        return 3
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="own", choices=["own", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS), help="c3 = configs[2] (headline), c2 = configs[1]")
    ap.add_argument("--no-secondary", dest="secondary", action="store_false", help="skip the configs[1] measurement")
    ap.add_argument("--cnn-mode", type=int, default=3, help="0 fp32 window, 2 tcgen05 window, 3 tcgen05 fused incremental")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--gather", default="nccl-overlap", choices=["nccl", "nccl-overlap", "peer"],
                    help="N>1: per-step score gather: NCCL all-gather on the compute stream, NCCL all-gather on a side stream "
                         "overlapped with the next step (default), or peer-memory stores + counters (rank 0 only)")
    ap.add_argument("--no-fuse", action="store_true", help="mode 3: keep mel / CNN / append / heads as separate launches (stage breakdown)")
    ap.add_argument("--no-tc-heads", action="store_true", help="heads on CUDA cores (heads.cu)")
    ap.add_argument("--tc-heads-terms", type=int, default=3, choices=[1, 3])
    ap.add_argument("--no-variants", dest="variants", action="store_false",
                    help="skip the split_from 15 / 20 variants of the headline workload (N=1, default split only)")
    ap.add_argument("--split-from", type=int, default=0,
                    help="first conv layer on fp16 hi/lo split operands (11 = default, scores within ~2e-4 of the fp32 graph; "
                         "20 = plain fp16 everywhere and the whole step as one fused launch, ~9e-4)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the scores each timed path returned in its last step as DIR/<name>.npy "
                         "(float32; inputs are seeded, so runs with the same arguments can be compared output for output)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference_arm(args)
    return run_own_arm(args)


if __name__ == "__main__":
    sys.exit(main())
