#!/usr/bin/env python
"""bench.py -- text-line-pixels/sec of one full training step of clstm's hot path on B200.

A "step" = one pass of the hot path over one minibatch of synthetic text lines:
    forward (bidi NPLSTM + Softmax) -> CTC alignment -> backward -> [derivative exchange] -> clip+SGD update -> decode
Default workload (BASELINE.json configs[1], "cfg2"): nhidden=100, H=48, T=500, 32 lines per GPU, 83 classes, fp32.
`--config cfg3|cfg4` select BASELINE configs[2] / [3]:
    cfg3: nhidden=200, 128 ragged lines (T = 200..2000) per GPU
    cfg4: nhidden=400, 256 ragged lines in the GLOBAL minibatch, split 256/N per GPU (strong scaling), derivative sum over
          NVLink (share_deltas, /root/reference/clstm.cc:731-744)
(configs[4], the nhidden x T sweep, is tools/sweep_cfg5.py, which calls this file once per cell.)
Multi-GPU: one process per GPU (torchrun), lines sharded per rank, ONE fused all-reduce + clip + update kernel over NVLink
peer memory per step (CLSTM_B200_DP=nccl selects ncclAllReduce + update instead).

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
           bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference --gpus 1 --steps 3 --warmup 1     # the reference's CPU path (oracle port)

Prints ONE JSON line (rank 0).  Timing: --steps training steps are timed, each bracketed by CUDA events on the handle's
stream, L2 is flushed in between; the reported step is the MEDIAN over the steps of the per-step maximum over ranks (the
mean and the full list are in the line as well).  --dump-outputs DIR writes what the last timed step returned (see
dump_outputs) so that two builds can be compared output for output on identical seeded inputs.
`value` = whole-job px/s with the batch resident in HBM; `e2e` = the same through the input pipeline with pinned host
buffers (H2D of the lines, D2H of the decoded result inside the timed region);
`roofline` for the dominant kernel from live CUDA-event phase timings; `cpu_baseline` = the CPU oracle port timed on this
box's host cores on a bounded sample.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from clstm_b200 import synth  # noqa: E402

LR, MOM, CLIP = 1e-4, 0.9, 100.0   # clstmocrtrain defaults (clstmocrtrain.cc:99-115), gradient_clip clstm.cc:204

CONFIGS = {   # BASELINE.json configs[1..3]
    "cfg2": dict(nhidden=100, batch=32, T=500, Tmax=0, split=False),
    "cfg3": dict(nhidden=200, batch=128, T=200, Tmax=2000, split=False),
    "cfg4": dict(nhidden=400, batch=256, T=200, Tmax=2000, split=True),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default=None, choices=sorted(CONFIGS), help="BASELINE.json config preset")
    ap.add_argument("--nhidden", type=int, default=None)
    ap.add_argument("--batch", type=int, default=None, help="lines per GPU (global lines with --split)")
    ap.add_argument("--T", type=int, default=None)
    ap.add_argument("--Tmax", type=int, default=None, help="if > T: variable lengths uniform in [T, Tmax]")
    ap.add_argument("--split", action="store_true", default=None,
                    help="--batch is the GLOBAL minibatch, split over the ranks (strong scaling)")
    ap.add_argument("--nclasses", type=int, default=83)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step as DIR/<name>.npy (float32, at most 64 MB in all)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the normalizer leg and the synchronous e2e form")
    a = ap.parse_args()
    preset = CONFIGS[a.config or "cfg2"]
    for k, v in preset.items():
        if getattr(a, k) is None:
            setattr(a, k, v)
    a.config = a.config or ("cfg2" if all(getattr(a, k) == v for k, v in CONFIGS["cfg2"].items()) else "custom")
    return a


def workload_name(a, world=1):
    t = "T=%d" % a.T if a.Tmax <= a.T else "T=%d..%d" % (a.T, a.Tmax)
    b = ("batch=%d global (%d/GPU)" % (a.batch, a.batch // world)) if a.split else "batch=%d/GPU" % a.batch
    tag = (a.config + " ") if a.config != "custom" else ""
    return "%sbidi-LSTM nhidden=%d H=48 %s %s nclasses=%d fwd+CTC+bwd+update" % (tag, a.nhidden, t, b, a.nclasses)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "src": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "src": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clock / throttle-reason samples; started well before the timed region (the process spawn must not sit
    between the barrier and the first timed step), filtered to the timed window afterwards."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for (t, r) in self.rows if t0 - 0.05 <= t <= t1 + 0.15] or [r for (_, r) in self.rows]
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except Exception:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def lines_T(a):
    return (a.T, a.Tmax) if a.Tmax > a.T else a.T


def make_batch(a, rank, world=1):
    """The lines of `rank`.  Weak scaling: every rank draws its own a.batch lines.  --split: the global minibatch of
    a.batch lines (seed 1000) is sorted by length and dealt round-robin to the ranks (SURVEY.md section 8(e))."""
    if not a.split:
        return synth.make_lines(a.batch, lines_T(a), 48, a.nclasses, seed=1000 + rank)
    x, T, labels, L = synth.make_lines(a.batch, lines_T(a), 48, a.nclasses, seed=1000)
    if world == 1:
        return x, T, labels, L
    offs = np.concatenate([[0], np.cumsum(T)])
    loffs = np.concatenate([[0], np.cumsum(L)])
    order = np.argsort(-T, kind="stable")
    mine = order[rank::world]
    xs = np.concatenate([x[offs[b]:offs[b + 1]] for b in mine], 0)
    labs = np.concatenate([labels[loffs[b]:loffs[b + 1]] for b in mine])
    return np.ascontiguousarray(xs), T[mine].copy(), labs.astype(np.int32), L[mine].copy()


DUMP_BYTES = 64 << 20


def dump_outputs(d, net, mpl):
    """What a caller of the timed step receives after it (rank 0): the decoded transcripts (clstm_b200_fetch_decoded,
    classes and column locations per line, padded with -1), the updated weights and the momentum buffer, as float32
    DIR/<name>.npy.  An array above its share of DUMP_BYTES is replaced by a sample of its elements at seeded positions
    (the same for the same arguments)."""
    dec = net.fetch_decoded(mpl)
    cls = np.full((len(dec), mpl), -1, np.float32)
    locs = np.full((len(dec), mpl), -1, np.float32)
    for b, (c, l) in enumerate(dec):
        cls[b, :len(c)] = c
        locs[b, :len(l)] = l
    outs = {"decoded_classes": cls, "decoded_locations": locs, "params": net.get_params(), "momentum": net.get_derivs()}
    os.makedirs(d, exist_ok=True)
    cap = DUMP_BYTES // len(outs) // 4
    for name, v in outs.items():
        if v.size > cap:
            v = v.ravel()[np.sort(np.random.default_rng(0).choice(v.size, cap, replace=False))]
        np.save(os.path.join(d, name + ".npy"), v)


# ------------------------------------------------------------------------------------------ reference arm (CPU)
def cpu_reference(a, budget_s, threads):
    """Times the CPU oracle port (reference algorithm, oracle/clstm_oracle.cc) on a bounded sample of the workload:
    `threads` host threads each run whole lines (fwdbwd per line, one sgd_update per repetition).  The sample holds at
    least as many lines as threads (several minibatches' worth if the workload's batch is smaller), so every thread has
    work."""
    from oracle import binding as ob
    net = ob.BidiOracle(48, a.nhidden, a.nclasses, seed=0.222)
    nl = max(1, threads)
    parts = []
    k = 0
    while sum(len(p[1]) for p in parts) < nl:
        parts.append(synth.make_lines(a.batch, lines_T(a), 48, a.nclasses, seed=1000 + k))
        k += 1
    x = np.concatenate([p[0] for p in parts], 0); T = np.concatenate([p[1] for p in parts])
    labels = np.concatenate([p[2] for p in parts]); L = np.concatenate([p[3] for p in parts])
    n_cols = int(T[:nl].sum())
    xs, Ts, Ls = x[: n_cols], T[:nl], L[:nl]
    labs = labels[: int(L[:nl].sum())]
    t = net.train_lines(xs, Ts, labs, Ls, LR, MOM, threads=threads, reps=1)      # warm-up + calibration
    reps = int(max(1, min(50, budget_s / max(t, 1e-3))))
    t = net.train_lines(xs, Ts, labs, Ls, LR, MOM, threads=threads, reps=reps)
    px = reps * n_cols * 48
    return {"value": px / t, "unit": "px/s", "cores": threads, "kind": "port",
            "sample": "%d line(s) x %d rep(s) of the workload (%s), %d host thread(s), fwdbwd per line + one "
                      "sgd_update per rep; reference's O(T^2) anynan asserts excluded" % (
                          nl, reps, ("T=%d" % a.T) if a.Tmax <= a.T else "T=%d..%d" % (a.T, a.Tmax), threads),
            "seconds": t}


def normalizer_leg(net, a):
    """Side measurement (not part of `value`): the step in front of the path, CenterNormalizer measure + normalize of
    one batch of raw 60-row line images from host memory into the resident input batch (clstm_b200_normalize_batch),
    next to the CPU restatement of extras.cc on one line."""
    B, h, w = min(a.batch, 32), 60, 640
    imgs = [synth.make_raw_line(w, h, seed=900 + b) for b in range(B)]
    net.normalize_batch(imgs, "center")
    net.profile(True)
    reps = 5
    t0 = time.perf_counter()
    for _ in range(reps):
        T = net.normalize_batch(imgs, "center")
    dt = (time.perf_counter() - t0) / reps
    stats = net.phase_stats()
    net.profile(False)
    dev_ms = stats.get("normalize", (0.0, 0))[0] / reps
    res = {"kind": "center", "lines": B, "raw_shape": [h, w], "normalized_columns": int(T.sum()),
           "ms_per_batch_host_to_resident": dt * 1e3, "device_ms_per_batch": dev_ms,
           "value": B * w * h / dt, "unit": "raw px/s", "launches_per_batch": stats.get("normalize", (0.0, 0))[1] / reps}
    # training straight from raw lines through the two-deep input pipeline: normalisation of batch i+1 runs on the copy
    # stream underneath step i (clstm_b200_prefetch_raw_batch / step_prefetched / fetch_decoded)
    rng = np.random.default_rng(5)
    L = [20] * B
    labels = rng.integers(1, a.nclasses, 20 * B).astype(np.int32)
    mpl = int(T.max()) // 2 + 1
    net.prefetch_raw_batch(imgs, labels, L)

    def raw_step():
        net.step_prefetched(LR, MOM, CLIP)
        net.prefetch_raw_batch(imgs, labels, L)
        net.fetch_decoded(mpl)
    for _ in range(3):
        raw_step()
    t0 = time.perf_counter()
    for _ in range(10):
        raw_step()
    res["train_from_raw_ms_per_step"] = (time.perf_counter() - t0) / 10 * 1e3
    res["train_from_raw_note"] = "wall clock per step incl. H2D of the raw pixels, device normalisation of the next batch, the training step on %d normalised columns and the D2H of its result" % int(T.sum())
    if not a.no_cpu_baseline:
        from oracle import binding as ob
        t0 = time.perf_counter()
        ob.center_line(imgs[0])
        res["cpu_port_px_per_s"] = w * h / (time.perf_counter() - t0)
    return res


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ncpu = os.cpu_count() or 1
    vals = []
    # a sample of the big configs is long: bound every repetition
    per_step = 2.0 if a.nhidden <= 100 else 6.0
    # best-effort CPU arm: all hardware threads are not always the fastest (SMT siblings, memory bandwidth), so the thread
    # count is calibrated on short samples (this doubles as the warm-up) and the best one is timed
    cand = sorted({ncpu, max(1, ncpu // 2), max(1, ncpu // 4)}, reverse=True)
    calib = {th: cpu_reference(a, 0.5, th)["value"] for th in cand}
    cores = max(calib, key=calib.get)
    for _ in range(max(1, min(a.steps, 5))):
        vals.append(cpu_reference(a, per_step, cores))
    px = sum(v["value"] * v["seconds"] for v in vals)
    sec = sum(v["seconds"] for v in vals)
    val = px / sec
    out = {"impl": "reference", "metric": "text-line-pixels/sec (fwd+bwd+CTC+update)", "value": val, "unit": "px/s",
           "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1000.0 * sec / max(1, len(vals)),
           "higher_is_better": True, "scaling": "strong" if a.split else "weak", "vs_baseline": None, "dtype": "f32",
           "data": "synthetic",
           "config": {"workload": workload_name(a, max(1, a.gpus)), "note": "reference CPU path = oracle port (Eigen absent, "
                      "reference not buildable); each step = bounded sample (>= one line per host thread), all host threads",
                      "samples_timed": len(vals), "host_threads_available": ncpu,
                      "thread_calibration_px_per_s": {str(k): v for k, v in calib.items()}},
           "cpu_baseline": {"value": val, "unit": "px/s", "cores": cores, "kind": "port", "sample": vals[-1]["sample"]},
           "e2e": {"value": val, "unit": "px/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out))


# ------------------------------------------------------------------------------------------ B200 arm
def run_b200(a):
    import torch
    import torch.distributed as dist
    import clstm_b200

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != a.gpus and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (a.gpus, world))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 path has no CPU fallback")
    if a.split and a.batch % world:
        raise SystemExit("--split: global batch %d not divisible by %d ranks" % (a.batch, world))
    torch.cuda.set_device(local)
    sampler = ClockSampler(local)                       # every rank, long before the timed region
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    dp_mode = "none"
    init = synth.reference_init(48, a.nhidden, a.nclasses, seed=0.222)
    net = clstm_b200.Net(48, a.nhidden, a.nclasses, device=local)
    net.set_params(init)
    if world > 1:
        idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(clstm_b200.Net.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0)
        net.comm_init(bytes(idt.cpu().numpy().tobytes()), rank, world)
        if os.environ.get("CLSTM_B200_DP", "p2p") != "nccl" and world <= 8:
            # NVLink peer-memory path: one fused kernel reads every rank's derivatives and applies the update
            mine = torch.frombuffer(bytearray(net.p2p_handle()), dtype=torch.uint8).cuda()
            allh = [torch.zeros(64, dtype=torch.uint8, device="cuda") for _ in range(world)]
            dist.all_gather(allh, mine)
            net.p2p_connect([bytes(h.cpu().numpy().tobytes()) for h in allh], rank, world)
            dp_mode = "p2p-fused"
        else:
            dp_mode = "nccl"

    x, T, labels, L = make_batch(a, rank, world)
    N = int(T.sum())
    cols = torch.tensor([N], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(cols)
    px_per_step = float(cols.item()) * 48                 # whole job, all ranks
    hx = clstm_b200.pinned_array(x.shape, np.float32); hx[...] = x   # pinned host copy for the end-to-end path
    stream = torch.cuda.ExternalStream(net.stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # > 126 MB L2

    def l2_flush():
        with torch.cuda.stream(stream):
            flush.zero_()

    def timed(fn, iters):
        """per-iteration device time (ms) of `iters` calls, each after an L2 flush; elementwise max over ranks"""
        evs = []
        for _ in range(iters):
            l2_flush()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            fn()
            e1.record(stream)
            evs.append((e0, e1))
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1) for e0, e1 in evs], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.cpu().numpy()

    # ---- resident-batch measurement (value)
    net.upload_batch(hx, T, labels, L)
    step_res = lambda: net.step_resident(LR, MOM, CLIP)  # noqa: E731
    warm = max(3, a.warmup)
    timed(step_res, warm)                                 # warm-up
    if dp_mode == "p2p-fused":
        net.peer_stats()                                  # arm the in-kernel counters of the fused all-reduce + update
    iters = a.steps
    net.synchronize()
    barrier()
    t0 = time.time()
    ms_it = timed(step_res, iters)                # the timed region of `value`: no phase events, nothing but the step
    barrier()
    t1 = time.time()
    clocks = sampler.stop(t0, t1)
    ms_step = float(np.median(ms_it))
    value = px_per_step / (ms_step / 1000.0)
    peer = net.peer_stats() if dp_mode == "p2p-fused" else None
    mpl = int(T.max()) // 2 + 1
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, net, mpl)
    # second pass with per-phase CUDA events for the kernel table / roofline (everything on one stream)
    net.profile(True)
    prof_iters = min(iters, max(3, a.steps))
    timed(step_res, prof_iters)
    stats = net.phase_stats()
    net.profile(False)

    # ---- end to end through the public C ABI with host buffers.  Two ways a caller can drive it:
    #  pipeline : the training-loop form -- while step i runs, batch i+1 is staged from pinned host memory on the copy
    #             stream (clstm_b200_prefetch_batch), then clstm_b200_fetch_decoded(i) reads the result back.
    #  sync     : clstm_b200_train_step per batch (upload, step, fetch; nothing overlaps)
    # Every timed iteration contains one full H2D of a batch and one D2H of a step's decoded result.
    def pipe_fn():
        net.step_prefetched(LR, MOM, CLIP)          # batch i (staged during step i-1)
        net.prefetch_batch(hx, T, labels, L)        # H2D of batch i+1 overlaps the kernels of step i
        net.fetch_decoded(mpl)                      # D2H of step i's result, synchronises
    net.prefetch_batch(hx, T, labels, L)
    for _ in range(3):
        pipe_fn()
    barrier()
    ms_e2e_it = timed(pipe_fn, iters)
    barrier()
    ms_e2e = float(np.median(ms_e2e_it))
    e2e = px_per_step / (ms_e2e / 1000.0)
    e2e_obj = {"value": e2e, "unit": "px/s", "ms_per_step": ms_e2e, "ms_per_step_mean": float(ms_e2e_it.mean()),
               "h2d_bytes_per_step": int(x.nbytes + T.nbytes * 5 + labels.nbytes + 8 * len(T)),
               "d2h_bytes_per_step": int(len(T) * 4 + 2 * len(T) * mpl * 4 + 4),
               "bytes_note": "per rank", "mode": "input pipeline: prefetch_batch(i+1) on the copy stream during step i, fetch_decoded(i)"}
    if not a.no_extras:
        sync_fn = lambda: net.train_step(hx, T, labels, L, LR, MOM, CLIP, max_per_line=mpl)  # noqa: E731
        for _ in range(3):
            sync_fn()
        barrier()
        ms_sync = float(np.median(timed(sync_fn, iters)))
        barrier()
        e2e_obj.update(sync_value=px_per_step / (ms_sync / 1000.0), sync_ms_per_step=ms_sync,
                       sync_mode="clstm_b200_train_step per batch, nothing overlapped")

    # ---- data-parallel check (N > 1): one update from the same start on (a) the N ranks, each on its shard, and (b) one
    # GPU on the whole minibatch must give the same weights (share_deltas semantics, clstm.cc:731-744; SURVEY 8(d) cfg4)
    dp_check = None
    if world > 1:
        net.set_params(init)
        net.clear_derivs()
        net.upload_batch(hx, T, labels, L)
        net.step_resident(LR, MOM, CLIP)
        p_dp = net.get_params()
        dig = np.frombuffer(hashlib.sha256(p_dp.tobytes()).digest()[:8], dtype=np.int64).copy()
        digs = [torch.zeros(1, dtype=torch.int64, device="cuda") for _ in range(world)]
        dist.all_gather(digs, torch.from_numpy(dig).cuda())
        same = all(int(d.item()) == int(digs[0].item()) for d in digs)
        dp_check = {"ranks_bit_identical": bool(same)}
        if rank == 0:
            shards = [make_batch(a, r, world) for r in range(world)]
            gx = np.concatenate([s[0] for s in shards], 0); gT = np.concatenate([s[1] for s in shards])
            gl = np.concatenate([s[2] for s in shards]); gL = np.concatenate([s[3] for s in shards])
            single = clstm_b200.Net(48, a.nhidden, a.nclasses, device=local)
            single.set_params(init)
            single.upload_batch(gx, gT, gl, gL)
            single.step_resident(LR, MOM, CLIP)
            p1 = single.get_params()
            single.close()
            # how far two single-GPU evaluations of the SAME minibatch are apart when only the fp32 summation order of the
            # derivative products differs (tcgen05 split-K tiles vs fp32 SIMT tiles): the noise floor of this comparison
            os.environ["CLSTM_B200_GEMM"] = "simt"
            alt = clstm_b200.Net(48, a.nhidden, a.nclasses, device=local)
            os.environ.pop("CLSTM_B200_GEMM", None)
            alt.set_params(init)
            alt.upload_batch(gx, gT, gl, gL)
            alt.step_resident(LR, MOM, CLIP)
            p2 = alt.get_params()
            alt.close()
            dp_check["fp32_order_noise_1gpu_rel"] = float(np.abs(p2 - p1).max() / max(np.abs(p1).max(), 1e-30))
            dp_check["max_rel_err_vs_1gpu"] = float(np.abs(p_dp - p1).max() / max(np.abs(p1).max(), 1e-30))
            dp_check["max_rel_update_err_vs_1gpu"] = float(np.abs((p_dp - init) - (p1 - init)).max() / max(np.abs(p1 - init).max(), 1e-30))
            dp_check["note"] = ("one update from the reference init: N ranks on their shards (fused NVLink all-reduce + update) "
                                "vs one GPU on the concatenated minibatch; bar 1e-5 relative (SURVEY 8(d)) -- met where the derivative sums are short "
                                "(cfg2: 16 000 columns); for 282 000-column sums (cfg4) read it against fp32_order_noise_1gpu_rel, the distance "
                                "between two single-GPU evaluations that differ only in fp32 summation order")
        barrier()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel from the live phase timings
    pk = peaks()
    no, ni, nc = a.nhidden, 48, a.nclasses
    P = synth.nparams(ni, no, nc)
    alg = {   # per launch of the phase (one step, this rank): (flops, bytes, bound)
        "xproj_gemm": (2.0 * 2 * N * 4 * no * ni, None, "tensor"),
        "lstm_fwd": (2.0 * 2 * N * 4 * no * no, None, "tensor"),
        "softmax_fwd": (2.0 * N * nc * 2 * no, None, "tensor"),
        "ctc_align": (None, 8.0 * N * nc, "hbm"),
        "softmax_bwd": (2.0 * 2 * N * nc * 2 * no, None, "tensor"),
        "lstm_bwd": (2.0 * 2 * N * 4 * no * no, None, "tensor"),
        "wgrad_gemm": (2.0 * 2 * N * 4 * no * (ni + no), None, "tensor"),
        "dx_gemm": (2.0 * 2 * N * 4 * no * ni, None, "tensor"),
        "sgd_update": (None, 16.0 * P, "hbm"),
        "decode": (None, 8.0 * N, "hbm"),          # per-column argmax index + value (DESIGN.md section 3)
    }
    kernels = {}
    for name, (ms, launches) in stats.items():
        if name in alg and ms > 0:
            fl, by, bound = alg[name]
            per = ms / prof_iters / 1000.0
            if bound == "tensor":
                ach = fl / per / 1e12; peak = pk["bf16_tflops"]; unit = "TFLOP/s"
            else:
                ach = by / per / 1e9; peak = pk["hbm_gbs"]; unit = "GB/s"
            kernels[name] = {"ms_per_step": ms / prof_iters, "launches_per_step": launches / prof_iters, "bound": bound,
                             "achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak}
    dom = max(kernels, key=lambda k: kernels[k]["ms_per_step"])
    roof = dict(kernels[dom]); roof["kernel"] = dom; roof["traffic"] = None
    try:   # DRAM bytes per launch of that kernel from the committed `ncu --set full` capture of the same configuration
        summ = json.load(open(os.path.join(ROOT, "profiles", "r2_summary.json")))
        for cap in summ.get("full_capture", []):
            if cap.get("config") == a.config and cap.get("phase") == dom:
                roof["traffic"] = cap["dram_bytes_per_launch"]
                roof["traffic_unit"] = "bytes per launch (ncu --set full, profiles/r2_summary.json)"
    except Exception:
        pass
    roof["peak_source"] = pk["src"]
    roof.pop("ms_per_step"); roof.pop("launches_per_step")
    roof["kernel_ms"] = kernels[dom]["ms_per_step"]
    roof["lstm_kernel"] = net.lstm_variant
    launches = int(round(sum(c for (_, c) in stats.values()) / prof_iters))

    out = {"metric": "text-line-pixels/sec (fwd+bwd+CTC+update)", "value": value, "unit": "px/s", "n_gpus": world,
           "steps": a.steps, "warmup": warm, "ms_per_step": ms_step, "ms_per_step_mean": float(ms_it.mean()),
           "ms_per_step_min": float(ms_it.min()), "ms_per_step_max": float(ms_it.max()),
           "step_ms": [round(float(v), 4) for v in ms_it[:400]],
           "higher_is_better": True, "scaling": "strong" if a.split else "weak", "vs_baseline": None, "dtype": "f32",
           "data": "synthetic",
           "config": {"workload": workload_name(a, world), "config": a.config,
                      "lines_per_gpu": len(T), "global_lines": a.batch if a.split else a.batch * world,
                      "columns_per_gpu": N, "global_columns": int(px_per_step // 48),
                      "l2": "flushed between timed iterations (256 MiB memset)",
                      "timing": "median over %d steps, each its own CUDA-event pair, per-step max over ranks" % a.steps,
                      "weights": "reference LCG init (negbiased, 0.01), seed 0.222", "lr": LR, "momentum": MOM,
                      "lstm_kernel": net.lstm_variant, "parallelism": "dp%d" % world,
                      "grad_exchange": dp_mode},
           "e2e": e2e_obj,
           "gpu_launches": launches, "clocks": clocks, "roofline": roof, "kernels": kernels,
           "allreduce_ms_per_step": (stats.get("allreduce", (0.0, 0))[0] / prof_iters) if world > 1 else 0.0}
    if dp_check is not None:
        out["dp_check"] = dp_check
    if peer is not None and peer["launches"] > 0:
        peer["nvlink_read_gbs"] = peer["nvlink_bytes_per_launch"] / max(peer["data_us"], 1e-9) / 1e3
        peer["note"] = ("peer_allreduce_update_kernel, rank 0, in-kernel %globaltimer: wait_us = arrive-flag spin until the slowest rank "
                        "published its derivatives, data_us = peer reads over NVLink + clip + update (block 0's share of the grid-stride loop)")
        out["fused_allreduce"] = peer
    if world == 1 and not a.no_extras:
        out["normalizer"] = normalizer_leg(net, a)
    if world == 1 and not a.no_cpu_baseline:
        cb = cpu_reference(a, a.cpu_seconds, 1)
        cb.pop("seconds")
        out["cpu_baseline"] = cb
    else:
        out["cpu_baseline"] = None
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)
