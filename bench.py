#!/usr/bin/env python
"""bench.py - MUSIC DOA windows/s on B200 (BASELINE.json metric), one JSON line on stdout.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config 2] [--impl ours|reference] [--dump-outputs DIR]
  N > 1:  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path (covariance -> eigenvectors -> pseudospectrum -> peak pick) over one batch of
synthetic windows per GPU: BASELINE.json configs[1] = M=4 antennas, 4096-snapshot windows, 3600-angle grid, 10 000
windows (1.31 GB, larger than the 126 MB L2, so every step streams from HBM).

  value     windows/s, whole job, inputs resident in HBM, device-timed (CUDA events on the launch stream), max over ranks.
  e2e       same metric through the reference-facing block API (music_doa.work -> C ABI process_host) with HOST buffers:
            H2D of the windows and D2H of the results are inside the timed region.  N = 1: one block on one GPU, pinned
            input (value) and pageable input (registered by the library on first sight).  N > 1: ONE block whose handle
            owns all N GPUs (music_b200_create_multi), one work() call per step from rank 0's process; the per-rank-blocks
            figure (N processes, one block each) is reported beside it.
  roofline  the dominant (HBM-touching) kernel; algorithmic bytes per window (8*M*N + 8*n + 4*n, SURVEY.md 8d) x windows
            per launch / its measured duration.
  cpu_baseline  the C oracle (a port of the reference's work()) timed on the host cores, one PROCESS per hardware thread.
  other_configs BASELINE configs[2..4] (M=8 / M=16 shapes) at their stated window counts: windows/s, HBM and FP64-pipe
            fractions, and a peak-bin comparison with the C oracle on sampled windows.
  --impl reference  times that same CPU port with all host threads (the reference arm).

Multi-GPU: windows shard round-robin (w -> GPU w mod G, SURVEY.md 8e); weak scaling (each GPU keeps its 10 000
windows/step).  The all-gather of the int32 peak bins is fused into the scan epilogue: every GPU stores its bins straight
into every peer's stream-ordered buffer over NVLink (peer-mapped memory, music_b200_gather_*); no collective kernel runs
inside the timed region.  ncclAllGather of the same bins is the check (after the timed region).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from gr_baz_b200 import sharding, synth  # noqa: E402
from gr_baz_b200.music_doa_helper import calculate_antenna_array_response  # noqa: E402

FP64_DFMA_PER_CLK_PER_SM = 64.0  # measured, profiles/r01_microbench.txt (DESIGN.md section 3)
POOL_WINDOWS = 4096              # distinct synthetic windows behind the large (configs 3-5) streams
DUMP_BYTES = 64 << 20            # --dump-outputs: at most this much in all


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, help="BASELINE.json config index (1-based, default 2)")
    ap.add_argument("--windows", type=int, default=0, help="windows per step per GPU (default: config's, capped by memory)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-next-rows", action="store_true", help="skip the planar-input and device-retune legs (SURVEY 8(f) rows)")
    ap.add_argument("--no-other-configs", action="store_true", help="skip BASELINE configs[2..4]")
    ap.add_argument("--nccl-gather", action="store_true", help="N > 1: all-gather the bins with NCCL instead of the fused peer stores (A/B)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (rank 0's windows: angles, levels, bins) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return args


def dump_outputs(out_dir, arrays, limit=DUMP_BYTES):
    """arrays: name -> (W, ...) device tensor.  Angles and levels are written as float32, bins as float64 (exact).  Above
    `limit` bytes in all, a fixed seeded sample of the windows is written, with its indices as window_index.npy."""
    host = {k: v.cpu().numpy().astype(np.float64 if k == "bins" else np.float32) for k, v in arrays.items()}
    W = len(host["bins"])
    per_window = sum(a[:1].nbytes for a in host.values())
    if W * per_window > limit:
        keep = np.sort(np.random.default_rng(0).choice(W, limit // (per_window + 8), replace=False))
        host = {k: a[keep] for k, a in host.items()}
        host["window_index"] = keep.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in host.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def workload(cfg_id, windows_override=0):
    cfg = synth.config(cfg_id)
    W = windows_override or min(cfg["windows"], {2: 10000, 3: 4096, 4: 8192, 5: 4096}.get(cfg_id, 10000))
    return cfg, W


def bytes_per_window(cfg):
    return 8 * cfg["m"] * cfg["snapshots"] + 8 * cfg["n"] + 4 * cfg["n"]


def dfma_per_window(cfg):
    """fp64 multiply-adds the path cannot avoid: Hermitian-half covariance (2*M^2 per snapshot) + the complement-form
    scan (4*M*n + 2 per bin) for n < M - n, the direct form otherwise (SURVEY.md section 8d's flop count / 2)."""
    M, N, K, n = cfg["m"], cfg["snapshots"], cfg["resolution"], cfg["n"]
    scan = (4 * M * n + 2) if n < M - n else (4 * M * (M - n) + 2 * (M - n))
    return 2 * M * M * N + K * scan


def table_for(cfg):
    arr = [[synth.SPACING * x, synth.SPACING * y] for x, y in cfg["antenna_array"]]
    resp = calculate_antenna_array_response(arr, cfg["resolution"], synth.C_LIGHT / synth.FREQUENCY)
    return resp, np.asarray(resp, dtype=np.complex128).astype(np.complex64)


def metric_name(cfg):
    return "MUSIC windows/sec (M=%d ant x %d snap x %d angle)" % (cfg["m"], cfg["snapshots"], cfg["resolution"])


def workload_name(cfg, cfg_id, W):
    return "BASELINE configs[%d]: M=%d, %d-snapshot windows, %d-angle grid, n=%d, %d windows/step/GPU" % (
        cfg_id - 1, cfg["m"], cfg["snapshots"], cfg["resolution"], cfg["n"], W)


def config_dict(cfg, cfg_id, W, G):
    """The `config` object - identical in the GPU arm and the reference arm (the driver compares them)."""
    return {"workload": workload_name(cfg, cfg_id, W), "windows_per_step": W * G,
            "l2": "inputs %.2f GB/step/GPU > 126 MB L2 (no flush needed)" % (W * cfg["nsamples"] * 8 / 1e9),
            "sharding": "round-robin w mod G, peak bins gathered on every GPU" if G > 1 else "single GPU",
            "snr_db": cfg["snr_db"], "geometry": cfg["geometry"]}


# ------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": float(max(pw))}


# ------------------------------------------------------------------------------------------
# CPU arm: the C port of the reference's work(), one PROCESS per hardware thread.  (Round 1 ran 128 threads in one
# process and measured 8 % to 45 % parallel efficiency depending on the box: the port keeps the reference's per-window
# 256 KiB allocation, and one address space serialises those; independent processes - which is also how independent
# GNU Radio flowgraphs would run - do not.)
_W = {}


def _cpu_worker_init(cfg_id, over, seed, first, count):
    from oracle import c_oracle

    c_oracle.lib()
    cfg = synth.config(cfg_id, **over)
    _W["cfg"] = cfg
    _W["table"] = table_for(cfg)[1]
    _W["x"] = synth.gen_windows_numpy(cfg, seed, first, count)
    _W["co"] = c_oracle


def _cpu_worker_run(reps):
    cfg = _W["cfg"]
    t = time.perf_counter()
    for _ in range(reps):
        _W["co"].work_batch(_W["x"], cfg["m"], cfg["n"], _W["table"], want_P=False)
    return time.perf_counter() - t


def _cpu_worker_entry(conn, cfg_id, over, seed, first, count):
    try:
        try:
            os.sched_setaffinity(0, os.sched_getaffinity(0))
        except Exception:
            pass
        _cpu_worker_init(cfg_id, over, seed, first, count)
        conn.send("ready")
        while True:
            msg = conn.recv()
            if msg is None:
                break
            conn.send(_cpu_worker_run(msg))
    except Exception as e:  # pragma: no cover
        try:
            conn.send(("error", repr(e)))
        except Exception:
            pass


class CpuArm:
    """`procs` worker processes, each holding `per` windows of the config's stream; run(reps) = one synchronous pass of
    every worker over its windows `reps` times; returns the wall-clock seconds of the slowest-started-to-last-finished."""

    def __init__(self, cfg_id, seed, procs, per):
        import multiprocessing as mp

        ctx = mp.get_context("spawn")  # never fork a process that holds a CUDA context
        self.procs, self.per = procs, per
        self.conns, self.ps = [], []
        for i in range(procs):
            a, b = ctx.Pipe()
            p = ctx.Process(target=_cpu_worker_entry, args=(b, cfg_id, {}, seed, i * per, per), daemon=True)
            p.start()
            self.conns.append(a)
            self.ps.append(p)
        for c in self.conns:
            msg = c.recv()
            if msg != "ready":
                raise RuntimeError("CPU worker failed: %r" % (msg,))

    def run(self, reps):
        t = time.perf_counter()
        for c in self.conns:
            c.send(reps)
        inner = [c.recv() for c in self.conns]
        dt = time.perf_counter() - t
        for v in inner:
            if isinstance(v, tuple):
                raise RuntimeError("CPU worker failed: %r" % (v,))
        return dt, inner

    def close(self):
        for c in self.conns:
            try:
                c.send(None)
            except Exception:
                pass
        for p in self.ps:
            p.join(timeout=5)


def cgroup_cpu_quota():
    """CPUs this container may use according to its cgroup (v2 cpu.max or v1 cfs quota), or None if unlimited / unknown."""
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            return float(q) / float(per)
    except Exception:
        pass
    try:
        q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        if q > 0 and per > 0:
            return q / per
    except Exception:
        pass
    return None


def host_threads():
    """Worker processes of the CPU arm: the CPUs this process may run on, capped by the container's CPU quota (an affinity
    mask of 128 under a 10-CPU quota would only oversubscribe the quota and report a core count the arm never had)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    q = cgroup_cpu_quota()
    if q:
        n = max(1, min(n, int(q + 0.999)))
    return n


def one_core_rate(cfg, table_c64, seed):
    from oracle import c_oracle

    c_oracle.lib()
    x0 = synth.gen_windows_numpy(cfg, seed, 0, 8)
    c_oracle.work_batch(x0, cfg["m"], cfg["n"], table_c64, want_P=False)
    t = time.perf_counter()
    c_oracle.work_batch(x0, cfg["m"], cfg["n"], table_c64, want_P=False)
    return 8.0 / (time.perf_counter() - t)


def cpu_port_throughput(cfg_id, cfg, table_c64, seed, budget_s, procs):
    """windows/s of the C port on `procs` worker processes over a bounded sample of the same synthetic stream."""
    r1 = one_core_rate(cfg, table_c64, seed)
    per = int(max(4, min(64, budget_s * r1 / 4)))  # windows held by each worker
    arm = CpuArm(cfg_id, seed, procs, per)
    try:
        dt, _ = arm.run(1)  # warm-up, and the pass time that sizes the timed run
        reps = int(max(1, min(400, round(budget_s / max(dt, 1e-3)))))
        dt, inner = arm.run(reps)
    finally:
        arm.close()
    total = procs * per * reps
    return {"value": total / dt, "windows": total, "seconds": dt, "value_1core": r1, "procs": procs, "per_proc": per, "reps": reps,
            "parallel_efficiency": (total / dt) / (r1 * procs), "slowest_worker_s": max(inner), "fastest_worker_s": min(inner)}


def reference_source_rate(cfg, table, seed, threads):
    """Informational: the reference's own work() source where oracle/_ref was prebuilt (it runs behind a stand-in Armadillo
    header, so it is NOT the reference's real speed - DESIGN.md section 2)."""
    try:
        from concurrent.futures import ThreadPoolExecutor

        from oracle import ref_build

        if not ref_build.available():
            return {"unavailable": "oracle/_ref not built"}
        os.environ.setdefault("OPENBLAS_NUM_THREADS", "1")
        ref_build.lib()
        S2 = threads * 2
        x = synth.gen_windows_numpy(cfg, seed, 0, S2)
        parts = np.array_split(np.arange(S2), threads)

        def job(idx):
            return ref_build.work_batch(x[idx[0]:idx[-1] + 1], cfg["m"], cfg["n"], table, want_spectrum=False)["angles"]

        with ThreadPoolExecutor(threads) as ex:
            list(ex.map(job, parts))
            t2 = time.perf_counter()
            list(ex.map(job, parts))
            dt2 = time.perf_counter() - t2
        return {"value": S2 / dt2, "unit": "windows/s", "cores": threads, "windows": S2,
                "what": "reference lib/baz_music_doa.cc compiled unmodified against stand-in GNU Radio/Armadillo headers "
                        "(LAPACK zheevd / BLAS zgemm from scipy's OpenBLAS), threads in one process; informational"}
    except Exception as e:  # informational leg: never let it take the reference arm down
        return {"unavailable": str(e)[:200]}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cfg, W = workload(args.config, args.windows)
    _, table = table_for(cfg)
    seed = synth.BASE_SEED + args.config
    procs = host_threads()
    r1 = one_core_rate(cfg, table, seed)
    total = args.steps + max(args.warmup, 1)
    # each step: every worker passes once over its windows; sized so that the whole run stays within ~1.5 min
    per = int(max(2, min(256, (80.0 / total) * r1)))
    arm = CpuArm(args.config, seed, procs, per)
    try:
        for _ in range(max(args.warmup, 1)):
            arm.run(1)
        t = time.perf_counter()
        for _ in range(args.steps):
            arm.run(1)
        dt = time.perf_counter() - t
    finally:
        arm.close()
    S = procs * per
    value = S * args.steps / dt
    sample = ("%d windows/step of the config-%d stream (first %d of %d), %d worker processes x %d windows, C port of work() "
              "(-O3 -DNDEBUG), parallel efficiency %.2f vs %d x the 1-core rate %.0f/s" % (S, args.config, S, W, procs, per, value / (r1 * procs), procs, r1))
    line = {
        "impl": "reference", "metric": metric_name(cfg), "value": value, "unit": "windows/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_dict(cfg, args.config, W, args.gpus),
        "cpu_baseline": {"value": value, "unit": "windows/s", "cores": procs, "kind": "port", "sample": sample,
                         "value_1core": r1, "parallel_efficiency": value / (r1 * procs), "effective_cores": value / r1,
                         "cgroup_cpu_quota": cgroup_cpu_quota()},
        "e2e": {"value": value, "unit": "windows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "reference_source": reference_source_rate(cfg, table, seed, procs),
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------
def interleave_host_memory():
    """Best effort: spread the pages of host buffers allocated from here on over all NUMA nodes (set_mempolicy
    MPOL_INTERLEAVE), so that N PCIe links pulling from ONE buffer are not all served by one socket's memory."""
    try:
        import ctypes

        nodes = [int(d[4:]) for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit()]
        if len(nodes) < 2:
            return "single NUMA node"
        mask = ctypes.c_ulong(sum(1 << n for n in nodes))
        libc = ctypes.CDLL(None, use_errno=True)
        rc = libc.syscall(238, 3, ctypes.byref(mask), ctypes.c_ulong(max(nodes) + 2))  # __NR_set_mempolicy, MPOL_INTERLEAVE
        return "interleaved over %d NUMA nodes" % len(nodes) if rc == 0 else "set_mempolicy failed (errno %d)" % ctypes.get_errno()
    except Exception as e:
        return "not set (%s)" % e


def default_host_memory():
    try:
        import ctypes

        ctypes.CDLL(None).syscall(238, 0, None, ctypes.c_ulong(0))  # MPOL_DEFAULT
    except Exception:
        pass


def time_work(blk, We, x_np, outs, steps, sync):
    for _ in range(2):
        blk.work(We, [x_np], outs)
    sync()
    t0 = time.perf_counter()
    for _ in range(steps):
        blk.work(We, [x_np], outs)  # synchronous: returns when the results are in host memory
    return time.perf_counter() - t0


def run_other_config(cid, args, torch, dist, dev, local, rank, G, peak_hbm, sm_mhz):
    """One of BASELINE configs[2..4] at its stated window count (per GPU: count / G), device resident."""
    from gr_baz_b200.music_doa import music_doa
    from oracle import c_oracle

    cfg = synth.config(cid)
    resp, table = table_for(cfg)
    seed = synth.BASE_SEED + cid
    n, K = cfg["n"], cfg["resolution"]
    total = cfg["windows"]
    # C3 is a 1-GPU config (100 k windows); C4 / C5 are 1 M windows over 8 GPUs = 125 k per GPU, which is also what one
    # GPU runs here when N < 8 (weak scaling, like the headline)
    W = total if cid == 3 else total // 8
    free_b, _ = torch.cuda.mem_get_info()
    W = int(min(W, (free_b - (6 << 30)) // (cfg["nsamples"] * 8)))
    pool = min(POOL_WINDOWS, W)
    blk = music_doa(cfg["m"], n, cfg["nsamples"], resp, K, device=local)
    d_in = torch.empty((W, cfg["nsamples"] * 2), dtype=torch.float32, device=dev)
    # this rank's windows are i * G + rank; a pool of distinct windows is generated (bit-identical to the numpy
    # generator) and replicated device-to-device: every window has its own HBM address, the pool is >> L2
    widx = sharding.shard_indices(pool * G, G, rank)
    synth.gen_windows_torch(cfg, seed, 0, pool, dev, out=d_in[:pool], indices=widx)
    for w0 in range(pool, W, pool):
        c = min(pool, W - w0)
        d_in[w0:w0 + c].copy_(d_in[:c])
    d_ang = torch.empty((W, n), dtype=torch.float32, device=dev)
    d_lvl = torch.empty((W, n), dtype=torch.float32, device=dev)
    d_bins = torch.empty((W, n), dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream()

    d_all = torch.empty((G, W, n), dtype=torch.int32, device=dev) if G > 1 else None

    def step():
        blk.process_device(d_in.data_ptr(), W, d_ang.data_ptr(), d_lvl.data_ptr(), None, d_bins.data_ptr(), stream=stream.cuda_stream)
        if G > 1:  # BASELINE configs[3], [4]: "NCCL all-gather of peak indices" (gathered[r][i] <-> stream window i * G + r)
            dist.all_gather_into_tensor(d_all.view(-1), d_bins.view(-1))

    for _ in range(2):
        step()
    torch.cuda.synchronize()
    if G > 1:
        dist.barrier()
    reps = 3
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(reps):
        step()
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    if G > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    gathered_ok = None
    if G > 1:  # every rank's bins arrived in every rank's buffer
        gathered_ok = bool(torch.equal(d_all[rank], d_bins))
    # stage split of the same step (separate pass)
    blk.set_stage_timing(True)
    step()
    torch.cuda.synchronize()
    ms4, chunks = blk.stage_times_ms()
    blk.set_stage_timing(False)
    # peak bins against the C oracle on sampled windows of the pool (all of them distinct inputs)
    ns = min(256, pool)
    rng = np.random.default_rng(cid)
    sel = np.unique(np.concatenate([np.arange(min(16, pool)), rng.integers(0, pool, ns)]))
    x = d_in[torch.from_numpy(sel).to(dev)].cpu().numpy().view(np.complex64)
    got = d_bins[torch.from_numpy(sel).to(dev)].cpu().numpy()
    base = (W - 1) // pool * pool  # the last (possibly partial) replica of the pool holds the same inputs
    sel_last = sel[base + sel < W]
    last = d_bins[torch.from_numpy(base + sel_last).to(dev)].cpu().numpy()
    from concurrent.futures import ThreadPoolExecutor

    th = min(host_threads(), 32)
    parts = [p for p in np.array_split(np.arange(len(sel)), th) if len(p)]
    with ThreadPoolExecutor(th) as ex:
        refs = list(ex.map(lambda p: c_oracle.work_batch(x[p], cfg["m"], n, table, want_P=False)["bins"], parts))
    ref = np.concatenate(refs)
    mism = int(np.sum(np.any(got != ref, axis=1)))
    mism_last = int(np.sum(np.any(last != ref[:len(sel_last)], axis=1)))  # (sel is sorted: sel_last is its prefix)
    value = W * G / (ms * 1e-3)
    per_gpu = W / (ms * 1e-3)
    out = {"metric": metric_name(cfg), "value": value, "unit": "windows/s", "ms_per_step": ms, "windows_per_step": W * G,
           "windows_per_gpu": W, "distinct_windows_per_gpu": pool,
           "data": "synthetic; %d distinct windows per GPU (%.1f GB >> L2) replicated device-to-device to %d" % (pool, pool * cfg["nsamples"] * 8 / 1e9, W),
           "hbm_frac": bytes_per_window(cfg) * per_gpu / 1e9 / peak_hbm,
           "fp64_pipe_frac": dfma_per_window(cfg) * per_gpu / (FP64_DFMA_PER_CLK_PER_SM * 148 * sm_mhz * 1e6),
           "stages_ms": {"cov": ms4[0], "eig": ms4[1], "scan": ms4[2], "topn": ms4[3], "chunks": chunks},
           "bins_checked": int(len(sel)), "bins_mismatch": mism, "bins_mismatch_last_replica": mism_last,
           "checker": "C oracle (port of work()) on the same bytes"}
    if G > 1:
        out["gather"] = {"how": "ncclAllGather of int32 bins per step inside the timed region", "own_shard_ok": gathered_ok}
    blk.close()
    del d_in, d_ang, d_lvl, d_bins
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    _t00 = time.perf_counter()

    def leg(msg):  # progress of the legs on stderr (BENCH_VERBOSE=1); BENCH_WATCHDOG=<s> dumps every thread's stack every <s> seconds
        if os.environ.get("BENCH_VERBOSE"):
            print("[bench rank %s +%.1fs] %s" % (os.environ.get("RANK", "0"), time.perf_counter() - _t00, msg), file=sys.stderr, flush=True)

    if os.environ.get("BENCH_WATCHDOG"):
        import faulthandler

        faulthandler.dump_traceback_later(int(os.environ["BENCH_WATCHDOG"]), repeat=True, file=sys.stderr)

    from gr_baz_b200.music_doa import music_doa

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the product has no CPU path (use --impl reference for the CPU arm)")
    if world != args.gpus and world > 1:
        raise SystemExit("WORLD_SIZE (%d) != --gpus (%d)" % (world, args.gpus))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    cfg, W = workload(args.config, args.windows)
    resp, table = table_for(cfg)
    seed = synth.BASE_SEED + args.config
    n, K = cfg["n"], cfg["resolution"]
    G = world

    # this rank's shard of the global stream: windows w = i*G + rank  (round-robin)
    blk = music_doa(cfg["m"], n, cfg["nsamples"], resp, K, device=local)
    d_in = torch.empty((W, cfg["nsamples"] * 2), dtype=torch.float32, device=dev)
    widx = sharding.shard_indices(W * G, G, rank)  # round-robin: this rank's windows i*G + rank
    synth.gen_windows_torch(cfg, seed, 0, W, dev, out=d_in, indices=widx)
    d_ang = torch.empty((W, n), dtype=torch.float32, device=dev)
    d_lvl = torch.empty((W, n), dtype=torch.float32, device=dev)
    d_bins = torch.empty((W, n), dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream()

    # ---- the bins all-gather ---------------------------------------------------------------------------------------
    # default: fused into the scan epilogue (peer stores into every rank's stream-ordered buffer, epoch flags);
    # --nccl-gather: the round-1 form (async double-buffered ncclAllGather overlapping the next step), kept for A/B.
    fused_gather = G > 1 and not args.nccl_gather
    gathered = None  # torch view of this rank's stream-ordered gather buffer
    gather_fallback = None
    if fused_gather:
        # every rank takes every collective below whatever happens locally; if any rank cannot set the peer mapping up
        # (IPC refused, ...), ALL ranks fall back to the NCCL all-gather together
        ok, why = 1, ""
        mine = np.zeros(128, np.uint8)
        try:
            mine = np.frombuffer(blk.gather_create(W * G), dtype=np.uint8).copy()
        except Exception as e:
            ok, why = 0, repr(e)[:200]
        t_mine = torch.from_numpy(mine).to(dev)
        t_all = torch.empty((G, 128), dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(t_all.view(-1), t_mine)
        if ok:
            try:
                blk.gather_attach(G, rank, [bytes(t_all[r].cpu().numpy().tobytes()) for r in range(G)])
            except Exception as e:
                ok, why = 0, repr(e)[:200]
        t_ok = torch.tensor([ok], dtype=torch.int32, device=dev)
        dist.all_reduce(t_ok, op=dist.ReduceOp.MIN)
        if int(t_ok.item()) == 0:
            fused_gather = False
            gather_fallback = "fused all-gather unavailable on at least one rank (%s): ncclAllGather instead" % (why or "another rank")
            if rank == 0:
                print("[bench] " + gather_fallback, file=sys.stderr, flush=True)
    d_all2 = [torch.empty((G, W, n), dtype=torch.int32, device=dev), torch.empty((G, W, n), dtype=torch.int32, device=dev)] if (G > 1 and not fused_gather) else None
    d_bins2 = [d_bins, torch.empty_like(d_bins)]
    pending = [None, None]
    stepno = [0]

    def step():
        b = stepno[0] & 1 if (G > 1 and not fused_gather) else 0
        stepno[0] += 1
        if pending[b] is not None:
            pending[b].wait()
            pending[b] = None
        blk.process_device(d_in.data_ptr(), W, d_ang.data_ptr(), d_lvl.data_ptr(), None, d_bins2[b].data_ptr(),
                           stream=stream.cuda_stream)
        if G > 1 and not fused_gather:
            # gathered[r][i] <-> stream window w = i*G + r  (sharding.gathered_to_stream restores stream order)
            pending[b] = dist.all_gather_into_tensor(d_all2[b].view(-1), d_bins2[b].view(-1), async_op=True)

    def drain():
        if fused_gather:
            blk.gather_wait(stream.cuda_stream)  # returns (on the stream) when every rank's bins of the last step are here
        for b in range(2):
            if pending[b] is not None:
                pending[b].wait()
                pending[b] = None

    def sync_all():
        drain()
        torch.cuda.synchronize()
        if G > 1:
            dist.barrier()
        torch.cuda.synchronize()

    leg('setup done, warm-up')
    for _ in range(max(args.warmup, 3)):
        step()
    sync_all()

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    l0 = blk.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    e0.record(stream)
    for _ in range(args.steps):
        step()
    drain()  # the timed region ends when every rank holds every step's gathered bins
    e1.record(stream)
    sync_all()
    leg('timed region done')
    ms = e0.elapsed_time(e1)
    launches = blk.launch_count() - l0
    clocks = sampler.stop() if sampler else None
    if G > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        lt = torch.tensor([launches], dtype=torch.int64, device=dev)
        dist.all_reduce(lt)
        launches = int(lt.item())
    value = W * G * args.steps / (ms * 1e-3)

    leg('gather check')
    # the gathered bins against the collective they replace (outside the timed region)
    gather_check = None
    last_bins = d_bins2[(stepno[0] - 1) & 1 if (G > 1 and not fused_gather) else 0]
    if args.dump_outputs and rank == 0:  # before the untimed legs below reuse the output buffers
        dump_outputs(args.dump_outputs, {"angles": d_ang, "levels": d_lvl, "bins": last_bins})
    if G > 1:
        ref_all = torch.empty((G, W, n), dtype=torch.int32, device=dev)
        dist.all_gather_into_tensor(ref_all.view(-1), last_bins.view(-1))
        ref_stream = sharding.gathered_to_stream(ref_all, W * G)
        if fused_gather:
            torch.cuda.synchronize()
            mine_all = torch.from_numpy(blk.gather_read(W * G)).to(dev)
            gather_check = {"how": "peer stores from the scan epilogue into every rank's buffer + epoch flags (music_b200_gather_*)",
                            "equals_nccl_all_gather": bool(torch.equal(mine_all, ref_stream))}
        else:
            gather_check = {"how": "async double-buffered ncclAllGather", "equals_nccl_all_gather": True}
            if gather_fallback:
                gather_check["fallback"] = gather_fallback

    # sanity: the result of the timed work is a real answer (mirror-folded true bins at 20 dB)
    bins_h = last_bins.cpu().numpy()
    ok_frac = None
    if rank == 0 and not cfg.get("fixed_sources"):
        tb = synth.true_bins(cfg, seed, indices=widx)[:, 0]
        if cfg["geometry"] == "ula_x":
            tb = np.minimum(tb, (K - tb) % K)
        ok_frac = float(np.mean(np.abs(bins_h[:, 0] - tb) <= 2))

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    sm_mhz = float((clocks or {}).get("sm_mhz") or peaks.get("sm_max_mhz", 1965.0))

    leg('roofline leg')
    # ---- roofline leg: stage timing of the same step (separate, untimed passes) -------------
    roof = None
    stages = None
    fused = cfg["m"] == 4 and n == 1 and os.environ.get("MUSIC_B200_FUSED", "1") != "0"
    b2b_ms = None
    if fused and G > 1:
        # back-to-back launches of the dominant kernel alone (no gather wait in the timed region).  EVERY rank runs
        # them: the fused all-gather counts calls per rank (epochs), a rank that made extra calls would wait forever
        # for peers that did not.
        for _ in range(3):
            blk.process_device(d_in.data_ptr(), W, d_ang.data_ptr(), d_lvl.data_ptr(), None, d_bins.data_ptr(), stream=stream.cuda_stream)
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        r0.record(stream)
        for _ in range(args.steps):
            blk.process_device(d_in.data_ptr(), W, d_ang.data_ptr(), d_lvl.data_ptr(), None, d_bins.data_ptr(), stream=stream.cuda_stream)
        r1.record(stream)
        sync_all()
        b2b_ms = r0.elapsed_time(r1) / args.steps
    if rank == 0:
        def time_stages(b, reps=5):
            b.set_stage_timing(True)
            for _ in range(reps):
                b.process_device(d_in.data_ptr(), W, d_ang.data_ptr(), d_lvl.data_ptr(), None, d_bins.data_ptr(),
                                 stream=stream.cuda_stream)
            torch.cuda.synchronize()
            ms4, chunks = b.stage_times_ms()
            b.set_stage_timing(False)
            return [m / reps for m in ms4], chunks // reps

        # the three stages timed separately on a second handle that runs the unfused kernels
        old_env = os.environ.get("MUSIC_B200_FUSED")
        os.environ["MUSIC_B200_FUSED"] = "0"
        blk3 = music_doa(cfg["m"], n, cfg["nsamples"], resp, K, device=local)
        if old_env is None:
            del os.environ["MUSIC_B200_FUSED"]
        else:
            os.environ["MUSIC_B200_FUSED"] = old_env
        for _ in range(2):
            blk3.process_device(d_in.data_ptr(), W, d_ang.data_ptr(), d_lvl.data_ptr(), None, d_bins.data_ptr(),
                                stream=stream.cuda_stream)
        s4, nl = time_stages(blk3)
        blk3.close()
        if fused:
            # nothing but back-to-back launches of this kernel, CUDA events on its stream: at N = 1 the timed region itself
            dom_ms = ms / args.steps if G == 1 else b2b_ms
            dom_how = "CUDA events around %d back-to-back launches on the launch stream (the step is this one kernel)" % args.steps
            kernel = "music4_fused_kernel (K1 covariance + K2 eigenvectors + K3 scan in one persistent launch)"
        else:
            ms4, _ = time_stages(blk)
            dom_ms = ms4[0]
            dom_how = "per-launch CUDA events, separate passes of the same step"
            kernel = "K1 covariance (cov4_tma_kernel / covN_tma_kernel / cov_tile_kernel)"
        stages = {"unfused_cov_ms": s4[0], "unfused_eig_ms": s4[1], "unfused_scan_ms": s4[2], "unfused_topn_ms": s4[3],
                  "default_path_kernel_ms": dom_ms, "default_path": "fused" if fused else "three kernels"}
        achieved = bytes_per_window(cfg) * W / (dom_ms * 1e-3) / 1e9
        traffic, traffic_src = None, None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
            traffic = tj.get("config%d" % args.config)
            traffic_src = {k: tj.get(k) for k in ("capture", "capture_commit", "unit")}
        except Exception:
            pass
        roof = {"bound": "hbm", "kernel": kernel, "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": achieved / peak,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (burst copy), of measured" if peaks else "fallback 6650 GB/s, of fallback",
                "traffic": traffic, "traffic_source": traffic_src, "bytes_per_window": bytes_per_window(cfg), "windows_per_launch": W,
                "launch_ms": dom_ms, "launch_ms_source": dom_how,
                "whole_step_frac": (bytes_per_window(cfg) * value / G / 1e9) / peak,
                "fp64_pipe_frac": dfma_per_window(cfg) * (W / (dom_ms * 1e-3)) / (FP64_DFMA_PER_CLK_PER_SM * 148 * sm_mhz * 1e6),
                "unfused_cov_kernel_frac": bytes_per_window(cfg) * W / (s4[0] * 1e-3) / 1e9 / peak}

    # ---- e2e: block API with HOST buffers (H2D + D2H inside the timed region) --------------------------------------
    leg('e2e leg')
    e2e = None
    if not args.no_e2e:
        We = W
        esteps = max(3, min(args.steps, 20))
        in_bytes = We * cfg["nsamples"] * 8

        def host_copy_of(shard, pinned):
            h = torch.empty((We, cfg["nsamples"] * 2), dtype=torch.float32)
            if pinned:
                h = h.pin_memory()
            h.copy_(shard[:We].cpu())
            return h

        h_in = host_copy_of(d_in, True)
        h_ang = torch.empty((We, n), dtype=torch.float32).pin_memory()
        h_lvl = torch.empty((We, n), dtype=torch.float32).pin_memory()
        x_np = h_in.numpy().view(np.complex64)
        a_np, l_np = h_ang.numpy(), h_lvl.numpy()
        sync_all()
        dt = time_work(blk, We, x_np, [a_np, l_np], esteps, torch.cuda.synchronize)
        assert np.array_equal(blk.last_bins(), bins_h[:We]), "host path and device path disagree"
        if G > 1:
            t = torch.tensor([dt], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        per_rank_value = We * G * esteps / dt
        # the PCIe roof of this leg: the same host buffer copied to the device and nothing else
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        d_tmp = d_in[:We]  # h_in holds exactly these windows: the copy does not change the data
        for _ in range(2):
            d_tmp.copy_(h_in, non_blocking=True)
        torch.cuda.synchronize()
        c0.record(stream)
        for _ in range(3):
            d_tmp.copy_(h_in, non_blocking=True)
        c1.record(stream)
        torch.cuda.synchronize()
        h2d_gbs = 3 * in_bytes / (c0.elapsed_time(c1) * 1e-3) / 1e9
        e2e = {"value": per_rank_value, "unit": "windows/s", "h2d_bytes_per_step": int(in_bytes * G),
               "d2h_bytes_per_step": int(We * n * 4 * 3 * G), "windows_per_step": We * G, "steps": esteps,
               "api": "music_doa.work() -> music_b200_process_host, pinned host input, one block per GPU",
               "h2d_copy_only_gbs": h2d_gbs, "e2e_input_gbs": in_bytes * G * esteps / dt / 1e9}
        # pageable input (what GNU Radio and numpy hand over): pinned by the library on first sight, cached afterwards
        if G == 1:
            h_pg = host_copy_of(d_in, False)
            a2, l2 = np.zeros((We, n), np.float32), np.zeros((We, n), np.float32)
            t_first = time.perf_counter()
            blk.work(We, [h_pg.numpy().view(np.complex64)], [a2, l2])
            t_first = time.perf_counter() - t_first
            dtp = time_work(blk, We, h_pg.numpy().view(np.complex64), [a2, l2], esteps, torch.cuda.synchronize)
            assert np.array_equal(a2, a_np)
            e2e["pageable_value"] = We * esteps / dtp
            e2e["pageable_over_pinned"] = (We * esteps / dtp) / per_rank_value
            e2e["pageable_first_call_s"] = t_first
            e2e["pageable_how"] = "numpy (malloc) input and outputs; cudaHostRegister on the first call, cache hits afterwards"
            del h_pg
        del h_in
        # N > 1: ONE block over all N GPUs, one work() call per step, driven by rank 0 alone
        if G > 1:
            leg('e2e: single block over all GPUs')
            dist.barrier()
            single = None
            if rank == 0:
                try:  # a reported extra: it must not take the headline line down
                    policy = interleave_host_memory()
                    Wm = We * G
                    hm = torch.empty((Wm, cfg["nsamples"] * 2), dtype=torch.float32).pin_memory()
                    default_host_memory()
                    xg = synth.gen_windows_torch(cfg, seed, 0, min(Wm, 4096), dev)  # stream windows 0..4095 (all shards), replicated
                    for w0 in range(0, Wm, xg.shape[0]):
                        c = min(xg.shape[0], Wm - w0)
                        hm[w0:w0 + c].copy_(xg[:c])
                    del xg
                    am, lm = np.zeros((Wm, n), np.float32), np.zeros((Wm, n), np.float32)
                    mblk = music_doa(cfg["m"], n, cfg["nsamples"], resp, K, devices=list(range(G)))
                    msteps = max(3, min(esteps, 5))  # (10.5 GB per call at 8 GPUs: a few calls are enough)
                    dtm = time_work(mblk, Wm, hm.numpy().view(np.complex64), [am, lm], msteps, torch.cuda.synchronize)
                    # same answers as the single-GPU block on the same windows
                    chk = min(Wm, 2048)
                    ac = np.zeros((chk, n), np.float32)
                    blk.work(chk, [hm[:chk].numpy().view(np.complex64)], [ac])
                    single = {"value": Wm * msteps / dtm, "windows_per_step": Wm, "steps": msteps, "input_gbs": Wm * cfg["nsamples"] * 8 * msteps / dtm / 1e9,
                              "host_buffer": "one pinned buffer, " + policy, "equals_single_gpu_block": bool(np.array_equal(ac, am[:chk])),
                              "api": "ONE music_doa.work() call per step on a multi-device handle (music_b200_create_multi, windows dealt w mod %d)" % G}
                    mblk.close()
                    del hm
                except Exception as e:
                    default_host_memory()
                    single = {"error": repr(e)[:300]}
            dist.barrier()
            if rank == 0:
                # headline e2e at N GPUs: one block per GPU, each fed by its own host process (the launch the driver makes);
                # the ONE-block-over-all-GPUs form (one host thread, one buffer) is reported beside it
                e2e["per_rank_blocks_value"] = per_rank_value
                e2e["single_block_all_gpus"] = single

    # ---- SURVEY 8(f) rows built so far, same workload (untimed w.r.t. the headline; rank 0, N = 1) ----------
    next_rows = None
    if rank == 0 and G == 1 and not args.no_next_rows:
        next_rows = {}
        N, M = cfg["snapshots"], cfg["m"]
        # (f2) planar antenna streams: the same samples as d_in, de-interleaved once (setup, untimed)
        Wp = W
        planar = d_in[:Wp].view(Wp, N, M, 2).permute(2, 0, 1, 3).contiguous().view(M, Wp * N * 2)
        ptrs = [planar[r].data_ptr() for r in range(M)]
        d_bp = torch.empty((2 * Wp, n), dtype=torch.int32, device=dev)
        d_ap = torch.empty((2 * Wp, n), dtype=torch.float32, device=dev)
        for name, hop, Wn in (("planar_hop_N", N, Wp), ("planar_hop_N_over_2", N // 2, 2 * Wp - 1)):
            for _ in range(2):
                blk.process_planar_device(ptrs, hop, Wn, d_ap.data_ptr(), None, None, d_bp.data_ptr(), stream.cuda_stream)
            torch.cuda.synchronize()
            p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = max(3, min(args.steps, 10))
            p0.record(stream)
            for _ in range(reps):
                blk.process_planar_device(ptrs, hop, Wn, d_ap.data_ptr(), None, None, d_bp.data_ptr(), stream.cuda_stream)
            p1.record(stream)
            torch.cuda.synchronize()
            pms = p0.elapsed_time(p1) / reps
            row = {"value": Wn / (pms * 1e-3), "unit": "windows/s", "ms_per_step": pms, "windows_per_step": Wn, "hop": hop,
                   "hbm_bytes_per_window": 8 * M * hop + 12 * n,
                   "api": "music_b200_process_planar_device (M device streams, no interleaved copy)"}
            if hop == N:
                row["bins_equal_interleaved_path"] = bool(torch.equal(d_bp[:Wp], last_bins[:Wp]))
            next_rows[name] = row
        del planar
        # (f1) retune: device table build vs the reference's Python loop + re-marshalling
        pos = [[synth.SPACING * x, synth.SPACING * y] for x, y in cfg["antenna_array"]]
        lam = synth.C_LIGHT / (synth.FREQUENCY * 1.01)
        blkx = music_doa(M, n, cfg["nsamples"], resp, K, device=local)
        t0 = time.perf_counter()
        tab = calculate_antenna_array_response(pos, K, lam)
        blkx.set_array_response(tab)
        t_py = time.perf_counter() - t0
        blkx.set_array_geometry(pos, lam)
        ts = []
        for i in range(5):
            t0 = time.perf_counter()
            guarded = blkx.set_array_geometry(pos, lam * (1.0 + 1e-3 * i))
            ts.append(time.perf_counter() - t0)
        same = bool(np.array_equal(blkx.array_response_c64().view(np.uint32),
                                   np.asarray(calculate_antenna_array_response(pos, K, lam * (1.0 + 1e-3 * 4))).astype(np.complex64).view(np.uint32)))
        blkx.close()
        next_rows["retune"] = {"device_ms": 1e3 * sorted(ts)[2], "python_helper_ms": 1e3 * t_py, "entries": 2 * M * K,
                               "guarded_entries": guarded, "table_bit_identical": same,
                               "api": "music_b200_set_geometry vs calculate_antenna_array_response + set_array_response"}

    leg('other configs')
    # ---- BASELINE configs[2..4] ---------------------------------------------------------------------------------
    other = None
    if not args.no_other_configs and args.config == 2:
        blk.close()
        del d_in
        torch.cuda.empty_cache()
        other = {}
        for cid in (3, 4, 5):
            if cid == 3 and G > 1:
                continue  # configs[2] is a 1-GPU config
            try:
                res = run_other_config(cid, args, torch, dist, dev, local, rank, G, peak, sm_mhz)
            except Exception as e:  # a reported leg must not take the headline down
                res = {"error": repr(e)[:300]}
                torch.cuda.empty_cache()
            other["C%d" % cid] = res
        blk = None

    cpu = None
    if rank == 0 and G == 1 and not args.no_cpu_baseline:
        procs = host_threads()
        r = cpu_port_throughput(args.config, cfg, table, seed, budget_s=10.0, procs=procs)
        cpu = {"value": r["value"], "unit": "windows/s", "cores": procs, "kind": "port",
               "sample": "%d windows (%d worker processes x %d windows of the same synthetic stream x %d passes), %.2f s wall, C port of work() (-O3 -DNDEBUG)"
                         % (r["windows"], procs, r["per_proc"], r["reps"], r["seconds"]),
               "value_1core": r["value_1core"], "parallel_efficiency": r["parallel_efficiency"],
               "effective_cores": r["value"] / r["value_1core"], "cgroup_cpu_quota": cgroup_cpu_quota(),
               "note": "effective_cores = value / value_1core: what the box actually gave the arm (affinity masks on shared hosts "
                       "list more CPUs than the container's share; the arm cannot go faster than that share)",
               "slowest_worker_s": r["slowest_worker_s"], "fastest_worker_s": r["fastest_worker_s"]}

    if rank == 0:
        line = {
            "metric": metric_name(cfg), "value": value, "unit": "windows/s", "n_gpus": G, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_dict(cfg, args.config, W, G),
            "e2e": e2e, "gpu_launches": launches, "clocks": clocks, "roofline": roof, "cpu_baseline": cpu,
            "stages": stages, "sanity_bins_within_2_of_truth": ok_frac, "gather": gather_check, "next_rows": next_rows,
            "other_configs": other,
        }
        print(json.dumps(line))
    if blk is not None:
        blk.close()
    if G > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
