#!/usr/bin/env python
"""Benchmark of the NCuts hot path (BASELINE.json metric: NCuts chunks/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
                    [--config tarl_spatial|spatial|tarl_spatial_dino] [--workload batch|map] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Default workload (BASELINE.json configs[1]): config_tarl_spatial (alpha 1.0, theta 0.5, T 0.03) on synthetic
SemanticKITTI-shaped chunks of about 8192 major points with random 96-d TARL features.  One step = one pass of the
whole path (affinity -> degrees -> Lanczos -> N-cut scan -> partition, recursively, -> labels) over one batch of
`--batch` chunks per GPU.  Multi-GPU is weak scaling: every rank segments the SAME batch (identical per-GPU work, so
the max over ranks is not a straggler lottery); after segmenting, the ranks all-gather the label arrays (NCCL) and
rank 0 takes them to the host, as the map merge needs them (SURVEY.md §8e).
`--workload map` is BASELINE.json configs[3]: ONE synthetic first map of 40 chunks (N in [3 k, 12 k]) sharded
longest-first over the ranks (strong scaling), labels gathered once, merged and scored on rank 0.

The JSON line carries: value (inputs resident in HBM), e2e (host buffers through the C ABI entry
`ancuts_segment_chunks_host`: H2D of points+features and D2H of labels inside the timed region), roofline (dominant
kernel: the dense matvec of the persistent Lanczos kernels, CUDA events around every level launch, algorithmic bytes
of SURVEY.md §8d, with the sparse lower bound next to it), cpu_baseline (the oracle port of the reference's CPU path
on one host core, whose pinned labels also give `parity_ok` for that chunk), clocks.
`--impl reference` times only the CPU oracle port on all host cores (the reference is pure Python; `oracle/` is its
restatement, proven bit-equal to the unmodified reference by oracle/make_golden.py).
"""
from __future__ import annotations

import argparse
import json
import os
import platform
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "ncuts_chunks_per_sec"
UNIT = "chunks/s"
FEATURES = {"spatial": "", "tarl_spatial": "tarl", "tarl_spatial_dino": "tarl_dino"}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def make_batch(batch, n_target, seed0, config):
    from autoinst_b200.synthetic import make_chunk
    return [make_chunk(seed0 + i, n_target=n_target, features=FEATURES[config] or "tarl") for i in range(batch)]


def config_block(args):
    """The `config` object: identical in the b200 and the reference arm (the driver compares them)."""
    from autoinst_b200.synthetic import CONFIGS
    cfg = CONFIGS[args.config]
    feat = {"spatial": "no features", "tarl_spatial": "96-d TARL features",
            "tarl_spatial_dino": "96-d TARL + 384-d DINOv2 features"}[args.config]
    if args.workload == "map":
        w = (f"config_{args.config} NCuts (alpha {cfg['alpha']}, theta {cfg['theta']}, gamma {cfg['gamma']}, T {cfg['T']}), "
             f"one synthetic first map: {args.map_chunks} chunks of {args.map_lo}-{args.map_hi} major points, {feat}")
    else:
        w = (f"config_{args.config} NCuts (alpha {cfg['alpha']}, theta {cfg['theta']}, T {cfg['T']}), "
             f"synthetic SemanticKITTI-shaped chunks n_target={args.n_target}, {feat}")
    return {"workload": w}


def host_info():
    info = {"os_cpu_count": os.cpu_count(), "python": platform.python_version()}
    try:
        info["sched_affinity"] = len(os.sched_getaffinity(0))
    except Exception:
        pass
    try:
        out = subprocess.run(["lscpu"], capture_output=True, text=True, timeout=10).stdout
        for line in out.splitlines():
            if line.startswith("Model name"):
                info["lscpu_model"] = line.split(":", 1)[1].strip()
                break
    except Exception:
        pass
    try:
        import psutil
        vm = psutil.virtual_memory()
        info["ram_total_gb"] = round(vm.total / 2 ** 30, 1)
        info["ram_available_gb"] = round(vm.available / 2 ** 30, 1)
    except Exception:
        pass
    try:
        import scipy
        info["numpy"], info["scipy"] = np.__version__, scipy.__version__
    except Exception:
        pass
    return info


# ------------------------------------------------------------------------------------------------
# CPU side: the oracle port of the reference path, one chunk per call.  Only what the reference's ncuts_chunk
# computes is timed (affinity -> csr_matrix -> normalized_cut, ncuts_utils.py:56-174): inputs are in memory.
# ------------------------------------------------------------------------------------------------
def _cpu_init():
    os.environ["OMP_NUM_THREADS"] = "1"
    os.environ["OPENBLAS_NUM_THREADS"] = "1"
    os.environ["MKL_NUM_THREADS"] = "1"
    import scipy.sparse  # noqa: F401
    import scipy.sparse.linalg  # noqa: F401
    import scipy.spatial.distance  # noqa: F401
    from oracle import affinity_ref, ncut_ref  # noqa: F401


def _cpu_compute(task):
    """task = (points, tarl, dino, config name, pinned).  Returns (seconds, n, labels)."""
    pts, tarl, dino, name, pinned = task
    import contextlib
    import scipy.sparse as sp
    from autoinst_b200.synthetic import CONFIGS
    from oracle import ncut_ref as R
    from oracle.affinity_ref import affinity_ref, drop_isolated
    cfg = CONFIGS[name]
    n = pts.shape[0]
    t0 = time.perf_counter()
    A = affinity_ref(pts, tarl, dino, alpha=cfg["alpha"], theta=cfg["theta"], gamma=cfg["gamma"])
    _keep, A = drop_isolated(A)
    w = sp.csr_matrix(A)
    with (R.pinned_eigsh() if pinned else contextlib.nullcontext()):
        groups = R.normalized_cut_ref(w, n, np.arange(n), T=cfg["T"], split_lim=0.01, faithful=True)
    dt = time.perf_counter() - t0
    return dt, n, R.labels_from_groups(groups, n)


def chunk_task(ch, name, pinned=False):
    from autoinst_b200.synthetic import CONFIGS
    cfg = CONFIGS[name]
    return (ch.points, ch.tarl if cfg["theta"] else None, ch.dino if cfg["gamma"] else None, name, pinned)


def host_workers(n_points):
    """Worker processes for the all-core figure: every core the process may use, bounded by RAM
    (about 10 live dense float64 N x N arrays per worker, SURVEY §6.2)."""
    try:
        cores = len(os.sched_getaffinity(0))
    except Exception:
        cores = os.cpu_count() or 1
    try:
        import psutil
        avail = psutil.virtual_memory().available
    except Exception:
        avail = 64 << 30
    per_worker = 10 * 8 * float(n_points) ** 2
    return int(max(1, min(cores, avail * 0.7 // per_worker)))


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation (oracle port, `kind: "port"`; oracle/make_golden.py proves it
    bit-equal to the unmodified pipeline/ncuts code) on ALL host cores.  A persistent pool of single-threaded workers is
    created, warmed up and handed the pre-generated chunks BEFORE the clock starts; the K steps are submitted back to
    back (a worker that finishes a chunk takes the next one, no per-step barrier), ms_per_step = wall / K."""
    if rank != 0:
        return
    import multiprocessing as mp
    cfgb = config_block(args)
    if args.workload == "map":
        from autoinst_b200.synthetic import make_map
        chunks = make_map(args.map_chunks, (args.map_lo, args.map_hi), features=FEATURES[args.config] or "tarl", seed=args.seed)
        nmax = max(c.n for c in chunks)
        workers = host_workers(nmax)
        per_step = len(chunks)
    else:
        nmax = int(args.n_target * 1.15)
        workers = host_workers(nmax)
        per_step = args.ref_chunks if args.ref_chunks > 0 else workers       # upper bound; trimmed to the time budget below
        chunks = make_batch(per_step, args.n_target, args.seed, args.config)
    tasks = [chunk_task(c, args.config) for c in chunks]
    pool = mp.get_context("spawn").Pool(workers, initializer=_cpu_init)
    try:
        # warm-up: imports and page-in on every worker (tiny chunks), then ONE full-size chunk alone on an otherwise idle
        # machine = the 1-core figure (what run_pipeline.py does: one chunk after the other on one core)
        from autoinst_b200.synthetic import make_chunk
        tiny = chunk_task(make_chunk(1, n_target=600, features=FEATURES[args.config] or "tarl"), args.config)
        for _ in range(max(args.warmup, 1)):
            pool.map(_cpu_compute, [tiny] * workers, chunksize=1)
        one = None
        if not args.no_one_core:
            dt1, n1, _ = pool.apply(_cpu_compute, (tasks[0],))
            one = {"value": 1.0 / dt1, "unit": UNIT, "cores": 1, "seconds_per_chunk": dt1, "points": n1}
        if args.workload != "map" and args.ref_chunks <= 0:
            # bounded sample: K steps must end within --ref-budget-s.  A chunk takes about twice its idle-machine time when
            # every core runs one (memory-bound dense ncut_cost); `rounds` chunks per worker fit the budget.
            t_c = 2.0 * (one["seconds_per_chunk"] if one else 25.0)
            rounds = max(1, int(args.ref_budget_s // t_c))
            per_step = int(min(workers, max(1, rounds * workers // max(args.steps, 1))))
            chunks, tasks = chunks[:per_step], tasks[:per_step]
        pts_step = int(sum(c.n for c in chunks))
        t0 = time.perf_counter()
        res = pool.map(_cpu_compute, tasks * args.steps, chunksize=1)
        wall = time.perf_counter() - t0
    finally:
        pool.terminate()
    ms = 1e3 * wall / args.steps
    value = per_step * args.steps / wall
    each = [r[0] for r in res]
    sample = (f"{per_step} chunk(s) per step ({pts_step} major points), {args.steps} steps submitted back to back to a "
              f"persistent pool of {workers} single-threaded worker processes (pool start, imports and chunk generation "
              f"outside the clock); oracle port with the reference's dense ncut_cost (faithful=True); "
              f"mean {np.mean(each):.1f} s per chunk under load")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "strong" if args.workload == "map" else "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": cfgb,
        "detail": {"chunks_per_step": per_step, "points_per_sec": pts_step * args.steps / wall,
                   "seconds_per_chunk_under_load": {"mean": float(np.mean(each)), "min": float(np.min(each)),
                                                    "max": float(np.max(each))},
                   "cpu_seconds_total": float(np.sum(each)), "one_core": one, "host": host_info()},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": workers, "kind": "port", "sample": sample,
                         "one_core_value": one["value"] if one else None},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    QUERY = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.gpu_index)], stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self, t_begin=None, t_end=None):
        """Median SM clock over the samples taken inside [t_begin, t_end] (wall clock); all samples if none fall inside."""
        import datetime
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        rows = []
        try:
            for line in open(self.path):
                p = [x.strip() for x in line.split(",")]
                if len(p) < 9:
                    continue
                try:
                    ts = datetime.datetime.strptime(p[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                    rows.append((ts, float(p[1]), float(p[2]), float(p[3]) if p[3].replace(".", "").isdigit() else 0.0, p[5:9]))
                except ValueError:
                    continue
            os.unlink(self.path)
        except Exception:
            pass
        inside = [r for r in rows if t_begin is not None and t_begin - 0.05 <= r[0] <= t_end + 0.05]
        use = inside if inside else rows
        reasons = set()
        for r in use:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if use:
            out.update(sm_mhz=float(np.median([r[1] for r in use])), sm_max_mhz=float(max(r[2] for r in use)),
                       reasons=sorted(reasons), samples=len(use), samples_in_timed_region=len(inside),
                       power_w_max=float(max(r[3] for r in use)))
        return out


TRAFFIC_FILE = "r2_cluster_dram_b128.csv"        # ncu DRAM bytes of the cluster kernels, same build (tools/gpu_evidence.sh)


def measured_traffic(args, launches_per_step):
    """DRAM bytes per timed launch of the dominant kernel from the committed ncu list (two passes over 128 chunks of
    n_target 8192, config_tarl_spatial, dense matvec), or None when the workload differs."""
    path = os.path.join(ROOT, "profiles", TRAFFIC_FILE)
    if (args.batch != 128 or args.n_target != 8192 or args.config != "tarl_spatial" or args.workload != "batch"
            or not os.path.exists(path) or launches_per_step <= 0):
        return None
    total = 0.0
    for line in open(path):
        f = line.strip().split(",")
        if len(f) >= 7 and f[0].startswith("k_lanczos_cluster"):      # the kernel name itself contains a comma
            total += (float(f[-2]) + float(f[-1])) * 1e9
    return total / 2.0 / launches_per_step if total else None


_REAL_STDOUT = None


def protect_stdout():
    """Libraries (NCCL banner, torchrun) may write to fd 1; the contract is ONE JSON line on stdout.
    fd 1 is pointed at stderr for the whole run and the line is written to the saved descriptor."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line: dict):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """--dump-outputs: write every array of `arrays` (name -> numpy array) as out_dir/<name>.npy, float64 arrays as float64
    and everything else as float32 (integers up to 2^24 are exact there, labels included), at most DUMP_BYTES in all.
    Beyond that, every array over 1 MB is replaced by the same seeded sample of its flattened elements, in index order, and
    <name>_index.npy (float64) says which elements were kept, so that two runs with the same arguments stay comparable."""
    out = {}
    for name, a in arrays.items():
        a = np.asarray(a)
        wide = a.dtype == np.float64 or (a.dtype.kind in "iu" and a.size and int(np.abs(a).max()) >= 1 << 24)
        out[name] = a.astype(np.float64 if wide else np.float32)
    big = [n for n, a in out.items() if a.nbytes > 1 << 20]
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_BYTES:
        room = DUMP_BYTES - sum(out[n].nbytes for n in out if n not in big)
        frac = room / sum(out[n].nbytes + 8 * out[n].size for n in big)         # + the float64 index of every kept element
        for n in big:
            a = out[n].reshape(-1)
            idx = np.sort(np.random.default_rng(0).choice(a.size, int(a.size * frac), replace=False))
            out[n] = a[idx]
            out[n + "_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


class Dist:
    """Rank bookkeeping + the timing helper of the contract (barrier + synchronize on both sides, CUDA events on the
    current stream, MAX over ranks; min / mean over ranks reported next to it)."""

    def __init__(self):
        import torch
        self.torch = torch
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        assert torch.cuda.is_available(), "bench.py needs a CUDA device; there is no CPU fallback"
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            import datetime
            import torch.distributed as dist
            # a mismatched collective must fail in minutes, not hold the box for the default 10-minute watchdog
            dist.init_process_group("nccl", device_id=self.dev, timeout=datetime.timedelta(seconds=180))

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def over_ranks(self, x):
        """(max, min, mean) of a per-rank scalar."""
        if self.world == 1:
            return float(x), float(x), float(x)
        import torch.distributed as dist
        t = self.torch.tensor([float(x)], dtype=self.torch.float64, device=self.dev)
        all_ = self.torch.empty(self.world, dtype=self.torch.float64, device=self.dev)
        dist.all_gather_into_tensor(all_, t)
        a = all_.cpu().numpy()
        return float(a.max()), float(a.min()), float(a.mean())

    def timed(self, fn, steps):
        torch = self.torch
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        self.barrier()
        ms = e0.elapsed_time(e1) / steps
        return self.over_ranks(ms)

    def close(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
            dist.destroy_process_group()


def sparse_bound(stats, nnz_per_row):
    """SURVEY.md §8d last sentence: bytes per chunk a sparse matvec would move for the same Lanczos steps,
    (4 + 4) bytes per stored entry, next to the dense 4 n^2 + 8 n."""
    if stats is None or nnz_per_row is None:
        return None
    n = stats["n"].astype(np.float64)
    k = stats["steps"].astype(np.float64)
    return float((k * 8.0 * nnz_per_row * n).sum())


def run_batch(args):
    import torch
    from autoinst_b200 import api, sharding
    from autoinst_b200._lib import MATVEC_DENSE, MATVEC_SPARSE, OPT_CLUSTER_MAP, OPT_MATVEC, OPT_PAIR_SEARCH
    from autoinst_b200.synthetic import CONFIGS
    D = Dist()
    rank, world, dev = D.rank, D.world, D.dev
    cfg = CONFIGS[args.config]
    kw = dict(alpha=cfg["alpha"], theta=cfg["theta"], gamma=cfg["gamma"], T=cfg["T"])

    chunks = make_batch(args.batch, args.n_target, args.seed, args.config)       # the same batch on every rank
    packed = api.PackedChunks([c.points for c in chunks], [c.tarl for c in chunks] if cfg["theta"] else None,
                              [c.dino for c in chunks] if cfg["gamma"] else None, theta=cfg["theta"], gamma=cfg["gamma"],
                              pin=True)
    local_ids = [rank * args.batch + i for i in range(args.batch)]
    total_chunks = args.batch * world
    gat = sharding.LabelGather(local_ids, packed.sizes, total_chunks, device=dev, dst=0) if world > 1 else None
    dev_chunks = packed.to_device(dev, labels=gat.send_view() if gat else None)
    hd = api.Handle.get(dev)
    hd.set_option(OPT_MATVEC, MATVEC_DENSE if args.matvec == "dense" else MATVEC_SPARSE)
    hd.set_option(OPT_PAIR_SEARCH, 1 if args.pairs == "shuffled" else 0)
    hd.set_option(OPT_CLUSTER_MAP, args.cluster_map)
    gather_host_ms = []

    def gather():
        if gat is None:
            return
        t0 = time.perf_counter()
        gat.start()
        gat.finish()
        gather_host_ms.append(1e3 * (time.perf_counter() - t0))

    last = {}

    def step_resident():
        last["res"] = api.segment_packed(packed, dev_chunks=dev_chunks, **kw)
        gather()

    def step_single_call():             # host buffers through ONE synchronous C call: upload, cut, labels back
        res = api.segment_packed(packed, device=dev, **kw)
        if gat is not None:
            gat.load_flat(packed.labels)
            gather()
        return res

    # e2e: successive batches through api.SegmentStream -- every step uploads one batch from pinned host memory (for the
    # NEXT step, on a side stream, while this step's batch is cut), cuts one batch and reads its labels back to the host
    stream = api.SegmentStream(device=dev, **kw)

    def step_e2e():
        stream.submit(packed, labels=gat.send_view() if gat is not None else None)     # labels land in the gather's send buffer
        res = stream.result()
        gather()
        return res

    sampler = ClockSampler(D.local_rank)
    if rank == 0:
        sampler.start()                 # nvidia-smi needs ~1 s before its first sample: start before the warm-up
    for _ in range(args.warmup):        # warm-up (also sizes the workspace)
        step_resident()
    step_single_call()
    stream.submit(packed, labels=gat.send_view() if gat is not None else None)      # prime the pipeline: one batch is always uploaded ahead
    step_e2e()
    t_begin = time.time()
    # timed region 1: inputs resident in HBM.  CUDA events around every level launch of the Lanczos kernels (timing
    # mode 2) give the roofline of the dominant kernel over exactly this region.
    hd.set_stage_timing(2)
    hd.launch_count(reset=True)
    mv = dict(bytes=0.0, ms=0.0, launches=0)
    acc_all = {s: dict(bytes=0.0, launches=0) for s in api.STAGES}

    def step_resident_acct():
        step_resident()
        acc = hd.accounting()
        for k in mv:
            mv[k] += acc["matvec"][k]
        for s in api.STAGES:
            acc_all[s]["bytes"] += acc[s]["bytes"]; acc_all[s]["launches"] += acc[s]["launches"]

    gather_host_ms.clear()
    sparse_acc = dict(entry_steps=0.0, entries=0.0)
    _plain_acct = step_resident_acct

    def step_resident_acct():        # noqa: F811  (adds the sparse-form counters of every step)
        _plain_acct()
        sa = hd.sparse_accounting()
        sparse_acc["entry_steps"] += sa["entry_steps"]; sparse_acc["entries"] += sa["entries"]

    ms_step, ms_min, ms_mean = D.timed(step_resident_acct, args.steps)
    launches = hd.launch_count(reset=True)
    hd.set_stage_timing(0)
    outputs = None
    if args.dump_outputs and rank == 0:     # the label buffer of the last timed step, before the later legs overwrite it
        outputs = {"labels": dev_chunks.labels[:int(packed.off[-1])].cpu().numpy(),
                   "num_segments": last["res"].num_segments.copy()}
    mv_default = dict(mv)
    g_res = list(gather_host_ms)
    gather_host_ms.clear()
    # timed region 2: the same steps through the host-buffer entry point
    ms_e2e, ms_e2e_min, ms_e2e_mean = D.timed(step_e2e, args.steps)
    g_e2e = list(gather_host_ms)
    res_last = stream.result()          # drain the batch uploaded by the last timed step (outside the region)
    ms_single, _, _ = D.timed(step_single_call, min(args.steps, 3))
    t_end = time.time()
    clocks = sampler.stop(t_begin, t_end) if rank == 0 else None
    gmax = D.over_ranks(float(np.mean(g_res)) if g_res else 0.0)

    # roofline leg: the north-star DENSE matvec form (W streamed from HBM every Lanczos step) on the same batch, same process,
    # CUDA events around every level launch.  When the timed region itself ran the dense form this is that region.
    roof_src = "the timed region (value)"
    roof_steps_used = args.steps
    if args.matvec != "dense" and args.roof_steps > 0:
        roof_steps_used = args.roof_steps
        hd.set_option(OPT_MATVEC, MATVEC_DENSE)
        api.segment_packed(packed, dev_chunks=dev_chunks, **kw)              # warm-up of the dense kernels
        hd.set_stage_timing(2)
        for k in mv:
            mv[k] = 0.0
        for _ in range(args.roof_steps):
            api.segment_packed(packed, dev_chunks=dev_chunks, **kw)
            acc = hd.accounting()
            for k in mv:
                mv[k] += acc["matvec"][k]
        hd.set_stage_timing(0)
        hd.set_option(OPT_MATVEC, MATVEC_SPARSE)
        roof_src = f"a separate leg of {args.roof_steps} steps with ANCUTS_OPT_MATVEC = dense after the timed regions (the default form keeps W in shared memory)"
    # outside the timed regions: node statistics, per-stage shares, the Python-list surface, the parity spot check
    res = api.segment_packed(packed, device=dev, want_stats=True, **kw)
    stats = res.stats
    if not all(np.array_equal(a, b) for a, b in zip(res.labels, res_last.labels)):
        raise SystemExit("bench: labels of the streamed e2e path differ from the single host call")
    hd.set_stage_timing(1)
    api.segment_packed(packed, dev_chunks=dev_chunks, **kw)
    stage_ms = {s: v["ms"] for s, v in hd.accounting().items()}
    hd.set_stage_timing(0)
    py_ms = None
    if rank == 0 and not args.no_python_surface:
        lists = ([c.points for c in chunks], [c.tarl for c in chunks] if cfg["theta"] else None,
                 [c.dino for c in chunks] if cfg["gamma"] else None)
        api.segment_chunks(*lists, device=dev, **kw)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for _ in range(2):
            api.segment_chunks(*lists, device=dev, **kw)
        py_ms = 1e3 * (time.perf_counter() - t0) / 2

    if rank == 0:
        peak, peak_src = peaks()
        value = total_chunks / (ms_step / 1e3)
        pts_total = int(packed.off[-1]) * world
        achieved = (mv["bytes"] / mv["launches"]) / ((mv["ms"] / mv["launches"]) * 1e-3) / 1e9 if mv["launches"] else 0.0
        cpu = None
        parity = None
        nnz_row = None
        if args.cpu_chunks > 0 and world == 1:          # the CPU leg (and with it the parity spot check) runs at N = 1 only
            # the oracle port on one host core, pinned eigsh start vector: its labels are also the parity spot check of the
            # timed batch (same chunks, GPU labels of the e2e call above)
            t0 = time.perf_counter()
            outs = [_cpu_compute(chunk_task(chunks[i], args.config, pinned=True)) for i in range(args.cpu_chunks)]
            wall = time.perf_counter() - t0
            from oracle import ncut_ref as R
            ok = [bool(R.same_partition(res.labels[i], outs[i][2])) for i in range(args.cpu_chunks)]
            parity = {"parity_ok": all(ok), "chunks_checked": len(ok), "identical": int(sum(ok)),
                      "against": "oracle port under the eigsh pin (v0 = ones), partition equality up to label permutation"}
            from oracle.affinity_ref import affinity_ref
            c0 = chunks[0]
            A = affinity_ref(c0.points, c0.tarl if cfg["theta"] else None, c0.dino if cfg["gamma"] else None,
                             alpha=cfg["alpha"], theta=cfg["theta"], gamma=cfg["gamma"])
            nnz_row = float(np.count_nonzero(A)) / c0.n
            compute_s = float(sum(o[0] for o in outs))
            cpu = {"value": args.cpu_chunks / compute_s, "unit": UNIT, "cores": 1, "kind": "port",
                   "sample": f"{args.cpu_chunks} chunk(s) of the timed batch (seed {args.seed}.., {sum(o[1] for o in outs)} major "
                             f"points), oracle port with the reference's dense ncut_cost (faithful=True), single thread, "
                             f"{compute_s:.1f} s of affinity + csr + normalized_cut",
                   "host": host_info()}
        sp_bytes = sparse_bound(stats, nnz_row)
        dense_bytes = float(((4.0 * stats["n"].astype(np.float64) ** 2 + 8.0 * stats["n"]) * stats["steps"]).sum()) if stats is not None else None
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": config_block(args),
            "detail": {"chunks_per_gpu_per_step": args.batch, "points_per_step": pts_total,
                       "points_per_sec": pts_total / (ms_step / 1e3),
                       "ms_per_step_over_ranks": {"max": ms_step, "min": ms_min, "mean": ms_mean},
                       "gather_ms": {"host_timer_mean_rank0": float(np.mean(g_res)) if g_res else 0.0,
                                     "max_over_ranks": gmax[0], "e2e_mean_rank0": float(np.mean(g_e2e)) if g_e2e else 0.0,
                                     "what": "one all_gather_into_tensor of the padded label buffers + one async D2H into "
                                             "pinned memory on rank 0; tables exchanged once before the clock"},
                       "matvec_form": "dense blocks streamed from HBM every Lanczos step" if args.matvec == "dense" else
                                      "row slices compressed into shared memory once per node (nodes <= 2048 points)",
                       "pair_search": args.pairs,
                       "l2": "inputs larger than L2: every step rebuilds the float32 affinity blocks of all recursion nodes "
                             "(%.1f GB per GPU, 126 MB of L2) and streams them from HBM once per Lanczos step"
                             % (acc_all["degree"]["bytes"] / max(args.steps, 1) / 1e9),
                       "arithmetic": "W float32 in HBM; vectors, degrees, dots and cut sums float64",
                       "segments_per_chunk": float(np.mean(res.num_segments)),
                       "eig_nodes_per_chunk": (len(stats) / args.batch) if stats is not None else None,
                       "lanczos_steps_per_chunk": (float(stats["steps"].sum()) / args.batch) if stats is not None else None,
                       "unconverged_nodes": int(res.unconverged),
                       "stage_ms_one_step": stage_ms,
                       "stage_algorithmic_gb_per_step": {s: acc_all[s]["bytes"] / args.steps / 1e9 for s in api.STAGES},
                       "python_list_surface": None if py_ms is None else {
                           "value": args.batch / (py_ms / 1e3), "unit": UNIT, "ms_per_step": py_ms,
                           "what": "api.segment_chunks(lists of numpy arrays): packing into host buffers (float64 -> float32 "
                                   "features, pageable) + the C ABI host call, rank 0 alone, outside the timed regions"}},
            "parity": parity,
            "e2e": {"value": total_chunks / (ms_e2e / 1e3), "unit": UNIT, "ms_per_step": ms_e2e,
                    "ms_per_step_over_ranks": {"max": ms_e2e, "min": ms_e2e_min, "mean": ms_e2e_mean},
                    "h2d_bytes_per_step": packed.h2d_bytes() * world, "d2h_bytes_per_step": packed.d2h_bytes() * world,
                    "how": "api.SegmentStream: every step uploads one batch from pinned host memory on a side stream (the batch "
                           "the next step cuts), cuts the batch uploaded one step earlier through the C ABI and copies its labels "
                           "to pinned host memory; K uploads, K cuts, K read-backs inside the K timed steps",
                    "single_call": {"value": total_chunks / (ms_single / 1e3), "unit": UNIT, "ms_per_step": ms_single,
                                    "steps": min(args.steps, 3),
                                    "what": "ancuts_segment_chunks_host, one synchronous call per batch: upload, cut and "
                                            "read-back in sequence (points first, features overlap the pair stage)"}},
            "gpu_launches": int(launches) * world,
            "sparse": None if args.matvec == "dense" else {
                "what": "default matvec form: the CTA's row slice as CSR (float32 value + uint16 column) in shared memory, built once "
                        "per node from the dense block; its Lanczos kernels over the timed region (value)",
                "entry_steps_per_step": sparse_acc["entry_steps"] / max(args.steps, 1),
                "lower_bound_bytes_per_step": 8.0 * sparse_acc["entry_steps"] / max(args.steps, 1),
                "hbm_bytes_per_step": mv_default["bytes"] / max(args.steps, 1),
                "lanczos_ms_per_step": mv_default["ms"] / max(args.steps, 1),
                "lower_bound_gbs": (8.0 * sparse_acc["entry_steps"] / (mv_default["ms"] * 1e-3) / 1e9) if mv_default["ms"] else None,
                "note": "the sparse matvec reads shared memory, not HBM: its Lanczos phase is bound by Gram-Schmidt, barriers and the "
                        "convergence checks (profiles/), not by a memory roofline; lower_bound_gbs is the (4+4)-byte-per-entry "
                        "bound of SURVEY.md §8d divided by the measured Lanczos time"},
            "roofline": {"bound": "hbm", "kernel": "k_lanczos_cluster<C, 6> (dense matvec of the persistent Lanczos kernels, one timed "
                                                    "launch = the concurrent kernels of one recursion level)",
                         "measured_over": roof_src,
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": measured_traffic(args, mv["launches"] / max(roof_steps_used, 1)),
                         "traffic_source": "ncu dram__bytes_read.sum + dram__bytes_write.sum of the cluster kernels, "
                                           "profiles/" + TRAFFIC_FILE + ", per level like achieved",
                         "peak_source": peak_src,
                         "launches_timed": mv["launches"], "avg_launch_us": 1e3 * mv["ms"] / max(mv["launches"], 1),
                         "algorithmic_bytes_per_launch": mv["bytes"] / max(mv["launches"], 1),
                         "dense_matvec_bytes_per_chunk": dense_bytes / args.batch if dense_bytes else None,
                         "sparse_lower_bound_bytes_per_chunk": sp_bytes / args.batch if sp_bytes else None,
                         "dense_over_sparse": (dense_bytes / sp_bytes) if (dense_bytes and sp_bytes) else None,
                         "nnz_per_row": nnz_row,
                         "note": "algorithmic bytes = sum over running nodes of 4 n^2 + 8 n per Lanczos step (SURVEY.md §8d), summed "
                                 "over the steps the kernels of one level take; the blocks of small nodes stay in L2, so the DRAM "
                                 "traffic is below the algorithmic bytes.  The sparse lower bound is (4+4) bytes per stored entry "
                                 "per step for the same steps: the fraction of the HBM peak says how well the DENSE design "
                                 "streams, not that streaming zeros is optimal"},
            "cpu_baseline": cpu,
            "clocks": clocks,
        }
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        emit(line)
    D.close()


def run_map(args):
    """BASELINE.json configs[3]: one synthetic first map, chunks sharded longest-first over the ranks (strong scaling),
    labels gathered once per pass to rank 0, merged (N2) and scored (N4) there on the device."""
    import torch
    from autoinst_b200 import api, sharding
    from autoinst_b200._lib import MATVEC_DENSE, MATVEC_SPARSE, OPT_CLUSTER_MAP, OPT_MATVEC, OPT_PAIR_SEARCH
    from autoinst_b200.synthetic import CONFIGS, make_map
    D = Dist()
    rank, world, dev = D.rank, D.world, D.dev
    cfg = CONFIGS[args.config]
    kw = dict(alpha=cfg["alpha"], theta=cfg["theta"], gamma=cfg["gamma"], T=cfg["T"])
    chunks = make_map(args.map_chunks, (args.map_lo, args.map_hi), features=FEATURES[args.config] or "tarl", seed=args.seed)
    sizes = [c.n for c in chunks]
    shards = sharding.shard_chunks(sizes, world)
    mine = shards[rank]
    loc = [chunks[i] for i in mine]
    packed = api.PackedChunks([c.points for c in loc], [c.tarl for c in loc] if cfg["theta"] else None,
                              [c.dino for c in loc] if cfg["gamma"] else None, theta=cfg["theta"], gamma=cfg["gamma"], pin=True)
    gat = sharding.LabelGather(mine, packed.sizes, len(chunks), device=dev, dst=0)
    dev_chunks = packed.to_device(dev, labels=gat.send_view())
    hd = api.Handle.get(dev)
    hd.set_option(OPT_MATVEC, MATVEC_DENSE if args.matvec == "dense" else MATVEC_SPARSE)
    hd.set_option(OPT_PAIR_SEARCH, 1 if args.pairs == "shuffled" else 0)
    hd.set_option(OPT_CLUSTER_MAP, args.cluster_map)
    post = api.MapPost(chunks, device=dev, min_points=args.min_points) if rank == 0 else None
    last = {}
    src_index = None
    if rank == 0:
        # where every chunk's labels sit in the gathered buffer (rank r's padded segment), in chunk order
        where = {}
        for r, (ids, szs) in enumerate(gat.tables):
            o = r * gat.pad
            for cid, n in zip(ids, szs):
                where[cid] = (o, n)
                o += n
        src_index = torch.as_tensor(np.concatenate([np.arange(where[c][0], where[c][0] + where[c][1]) for c in range(len(chunks))]),
                                    dtype=torch.int64).to(dev)

    def finish(labels):
        if rank == 0:
            # merge + metrics consume the gathered labels where the collective left them (device); the host copy of
            # LabelGather is what a caller that writes the map to disk would take
            last["metrics"] = post.merge_and_score(gat.recv[src_index])

    def step_resident():
        api.segment_packed(packed, dev_chunks=dev_chunks, **kw)
        gat.start()
        finish(gat.finish())

    def step_single_call():
        api.segment_packed(packed, device=dev, **kw)
        gat.load_flat(packed.labels)
        gat.start()
        finish(gat.finish())

    stream = api.SegmentStream(device=dev, **kw)      # successive maps: the next map's chunks upload while this one is cut

    def step_e2e():
        stream.submit(packed)
        stream.result()
        gat.load_flat(packed.labels)
        gat.start()
        finish(gat.finish())

    sampler = ClockSampler(D.local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        step_resident()
    step_single_call()
    stream.submit(packed)
    step_e2e()
    t_begin = time.time()
    hd.launch_count(reset=True)
    ms_step, ms_min, ms_mean = D.timed(step_resident, args.steps)
    launches = hd.launch_count(reset=True)
    outputs = None
    if args.dump_outputs and rank == 0:     # gathered labels (chunk order) and metrics of the last timed step
        outputs = {"labels": gat.recv[src_index].cpu().numpy()}
        outputs.update({"metrics_" + k: np.float64(v) for k, v in last["metrics"].items()})
    ms_e2e, ms_e2e_min, ms_e2e_mean = D.timed(step_e2e, args.steps)
    stream.result()
    ms_single, _, _ = D.timed(step_single_call, min(args.steps, 3))
    t_end = time.time()
    clocks = sampler.stop(t_begin, t_end) if rank == 0 else None
    # where one resident pass spends its time (host timer with a device synchronisation after every part, one extra pass)
    D.barrier()
    t0 = time.perf_counter()
    api.segment_packed(packed, dev_chunks=dev_chunks, **kw)
    torch.cuda.synchronize(dev)
    t1 = time.perf_counter()
    gat.start()
    lab_h = gat.finish()
    torch.cuda.synchronize(dev)
    t2 = time.perf_counter()
    finish(lab_h)
    torch.cuda.synchronize(dev)
    t3 = time.perf_counter()
    seg_ms = D.over_ranks(1e3 * (t1 - t0))
    breakdown = {"segment_ms_max_over_ranks": seg_ms[0], "segment_ms_min_over_ranks": seg_ms[1],
                 "gather_ms_rank0": 1e3 * (t2 - t1), "merge_metrics_ms_rank0": 1e3 * (t3 - t2)}
    # single-chunk latency through the array-level call the drop-in ncuts_chunk makes (one chunk per call)
    lat = None
    if rank == 0:
        c = chunks[int(np.argsort(sizes)[len(sizes) // 2])]
        for _ in range(2):
            api.segment_chunk(c.points, c.tarl if cfg["theta"] else None, c.dino if cfg["gamma"] else None, device=dev, **kw)
        t0 = time.perf_counter()
        for _ in range(5):
            api.segment_chunk(c.points, c.tarl if cfg["theta"] else None, c.dino if cfg["gamma"] else None, device=dev, **kw)
        lat = {"ms": 1e3 * (time.perf_counter() - t0) / 5, "n": c.n,
               "what": "api.segment_chunk (host arrays in, host labels out), the call ncuts.ncuts_utils.ncuts_chunk makes"}
    load = D.over_ranks(float(sum(sizes[i] ** 2 for i in mine)))
    h2d_mean = D.over_ranks(packed.h2d_bytes())[2]          # (collectives on every rank, outside the rank-0 block)
    if rank == 0:
        pts_total = int(sum(sizes))
        line = {
            "metric": METRIC, "value": len(chunks) / (ms_step / 1e3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": config_block(args),
            "detail": {"chunks": len(chunks), "points": pts_total, "points_per_sec": pts_total / (ms_step / 1e3),
                       "chunk_sizes": {"min": int(min(sizes)), "max": int(max(sizes)), "mean": float(np.mean(sizes))},
                       "chunks_per_rank": [len(s) for s in shards],
                       "load_n2_over_ranks": {"max": load[0], "min": load[1], "mean": load[2]},
                       "ms_per_step_over_ranks": {"max": ms_step, "min": ms_min, "mean": ms_mean},
                       "step": "segment the rank's shard -> all-gather labels -> D2H on rank 0 -> merge + metrics on rank 0"
                               + (" (device: ancuts_merge_chunks / ancuts_instance_metrics)" if post is not None else
                                  " (merge/metrics not in this build)"),
                       "breakdown_one_pass": breakdown,
                       "metrics": last.get("metrics"), "single_chunk_latency": lat},
            "e2e": {"value": len(chunks) / (ms_e2e / 1e3), "unit": UNIT, "ms_per_step": ms_e2e,
                    "ms_per_step_over_ranks": {"max": ms_e2e, "min": ms_e2e_min, "mean": ms_e2e_mean},
                    "h2d_bytes_per_step": int(h2d_mean * world),
                    "d2h_bytes_per_step": int(4 * pts_total),
                    "how": "api.SegmentStream: the chunks of the next map upload on a side stream while this map is cut; every "
                           "step uploads one map, cuts one map and reads its labels back",
                    "single_call": {"value": len(chunks) / (ms_single / 1e3), "unit": UNIT, "ms_per_step": ms_single,
                                    "steps": min(args.steps, 3),
                                    "what": "one synchronous ancuts_segment_chunks_host call per map"}},
            "gpu_launches": int(launches) * world, "roofline": None, "cpu_baseline": None, "clocks": clocks,
        }
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        emit(line)
    D.close()


def main():
    protect_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="tarl_spatial", choices=list(FEATURES))
    ap.add_argument("--workload", default="batch", choices=["batch", "map"])
    ap.add_argument("--batch", type=int, default=128, help="chunks per GPU per step")
    ap.add_argument("--n-target", dest="n_target", type=int, default=8192)
    ap.add_argument("--seed", type=int, default=1000)
    ap.add_argument("--matvec", default="sparse", choices=["sparse", "dense"],
                    help="ANCUTS_OPT_MATVEC: row slices in shared memory (default) or dense blocks from HBM every step")
    ap.add_argument("--pairs", default="sorted", choices=["sorted", "shuffled"], help="ANCUTS_OPT_PAIR_SEARCH")
    ap.add_argument("--cluster-map", dest="cluster_map", type=int, default=0, help="ANCUTS_OPT_CLUSTER_MAP (tuning)")
    ap.add_argument("--roof-steps", dest="roof_steps", type=int, default=3,
                    help="steps of the dense-matvec leg that measures the roofline of the north-star kernel (0 = skip)")
    ap.add_argument("--cpu-chunks", type=int, default=1, help="chunks in the cpu_baseline sample / parity check (0 = skip)")
    ap.add_argument("--ref-chunks", type=int, default=0, help="--impl reference: chunks per step (0 = half the workers)")
    ap.add_argument("--no-one-core", action="store_true", help="--impl reference: skip the separate 1-core measurement")
    ap.add_argument("--ref-budget-s", dest="ref_budget_s", type=float, default=420.0,
                    help="--impl reference: wall-clock budget of the timed steps (bounded sample)")
    ap.add_argument("--no-python-surface", action="store_true")
    ap.add_argument("--map-chunks", type=int, default=40)
    ap.add_argument("--map-lo", type=int, default=3000)
    ap.add_argument("--map-hi", type=int, default=12000)
    ap.add_argument("--min-points", type=int, default=20, help="map workload: Metrics min_points at the major level")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (labels; metrics of the map workload) as DIR/<name>.npy "
                         "in float32 / float64, at most 64 MB (a seeded sample of larger outputs), for comparing two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the CUDA path; the reference arm sizes its batch by a time budget")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    elif args.workload == "map":
        run_map(args)
    else:
        run_batch(args)


if __name__ == "__main__":
    main()
