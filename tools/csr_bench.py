"""Throughput of the CSR front end (`api.segment_graphs`, ancuts_segment_csr_f32) on the bench.py batch.

The batch is bench.py's: 128 chunks, n_target 8192, config_tarl_spatial, seed 1000.  Every chunk's affinity is built once
on the device (api.affinity), outside the clock, and kept as a CUDA sparse-CSR tensor.  Timed with CUDA events after a
warm-up:
  (a) segment_graphs on the whole batch (one batched call);
  (b) segment_dense once per chunk, the only way to cut caller graphs before the CSR entry;
  (c) segment_packed with resident inputs (the points path), for reference.
Also the drop-in `normalized_cut` on one host scipy CSR chunk: the old route (toarray() + segment_dense) against the new.
Prints one JSON object: chunks/s, per-stage accounting of (a), the share of chunks whose partitions agree between (a) and
(b), the card and its power limit (a query only).

    python tools/csr_bench.py [--batch 128] [--reps 3] [--out profiles/csr_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        return float(r.stdout.strip().splitlines()[0])
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=128)
    ap.add_argument("--n-target", type=int, default=8192)
    ap.add_argument("--seed", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import scipy.sparse as sp
    import torch
    from autoinst_b200 import api
    from autoinst_b200.synthetic import CONFIGS, make_chunk
    from ncuts.normalized_cut import _to_device_matrix, normalized_cut
    from oracle import ncut_ref as R

    cfg = CONFIGS["tarl_spatial"]
    dev = torch.device("cuda", 0)
    chunks = [make_chunk(args.seed + i, n_target=args.n_target, features="tarl") for i in range(args.batch)]
    graphs = []
    for ch in chunks:
        W = api.affinity(ch.points, ch.tarl, alpha=cfg["alpha"], theta=cfg["theta"], device=dev)
        graphs.append(W.contiguous().to_sparse_csr())
        del W
    nnz = sum(int(g.values().numel()) for g in graphs)
    torch.cuda.synchronize()

    def timed(fn):
        fn()                                                      # warm-up
        best = []
        for _ in range(args.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn()
            e1.record()
            torch.cuda.synchronize()
            best.append(e0.elapsed_time(e1))
        return out, float(np.median(best)), best

    hd = api.Handle.get(dev, 0)
    hd.set_stage_timing(0)
    res_a, ms_a, all_a = timed(lambda: api.segment_graphs(graphs, T=cfg["T"], device=dev))
    hd.set_stage_timing(1)
    api.segment_graphs(graphs, T=cfg["T"], device=dev)
    acct = hd.accounting()
    sparse = hd.sparse_accounting()
    hd.set_stage_timing(0)

    def run_b():
        out = []
        for g in graphs:
            Wd = g.to_dense()
            out.append(api.segment_dense(Wd, T=cfg["T"]))
            del Wd
        return out
    res_b, ms_b, all_b = timed(run_b)
    agree = sum(R.same_partition(a, b) for a, b in zip(res_a.labels, res_b))

    packed = api.PackedChunks([c.points for c in chunks], [c.tarl for c in chunks], None, theta=cfg["theta"])
    dc = packed.to_device(dev)
    kw = dict(alpha=cfg["alpha"], theta=cfg["theta"], T=cfg["T"], device=dev)
    _, ms_c, all_c = timed(lambda: api.segment_packed(packed, dev_chunks=dc, **kw))

    # drop-in, one host scipy CSR chunk: old route (densify on the host, n^2 floats to the device) against the new one
    g0 = graphs[0].cpu()
    A = sp.csr_matrix((g0.values().numpy(), g0.col_indices().numpy(), g0.crow_indices().numpy()), shape=tuple(g0.shape))
    n0 = A.shape[0]

    def wall(fn, reps=args.reps):
        fn()
        t = []
        for _ in range(reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            t.append((time.perf_counter() - t0) * 1e3)
        return float(np.median(t))
    old_ms = wall(lambda: api.segment_dense(_to_device_matrix(A), num_points_orig=n0, T=cfg["T"], strict=True))
    new_ms = wall(lambda: normalized_cut(A, n0, np.arange(n0), T=cfg["T"]))

    B = args.batch
    out = {
        "workload": f"{B} chunks, n_target {args.n_target}, config_tarl_spatial, seed {args.seed}; caller graphs = "
                    "device affinities as CUDA sparse-CSR tensors",
        "points": int(sum(c.n for c in chunks)), "nnz": nnz,
        "a_segment_graphs": {"ms": ms_a, "ms_all": all_a, "chunks_per_s": B / ms_a * 1e3},
        "b_segment_dense_per_chunk": {"ms": ms_b, "ms_all": all_b, "chunks_per_s": B / ms_b * 1e3},
        "c_segment_packed_resident": {"ms": ms_c, "ms_all": all_c, "chunks_per_s": B / ms_c * 1e3},
        "a_stages": acct, "a_sparse_entries": sparse["entries"],
        "partitions_agree_a_b": f"{agree}/{B}",
        "dropin_one_chunk": {"n": n0, "nnz": int(A.nnz), "old_toarray_segment_dense_ms": old_ms,
                             "new_csr_ms": new_ms},
        "device": torch.cuda.get_device_name(dev), "power_limit_w": power_limit(),
    }
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
