#!/usr/bin/env python
"""Per-level trace of one bench step: active nodes per size bin, cluster sizes, time of the concurrent
cluster kernels, and per-level node statistics (sum n^2, steps) from the node table; the Lanczos steps of the
persistent kernel and how many of them took the full Gram-Schmidt pass.  With ANCUTS_PHASES=1 also the phase clocks of
the cluster kernel per cluster size, in total and per Lanczos step (steps of the nodes that ran at that cluster size,
from the node table: n -> size bin -> the level's cluster map).

    python tools/level_profile.py --batch 64 --out gpurun_out/levels_b64.json
"""
import argparse, json, os, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

BIN_LIMITS = (320, 512, 640, 1024, 2048, 4096)     # kernels_graph.cuh cluster_class: node size bins of the cluster kernel


def cluster_class(n):
    for b, lim in enumerate(BIN_LIMITS):
        if n <= lim:
            return b
    return -1


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--n-target", dest="n_target", type=int, default=8192)
    ap.add_argument("--seed", type=int, default=1000)
    ap.add_argument("--out", default="gpurun_out/levels.json")
    ap.add_argument("--matvec", type=int, default=0, help="ANCUTS_OPT_MATVEC: 0 shared-memory sparse (default), 1 dense")
    ap.add_argument("--pairs", type=int, default=0, help="ANCUTS_OPT_PAIR_SEARCH: 0 cell-sorted (default), 1 shuffled")
    ap.add_argument("--map", type=int, default=0, help="chunks of one synthetic map (N in [3 k, 12 k]) instead of --batch equal chunks")
    args = ap.parse_args()
    import torch
    from autoinst_b200 import api
    from autoinst_b200.synthetic import CONFIGS, make_chunk
    dev = torch.device("cuda", 0)
    cfg = CONFIGS["tarl_spatial"]
    kw = dict(alpha=cfg["alpha"], theta=cfg["theta"], T=cfg["T"])
    if args.map:
        from autoinst_b200.synthetic import make_map
        chunks = make_map(args.map, (3000, 12000), features="tarl", seed=args.seed)
    else:
        chunks = [make_chunk(args.seed + i, n_target=args.n_target, features="tarl") for i in range(args.batch)]
    packed = api.PackedChunks([c.points for c in chunks], [c.tarl for c in chunks], None, theta=cfg["theta"])
    devc = packed.to_device(dev)
    hd = api.Handle.get(dev)
    from autoinst_b200._lib import OPT_MATVEC, OPT_PAIR_SEARCH
    hd.set_option(OPT_MATVEC, args.matvec)
    hd.set_option(OPT_PAIR_SEARCH, args.pairs)
    for _ in range(2):
        api.segment_packed(packed, dev_chunks=devc, **kw)
    hd.set_stage_timing(2)
    api.segment_packed(packed, dev_chunks=devc, **kw)
    lv = hd.levels()
    acc = hd.accounting()
    hd.set_stage_timing(0)
    phases = None
    if os.environ.get("ANCUTS_PHASES"):
        hd.debug_phases(reset=True)
        api.segment_packed(packed, dev_chunks=devc, **kw)
        phases = hd.debug_phases()
        for c, d in phases.items():
            tot = sum(d.values()) or 1.0
            print("cluster size", c, {k: round(100 * v / tot, 1) for k, v in d.items()}, "Mcycles %.1f" % (tot / 1e6), flush=True)
    res = api.segment_packed(packed, device=dev, want_stats=True, **kw)
    st = res.stats
    ra = hd.reorth_accounting()
    print("cluster kernel: Lanczos steps %d, steps with the full Gram-Schmidt pass %d (%.1f %%)"
          % (ra["steps"], ra["full_passes"], 100.0 * ra["full_passes"] / max(ra["steps"], 1)), flush=True)
    rows = []
    steps_per_c = {}
    for i, l in enumerate(lv):
        m = st[st["level"] == i + 1] if (st["level"].min() >= 1) else st[st["level"] == i]
        if len(m) == 0:
            m = st[st["level"] == i]
        n = m["n"].astype(np.float64)
        k = m["steps"].astype(np.float64)
        bytes_ = float((k * (4 * n * n + 8 * n)).sum())
        for nn, kk in zip(m["n"], m["steps"]):
            b = cluster_class(int(nn))
            if b >= 0:
                c = int(l["cluster"][b])
                steps_per_c[c] = steps_per_c.get(c, 0) + int(kk)
        l.update(level=i, nodes_in_stats=int(len(m)), sum_n2=float((n * n).sum()), max_n=int(n.max()) if len(n) else 0,
                 max_steps=int(k.max()) if len(k) else 0, mean_steps=float(k.mean()) if len(k) else 0.0,
                 gb=bytes_ / 1e9, gbs=bytes_ / 1e9 / (l["ms"] * 1e-3) if l["ms"] > 0 else 0.0,
                 longest_node_us_per_step=(l["ms"] * 1e3 / k.max()) if len(k) else 0.0)
        rows.append(l)
        print(json.dumps(l), flush=True)
    phases_per_step = None
    if phases:
        phases_per_step = {c: {k_: v / steps_per_c[c] for k_, v in d.items()} for c, d in phases.items() if steps_per_c.get(c)}
        for c, d in phases_per_step.items():
            print("cluster size", c, "steps", steps_per_c[c], "cycles per step",
                  {k_: round(v) for k_, v in d.items()}, "total %d" % round(sum(d.values())), flush=True)
    out = dict(batch=args.batch, n_target=args.n_target, levels=rows, matvec_ms=acc["matvec"]["ms"],
               stat_levels=sorted(set(int(x) for x in st["level"])), phases=phases, steps_per_cluster_size=steps_per_c,
               phases_per_step=phases_per_step, reorth=ra)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    json.dump(out, open(args.out, "w"), indent=1)
    print("total matvec ms", acc["matvec"]["ms"], "levels", out["stat_levels"])
    print("stage ms", {k: round(v["ms"], 3) for k, v in acc.items()})


if __name__ == "__main__":
    main()
