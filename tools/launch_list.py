#!/usr/bin/env python
"""Kernel launch list of bench steps with inputs resident in HBM, from torch.profiler (CUDA activities): launches, total
and mean device time per kernel over the profiled passes, largest first, as CSV on stdout (and in --out when given).  One
warm-up pass runs outside the profile.

    python tools/launch_list.py --batch 128 --passes 2 --out launch_list_b128.csv
"""
import argparse, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
from torch.profiler import ProfilerActivity, profile
from autoinst_b200 import api
from autoinst_b200.synthetic import CONFIGS, make_chunk
ap = argparse.ArgumentParser()
ap.add_argument("--batch", type=int, default=128)
ap.add_argument("--n-target", dest="n_target", type=int, default=8192)
ap.add_argument("--seed", type=int, default=1000)
ap.add_argument("--passes", type=int, default=2)
ap.add_argument("--matvec", type=int, default=0, help="ANCUTS_OPT_MATVEC: 0 shared-memory sparse (default), 1 dense from HBM")
ap.add_argument("--out", default=None, help="also write the CSV to this file")
args = ap.parse_args()
dev = torch.device("cuda", 0)
cfg = CONFIGS["tarl_spatial"]
chunks = [make_chunk(args.seed + i, n_target=args.n_target, features="tarl") for i in range(args.batch)]
packed = api.PackedChunks([c.points for c in chunks], [c.tarl for c in chunks], None, theta=cfg["theta"])
devc = packed.to_device(dev)
from autoinst_b200._lib import OPT_MATVEC
api.Handle.get(dev).set_option(OPT_MATVEC, args.matvec)


def one_pass():
    api.segment_packed(packed, dev_chunks=devc, alpha=cfg["alpha"], theta=cfg["theta"], T=cfg["T"])


one_pass()
torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(args.passes):
        one_pass()
    torch.cuda.synchronize()
agg = {}
for ev in prof.events():
    if ev.device_type != torch.autograd.DeviceType.CUDA or ev.name.startswith("Memcpy") or ev.name.startswith("Memset"):
        continue
    n, t = agg.get(ev.name, (0, 0.0))
    agg[ev.name] = (n + 1, t + ev.time_range.elapsed_us())
total = sum(t for _, t in agg.values())
launches = sum(n for n, _ in agg.values())
lines = [f"# {args.passes} passes of {args.batch} chunks, matvec {args.matvec}: launches {launches}, kernel time "
         f"{total / 1e3:.1f} ms (device time summed over kernels; concurrent kernels overlap), "
         f"{torch.cuda.get_device_name(dev)}", "kernel,launches,total_us,avg_us,share_pct"]
for name, (n, t) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
    lines.append(f"\"{name}\",{n},{t:.1f},{t / n:.2f},{100.0 * t / total:.1f}")
text = "\n".join(lines) + "\n"
if args.out:
    with open(args.out, "w") as f:
        f.write(text)
print(text, end="")
