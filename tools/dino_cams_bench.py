"""Cost of a second DINOv2 camera on the bench.py batch: config_tarl_spatial_dino, 128 chunks, n_target 8192, the chunks of
bench.make_batch (seeds 1000..).  Camera 0 of a "tarl_dino2" chunk is bench.py's DINOv2 array bit for bit; the 2-camera
runs add the synthetic second camera.  The two camera counts run alternately in every leg:
  (a) inputs resident in HBM (segment_packed with dev_chunks), CUDA events around each call;
  (b) through segment_stream (SegmentStream: upload of the next batch from pinned memory overlapping the cut), host clock
      over `--stream-steps` batches after a primed pipeline, synchronised at both ends;
  (c) stage timing on (CUDA events around every launch), a leg of its own: milliseconds and algorithmic bytes of the
      affinity stage from ancuts_last_accounting.
Prints one JSON object with chunks/s, the affinity stage, the H2D bytes per batch, the card and its power limit.

    python tools/dino_cams_bench.py [--batch 128] [--reps 5] [--stream-steps 4] [--out profiles/r6_dino_cams_bench.json]
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
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--stream-steps", type=int, default=4)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from autoinst_b200 import api
    from autoinst_b200.synthetic import CONFIGS, make_chunk

    cfg = CONFIGS["tarl_spatial_dino"]
    kw = dict(alpha=cfg["alpha"], theta=cfg["theta"], gamma=cfg["gamma"], T=cfg["T"])
    dev = torch.device("cuda", 0)
    chunks = []
    for i in range(args.batch):
        ch = make_chunk(args.seed + i, n_target=args.n_target, features="tarl_dino2")
        ch.dino = [g.astype(np.float32) for g in ch.dino]      # float32-representable: same values, half the host memory
        ch.tarl = ch.tarl.astype(np.float32)
        chunks.append(ch)
    pts, tarl = [c.points for c in chunks], [c.tarl for c in chunks]
    packed = {1: api.PackedChunks(pts, tarl, [c.dino[0] for c in chunks], theta=cfg["theta"], gamma=cfg["gamma"]),
              2: api.PackedChunks(pts, tarl, [c.dino for c in chunks], theta=cfg["theta"], gamma=cfg["gamma"])}
    del chunks
    resident = {k: p.to_device(dev) for k, p in packed.items()}
    streams = {k: api.SegmentStream(device=dev, **kw) for k in packed}
    hd = api.Handle.get(dev)
    hd.set_stage_timing(0)

    def run_resident(k):
        return api.segment_packed(packed[k], dev_chunks=resident[k], **kw)

    for k in packed:                                            # warm-up: workspace sizes, module load, pinned pools
        run_resident(k)
        streams[k].submit(packed[k])
        streams[k].result()
    torch.cuda.synchronize()

    ms = {1: [], 2: []}
    for _ in range(args.reps):
        for k in (1, 2):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            run_resident(k)
            e1.record()
            torch.cuda.synchronize()
            ms[k].append(e0.elapsed_time(e1))

    stream_ms = {1: [], 2: []}
    for _ in range(max(1, args.reps // 2)):
        for k in (1, 2):
            ss = streams[k]
            ss.submit(packed[k])                                # primed: one batch always uploads ahead
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(args.stream_steps):
                ss.submit(packed[k])
                ss.result()
            torch.cuda.synchronize()
            stream_ms[k].append((time.perf_counter() - t0) * 1e3 / args.stream_steps)
            ss.result()                                         # drain outside the clock

    stage = {1: [], 2: []}
    hd.set_stage_timing(1)
    try:
        for _ in range(max(1, args.reps // 2)):
            for k in (1, 2):
                run_resident(k)
                acc = hd.accounting()["affinity"]
                stage[k].append(dict(ms=acc["ms"], bytes=acc["bytes"], launches=acc["launches"]))
    finally:
        hd.set_stage_timing(0)

    B = args.batch
    out = {
        "workload": f"{B} chunks, n_target {args.n_target}, config_tarl_spatial_dino, seeds {args.seed}..{args.seed + B - 1} "
                    "(bench.make_batch); camera 0 = bench.py's DINOv2 rows, camera 1 = the synthetic second camera",
        "points": int(packed[1].off[-1]),
        "dino_bytes_per_pair_ratio": (96 + 2 * 384) / (96 + 384),
    }
    for k in (1, 2):
        r, s = float(np.median(ms[k])), float(np.median(stream_ms[k]))
        out[f"cams_{k}"] = {
            "resident": {"ms": r, "ms_all": ms[k], "chunks_per_s": B / r * 1e3},
            "segment_stream": {"ms_per_batch": s, "ms_all": stream_ms[k], "chunks_per_s": B / s * 1e3},
            "affinity_stage": {"ms": float(np.median([x["ms"] for x in stage[k]])), "ms_all": [x["ms"] for x in stage[k]],
                               "bytes": stage[k][0]["bytes"], "launches": stage[k][0]["launches"]},
            "h2d_bytes_per_batch": int(packed[k].h2d_bytes()),
        }
    out["affinity_stage_ratio_2_over_1"] = out["cams_2"]["affinity_stage"]["ms"] / out["cams_1"]["affinity_stage"]["ms"]
    out["device"] = torch.cuda.get_device_name(dev)
    out["power_limit_w"] = power_limit()
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
