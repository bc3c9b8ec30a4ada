"""Digest of what one segment call returns for the bench batch (labels, node records): to compare two builds of the
library (ANCUTS_LIB_PATH) that are meant to give bit-identical results.
    python tools/labels_digest.py [--batch 32] [--matvec 1] [--config tarl_spatial_dino]"""
import argparse
import hashlib
import os
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--n-target", dest="n_target", type=int, default=8192)
    ap.add_argument("--matvec", type=int, default=0, help="ANCUTS_OPT_MATVEC: 0 shared-memory sparse (default), 1 dense")
    ap.add_argument("--config", default="tarl_spatial", choices=["spatial", "tarl_spatial", "tarl_spatial_dino"])
    args = ap.parse_args()
    import torch
    from autoinst_b200 import api
    from autoinst_b200.synthetic import CONFIGS, make_chunk
    cfg = CONFIGS[args.config]
    chunks = [make_chunk(1000 + i, n_target=args.n_target, features="tarl_dino" if cfg["gamma"] else "tarl")
              for i in range(args.batch)]
    packed = api.PackedChunks([c.points for c in chunks], [c.tarl for c in chunks], [c.dino for c in chunks],
                              theta=cfg["theta"], gamma=cfg["gamma"])
    from autoinst_b200._lib import OPT_MATVEC
    hd = api.Handle.get(torch.device("cuda:0"))
    hd.set_option(OPT_MATVEC, args.matvec)
    res = api.segment_packed(packed, device=torch.device("cuda:0"), alpha=cfg["alpha"], theta=cfg["theta"],
                             gamma=cfg["gamma"], T=cfg["T"], want_stats=True)
    h = hashlib.sha1()
    for lab in res.labels:
        h.update(np.ascontiguousarray(lab).tobytes())
    st = res.stats
    # every field is a sort key: records of one level that agree on (chunk, n, n_side) are appended by concurrent CTAs in
    # no fixed order, so the digests are those of the set of records
    order = np.lexsort((st["lambda2"], st["mcut"], st["steps"], st["split"], st["best_k"], st["n_side"], st["n"], st["level"],
                        st["chunk"]))
    key = np.stack([st[k] for k in ("chunk", "level", "n", "n_side")], axis=1)
    ties = len(key) - len(np.unique(key, axis=0))
    h2 = hashlib.sha1()
    for k in ("chunk", "level", "n", "n_side", "best_k", "split", "steps"):
        h2.update(np.ascontiguousarray(st[k][order]).tobytes())
    h3 = hashlib.sha1(np.ascontiguousarray(st["mcut"][order]).tobytes())
    h4 = hashlib.sha1(np.ascontiguousarray(st["lambda2"][order]).tobytes())
    print("labels", h.hexdigest()[:16], "records", h2.hexdigest()[:16], "mcut", h3.hexdigest()[:16],
          "lambda2", h4.hexdigest()[:16], "nodes", len(st), "steps", int(st["steps"].sum()), "unconverged", res.unconverged,
          "reorth", hd.reorth_accounting(),
          "records tied on (chunk, level, n, n_side)", ties)


if __name__ == "__main__":
    main()
