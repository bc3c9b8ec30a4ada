"""Per-node reference of the device recursion (TEST INFRASTRUCTURE, see oracle/__init__.py).

`device_model.segment_model` restates the device algorithm step for step, Lanczos included, so it inherits the
eigensolver's own stopping error.  Here every node of the tree gets the exact quantities the device records for it
(`ancuts_node_stat`): each eigen-pair comes from DENSE `scipy.linalg.eigh` of the node's normalised Laplacian, every sum
is float64.  The recursion is the device's, not the reference's peeling (DESIGN.md §4.2):

* the root (level 0) is split into its connected components, which sit at level 1 (engine.cu::k_init_roots marks the
  root as split);
* a node is cut when it passes the size rule `n > 2 and n / (N + 1e-8) > lim` (`lim = split_lim` at the root, 0.01
  below) and its best N-cut value is below T; every side that passes the size rule is split into its components, one
  level below the node (`kernels_graph.cuh::k_new_ranges`);
* the ten thresholds are `t_k = k·step + min` with numpy's two roundings, a threshold's cost is
  `cut / vol_A + cut / vol_B`, the first strict minimum wins and `np.allclose(min, max)` leaves the node uncut.

Each record also carries the margins by which its outcome is decided.  A node whose margins are all far above the
eigensolver's tolerance (`node_is_clear`) has one correct outcome: a device result that differs there is wrong, not
rounded differently.
"""
from __future__ import annotations

import numpy as np
import scipy.linalg
from scipy.sparse import csr_matrix
from scipy.sparse.csgraph import connected_components

NUM_CUTS = 10
FIX_SHIFT = 40                    # csrc common.cuh: cut weights are summed in 2^-40 fixed point (DESIGN.md §4.4)

# csrc/kernels_cluster.cuh: shared-memory budget of the persistent eigensolver kernel and its slice geometry
CL_DYN_SMEM = 194 * 1024
CL_NMAX = 4096

# bounds of node_is_clear: 10^3 x or more above the 1e-10 residual tolerance of the Lanczos stop rule
CLEAR = dict(thr_margin=1e-7, sign_margin=1e-6, gap=1e-5, cost_margin=1e-6, T_margin=1e-6)


def _components(Wb):
    nc, lab = connected_components(csr_matrix(Wb != 0), directed=False)
    return [np.nonzero(lab == c)[0] for c in range(nc)]


def fix_shift(vol: float) -> int:
    """Fraction bits of a node's fixed-point cut sums (csrc kernels_ncut.cuh::fix_shift)."""
    return min(FIX_SHIFT, 61 - int(np.floor(np.log2(max(vol, 1.0)))))


def node_record(Wb: np.ndarray, T: float):
    """Eigen-pair, cut decision and margins of ONE connected node.  Wb: float64 block of w (unit diagonal).
    Returns (record, signed unit-norm Fiedler vector, mask side of the best threshold or None)."""
    n = Wb.shape[0]
    d = 1.0 + Wb.sum(axis=1)
    s = 1.0 / np.sqrt(d)
    L = np.eye(n) - s[:, None] * (Wb + np.eye(n)) * s[None, :]
    vals, vecs = scipy.linalg.eigh(L, subset_by_index=[0, 2])
    lam2, lam3 = float(vals[1]), float(vals[2])
    ev = vecs[:, 1] / np.linalg.norm(vecs[:, 1])
    if ev.sum() < 0:
        ev = -ev
    rec = dict(n=n, lambda2=lam2, lambda3=lam3, gap=lam3 - lam2, sign_margin=float(abs(ev.sum())),
               entries=(Wb != 0).sum(axis=1).astype(np.int64), best_k=-1, split=0, n_side=0, mcut=np.inf,
               costs=np.full(NUM_CUTS, np.inf), thr_margin=np.inf, cost_margin=np.inf, T_margin=np.inf, mcut_floor=0.0)
    mn, mx = ev.min(), ev.max()
    if np.allclose(mn, mx):
        return rec, ev, None
    step = (mx - mn) / NUM_CUTS
    t = np.arange(NUM_CUTS) * step + mn
    dist = np.abs(ev[:, None] - t[None, :])
    dist[ev == mn, 0] = np.inf                      # t_0 is min itself, in every rounding
    rec["thr_margin"] = float(dist.min() / np.abs(ev).max())
    bucket = (ev[:, None] > t[None, :]).sum(axis=1)
    iu, ju = np.nonzero(np.triu(Wb, 1))
    wv = Wb[iu, ju]
    lo = np.minimum(bucket[iu], bucket[ju])
    hi = np.maximum(bucket[iu], bucket[ju])
    costs = np.empty(NUM_CUTS)
    ncut_edges = np.empty(NUM_CUTS, dtype=np.int64)
    for k in range(NUM_CUTS):
        crossing = (lo <= k) & (hi > k)
        cut = wv[crossing].sum()
        vol_b = d[bucket <= k].sum()
        vol_a = d[bucket > k].sum()
        costs[k] = cut / vol_a + cut / vol_b
        ncut_edges[k] = crossing.sum()
    best_k = 0
    for k in range(1, NUM_CUTS):
        if costs[k] < costs[best_k]:
            best_k = k
    best = costs[best_k]
    # another threshold with the SAME mask has the same cost on the device too (integer cut sums, same volumes)
    cnt = np.bincount(bucket, minlength=NUM_CUTS + 1)
    other = [costs[k] for k in range(NUM_CUTS) if cnt[min(k, best_k) + 1:max(k, best_k) + 1].sum() > 0]
    side = bucket > best_k
    vol_a, vol_b = d[side].sum(), d[~side].sum()
    rec.update(best_k=best_k, mcut=float(best), costs=costs, split=int(best < T), n_side=int(side.sum()),
               cost_margin=float((min(other) - best) / best) if other and best > 0 else np.inf,
               T_margin=float(abs(best - T) / T),
               mcut_floor=float(ncut_edges[best_k] * 2.0 ** -fix_shift(d.sum()) * (1.0 / vol_a + 1.0 / vol_b)))
    return rec, ev, side


def node_tree(W32: np.ndarray, T: float, split_lim: float = 0.01, points=None):
    """Records of every eigensolver node of one chunk, and the chunk's labels.

    W32: the (N, N) float32 affinity the device holds (unit diagonal).  `points` is accepted for symmetry with
    `device_model.segment_model` and unused: dense eigen-pairs do not depend on a start vector.
    Returns (records, labels); records are dicts with level, n, n_side, best_k, split, lambda2, lambda3, mcut, the
    margins (thr_margin, sign_margin, gap, cost_margin, T_margin), mcut_floor, entries (stored entries per row) and idx
    (the node's point indices)."""
    del points
    W = np.asarray(W32, dtype=np.float32).astype(np.float64)
    N = W.shape[0]
    labels = np.full(N, -1, dtype=np.int32)
    records = []

    def passes(n, lim):
        return n > 2 and n / (N + 1e-8) > lim

    if not (passes(N, split_lim) and T > 0):
        labels[:] = 0
        return records, labels
    next_label = 0
    frontier = [(c, 1) for c in _components(W)]
    while frontier:
        nxt = []
        for idx, level in frontier:
            if not passes(idx.shape[0], 0.01):
                labels[idx] = next_label
                next_label += 1
                continue
            Wb = W[np.ix_(idx, idx)]
            rec, ev, side = node_record(Wb, T)
            rec.update(level=level, idx=idx)
            records.append(rec)
            if rec["split"]:
                for part in (idx[side], idx[~side]):
                    if passes(part.shape[0], 0.01):
                        nxt.extend((part[c], level + 1) for c in _components(W[np.ix_(part, part)]))
                    else:
                        nxt.append((part, level + 1))
            else:
                labels[idx] = next_label
                next_label += 1
        frontier = nxt
    return records, labels


def node_is_clear(rec: dict, bounds: dict = CLEAR) -> bool:
    """Every margin of the node above its bound: the node has one correct outcome (tree, threshold, decision)."""
    return all(rec[k] > v for k, v in bounds.items())


def slice_fits(entries, C: int):
    """Whether the node's CSR slices fit the shared memory of the persistent eigensolver kernel at C CTAs per node
    (csrc/kernels_cluster.cuh, MODE 7 set-up).  entries: stored entries of every row of the node (diagonal included).

    CTA r holds rows [r·rp, min(n, r·rp + rp)) of the node, rp = ceil(n / C), in the device's order of the node's points,
    which this side does not know.  Returns True when every CTA fits whatever the order (the rp largest rows fit), False
    when one CTA misfits whatever the order (rank 0 always holds rp rows: the rp smallest ones do not fit), None
    otherwise."""
    e = np.sort(np.asarray(entries, dtype=np.int64))
    n = e.shape[0]
    dyn_doubles = CL_DYN_SMEM // 8
    nz = (n + 8 + 3) & ~3                                  # zs: z of the whole node on its 16-byte window

    def misfit(rows):
        nr = rows.shape[0]
        total = int(((rows + 3) & ~3).sum())              # rows start at multiples of four entries
        ptr_d = (((nr + 1 + 1) // 2) + 1) & ~1             # row offsets (int), doubles, even
        val_d = (total + 1) // 2                           # float values
        col_d = (total + 3) // 4                           # 16-bit columns
        return nz + ptr_d + val_d + col_d > dyn_doubles

    rp = (n + C - 1) // C
    if not misfit(e[n - rp:]):
        return True
    if misfit(e[:rp]):
        return False
    return None
