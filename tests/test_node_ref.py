"""CPU checks of the per-node reference (`oracle/node_ref.py`) and of the designed chunks the GPU node-record tests run on.

`node_tree` gives every eigensolver node of a chunk its exact record (dense float64 eigen-pair, cut, decision) and the
margins by which that outcome is decided.  Here it is checked against the numpy model of the device algorithm and the
pinned reference, and every fixture chunk is shown to be usable: every node of its tree is clear (one correct outcome),
and the chunk reaches the eigensolver edges it is there for (tests/test_gpu_node_records.py):

* bins:  root components of exactly 320/321, 512/513, 640/641, 1024/1025, 2048/2049, 4096 points (the edges of the size
         bins of the persistent eigensolver kernel, kernels_graph.cuh::cluster_class) and one above 4096 (grid-wide path);
* tiny:  nodes of 3 to 7 points in a chunk of 250, so that they pass the 1 % size rule: Krylov exhaustion (k = n - 1) and,
         at 8 CTAs per node, CTAs without rows;
* dense: a node of 1000 points at about 120 stored entries per row whose CSR slices do not fit shared memory at 2 CTAs per
         node and do at 8: the in-kernel dense matvec and the separate cut kernels under one map, the CSR form and the
         fused cut under another;
* slow:  a long serpentine strip whose Fiedler vector needs more than the 256 steps of the persistent kernel: the hand-off
         to the multi-launch path;
* bench: two chunks of the benchmarked workload.
"""
import functools

import numpy as np
import pytest
from scipy.sparse import csr_matrix
from scipy.sparse.csgraph import connected_components

from conftest import CONFIG_NAMES, GOLDEN_SEEDS, load_golden
from autoinst_b200.synthetic import CONFIGS, make_chunk
from oracle import device_model as M
from oracle import ncut_ref as R
from oracle import node_ref as NR
from oracle.affinity_ref import affinity_ref
from test_partial_reorth import lanczos_fiedler_device

CFG = CONFIGS["tarl_spatial"]
CL_KMAX = 256                                   # csrc kernels_cluster.cuh: steps of the persistent eigensolver kernel ...
CL_NMAX = 4096                                  # ... and its largest node
BIN_EDGES = (320, 321, 512, 513, 640, 641, 1024, 1025, 2048, 2049, 4096, 4097)
ACCOUNTED_MAPS = (112248, 888888)               # ANCUTS_OPT_CLUSTER_MAP values under which the dense chunk is accounted


def ctas(cmap, n):
    """CTAs per node of n <= 4096 points under a cluster map (six digits: CTAs for the size bins up to BIN_EDGES)."""
    b = next(i for i, hi in enumerate(BIN_EDGES[0::2]) if n <= hi)
    return int(str(cmap)[b])


def _patch(rng, n, aspect, spacing):
    """n points of a jittered grid (pitch `spacing`) on an irregular oval patch of the given aspect, in the xy plane."""
    a, b = aspect, 1.0
    span = spacing * np.sqrt(n / (np.pi * a * b)) * 1.6
    gx = np.arange(-a * span, a * span, spacing)
    gy = np.arange(-b * span, b * span, spacing)
    X, Y = np.meshgrid(gx, gy)
    P = np.stack([X.ravel(), Y.ravel()], 1)
    P = P + rng.uniform(-0.3, 0.3, P.shape) * spacing
    ang = np.arctan2(P[:, 1] / b, P[:, 0] / a)
    ph = rng.uniform(0, 2 * np.pi, 2)
    r = np.hypot(P[:, 0] / a, P[:, 1] / b) / (1 + 0.15 * np.sin(3 * ang + ph[0]) + 0.1 * np.sin(5 * ang + ph[1]))
    assert P.shape[0] >= n
    P = P[np.argsort(r, kind="stable")[:n]]
    return np.column_stack([P, rng.normal(0, 0.03, n)])


def _line(rng, n):
    """n points along a line about 0.44 m apart: neighbours and next-neighbours linked, nothing further."""
    x = np.concatenate([[0.0], np.cumsum(rng.uniform(0.42, 0.46, n - 1))])
    return np.column_stack([x, rng.normal(0, 0.02, n), rng.normal(0, 0.02, n)])


def _serpentine(rng, n, legs, leg, pitch=2.0, width=0.4):
    """n points on a strip of the given width that runs `legs` times along x (`leg` metres), `pitch` apart in y."""
    V = np.array([(0.0 if (i % 2 == 0) == (j == 0) else leg, i * pitch) for i in range(legs) for j in range(2)])
    seg = np.diff(V, axis=0)
    ln = np.hypot(seg[:, 0], seg[:, 1])
    cum = np.concatenate([[0.0], np.cumsum(ln)])
    s = np.sort(rng.uniform(0, cum[-1], n))
    j = np.minimum(np.searchsorted(cum, s, side="right") - 1, len(seg) - 1)
    P = V[j] + ((s - cum[j]) / ln[j])[:, None] * seg[j]
    nrm = np.column_stack([-seg[j, 1], seg[j, 0]]) / ln[j][:, None]
    P = P + nrm * rng.uniform(-width / 2, width / 2, n)[:, None]
    return np.column_stack([P, rng.normal(0, 0.03, n)])


def designed_chunk(seed, objects, gap=1.6):
    """Chunk of separated objects of exact sizes (each one root component of that size), placed along x `gap` metres
    apart (proximity: 1 m).  objects: ("patch", n[, spacing]) irregular surface patch, about 40 stored entries per row at
    the default 0.27 m pitch; ("line", n); ("serpentine", n, legs).  TARL rows: one prototype per object plus noise, 5 %
    zero rows, as synthetic.make_chunk.  Returns (points, tarl, sizes)."""
    rng = np.random.default_rng(seed)
    pts, inst, x0 = [], [], 0.0
    for o, spec in enumerate(objects):
        kind, n = spec[0], spec[1]
        if kind == "patch":
            p = _patch(rng, n, rng.uniform(1.8, 2.6), spec[2] if len(spec) > 2 else 0.27)
        elif kind == "line":
            p = _line(rng, n)
        else:
            p = _serpentine(rng, n, spec[2], 24.0)
        p = p - p.min(axis=0) + np.array([x0, 0.0, 0.0])
        x0 = p[:, 0].max() + gap
        pts.append(p)
        inst.append(np.full(n, o))
    perm = rng.permutation(sum(len(p) for p in pts))
    points = np.concatenate(pts)[perm].astype(np.float32).astype(np.float64)
    im = np.concatenate(inst)[perm]
    proto = rng.normal(0, 1, size=(len(objects), 96))
    t = (proto[im] + 0.3 * rng.normal(0, 1, size=(len(im), 96))).astype(np.float32)
    t[rng.random(len(im)) < 0.05] = 0.0
    return points, t.astype(np.float64), [spec[1] for spec in objects]


# name -> (seed, objects); seeds chosen so that every node of every tree is clear (test_every_fixture_node_is_clear)
DESIGNED = {
    "bins_a": (1, [("patch", 4096), ("patch", 2049), ("patch", 513), ("patch", 320)]),
    "bins_b": (2, [("patch", 4200), ("patch", 2048), ("patch", 641), ("patch", 321)]),
    "bins_c": (3, [("patch", 1024), ("patch", 1025), ("patch", 512), ("patch", 640)]),
    "tiny": (4, [("line", 3), ("line", 4), ("line", 5), ("line", 6), ("line", 7), ("patch", 225)]),
    "dense": (5, [("patch", 1000, 0.15), ("patch", 700), ("patch", 900)]),
    "slow": (6, [("serpentine", 2100, 7), ("patch", 800)]),
}
BENCH_SEEDS = (6, 7)
FIXTURES = list(DESIGNED) + [f"bench_{s}" for s in BENCH_SEEDS]


@functools.lru_cache(maxsize=None)
def fixture_chunk(name):
    """(points, tarl, object sizes or None) of a fixture chunk."""
    if name.startswith("bench_"):
        ch = make_chunk(int(name.split("_")[1]), n_target=8192, features="tarl")
        return ch.points, ch.tarl, None
    seed, objects = DESIGNED[name]
    return designed_chunk(seed, objects)


@functools.lru_cache(maxsize=None)
def fixture_reference(name):
    """float32 affinity of the chunk (what the device holds), its node_tree records and labels."""
    points, tarl, _ = fixture_chunk(name)
    W32 = affinity_ref(points, tarl, None, alpha=CFG["alpha"], theta=CFG["theta"]).astype(np.float32)
    recs, labels = NR.node_tree(W32, CFG["T"])
    return W32, recs, labels


def _model(W32, points=None):
    """Labels and per-node stats of the numpy model of the device algorithm: the persistent kernel's step for nodes of up
    to 4096 points; a node it does not finish in 256 steps, or a larger one, starts over on the grid-wide path (the
    twice-CGS step with a check every 16 steps, kernels_lanczos.cuh::k_lanczos_init), up to 1024 steps."""
    stats = []
    grid = M.lanczos_fiedler

    def step(Wb32, d, *, kmax, stats, v0=None, **kw):
        n = Wb32.shape[0]
        if n <= CL_NMAX:
            st = []
            ev, lam2 = lanczos_fiedler_device(Wb32, d, kmax=CL_KMAX, stats=st, v0=v0, **kw)
            if st[0]["converged"]:
                stats.extend(st)
                return ev, lam2
        ev, lam2 = grid(Wb32, d, kmax=kmax, check_every=16, stats=stats, v0=v0, **kw)
        stats[-1]["grid"] = True
        return ev, lam2

    M.lanczos_fiedler = step
    try:
        lab = M.segment_model(W32, CFG["T"], stats=stats, kmax=1024, points=points)
    finally:
        M.lanczos_fiedler = grid
    return lab, stats


def _compare_with_model(recs, labels, W32, points=None):
    lab, stats = _model(W32, points)
    assert R.same_partition(lab, labels)
    ref = sorted((r["n"], r["best_k"], r["split"], r["lambda2"]) for r in recs)
    mod = sorted((s["n"], s["best_k"], int(s["best_k"] >= 0 and s["mcut"] < CFG["T"]), s["lam2"]) for s in stats)
    assert [r[:3] for r in ref] == [m[:3] for m in mod]
    assert all(m[3] == pytest.approx(r[3], abs=1e-9) for r, m in zip(ref, mod))
    assert all(s["converged"] for s in stats)


@pytest.mark.parametrize("name", FIXTURES)
def test_node_tree_matches_the_device_model(name):
    """Same partition, same nodes (size, threshold, decision) and lambda2 to 1e-9 as the Lanczos model of the device."""
    W32, recs, labels = fixture_reference(name)
    points = fixture_chunk(name)[0]
    _compare_with_model(recs, labels, W32, points)


@pytest.mark.parametrize("seed", GOLDEN_SEEDS)
@pytest.mark.parametrize("cfg", CONFIG_NAMES)
def test_node_tree_matches_the_reference_on_golden(seed, cfg):
    """Golden chunks: every root component exceeds the 1 % size limit, so the device recursion and the reference's
    give the same leaves (DESIGN.md §4.2)."""
    inp, out, A = load_golden(seed, cfg)
    W32 = A.toarray().astype(np.float32)
    recs, labels = NR.node_tree(W32, float(out["T"]))
    assert len(recs) > 0 and R.same_partition(labels, out["labels"])


@pytest.mark.parametrize("name", FIXTURES)
def test_every_fixture_node_is_clear(name):
    _, recs, _ = fixture_reference(name)
    unclear = [(r["level"], r["n"], {k: r[k] for k in NR.CLEAR if not r[k] > NR.CLEAR[k]}) for r in recs
               if not NR.node_is_clear(r)]
    assert not unclear
    assert len(recs) > 0


@pytest.mark.parametrize("name", list(DESIGNED))
def test_designed_objects_are_root_components_of_exact_size(name):
    W32, recs, _ = fixture_reference(name)
    _, _, sizes = fixture_chunk(name)
    nc, lab = connected_components(csr_matrix(W32 != 0), directed=False)
    assert sorted(np.bincount(lab).tolist()) == sorted(sizes)
    assert sorted(r["n"] for r in recs if r["level"] == 1) == sorted(s for s in sizes if s > 2)


def test_bins_reach_every_bin_edge():
    roots = [r["n"] for name in ("bins_a", "bins_b", "bins_c") for r in fixture_reference(name)[1] if r["level"] == 1]
    for edge in BIN_EDGES[:-1]:
        assert edge in roots, edge
    assert max(roots) >= BIN_EDGES[-1]


def test_tiny_nodes_exhaust_the_krylov_space():
    W32, recs, _ = fixture_reference("tiny")
    small = sorted(r["n"] for r in recs if r["n"] <= 7)
    assert small == [3, 4, 5, 6, 7]
    _, stats = _model(W32)
    assert all(s["k"] == s["n"] - 1 for s in stats if s["n"] <= 7)


def test_dense_node_misfits_at_two_ctas_and_fits_at_eight():
    _, recs, _ = fixture_reference("dense")
    big = [r for r in recs if r["n"] == 1000]
    assert len(big) == 1 and np.mean(big[0]["entries"]) > 100
    assert NR.slice_fits(big[0]["entries"], 2) is False
    assert NR.slice_fits(big[0]["entries"], 8) is True
    # the GPU test predicts the matvec bytes of every node of this chunk under these maps: no slice may be undecided
    for cmap in ACCOUNTED_MAPS:
        for r in recs:
            assert NR.slice_fits(r["entries"], ctas(cmap, r["n"])) is not None, (cmap, r["n"])
    assert NR.slice_fits(big[0]["entries"], ctas(ACCOUNTED_MAPS[0], 1000)) is False
    assert NR.slice_fits(big[0]["entries"], ctas(ACCOUNTED_MAPS[1], 1000)) is True


def test_slow_node_needs_more_steps_than_the_persistent_kernel_takes():
    W32, recs, _ = fixture_reference("slow")
    _, stats = _model(W32, fixture_chunk("slow")[0])
    slow = [s for s in stats if s["k"] > CL_KMAX and s["n"] <= CL_NMAX]
    assert slow and all(s["converged"] and s["grid"] for s in slow)
    assert max(s["k"] for s in stats) <= 1024 - 100


def test_bench_chunks_have_realistic_trees():
    for s in BENCH_SEEDS:
        _, recs, _ = fixture_reference(f"bench_{s}")
        assert len(recs) >= 20 and max(r["level"] for r in recs) >= 3
        assert sum(r["split"] for r in recs) >= 3 and any(not r["split"] for r in recs)


def test_slice_fit_follows_the_kernel_layout():
    """Hand-computed cases of the MODE 7 set-up arithmetic (194 KB = 24832 doubles)."""
    # 512 rows of 44 entries: z 4104 + ptr 258 + values 11264 + columns 5632 = 21258 doubles
    assert NR.slice_fits(np.full(4096, 44), 8) is True
    # 512 rows of 68 entries: 4104 + 258 + 17408 + 8704 = 30474 > 24832
    assert NR.slice_fits(np.full(4096, 68), 8) is False
    # half the rows 4, half 160 entries, 256 rows per CTA: fits with the small rows, not with the large ones
    assert NR.slice_fits(np.r_[np.full(256, 4), np.full(256, 160)], 2) is None
