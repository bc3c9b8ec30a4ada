"""CPU checks of the edge fixtures of the segment path's affinity (tests/test_gpu_affinity_edges.py).

The segment path builds W with its own pair search (cell-sorted counting sort, tile boxes, box pruning, float32
pre-filter, exact float64 test) and writes it through the root order after the root split.  The GPU file observes that W
through the node records of the segment path against `oracle.node_ref.node_tree` and through the stage entry against
`oracle.affinity_ref`.  Here every fixture is shown to be usable for that (every node of its tree, under every config the
GPU file runs it with, is clear: one correct outcome) and to reach the edge it is there for:

* threshold:  one pair at float64 distance exactly `proximity` joins two objects, one pair a float32 ulp beyond it does not
              join two others; the four objects sit in two z layers of the cell grid so that the tiles of the sweep are
              pure and the two tiles of the joining pair have boxes exactly `proximity` apart (the box-pruning edge);
              also scaled by 0.5 and 2 and run at those proximities;
* far:        a chunk in map-frame coordinates (centre (3456.5, -1234.25, 87.0));
* outlier:    one point 36 km away, first in input order and in cell order: the origin of the float32 relative coordinates of
              the first tile of both sweeps, whose rounding (up to 4e-3 m) only the 1e-2 m margin of the pre-filter covers;
* wide:       objects over 40 m along x and one point 300 m out: cell pitch above `proximity`, cells clamp;
* coincident: exactly repeated points (distance 0);
* tiles:      root components of 63/64/65, 127/128/129, 255/256/257 points; chunks of those sizes (n63 ... n257);
* isolated:   every point more than `proximity` from every other: an empty pair queue;
* features:   TARL widths 4 and 36, DINOv2 widths 12 and 768 (one and two cameras), 5 % zero TARL rows, 30 % zero DINOv2
              rows, one object whose TARL rows sit at the tensor-core form's cancellation cutoff.
"""
import functools

import numpy as np
import pytest
from scipy.sparse import csr_matrix
from scipy.sparse.csgraph import connected_components
from scipy.spatial.distance import cdist

from autoinst_b200.synthetic import CONFIGS
from oracle import node_ref as NR
from oracle.affinity_ref import affinity_ref
from test_node_ref import _patch

PS_T, AT = 128, 64              # csrc kernels_graph.cuh: tile sides of the cell-sorted sweep and of the shuffled sweep
PG_DIM = 25                     # cells per axis of the cell grid (k_pair_grid_b)
CENTRE = np.array([3456.5, -1234.25, 87.0])
TILE_SIZES = (63, 64, 65, 127, 128, 129, 255, 256, 257)
TC_SCALES = (0.1, 1.0, 3.0, 10.0)


def _f32(x):
    return np.asarray(x, dtype=np.float32).astype(np.float64)


def _place(rng, specs, gap=1.6, x0=0.0):
    """Patches ("patch", n[, spacing]) placed along x `gap` metres apart; returns their point arrays."""
    out = []
    for spec in specs:
        p = _patch(rng, spec[1], rng.uniform(1.8, 2.6), spec[2] if len(spec) > 2 else 0.27)
        p = p - p.min(axis=0) + np.array([x0, 0.0, 0.0])
        x0 = p[:, 0].max() + gap
        out.append(p)
    return out


def _features(rng, im, n_obj, tdim, ddim, cams=2, sigma=None):
    """TARL rows (one prototype per object plus noise `sigma[object]`, 5 % zero rows) and `cams` DINOv2 cameras (prototype
    plus 0.3 noise, 30 % zero rows each), as synthetic.make_chunk makes them; float32 values as float64."""
    n = len(im)
    sig = np.full(n_obj, 0.3) if sigma is None else np.asarray(sigma)
    t = rng.normal(0, 1, (n_obj, tdim))[im] + sig[im, None] * rng.normal(0, 1, (n, tdim))
    t[rng.random(n) < 0.05] = 0.0
    dino = []
    for _ in range(cams):
        g = rng.normal(0, 1, (n_obj, ddim))[im] + 0.3 * rng.normal(0, 1, (n, ddim))
        g[rng.random(n) < 0.30] = 0.0
        dino.append(_f32(g))
    return _f32(t), dino


def _chunk(rng, parts, first=None, **feat):
    """Objects -> (points, tarl, dino cameras, object sizes, object of every point); points permuted, float32-representable.
    `first`: one point put at input index 0 (its own object)."""
    sizes = [len(p) for p in parts]
    pts = np.concatenate(parts)
    im = np.repeat(np.arange(len(parts)), sizes)
    perm = rng.permutation(len(pts))
    pts, im = pts[perm], im[perm]
    if first is not None:
        pts = np.vstack([first[None, :], pts])
        im = np.concatenate([[len(parts)], im])
        sizes = sizes + [1]
    tarl, dino = _features(rng, im, len(sizes), **feat)
    return _f32(pts), tarl, dino, sizes, im


def _layered_pair(rng, n_low, n_high, x0, dz):
    """Two patches joined by ONE pair: the low one below z = 0 with its largest-x point a raised to z = 0, the high one
    above z = 1 + 0.02 extending from its point b = a + (0, 0, dz) towards +x.  Every other pair is at least 1.02 apart."""
    lo = _f32(_patch(rng, n_low, rng.uniform(1.8, 2.6), 0.27))
    lo[:, 0] += x0 - lo[:, 0].min()
    a = int(np.argmax(lo[:, 0]))
    lo[:, 2] = -_f32(0.02 + np.abs(rng.normal(0, 0.03, n_low)))
    lo[a, 2] = 0.0
    hi = _f32(_patch(rng, n_high, rng.uniform(1.8, 2.6), 0.27))
    b = int(np.argmin(hi[:, 0]))
    hi[:, :2] = _f32(hi[:, :2] - hi[b, :2] + lo[a, :2])
    hi[b, :2] = lo[a, :2]
    hi[:, 2] = _f32(1.02 + np.abs(rng.normal(0, 0.03, n_high)))
    hi[b, 2] = dz
    return lo, hi


def _threshold(seed, scale=1.0):
    rng = np.random.default_rng(seed)
    a_lo, a_hi = _layered_pair(rng, 256, 200, 0.0, 1.0)
    b_lo, b_hi = _layered_pair(rng, 256, 180, 0.0, float(np.nextafter(np.float32(1.0), np.float32(2.0))))
    dy = np.ceil(max(a_lo[:, 1].max(), a_hi[:, 1].max()) - min(b_lo[:, 1].min(), b_hi[:, 1].min()) + 1.6)
    b_lo[:, 1] += dy                             # side by side in y: the extent stays below 24 cells
    b_hi[:, 1] += dy
    pts, tarl, dino, sizes, im = _chunk(rng, [a_lo, a_hi, b_lo, b_hi], tdim=96, ddim=384)
    return pts * scale, tarl, dino, sizes, im       # scaling by a power of two is exact


def _far(seed):
    rng = np.random.default_rng(seed)
    parts = _place(rng, [("patch", 600), ("patch", 450), ("patch", 350)])
    c = np.concatenate(parts).mean(axis=0)
    return _chunk(rng, [p - c + CENTRE for p in parts], tdim=96, ddim=384)


def _outlier(seed):
    rng = np.random.default_rng(seed)
    parts = _place(rng, [("patch", 500), ("patch", 400), ("patch", 300)])
    lo = np.concatenate(parts).min(axis=0)
    return _chunk(rng, parts, first=lo - np.array([36000.0, 1.0, 1.0]), tdim=96, ddim=384)


def _wide(seed):
    rng = np.random.default_rng(seed)
    parts = _place(rng, [("patch", 130, 0.3)] * 8, gap=3.0)
    hi = np.concatenate(parts).max(axis=0)
    return _chunk(rng, parts, first=np.array([hi[0] / 2, 300.0, 0.0]), tdim=96, ddim=384)


def _coincident(seed):
    rng = np.random.default_rng(seed)
    a, b = _place(rng, [("patch", 300, 0.4), ("patch", 400)])
    dup = rng.random(len(b)) < 0.5
    return _chunk(rng, [np.repeat(a, 3, axis=0), np.vstack([b, b[dup]])], tdim=96, ddim=384)


def _tiles(seed):
    rng = np.random.default_rng(seed)
    return _chunk(rng, _place(rng, [("patch", n) for n in TILE_SIZES]), tdim=96, ddim=384)


def _one_object(seed, n):
    rng = np.random.default_rng(seed)
    return _chunk(rng, _place(rng, [("patch", n)]), tdim=96, ddim=384)


def _isolated(seed):
    rng = np.random.default_rng(seed)
    g = np.stack(np.meshgrid(*[np.arange(6) * 1.25] * 3, indexing="ij"), -1).reshape(-1, 3)
    return _chunk(rng, [g + rng.uniform(-0.05, 0.05, g.shape)], tdim=96, ddim=384)


def _features_chunk(seed, tdim=96, ddim=384):
    rng = np.random.default_rng(seed)
    parts = _place(rng, [("patch", 600), ("patch", 500), ("patch", 400)])
    return _chunk(rng, parts, tdim=tdim, ddim=ddim, sigma=[0.3, 0.1, 0.3])


# name -> (builder, seed, keywords); every node of every tree the GPU file runs is clear (test_every_node_is_clear)
FIXTURES = {
    "threshold": (_threshold, 1, {}),
    "threshold_x0.5": (_threshold, 1, {"scale": 0.5}),
    "threshold_x2": (_threshold, 1, {"scale": 2.0}),
    "far": (_far, 2, {}),
    "outlier": (_outlier, 3, {}),
    "wide": (_wide, 4, {}),
    "coincident": (_coincident, 5, {}),
    "tiles": (_tiles, 6, {}),
    **{f"n{n}": (_one_object, 10 + i, {"n": n}) for i, n in enumerate(TILE_SIZES)},
    **{f"n{n}": (_one_object, 30 + n, {"n": n}) for n in (1, 2, 3)},
    "isolated": (_isolated, 7, {}),
    "features": (_features_chunk, 8, {}),
    "feat_t4": (_features_chunk, 8, {"tdim": 4}),
    "feat_t36": (_features_chunk, 8, {"tdim": 36}),
    "feat_d12": (_features_chunk, 8, {"ddim": 12}),
    "feat_d768": (_features_chunk, 8, {"ddim": 768}),
}
PROXIMITY = {"threshold_x0.5": 0.5, "threshold_x2": 2.0}

# config name -> (synthetic.CONFIGS entry, DINOv2 cameras)
RUN_CONFIGS = {"spatial": ("spatial", 0), "tarl_spatial": ("tarl_spatial", 0),
               "tarl_spatial_dino": ("tarl_spatial_dino", 1), "tarl_spatial_dino2": ("tarl_spatial_dino", 2)}
GEOMETRY = ["threshold", "far", "outlier", "wide", "coincident", "tiles", "isolated", "features"] + \
           [f"n{n}" for n in TILE_SIZES]
# groups of (fixture, config) the GPU file runs as one batch each: same config, same feature widths
# coincident points under the spatial term alone have bit-identical rows, and the Fiedler entries of a repeated extreme
# point differ by rounding only: their threshold margin is ~1e-16, no node of that tree is clear
GROUPS = {f"geometry_{c}": (c, [f for f in GEOMETRY if (f, c) != ("coincident", "spatial")]) for c in RUN_CONFIGS}
GROUPS.update({f"{f}_{c}": (c, [f]) for f in ("feat_t4", "feat_t36")
               for c in ("tarl_spatial", "tarl_spatial_dino", "tarl_spatial_dino2")})
GROUPS.update({f"{f}_{c}": (c, [f]) for f in ("feat_d12", "feat_d768") for c in ("tarl_spatial_dino", "tarl_spatial_dino2")})
GROUPS.update({f"{f}_tarl_spatial": ("tarl_spatial", [f]) for f in PROXIMITY})
# one call: chunks of 1, 2 and 3 points, the empty queue and the tile-edge sizes between two larger fixtures
BATCH = ["n1", "threshold", "n2", "isolated", "n3"] + [f"n{n}" for n in TILE_SIZES] + ["far"]
GROUPS["batch_tarl_spatial"] = ("tarl_spatial", BATCH)
CASES = [(f, g[0]) for g in GROUPS.values() for f in g[1]]


@functools.lru_cache(maxsize=None)
def fixture(name):
    """(points, tarl, list of DINOv2 cameras, object sizes, object of every point) of an edge fixture."""
    build, seed, kw = FIXTURES[name]
    return build(seed, **kw)


def proximity(name):
    return PROXIMITY.get(name, 1.0)


def run_config(config):
    """(alpha, theta, gamma, T, cams) of a config."""
    base, cams = RUN_CONFIGS[config]
    c = CONFIGS[base]
    return dict(alpha=c["alpha"], theta=c["theta"], gamma=c["gamma"]), c["T"], cams


def inputs(name, config):
    """(points, tarl or None, DINOv2 cameras or None) as a config uses them."""
    pts, tarl, dino = fixture(name)[:3]
    gains, _, cams = run_config(config)
    return pts, (tarl if gains["theta"] else None), (dino[:cams] if gains["gamma"] else None)


@functools.lru_cache(maxsize=None)
def reference(name, config):
    """float64 affinity, its float32 rounding (what the device holds), node_tree records and labels."""
    pts, tarl, dino = inputs(name, config)
    gains, T, _ = run_config(config)
    A = affinity_ref(pts, tarl, dino, proximity=proximity(name), **gains)
    W32 = A.astype(np.float32)
    recs, labels = NR.node_tree(W32, T)
    return A, W32, recs, labels


# ---- models of the pair search's geometry (csrc kernels_graph.cuh) ------------------------------------------------
def cell_order(pts, prox):
    """k_pair_grid_b: cells of pitch max(prox, extent / 24), at most 25 per axis (clamped), x fastest; points of a cell by
    input index.  Returns the input index of every cell-sorted rank."""
    lo, hi = pts.min(axis=0), pts.max(axis=0)
    pitch = max(prox, (hi - lo).max() / (PG_DIM - 1))
    inv_h = 1.0 / pitch
    dims = np.minimum(PG_DIM, np.floor((hi - lo) * inv_h).astype(int) + 1)
    c = np.clip(np.floor((pts - lo) * inv_h).astype(int), 0, dims - 1)
    cell = (c[:, 2] * dims[1] + c[:, 1]) * dims[0] + c[:, 0]
    return np.lexsort((np.arange(len(pts)), cell)), pitch


def tile_boxes(spts):
    n = len(spts)
    return [(spts[t:t + PS_T].min(axis=0), spts[t:t + PS_T].max(axis=0)) for t in range(0, n, PS_T)]


def box_gap2(a, b):
    """k_pair_sweep's squared gap of two tile boxes."""
    d = np.maximum(0.0, np.maximum(a[0] - b[1], b[0] - a[1]))
    return float(d[0] * d[0] + d[1] * d[1] + d[2] * d[2])


def prefilter_d2(pts, org, i, j):
    """Squared float32 distance of the pre-filter (coordinates relative to the tile origin `org`, rounded to float32) before
    its final float32 rounding, which changes it by a few ulp at most."""
    r = (pts[i] - org).astype(np.float32).astype(np.float64)
    c = (pts[j] - org).astype(np.float32).astype(np.float64)
    return ((r - c) ** 2).sum(axis=1)


def lim32(prox, margin):
    return float(np.float32((prox + margin) * (prox + margin) * 1.001))


# ---- the fixtures are usable ------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,config", CASES, ids=[f"{f}-{c}" for f, c in CASES])
def test_every_node_is_clear(name, config):
    _, _, recs, _ = reference(name, config)
    unclear = [(r["level"], r["n"], {k: r[k] for k in NR.CLEAR if not r[k] > NR.CLEAR[k]}) for r in recs
               if not NR.node_is_clear(r)]
    assert not unclear
    assert len(recs) > 0 or name in ("isolated", "n1", "n2")


@pytest.mark.parametrize("name", list(FIXTURES))
def test_fixture_is_float32_and_small(name):
    pts, tarl, dino, sizes, _ = fixture(name)
    assert len(pts) == sum(sizes) <= 3000
    for x in [pts, tarl] + dino:
        assert np.array_equal(x, _f32(x))


@pytest.mark.parametrize("name", [n for n in FIXTURES if n not in ("isolated",)])
def test_objects_are_root_components_of_exact_size(name):
    pts, _, _, sizes, im = fixture(name)
    nc, lab = connected_components(csr_matrix(affinity_ref(pts, proximity=proximity(name)) != 0), directed=False)
    if name.startswith("threshold"):             # objects 0 and 1 are one component (test_threshold_pairs)
        im = np.where(im == 1, 0, im)
    assert nc == len(np.unique(im))
    for c in range(nc):                          # every component is exactly one object
        assert len(np.unique(im[lab == c])) == 1 and len(np.unique(lab[im == im[lab == c][0]])) == 1


# ---- the fixtures reach their edges -------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["threshold", "threshold_x0.5", "threshold_x2"])
def test_threshold_pairs(name):
    """One pair at exactly `prox` joins objects 0 and 1 (one root component), one pair at the next float32 value up leaves
    objects 2 and 3 apart (two); every other pair between them is 2 % beyond `prox`.  The two points of the joining pair
    lie in different tiles of the cell-sorted sweep whose boxes are exactly `prox` apart."""
    pts, _, _, sizes, inst = fixture(name)
    prox = proximity(name)
    d = cdist(pts, pts)
    link = d[np.ix_(inst == 0, inst == 1)]
    assert link.min() == prox and (link == prox).sum() == 1
    assert np.sort(link.ravel())[1] >= 1.02 * prox
    beyond = d[np.ix_(inst == 2, inst == 3)]
    assert beyond.min() == float(np.nextafter(np.float32(prox), np.float32(2 * prox)))
    assert np.sort(beyond.ravel())[1] >= 1.02 * prox
    nc, lab = connected_components(csr_matrix(d <= prox), directed=False)
    roots = sorted(np.bincount(lab).tolist())
    assert roots == sorted([sizes[0] + sizes[1], sizes[2], sizes[3]])
    # the cell-sorted sweep: layer 0 (objects 0 and 2) first, whole tiles; the joining pair's tile boxes exactly prox apart
    order, pitch = cell_order(pts, prox)
    assert pitch == prox
    low = np.isin(inst, (0, 2))
    assert low[order[:low.sum()]].all() and low.sum() % PS_T == 0
    rank = np.empty(len(pts), dtype=int)
    rank[order] = np.arange(len(pts))
    i, j = np.argwhere(d == prox)[0]
    ti, tj = sorted((rank[i] // PS_T, rank[j] // PS_T))
    assert ti != tj
    boxes = tile_boxes(pts[order])
    assert box_gap2(boxes[ti], boxes[tj]) == prox * prox


def test_far_chunk_is_in_map_frame_coordinates():
    pts = fixture("far")[0]
    assert np.allclose(pts.mean(axis=0), CENTRE, atol=1e-2)
    assert np.abs(pts).min(axis=0)[0] > 3000


def test_outlier_is_the_origin_of_the_first_tiles_and_needs_the_prefilter_margin():
    """The outlier (input index 0) is the first cell-sorted point: the origin of tile 0 in both sweeps.  Relative to it
    the pre-filter's float32 squared distance of some in-mask pairs exceeds (1.001 prox^2) (what the test would see without
    the 1e-2 margin) and of none the real limit ((prox + 1e-2)^2 x 1.001)."""
    pts = fixture("outlier")[0]
    order, pitch = cell_order(pts, 1.0)
    assert order[0] == 0 and pitch > 1000
    d = cdist(pts, pts)
    for rows in (order[:PS_T], np.arange(AT)):           # cell-sorted sweep, shuffled sweep (input order)
        i, j = np.nonzero((d[rows] <= 1.0) & (d[rows] > 0))
        i = rows[i]
        f = prefilter_d2(pts, pts[0], i, j)
        assert f.max() < lim32(1.0, 1e-2) * (1 - 1e-5)
        assert (f > lim32(1.0, 0.0) * (1 + 1e-5)).sum() >= 2


def test_wide_chunk_has_clamped_cells_coarser_than_prox():
    pts = fixture("wide")[0]
    order, pitch = cell_order(pts[1:], 1.0)
    assert np.ptp(pts[1:, 0]) > 24 * 1.0 and pitch > 1.0              # the objects alone: pitch above prox
    order, pitch = cell_order(pts, 1.0)
    assert pitch > 10.0                                                  # with the outlier: 25 cells cover 300 m


def test_coincident_points_repeat_exactly_and_keep_the_queue():
    pts = fixture("coincident")[0]
    _, counts = np.unique(pts, axis=0, return_counts=True)
    assert counts.max() == 3 and (counts == 2).sum() > 100
    A = reference("coincident", "spatial")[0]
    pairs = ((A != 0).sum() - len(pts)) / 2
    assert pairs < 96 * len(pts)                  # the pair queue holds 96 pairs per point


def test_tile_edge_sizes():
    recs = reference("tiles", "tarl_spatial")[2]
    assert sorted(r["n"] for r in recs if r["level"] == 1) == sorted(TILE_SIZES)
    for n in TILE_SIZES + (1, 2, 3):
        assert len(fixture(f"n{n}")[0]) == n


def test_isolated_chunk_has_no_pair():
    A = reference("isolated", "tarl_spatial")[0]
    assert np.array_equal(A != 0, np.eye(len(A), dtype=bool))


def test_feature_fixtures():
    """Widths and zero rows as synthetic.make_chunk makes them; the object of TARL noise 0.1 puts pairs on both sides of the
    tensor-core form's cancellation cutoff (|f_i - f_j|^2 < 1e-2 (|f_i|^2 + |f_j|^2))."""
    for name, (t, d) in {"features": (96, 384), "feat_t4": (4, 384), "feat_t36": (36, 384), "feat_d12": (96, 12),
                         "feat_d768": (96, 768)}.items():
        pts, tarl, dino = fixture(name)[:3]
        assert tarl.shape == (len(pts), t) and len(dino) == 2 and all(g.shape == (len(pts), d) for g in dino)
        assert 0.03 < (~tarl.any(axis=1)).mean() < 0.07
        assert all(0.25 < (~g.any(axis=1)).mean() < 0.35 for g in dino)
    pts, tarl = fixture("features")[:2]
    d = cdist(pts, pts)
    i, j = np.nonzero((d <= 1.0) & (d > 0))
    nz = tarl[i].any(axis=1) & tarl[j].any(axis=1)
    i, j = i[nz], j[nz]
    nrm = (tarl ** 2).sum(axis=1)
    ratio = ((tarl[i] - tarl[j]) ** 2).sum(axis=1) / (nrm[i] + nrm[j])
    assert (ratio < 1e-2).sum() > 100 and ((ratio >= 1e-2) & (ratio < 1.5e-2)).sum() > 100


@pytest.mark.parametrize("scale", TC_SCALES)
def test_tc_scale_sweep_stays_in_normal_float32(scale):
    """The scaled TARL rows of the tensor-core sweep keep every in-mask weight a normal float32, so the 1e-5 relative gate
    measures the kernel, not float32 underflow."""
    pts, tarl = fixture("features")[:2]
    A = affinity_ref(pts, _f32(tarl * scale), None, alpha=1.0, theta=0.5)
    assert A[A != 0].min() > 2.0 ** -126
