"""GPU tests: every eigensolver node the segment path records (`ancuts_node_stat`) against the dense float64 reference
`oracle.node_ref.node_tree`, across cluster maps, matvec forms, the fused and separate cut, and the grid-wide path.

The fixture chunks (tests/test_node_ref.py) are built so that every node of their trees is clear: its size, threshold,
decision and side size have one correct value, and lambda2 and the N-cut value are pinned far below the margins.  So a
record that differs from the reference by more than the eigensolver's tolerance is a wrong result, whatever the labels.
"""
import numpy as np
import pytest

from oracle import ncut_ref as R
from test_node_ref import ACCOUNTED_MAPS, CFG, CL_KMAX, CL_NMAX, FIXTURES, ctas, fixture_chunk, fixture_reference

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

MATVEC, CMAP, FUSED = 2, 3, 4                   # include/autoinst_ncuts.h: ANCUTS_OPT_*
# name -> (ancuts_set_option values, segment_packed keywords)
CONFIGS = {
    "default": ({}, {}),
    "map_112248": ({CMAP: 112248}, {}),
    "map_222448": ({CMAP: 222448}, {}),
    "map_444488": ({CMAP: 444488}, {}),
    "map_888888": ({CMAP: 888888}, {}),
    "ring_112248": ({MATVEC: 1, CMAP: 112248}, {}),
    "ring_888888": ({MATVEC: 1, CMAP: 888888}, {}),
    "separate_cut": ({FUSED: 1}, {}),
    "separate_cut_888888": ({FUSED: 1, CMAP: 888888}, {}),
    "grid_path": ({}, {"lanczos_impl": 1}),
}
FIELDS = ("chunk", "level", "n", "n_side", "best_k", "split", "steps", "converged", "lambda2", "mcut")


def _api():
    from autoinst_b200 import api
    return api


def _lane(dev, options, lane):
    hd = _api().Handle.get(dev, lane)
    for opt in (MATVEC, CMAP, FUSED):
        hd.set_option(opt, options.get(opt, 0))
    return hd


@pytest.fixture(scope="module")
def reference():
    return {name: fixture_reference(name) for name in FIXTURES}


@pytest.fixture(scope="module")
def packed():
    api = _api()
    ch = [fixture_chunk(name) for name in FIXTURES]
    return api.PackedChunks([c[0] for c in ch], [c[1] for c in ch], None, theta=CFG["theta"])


def _run(dev, packed, name, lane):
    api = _api()
    options, kw = CONFIGS[name]
    hd = _lane(dev, options, lane)
    res = api.segment_packed(packed, device=dev, lane=lane, alpha=CFG["alpha"], theta=CFG["theta"], T=CFG["T"],
                             want_stats=True, **kw)
    return res, hd


def _sorted_records(st):
    order = np.lexsort(tuple(np.asarray(st[f]) for f in reversed(FIELDS)))
    return st[order]


def check_records(st, reference, chunks):
    """Device records of `chunks` (indices into FIXTURES, in call order) against node_tree; returns the largest
    |d lambda2| and |d mcut| / mcut."""
    worst_l, worst_m = 0.0, 0.0
    for ci, name in enumerate(chunks):
        recs = reference[name][1]
        dev = st[st["chunk"] == ci]
        assert len(dev) == len(recs), (name, len(dev), len(recs))
        groups = {}
        for r in recs:
            groups.setdefault((r["level"], r["n"]), []).append(r)
        for (level, n), rs in groups.items():
            d = dev[(dev["level"] == level) & (dev["n"] == n)]
            assert len(d) == len(rs), (name, level, n)
            d = d[np.lexsort((d["lambda2"], d["n_side"]))]
            rs = sorted(rs, key=lambda r: (r["n_side"], r["lambda2"]))
            for a, r in zip(d, rs):
                where = (name, level, n)
                assert (int(a["n_side"]), int(a["best_k"]), int(a["split"])) == (r["n_side"], r["best_k"], r["split"]), where
                dl = abs(float(a["lambda2"]) - r["lambda2"])
                assert dl <= (1e-12 if n <= 7 else 1e-9), (where, dl)
                worst_l = max(worst_l, dl)
                if r["best_k"] < 0:
                    assert np.isinf(a["mcut"]), where
                else:
                    dm = abs(float(a["mcut"]) - r["mcut"])
                    assert dm <= 1e-9 * r["mcut"] + r["mcut_floor"], (where, dm)
                    worst_m = max(worst_m, dm / r["mcut"])
                assert a["converged"] == 1 and 1 <= a["steps"] <= min(1024, n - 1), where
    return worst_l, worst_m


def test_device_affinity_is_the_rounded_reference(cuda_device, reference):
    """The reference trees are built on float32(affinity_ref): the device's W may differ from it only at rounding ties,
    by one ulp, at a handful of entries."""
    api = _api()
    for name in FIXTURES:
        points, tarl, _ = fixture_chunk(name)
        W = api.affinity(points, tarl, alpha=CFG["alpha"], theta=CFG["theta"], device=cuda_device).cpu().numpy()
        W32 = reference[name][0]
        diff = np.nonzero(W != W32)
        assert len(diff[0]) <= 8, (name, len(diff[0]))
        ulps = np.abs(W[diff].view(np.int32).astype(np.int64) - W32[diff].view(np.int32).astype(np.int64))
        assert np.all(ulps <= 1), name


@pytest.mark.parametrize("config", list(CONFIGS))
def test_node_records_match_the_dense_reference(cuda_device, reference, packed, config, record_property):
    """One configuration, two runs over the batch of all fixture chunks: records equal the reference's (size, side size,
    threshold, decision; lambda2 and the N-cut value to the eigensolver's tolerance), labels are its partition, and the
    second run is bit-identical to the first (labels and every record)."""
    lane = 40 + list(CONFIGS).index(config)
    res, _ = _run(cuda_device, packed, config, lane)
    assert res.unconverged == 0
    worst = check_records(res.stats, reference, FIXTURES)
    record_property("max_dlambda2_and_rel_dmcut", worst)
    print(f"{config}: max |d lambda2| = {worst[0]:.3e}, max |d mcut| / mcut = {worst[1]:.3e}")
    for name, lab in zip(FIXTURES, res.labels):
        assert R.same_partition(lab, reference[name][2]), name
    st = res.stats
    if config != "grid_path":
        slow = st[(st["chunk"] == FIXTURES.index("slow")) & (st["steps"] > CL_KMAX) & (st["n"] <= CL_NMAX)]
        assert len(slow) >= 1                      # the hand-off of the persistent kernel to the multi-launch path
    assert (st["n"] > CL_NMAX).any()
    again, _ = _run(cuda_device, packed, config, lane)
    for a, b in zip(res.labels, again.labels):
        assert np.array_equal(a, b)
    assert np.array_equal(_sorted_records(res.stats), _sorted_records(again.stats))


def test_caller_w_records_match_the_dense_reference(cuda_device, reference):
    """segment_dense on each chunk's float32 reference affinity (caller-provided w, hash start vector)."""
    api = _api()
    for name in FIXTURES:
        W32 = reference[name][0]
        lab, st = api.segment_dense(torch.as_tensor(W32, device=cuda_device), T=CFG["T"], want_stats=True)
        st = st.copy()
        st["chunk"] = 0
        check_records(st, {name: reference[name]}, [name])
        assert R.same_partition(lab, reference[name][2]), name


@pytest.mark.parametrize("cmap", ACCOUNTED_MAPS)
def test_dense_node_takes_the_matvec_form_its_slice_allows(cuda_device, reference, cmap):
    """The dense chunk alone under a cluster map: its 1000-point node does not fit shared memory at 2 CTAs (in-kernel
    dense matvec, k (4 n^2 + 8 n) bytes, separate cut kernels) and does at 8 (CSR slices, 4 n^2 bytes, fused cut).  The
    matvec byte count of the call is the sum of these over the nodes, as node_ref.slice_fits predicts them."""
    from oracle import node_ref as NR
    api = _api()
    points, tarl, _ = fixture_chunk("dense")
    pk = api.PackedChunks([points], [tarl], None, theta=CFG["theta"])
    lane = 60 + ACCOUNTED_MAPS.index(cmap)
    hd = _lane(cuda_device, {CMAP: cmap}, lane)
    res = api.segment_packed(pk, device=cuda_device, lane=lane, alpha=CFG["alpha"], theta=CFG["theta"], T=CFG["T"],
                             want_stats=True)
    acc = hd.accounting()
    recs = reference["dense"][1]
    check_records(res.stats, {"dense": reference["dense"]}, ["dense"])
    st = res.stats
    expect = 0.0
    fits = {}
    for r in recs:
        fits.setdefault(r["n"], set()).add(NR.slice_fits(r["entries"], ctas(cmap, r["n"])))
    for a in st:
        n, k = float(a["n"]), float(a["steps"])
        (fit,) = fits[int(a["n"])]
        expect += 4 * n * n if fit else k * (4 * n * n + 8 * n)
    assert acc["matvec"]["bytes"] == pytest.approx(expect, rel=1e-12)
    assert fits[1000] == {ctas(cmap, 1000) == 8}
