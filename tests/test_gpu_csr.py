"""GPU tests of the CSR front end (`api.segment_graphs`, C ABI `ancuts_segment_csr_f32`): caller-supplied sparse affinity
graphs cut by the device recursion.

  * every node record of the fixture chunks (tests/test_node_ref.py) against the dense float64 reference, under the ten
    configurations of tests/test_gpu_node_records.py;
  * bit-identity with `segment_dense` on the densified graph under a fixed cluster map: same edge set -> same root layout,
    same blocks, and the integer widening of the library's own range is exact, so the CSR call (w_own = 1) and the dense
    call (w_own = 0) run the same sums;
  * device tensors, weights outside the library's range, per-graph num_points_orig, degenerate graphs, malformed input,
    the benchmarked size and the `normalized_cut` drop-in.
"""
import os
import re

import numpy as np
import pytest
import scipy.sparse as sp

from conftest import CONFIG_NAMES, GOLDEN, GOLDEN_SEEDS, load_golden
from oracle import ncut_ref as R
from test_gpu_node_records import CONFIGS, _sorted_records, check_records
from test_node_ref import CFG, FIXTURES, fixture_reference

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

MATVEC, CMAP, FUSED = 2, 3, 4                   # include/autoinst_ncuts.h: ANCUTS_OPT_*
FIXED = {MATVEC: 1, CMAP: 112248}               # dense blocks from HBM, CTAs per node fixed: batching changes no sum


def _api():
    from autoinst_b200 import api
    return api


def _options(hd, options):
    for opt in (MATVEC, CMAP, FUSED):
        hd.set_option(opt, options.get(opt, 0))


@pytest.fixture(scope="module")
def reference():
    return {name: fixture_reference(name) for name in FIXTURES}


@pytest.fixture
def fixed_lane0(cuda_device):
    """Lane 0 (the handle segment_dense uses) with the fixed form; restored afterwards."""
    hd = _api().Handle.get(cuda_device, 0)
    _options(hd, FIXED)
    yield hd
    _options(hd, {})


def _csr(W):
    return sp.csr_matrix(np.asarray(W, dtype=np.float32))


def _run(dev, graphs, lane, options, lanczos_impl=0, norig=None):
    """One batched call with the given options; returns (labels, stats, handle)."""
    api = _api()
    hd = api.Handle.get(dev, lane)
    _options(hd, options)
    pk = api.pack_graphs(graphs).to(dev)
    p = api.make_params(T=CFG["T"], lanczos_impl=lanczos_impl)
    labels, _nseg, stats = api._run_graphs(hd, pk, norig, p, True, dev)
    assert hd.last_unconverged() == 0
    return labels, stats, hd


def _dense(dev, W, norig=None):
    lab, st = _api().segment_dense(torch.as_tensor(np.asarray(W, dtype=np.float32), device=dev), num_points_orig=norig,
                                   T=CFG["T"], want_stats=True)
    return lab, st


def _same_records(a, b):
    a, b = a.copy(), b.copy()
    a["chunk"] = 0
    b["chunk"] = 0
    return _sorted_records(a).tobytes() == _sorted_records(b).tobytes()


@pytest.mark.parametrize("config", list(CONFIGS))
def test_records_match_the_dense_reference(cuda_device, reference, config):
    """Every fixture's float32 reference affinity as scipy CSR, one batched call: records equal the reference tree, labels
    are its partition, a second run is bit-identical.  The fixtures' weights all lie in {0} U [2^-126, 2) (they are the
    library's own affinity), so the default configuration takes the shared-memory CSR slices."""
    options, kw = CONFIGS[config]
    lane = 80 + list(CONFIGS).index(config)
    graphs = [_csr(reference[name][0]) for name in FIXTURES]
    labels, st, hd = _run(cuda_device, graphs, lane, options, **kw)
    check_records(st, reference, FIXTURES)
    for name, lab in zip(FIXTURES, labels):
        assert R.same_partition(lab, reference[name][2]), name
    if config == "default":
        assert hd.sparse_accounting()["entries"] > 0
    again, st2, _ = _run(cuda_device, graphs, lane, options, **kw)
    for a, b in zip(labels, again):
        assert np.array_equal(a, b)
    assert _sorted_records(st).tobytes() == _sorted_records(st2).tobytes()
    _options(hd, {})


def test_bit_identical_to_segment_dense(cuda_device, reference, fixed_lane0):
    labels, st, _ = _run(cuda_device, [_csr(reference[n][0]) for n in FIXTURES], 0, FIXED)
    for c, name in enumerate(FIXTURES):
        lab, dst = _dense(cuda_device, reference[name][0])
        assert np.array_equal(labels[c], lab), name
        assert _same_records(st[st["chunk"] == c], dst), name


def test_device_tensors_equal_scipy_input(cuda_device, reference):
    names = FIXTURES[:4]
    a, sa, _ = _run(cuda_device, [_csr(reference[n][0]) for n in names], 90, {})
    t = [torch.as_tensor(reference[n][0], device=cuda_device).to_sparse_csr() for n in names]
    b, sb, _ = _run(cuda_device, t, 90, {})
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    assert _sorted_records(sa).tobytes() == _sorted_records(sb).tobytes()
    res = _api().segment_graphs(t, T=CFG["T"], device=cuda_device, lane=90)
    for x, y in zip(a, res.labels):
        assert np.array_equal(x, y)


@pytest.mark.parametrize("value", [2.5, 1e-40], ids=["above_2", "denormal"])
def test_weights_outside_the_range_take_the_dense_form(cuda_device, reference, fixed_lane0, value):
    W = reference["tiny"][0].copy()
    i, j = [(i, j) for i, j in zip(*np.nonzero(W)) if i < j][7]
    W[i, j] = W[j, i] = np.float32(value)
    _options(fixed_lane0, {CMAP: 112248})           # default matvec form: the range alone must switch the slices off
    lab, st = _run(cuda_device, [_csr(W)], 0, {CMAP: 112248})[:2]
    assert fixed_lane0.sparse_accounting()["entries"] == 0
    dlab, dst = _dense(cuda_device, W)
    assert np.array_equal(lab[0], dlab)
    assert _same_records(st, dst)


def test_per_graph_num_points_orig(cuda_device, fixed_lane0):
    subs, norig = [], []
    for seed, name in zip(GOLDEN_SEEDS[:2], CONFIG_NAMES[:2]):
        _, out, A = load_golden(seed, name)
        idx = np.where(out["labels"] == 0)[0]
        subs.append(A[idx][:, idx])
        norig.append(A.shape[0])
    res = _api().segment_graphs(subs, num_points_orig=norig, T=CFG["T"], device=cuda_device)
    for s, no, lab in zip(subs, norig, res.labels):
        dlab = _api().segment_dense(torch.as_tensor(s.toarray().astype(np.float32), device=cuda_device), num_points_orig=no,
                                    T=CFG["T"])
        assert np.array_equal(lab, dlab)


def test_degenerate_graphs(cuda_device, reference, fixed_lane0):
    api = _api()
    eye = sp.identity(50, dtype=np.float32, format="csr")
    W = reference["tiny"][0].copy()
    iso = [3, 100, 249]
    W[iso, :] = 0
    W[:, iso] = 0
    W[iso, iso] = 1
    three = np.ones((3, 3), dtype=np.float32) * 0.5 + np.eye(3, dtype=np.float32) * 0.5
    mats = [eye.toarray(), W, three, reference["bins_c"][0], reference["dense"][0]]
    res = api.segment_graphs([sp.csr_matrix(m) for m in mats], T=CFG["T"], device=cuda_device)
    assert res.num_segments[0] == 50 and sorted(res.labels[0].tolist()) == list(range(50))
    for m, lab in zip(mats, res.labels):
        assert np.array_equal(lab, api.segment_dense(torch.as_tensor(m, device=cuda_device), T=CFG["T"]))
    assert len({int(res.labels[1][k]) for k in iso}) == 3


def _broken(kind, W):
    """(row_ptr, col, val, nnz) of the batch [3-point graph, W] with one rule of graph 1 broken."""
    api = _api()
    pk = api.pack_graphs([sp.csr_matrix(np.eye(3, dtype=np.float32)), sp.csr_matrix(W)])
    rp, col, val = pk.row_ptr.numpy().copy(), pk.col.numpy().copy(), pk.val.numpy().copy()
    nnz = len(col)
    r = 3 + 10                                       # row 10 of graph 1
    a, b = rp[r], rp[r + 1]
    off = [q for q in range(a, b) if col[q] != 10]
    if kind == "asymmetric":
        val[off[0]] = np.nextafter(val[off[0]], np.float32(1))
    elif kind == "missing_mirror":
        keep = np.ones(nnz, dtype=bool)
        keep[off[0]] = False
        col, val = col[keep], val[keep]
        rp[r + 1:] -= 1
        nnz -= 1
    elif kind == "unsorted":
        col[off[0]], col[off[1]] = col[off[1]], col[off[0]]
        val[off[0]], val[off[1]] = val[off[1]], val[off[0]]
    elif kind == "duplicate":
        col[a + 1] = col[a]
    elif kind == "column_high":
        col[b - 1] = W.shape[0]
    elif kind == "column_negative":
        col[a] = -1
    elif kind == "row_ptr_decreasing":
        rp[r + 1] = rp[r] - 1
    elif kind == "row_ptr_end":
        rp[-1] = nnz - 1
    else:
        q = [q for q in range(a, b) if col[q] == 10][0]
        val[q if kind == "diagonal" else off[0]] = {"diagonal": 0.5, "nan": np.nan, "inf": np.inf}[kind]
    return rp, col, val, nnz


@pytest.mark.parametrize("kind", ["asymmetric", "missing_mirror", "unsorted", "duplicate", "column_high", "column_negative",
                                  "row_ptr_decreasing", "row_ptr_end", "diagonal", "nan", "inf"])
def test_malformed_input_is_rejected(cuda_device, reference, kind):
    from autoinst_b200._lib import EINVAL, AncutsError
    api = _api()
    W = reference["tiny"][0]
    good = [sp.csr_matrix(np.eye(3, dtype=np.float32)), sp.csr_matrix(W)]
    before = api.segment_graphs(good, T=CFG["T"], device=cuda_device, lane=91).labels
    rp, col, val, nnz = _broken(kind, W)
    pk = api.PackedGraphs([3, W.shape[0]], np.array([0, 3, 3 + W.shape[0]], dtype=np.int64), torch.as_tensor(rp),
                          torch.as_tensor(col), torch.as_tensor(val)).to(cuda_device)
    hd = api.Handle.get(cuda_device, 91)
    with pytest.raises(AncutsError) as ex:
        api._run_graphs(hd, pk, None, api.make_params(T=CFG["T"]), False, cuda_device)
    assert ex.value.code == EINVAL
    m = re.search(r"graph (\d+), row (\d+)", str(ex.value))
    assert m and m.group(1) == "1", str(ex.value)
    after = api.segment_graphs(good, T=CFG["T"], device=cuda_device, lane=91).labels
    for x, y in zip(before, after):
        assert np.array_equal(x, y)


def test_bench_size_chunks_from_device_affinities(cuda_device):
    from autoinst_b200.synthetic import CONFIGS as SYN, make_chunk
    from oracle.make_parity_fixtures import SETS, tag
    api = _api()
    fix = np.load(os.path.join(GOLDEN, "parity_bench_size.npz"))
    for name, n_target, seed0, count, clutter in [s for s in SETS if s[1] == 8192 and s[4] == 0]:
        cfg = SYN[name]
        feats = "tarl_dino" if cfg["gamma"] else "tarl"
        seeds = list(range(seed0, seed0 + count))
        graphs, chunks = [], []
        for s in seeds:
            ch = make_chunk(s, n_target=n_target, features=feats, clutter=clutter)
            W = api.affinity(ch.points, ch.tarl if cfg["theta"] else None, ch.dino if cfg["gamma"] else None,
                             alpha=cfg["alpha"], theta=cfg["theta"], gamma=cfg["gamma"], device=cuda_device)
            graphs.append(W.contiguous().to_sparse_csr())
            chunks.append(ch)
            del W
        res = api.segment_graphs(graphs, T=cfg["T"], device=cuda_device, want_stats=True, lane=92)
        assert res.unconverged == 0 and int((res.stats["converged"] == 0).sum()) == 0
        for s, lab in zip(seeds, res.labels):
            t = tag(name, n_target, s, clutter)
            if bool(fix["stable_" + t]):
                assert R.same_partition(lab, fix["labels_" + t].astype(np.int32)), (name, s)


def test_normalized_cut_takes_the_csr_path(cuda_device, monkeypatch):
    from autoinst_b200 import api
    from ncuts.normalized_cut import normalized_cut
    seed, name = GOLDEN_SEEDS[0], CONFIG_NAMES[1]
    _, out, A = load_golden(seed, name)
    n = A.shape[0]
    T = float(out["T"])
    dense_groups = normalized_cut(A.toarray(), n, np.arange(n), T=T)

    def no_dense(*a, **k):
        raise AssertionError("segment_dense called for scipy input")
    monkeypatch.setattr(api, "segment_dense", no_dense)
    groups = normalized_cut(A, n, np.arange(n), T=T)
    assert R.same_partition(R.labels_from_groups(groups, n), out["labels"])
    assert R.same_partition(R.labels_from_groups(groups, n), R.labels_from_groups(dense_groups, n))
    bad = A.tolil()
    bad[0, 0] = 0.5
    with pytest.raises(ValueError, match=r"graph 0, row 0"):
        normalized_cut(bad.tocsr(), n, np.arange(n), T=T)
