"""GPU tests of the segment path's affinity at the edges of the pair search and the feature pass (fixtures and their CPU
checks: tests/test_affinity_edges.py).

The segment path builds W with the cell-sorted pair search (or the shuffled sweep, ANCUTS_OPT_PAIR_SEARCH = 1) and the
deferred feature pass, and no stage entry exposes that W.  It is observed through the node records (`want_stats`): every
node of every fixture tree is clear, so its size, side size, threshold and decision have one correct value and lambda2 is
pinned to 1e-9 -- a missing, extra or wrong entry in a node's block moves them.  The stage entry (`api.affinity`) is
compared entry by entry with the float64 reference on the same fixtures, in both forms (impl 0 exact, impl 1 tensor core).
"""
import numpy as np
import pytest
import scipy.sparse as sp

from oracle import ncut_ref as R
from oracle.affinity_ref import affinity_ref
from test_affinity_edges import (CASES, GROUPS, TC_SCALES, _f32, fixture, inputs, proximity, reference, run_config)
from test_gpu_node_records import FIELDS, check_records

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

PAIRS = 1                                        # include/autoinst_ncuts.h: ANCUTS_OPT_PAIR_SEARCH (0 cell-sorted, 1 shuffled)
EUNSUPPORTED = -5


def _api():
    from autoinst_b200 import api
    return api


def _lane(dev, pairs):
    """A handle of its own per pair search."""
    lane = 70 + pairs
    _api().Handle.get(dev, lane).set_option(PAIRS, pairs)
    return lane


def _refs(names, config):
    """name -> (W32, records, labels), as check_records reads them."""
    return {f: reference(f, config)[1:] for f in names}


def _packed(names, config):
    api = _api()
    gains, _, _ = run_config(config)
    ins = [inputs(f, config) for f in names]
    return api.PackedChunks([x[0] for x in ins], [x[1] for x in ins] if gains["theta"] else None,
                            [x[2] for x in ins] if gains["gamma"] else None, theta=gains["theta"], gamma=gains["gamma"])


def _segment(dev, names, config, lane, resident, packed=None):
    """Labels (per chunk) and records of one segment call through host buffers or with resident inputs."""
    api = _api()
    gains, T, _ = run_config(config)
    packed = packed if packed is not None else _packed(names, config)
    kw = dict(T=T, proximity=proximity(names[0]), want_stats=True, lane=lane, **gains)
    if resident:
        dc = packed.to_device(dev)
        res = api.segment_packed(packed, dev_chunks=dc, **kw)
        lab = dc.labels.cpu().numpy()
        labels = [lab[a:b].copy() for a, b in zip(packed.off[:-1], packed.off[1:])]
    else:
        res = api.segment_packed(packed, device=dev, **kw)
        labels = res.labels
    assert res.unconverged == 0
    return labels, res.stats


def _sorted(st):
    return st[np.lexsort(tuple(np.asarray(st[f]) for f in reversed(FIELDS)))]


@pytest.mark.parametrize("pairs", [0, 1])
@pytest.mark.parametrize("group", list(GROUPS))
def test_segment_records_match_the_dense_reference(cuda_device, group, pairs, record_property):
    """Every fixture of a group in one call: records and labels equal the reference's, through host buffers and with
    resident inputs, and the two calls agree bit for bit (labels and every field of every record)."""
    config, names = GROUPS[group]
    lane = _lane(cuda_device, pairs)
    refs = _refs(names, config)
    out = [_segment(cuda_device, names, config, lane, resident) for resident in (False, True)]
    for labels, st in out:
        worst = check_records(st, refs, names)
        for name, lab in zip(names, labels):
            assert R.same_partition(lab, refs[name][2]), name
    record_property("max_dlambda2_and_rel_dmcut", worst)
    (lh, sh), (ld, sd) = out
    for a, b in zip(lh, ld):
        assert np.array_equal(a, b)
    assert np.array_equal(_sorted(sh), _sorted(sd))


def _ulp_diff(W, W32):
    diff = np.nonzero(W != W32)
    ulps = np.abs(W[diff].view(np.int32).astype(np.int64) - W32[diff].view(np.int32).astype(np.int64))
    return len(diff[0]), (int(ulps.max()) if len(ulps) else 0)


@pytest.mark.parametrize("name,config", CASES, ids=[f"{f}-{c}" for f, c in CASES])
def test_stage_affinity_is_the_rounded_reference(cuda_device, name, config):
    """impl 0: W equals float32(affinity_ref) but for one ulp at a handful of rounding ties (the rule of
    test_gpu_node_records.test_device_affinity_is_the_rounded_reference)."""
    api = _api()
    pts, tarl, dino = inputs(name, config)
    gains, _, _ = run_config(config)
    W = api.affinity(pts, tarl, dino, proximity=proximity(name), device=cuda_device, **gains).cpu().numpy()
    count, ulps = _ulp_diff(W, reference(name, config)[1])
    assert count <= 8 and ulps <= 1, (count, ulps)


def _tc_gate(W, A):
    """Level-1 gate of the tensor-core form: the reference's zero pattern, 1e-5 relative error; returns the worst error."""
    W = W.double().cpu().numpy()
    assert np.array_equal(W != 0, A != 0)
    return float((np.abs(W - A)[A != 0] / A[A != 0]).max())


TC_CASES = [(f, c) for f, c in CASES if c in ("tarl_spatial", "tarl_spatial_dino") and fixture(f)[1].shape[1] <= 96]


@pytest.mark.parametrize("name,config", TC_CASES, ids=[f"{f}-{c}" for f, c in TC_CASES])
def test_stage_affinity_tensor_core_form(cuda_device, name, config):
    """impl 1 (TARL Gram matrix on tcgen05, one DINOv2 camera): TARL widths below 96 and not multiples of 32 leave hi.hi
    slices unused and zero-pad the operands."""
    api = _api()
    pts, tarl, dino = inputs(name, config)
    gains, _, _ = run_config(config)
    W = api.affinity(pts, tarl, dino, proximity=proximity(name), impl=1, device=cuda_device, **gains)
    assert _tc_gate(W, reference(name, config)[0]) <= 1e-5


def test_tensor_core_error_over_the_feature_scale(cuda_device, record_property):
    """The 3 x TF32 dot products err relative to |f|^2, not to the distance; the pairs of the fixture's 0.1-noise object sit
    on both sides of the cancellation cutoff, where that error weighs most.  The gate holds at TARL scales 0.1 to 10."""
    api = _api()
    pts, tarl, _ = inputs("features", "tarl_spatial")
    worst = {}
    for s in TC_SCALES:
        t = _f32(tarl * s)
        A = affinity_ref(pts, t, None, alpha=1.0, theta=0.5)
        worst[s] = _tc_gate(api.affinity(pts, t, None, alpha=1.0, theta=0.5, impl=1, device=cuda_device), A)
    record_property("worst_rel_err_per_scale", worst)
    print("tensor-core form, worst relative error of W per TARL scale:", worst)
    assert max(worst.values()) <= 1e-5, worst


def test_batch_with_one_overflowing_chunk_falls_back_whole(cuda_device):
    """One chunk whose pair queue overflows (more than 96 pairs per point: the blob of test_pair_queue_overflow_falls_back)
    among chunks whose queues do not: the whole call takes the one-kernel form (input-order positions, a fresh forest).
    Every chunk's labels equal the oracle's and the fixtures' records the reference's, through host buffers and with
    resident inputs."""
    api = _api()
    config = "tarl_spatial"
    gains, T, _ = run_config(config)
    names = ["threshold", "n3", "isolated", "n129", "far"]
    rng = np.random.default_rng(5)
    n = 900
    blob = (rng.normal(size=(n, 3)) * 0.2).astype(np.float32).astype(np.float64)
    blob[n // 2:] += 7.0
    bt = rng.normal(size=(n, 96)).astype(np.float32).astype(np.float64)
    A = affinity_ref(blob, bt, None, **gains)
    assert (A != 0).sum() > 2 * 96 * n
    with R.pinned_eigsh():
        g = R.normalized_cut_ref(sp.csr_matrix(A), n, np.arange(n), T=T)
    blob_ref = R.labels_from_groups(g, n)
    ins = [inputs(f, config) for f in names]
    packed = api.PackedChunks([x[0] for x in ins] + [blob], [x[1] for x in ins] + [bt], None, theta=gains["theta"])
    refs = _refs(names, config)
    for resident in (False, True):
        labels, st = _segment(cuda_device, names, config, 0, resident, packed=packed)
        check_records(st[st["chunk"] < len(names)], refs, names)
        for name, lab in zip(names, labels):
            assert R.same_partition(lab, refs[name][2]), (name, resident)
        assert R.same_partition(labels[-1], blob_ref), resident


@pytest.mark.parametrize("pairs", [0, 1])
def test_batch_labels_equal_single_chunk_calls(cuda_device, pairs):
    """Chunks of 1, 2 and 3 points, the empty queue and the tile-edge sizes between two fixtures: every chunk's labels in
    the batch equal its own single-chunk call bit for bit."""
    config, names = GROUPS["batch_tarl_spatial"]
    lane = _lane(cuda_device, pairs)
    batch, _ = _segment(cuda_device, names, config, lane, False)
    for name, lab in zip(names, batch):
        one, st = _segment(cuda_device, [name], config, lane, False)
        assert np.array_equal(lab, one[0]), name
        check_records(st, _refs([name], config), [name])


def test_refusals_carry_their_message(cuda_device):
    """A feature width that is not a multiple of 4 (both segment entries and the stage entry); the tensor-core form with
    more than 96 TARL dimensions or two DINOv2 cameras."""
    api = _api()
    from autoinst_b200._lib import AncutsError
    pts, tarl, dino = inputs("n257", "tarl_spatial_dino2")
    gains, T, _ = run_config("tarl_spatial_dino2")
    t6 = tarl[:, :6]
    with pytest.raises(AncutsError, match="multiples of 4") as e:
        api.affinity(pts, t6, None, alpha=1.0, theta=0.5, device=cuda_device)
    assert e.value.code == EUNSUPPORTED
    packed = api.PackedChunks([pts], [t6], None, theta=0.5)
    for dc in (None, packed.to_device(cuda_device)):
        with pytest.raises(AncutsError, match="multiples of 4") as e:
            api.segment_packed(packed, device=cuda_device, dev_chunks=dc, alpha=1.0, theta=0.5, T=T)
        assert e.value.code == EUNSUPPORTED
    t128 = np.hstack([tarl, tarl[:, :32]])
    with pytest.raises(AncutsError, match="up to 96 TARL dimensions") as e:
        api.affinity(pts, t128, None, alpha=1.0, theta=0.5, impl=1, device=cuda_device)
    assert e.value.code == EUNSUPPORTED
    with pytest.raises(AncutsError, match="one DINOv2 camera") as e:
        api.affinity(pts, tarl, dino, impl=1, device=cuda_device, **gains)
    assert e.value.code == EUNSUPPORTED
