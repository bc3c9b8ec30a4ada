"""GPU parity tests of the whole path (labels), through the C ABI, against the pinned oracle."""
import numpy as np
import pytest
import scipy.sparse as sp

from conftest import CONFIG_NAMES, GOLDEN, GOLDEN_SEEDS, load_golden
from autoinst_b200.synthetic import CONFIGS, make_chunk
from oracle import ncut_ref as R
from oracle.affinity_ref import affinity_ref

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


def _api():
    from autoinst_b200 import api
    return api


def oracle_labels(ch, cfg, v0="ones", seed=0):
    A = affinity_ref(ch.points, ch.tarl, ch.dino, alpha=cfg["alpha"], theta=cfg["theta"], gamma=cfg["gamma"])
    with R.pinned_eigsh(v0, seed):
        g = R.normalized_cut_ref(sp.csr_matrix(A), ch.n, np.arange(ch.n), T=cfg["T"], split_lim=0.01)
    return R.labels_from_groups(g, ch.n)


@pytest.mark.parametrize("seed", GOLDEN_SEEDS)
@pytest.mark.parametrize("name", CONFIG_NAMES)
def test_labels_match_reference_golden(cuda_device, seed, name):
    inp, out, A = load_golden(seed, name)
    lab = _api().segment_chunk(inp["points"], inp["tarl"], inp["dino"], alpha=float(out["alpha"]),
                               theta=float(out["theta"]), gamma=float(out["gamma"]), T=float(out["T"]),
                               device=cuda_device)
    assert lab.dtype == np.int32 and lab.min() == 0 and lab.max() + 1 == len(out["group_sizes"])
    assert R.same_partition(lab, out["labels"])


def test_known_answers_dense(cuda_device):
    kat = np.load(f"{GOLDEN}/known_answers.npz")
    for nm in sorted({k[:-2] for k in kat.files if k.endswith("_w")}):
        w, lab = kat[nm + "_w"], kat[nm + "_labels"]
        T = float(nm.split("_T")[1])
        got = _api().segment_dense(torch.as_tensor(w, dtype=torch.float32, device=cuda_device), T=T)
        if nm.startswith("one_clique"):
            assert len(set(got.tolist())) == 1
        else:
            assert R.same_partition(got, lab), (nm, got, lab)


@pytest.mark.parametrize("name", CONFIG_NAMES)
def test_labels_match_oracle_batched(cuda_device, name):
    """A batch of seeded chunks in one call: every oracle-stable chunk must match (north_star level 2)."""
    cfg = CONFIGS[name]
    feats = "tarl_dino" if cfg["gamma"] else "tarl"
    chunks = [make_chunk(100 + i, n_target=1200 + 300 * i, features=feats) for i in range(4)]
    res = _api().segment_chunks([c.points for c in chunks], [c.tarl for c in chunks],
                                [c.dino for c in chunks] if cfg["gamma"] else None,
                                alpha=cfg["alpha"], theta=cfg["theta"], gamma=cfg["gamma"], T=cfg["T"],
                                device=cuda_device, want_stats=True)
    assert res.stats is not None and len(res.stats) > 0 and res.stats["converged"].all()
    stable = matched = 0
    for ch, lab, ns in zip(chunks, res.labels, res.num_segments):
        assert lab.shape == (ch.n,) and lab.min() == 0 and lab.max() + 1 == ns
        ref = oracle_labels(ch, cfg)
        if not R.same_partition(ref, oracle_labels(ch, cfg, "random", 5)):
            continue                                                  # oracle-unstable chunk (SURVEY §7.3)
        stable += 1
        matched += R.same_partition(lab, ref)
    assert stable >= 3 and matched == stable


def test_multi_launch_path_gives_the_same_labels(cuda_device):
    """lanczos_impl=1 (grid-wide kernels for every node) against the default persistent cluster kernels."""
    cfg = CONFIGS["tarl_spatial"]
    from autoinst_b200 import api
    chunks = [make_chunk(400 + i, n_target=1500, features="tarl") for i in range(2)]
    pk = api.PackedChunks([c.points for c in chunks], [c.tarl for c in chunks], theta=cfg["theta"], pin=False)
    kw = dict(alpha=cfg["alpha"], theta=cfg["theta"], T=cfg["T"], device=cuda_device, want_stats=True)
    a = api.segment_packed(pk, lanczos_impl=0, **kw)
    b = api.segment_packed(pk, lanczos_impl=1, **kw)
    for la, lb in zip(a.labels, b.labels):
        assert R.same_partition(la, lb)
    assert a.stats["converged"].all() and b.stats["converged"].all()


def test_tensor_core_affinity_gives_the_same_labels(cuda_device):
    cfg = CONFIGS["tarl_spatial"]
    from autoinst_b200 import api
    chunks = [make_chunk(500 + i, n_target=1500, features="tarl") for i in range(2)]
    pk = api.PackedChunks([c.points for c in chunks], [c.tarl for c in chunks], theta=cfg["theta"], pin=False)
    kw = dict(alpha=cfg["alpha"], theta=cfg["theta"], T=cfg["T"], device=cuda_device)
    a = api.segment_packed(pk, affinity_impl=0, **kw)
    b = api.segment_packed(pk, affinity_impl=1, **kw)
    for la, lb in zip(a.labels, b.labels):
        assert R.same_partition(la, lb)
    # resident inputs give the labels of the host entry, whose features arrive chunk by chunk, bit for bit
    dev = pk.to_device(cuda_device)
    api.segment_packed(pk, affinity_impl=1, dev_chunks=dev, **{k: v for k, v in kw.items() if k != "device"})
    dl = dev.labels.cpu().numpy()
    for c, lb in enumerate(b.labels):
        assert np.array_equal(lb, dl[pk.off[c]:pk.off[c + 1]])


def test_batched_equals_single(cuda_device):
    cfg = CONFIGS["tarl_spatial"]
    chunks = [make_chunk(200 + i, n_target=900 + 200 * i, features="tarl") for i in range(3)]
    kw = dict(alpha=cfg["alpha"], theta=cfg["theta"], T=cfg["T"], device=cuda_device)
    res = _api().segment_chunks([c.points for c in chunks], [c.tarl for c in chunks], **kw)
    for ch, lab in zip(chunks, res.labels):
        single = _api().segment_chunk(ch.points, ch.tarl, **kw)
        assert R.same_partition(lab, single)
        assert np.array_equal(lab, single)                            # deterministic label numbering too


def test_edge_cases(cuda_device):
    api = _api()
    # n <= 2 and T <= 0: one segment (normalized_cut.py:39-40,56)
    assert api.segment_chunk(np.zeros((1, 3)), alpha=1.0, T=0.075, device=cuda_device).tolist() == [0]
    assert api.segment_chunk(np.array([[0, 0, 0], [5.0, 0, 0]]), alpha=1.0, T=0.075, device=cuda_device).tolist() == [0, 0]
    ch = make_chunk(300, n_target=800, features="tarl")
    assert set(api.segment_chunk(ch.points, alpha=1.0, T=0.0, device=cuda_device).tolist()) == {0}
    # cluttered chunk: tiny fragments; the oracle itself is order-dependent there, so only sanity is checked
    chc = make_chunk(301, n_target=1000, features="tarl", clutter=20)
    lab = api.segment_chunk(chc.points, chc.tarl, alpha=1.0, theta=0.5, T=0.03, device=cuda_device)
    assert lab.shape == (chc.n,) and lab.min() == 0 and len(set(lab.tolist())) == lab.max() + 1
    with pytest.raises(NotImplementedError):
        api.make_params(beta=0.5)


def test_map_level_metrics_match_oracle(cuda_device):
    """north_star level 3: AP, P/R/F1, S_assoc from GPU labels vs oracle labels, both through the same merge
    (oracle.merge_ref) and the same metrics (oracle.metrics_ref, pinned to the reference's Metrics class)."""
    from autoinst_b200.synthetic import make_map
    from oracle import merge_ref as M
    from oracle.metrics_ref import instance_metrics
    cfg = CONFIGS["tarl_spatial"]
    chunks = make_map(5, 2000, seed=9)
    res = _api().segment_chunks([c.points for c in chunks], [c.tarl for c in chunks], alpha=cfg["alpha"],
                                theta=cfg["theta"], T=cfg["T"], device=cuda_device)
    gt_pts, gt_lab = M.merge_unite_gt([(c.points, c.instance) for c in chunks])
    gt = M.compact_labels(gt_lab)

    def evaluate(per_chunk_labels):
        parts = [(c.points, M.globally_unique(c.chunk_id, M.canonical_labels(lab))) for c, lab in zip(chunks, per_chunk_labels)]
        pts, lab = M.merge_chunks_unite_instances(parts)
        assert np.array_equal(pts, gt_pts)
        allp = M.compact_labels(lab)
        inst = M.remove_semantics(gt, allp.copy())
        return instance_metrics(allp, inst, gt, min_points=20)      # major-level evaluation (SURVEY Appendix A item 10)

    got = evaluate(res.labels)
    ref = evaluate([oracle_labels(c, cfg) for c in chunks])
    for k in ("p", "r", "f1", "ap", "ap0.25", "ap0.5", "S_assoc"):
        assert abs(got[k] - ref[k]) <= 1e-3, (k, got[k], ref[k])    # 0.1 points
    assert ref["S_assoc"] > 0.3 and ref["ap0.25"] > 0.2              # the comparison is not vacuous


def test_segment_stream_equals_single_calls(cuda_device):
    """api.segment_stream (upload of batch k+1 overlaps the cut of batch k, two alternating sets of device input buffers)
    returns, batch by batch, the labels of the synchronous host call -- batches of different sizes and feature sets of
    one config, so that the slots are re-used with other shapes."""
    api = _api()
    cfg = CONFIGS["tarl_spatial"]
    kw = dict(alpha=cfg["alpha"], theta=cfg["theta"], gamma=cfg["gamma"], T=cfg["T"])
    batches = []
    for b, (count, n) in enumerate([(3, 1400), (1, 2600), (4, 900), (2, 2000), (1, 700)]):
        chunks = [make_chunk(900 + 10 * b + i, n_target=n, features="tarl") for i in range(count)]
        batches.append(api.PackedChunks([c.points for c in chunks], [c.tarl for c in chunks], None, theta=cfg["theta"]))
    want = [[l.copy() for l in api.segment_packed(pk, device=cuda_device, **kw).labels] for pk in batches]
    got = list(api.segment_stream(batches, device=cuda_device, **kw))
    assert len(got) == len(batches)
    for res, ref, pk in zip(got, want, batches):
        assert len(res.labels) == len(pk.sizes)
        for a, b in zip(res.labels, ref):
            assert np.array_equal(a, b)
    # the explicit form: never more than two batches in flight
    ss = api.SegmentStream(device=cuda_device, **kw)
    ss.submit(batches[0]); ss.submit(batches[1])
    with pytest.raises(RuntimeError):
        ss.submit(batches[2])
    assert np.array_equal(ss.result().labels[0], want[0][0])
    assert np.array_equal(ss.result().labels[0], want[1][0])
    with pytest.raises(RuntimeError):
        ss.result()
