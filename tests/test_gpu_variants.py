"""GPU tests of the alternative implementations behind the same C ABI (ancuts_set_option): pair search, matvec forms,
the stage entry's two-pass affinity and the pair-queue overflow fallback; non-convergence reporting; the per-level trace."""
import numpy as np
import pytest
import scipy.sparse as sp

from autoinst_b200.synthetic import CONFIGS, make_chunk
from oracle import ncut_ref as R
from oracle.affinity_ref import affinity_ref

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


def _api():
    from autoinst_b200 import api
    return api


def variant_lane(dev, options, lane):
    """A library handle of its own (`lane`) with the given ancuts_set_option values."""
    api = _api()
    hd = api.Handle.get(dev, lane)
    for opt, val in options.items():
        hd.set_option(opt, val)
    return lane


def check_affinity(W, A):
    W = W.double().cpu().numpy()
    assert np.array_equal(W != 0, A != 0)
    rel = np.abs(W - A)[A != 0] / A[A != 0]
    assert rel.max() <= 1e-5, rel.max()              # north_star level 1
    assert np.array_equal(W, W.T)


# include/autoinst_ncuts.h: ANCUTS_OPT_PAIR_SEARCH 1 (0 cell-sorted sweep, 1 shuffled sweep), ANCUTS_OPT_MATVEC 2 (0 shared-
# memory slices, 1 dense from HBM), ANCUTS_OPT_CLUSTER_MAP 3 (CTAs per node and size bin), ANCUTS_OPT_FUSED_CUT 4 (0 cut
# decision inside the sparse-form eigensolver kernel, 1 its own kernels); option 0 is retired
PAIRS, MATVEC, CMAP, FUSED = 1, 2, 3, 4
VARIANTS = {"default": {}, "shuffled_pairs": {PAIRS: 1}, "dense_matvec": {MATVEC: 1},
            "dense_matvec_shuffled_pairs": {MATVEC: 1, PAIRS: 1},
            "sparse_matvec_few_ctas": {CMAP: 112248}, "dense_matvec_many_ctas": {MATVEC: 1, CMAP: 224888},
            "separate_cut_kernels": {FUSED: 1}, "separate_cut_few_ctas": {FUSED: 1, CMAP: 112248}}


def host_and_device_labels(api, packed, **kw):
    """segment_packed through host buffers (ancuts_segment_chunks_host, inputs arriving on its copy stream) and with the
    inputs resident on the device (ancuts_segment_chunks); the labels must be bit-identical.  Returns the host call."""
    res = api.segment_packed(packed, **kw)
    dev = packed.to_device(kw["device"])
    api.segment_packed(packed, dev_chunks=dev, **{k: v for k, v in kw.items() if k != "device"})
    labels = dev.labels.cpu().numpy()
    for c, lab in enumerate(res.labels):
        assert np.array_equal(lab, labels[packed.off[c]:packed.off[c + 1]]), c
    return res


@pytest.mark.parametrize("variant", list(VARIANTS))
def test_variants_give_oracle_labels(cuda_device, variant):
    api = _api()
    lane = variant_lane(cuda_device, VARIANTS[variant], 10 + list(VARIANTS).index(variant))
    cfg = CONFIGS["tarl_spatial"]
    chunks = [make_chunk(300 + i, n_target=1500 + 700 * i, features="tarl") for i in range(3)]
    packed = api.PackedChunks([c.points for c in chunks], [c.tarl for c in chunks], None, theta=cfg["theta"])
    res = host_and_device_labels(api, packed, device=cuda_device, lane=lane, alpha=cfg["alpha"], theta=cfg["theta"],
                                 T=cfg["T"], want_stats=True)
    assert int((res.stats["converged"] == 0).sum()) == 0 and res.unconverged == 0
    for ch, lab in zip(chunks, res.labels):
        A = affinity_ref(ch.points, ch.tarl, None, alpha=cfg["alpha"], theta=cfg["theta"])
        with R.pinned_eigsh():
            g = R.normalized_cut_ref(sp.csr_matrix(A), ch.n, np.arange(ch.n), T=cfg["T"])
        assert R.same_partition(lab, R.labels_from_groups(g, ch.n)), variant


def test_fused_cut_takes_the_decisions_of_the_cut_kernels(cuda_device):
    """The cut fused into the sparse-form eigensolver kernel (default) and the separate cut kernels decide every node of the
    tree alike: same labels, same node records (size, best threshold, split, side size), N-cut values equal to rounding
    (the bucket volumes are summed in another order; the cut weights are integer sums and equal)."""
    api = _api()
    cfg = CONFIGS["tarl_spatial"]
    chunks = [make_chunk(330 + i, n_target=2500 + 900 * i, features="tarl") for i in range(3)]
    packed = api.PackedChunks([c.points for c in chunks], [c.tarl for c in chunks], None, theta=cfg["theta"])
    kw = dict(device=cuda_device, alpha=cfg["alpha"], theta=cfg["theta"], T=cfg["T"], want_stats=True)
    fused = api.segment_packed(packed, lane=0, **kw)
    sep = api.segment_packed(packed, lane=variant_lane(cuda_device, {FUSED: 1}, 31), **kw)
    for a, b in zip(fused.labels, sep.labels):
        assert np.array_equal(a, b)

    def table(st):
        order = np.lexsort((st["n_side"], st["n"], st["level"], st["chunk"]))
        return {k: np.asarray(st[k])[order] for k in ("chunk", "level", "n", "n_side", "best_k", "split", "steps", "mcut")}
    tf, ts = table(fused.stats), table(sep.stats)
    assert len(tf["n"]) == len(ts["n"]) > 20
    for k in ("chunk", "level", "n", "n_side", "best_k", "split", "steps"):
        assert np.array_equal(tf[k], ts[k]), k
    fin = np.isfinite(ts["mcut"])
    assert np.array_equal(fin, np.isfinite(tf["mcut"]))
    assert np.allclose(tf["mcut"][fin], ts["mcut"][fin], rtol=1e-12, atol=0)


def test_non_convergence_is_never_silent(cuda_device):
    """Nodes that stop at lanczos_max_steps are counted by every segment call: the array level warns, `strict`
    (what the drop-in `ncuts` package passes) raises, as the reference's eigsh would (ADVICE round 1)."""
    api = _api()
    from autoinst_b200._lib import AncutsNoConvergence
    cfg = CONFIGS["tarl_spatial"]
    ch = make_chunk(310, n_target=1500, features="tarl")
    kw = dict(alpha=cfg["alpha"], theta=cfg["theta"], T=cfg["T"], device=cuda_device, max_steps=4)
    with pytest.warns(RuntimeWarning, match="without converging"):
        res = api.segment_chunks([ch.points], [ch.tarl], want_stats=True, **kw)
    assert res.unconverged > 0 and res.unconverged == int((res.stats["converged"] == 0).sum())
    with pytest.raises(AncutsNoConvergence):
        api.segment_chunk(ch.points, ch.tarl, strict=True, **kw)
    A = affinity_ref(ch.points, ch.tarl, None, alpha=cfg["alpha"], theta=cfg["theta"])
    import ncuts.normalized_cut as NC
    with pytest.raises(AncutsNoConvergence):
        api.segment_dense(torch.as_tensor(A, dtype=torch.float32, device=cuda_device), T=cfg["T"], max_steps=4, strict=True)
    assert len(NC.normalized_cut(sp.csr_matrix(A), ch.n, np.arange(ch.n), T=cfg["T"])) > 1      # default limit: converges
    res = api.segment_chunks([ch.points], [ch.tarl], alpha=cfg["alpha"], theta=cfg["theta"], T=cfg["T"], device=cuda_device)
    assert res.unconverged == 0


def test_cut_sums_do_not_overflow_on_heavy_weights(cuda_device):
    """Caller-provided w with weights far above 1: the fixed-point cut sums scale with the node's volume
    (2^-40 steps would overflow int64 beyond a cut weight of 2^23; ADVICE round 1)."""
    api = _api()
    rng = np.random.default_rng(3)
    n = 600
    w = np.zeros((n, n))
    half = n // 2
    for lo, hi in ((0, half), (half, n)):
        blk = rng.uniform(2e4, 6e4, size=(hi - lo, hi - lo))
        w[lo:hi, lo:hi] = (blk + blk.T) / 2
    link = rng.uniform(1.0, 2.0, size=(half, n - half)) * (rng.random((half, n - half)) < 0.02)
    w[:half, half:] = link
    w[half:, :half] = link.T
    np.fill_diagonal(w, 1.0)
    w = w.astype(np.float32).astype(np.float64)
    with R.pinned_eigsh():
        g = R.normalized_cut_ref(sp.csr_matrix(w), n, np.arange(n), T=0.01)
    ref = R.labels_from_groups(g, n)
    assert len(set(ref.tolist())) == 2
    got, stats = api.segment_dense(torch.as_tensor(w, dtype=torch.float32, device=cuda_device), T=0.01, want_stats=True)
    assert R.same_partition(got, ref)
    top = stats[stats["n"] == n][0]
    cut = w[:half, half:].sum()
    volA, volB = w[:half].sum() + half, w[half:].sum() + (n - half)
    assert abs(top["mcut"] - (cut / volA + cut / volB)) <= 1e-6 * top["mcut"]


@pytest.mark.parametrize("name", ["tarl_spatial", "tarl_spatial_dino"])
def test_two_pass_affinity_agrees_with_the_oracle(cuda_device, name):
    """The stage entry's two-pass form (pairs, then the feature pass on the dense matrix).  The dense forms of the segment
    path are no longer options: option 0 is retired and raises."""
    api = _api()
    cfg = CONFIGS[name]
    ch = make_chunk(41, n_target=2500, features="tarl_dino" if cfg["gamma"] else "tarl")
    A = affinity_ref(ch.points, ch.tarl, ch.dino if cfg["gamma"] else None, alpha=cfg["alpha"], theta=cfg["theta"], gamma=cfg["gamma"])
    W = api.affinity(ch.points, ch.tarl, ch.dino if cfg["gamma"] else None, alpha=cfg["alpha"], theta=cfg["theta"],
                     gamma=cfg["gamma"], device=cuda_device, lane=0)
    check_affinity(W, A)
    with pytest.raises(RuntimeError, match="option 0 is retired"):
        api.Handle.get(cuda_device, 0).set_option(0, 0)


def test_pair_queue_overflow_falls_back(cuda_device):
    """More than 96 in-mask pairs per point on average: the queue of the two-pass form overflows and the one-kernel
    form takes over, in the stage entry point (conditional launch) and in the segment call (host read-back), through host
    buffers and with resident inputs alike, with TARL terms and with TARL and DINO terms."""
    api = _api()
    rng = np.random.default_rng(5)
    n = 900
    pts = (rng.normal(size=(n, 3)) * 0.2).astype(np.float32).astype(np.float64)       # one 1 m blob: almost every pair inside
    pts[n // 2:] += 7.0                                                                  # ... and a second one far away
    tarl = rng.normal(size=(n, 96)).astype(np.float32)
    dino_rows = rng.normal(size=(n, 384)).astype(np.float32)
    for name in ("tarl_spatial", "tarl_spatial_dino"):
        cfg = CONFIGS[name]
        dino = dino_rows if cfg["gamma"] else None
        kw = dict(alpha=cfg["alpha"], theta=cfg["theta"], gamma=cfg["gamma"])
        A = affinity_ref(pts, tarl.astype(np.float64), None if dino is None else dino.astype(np.float64), **kw)
        assert (A != 0).sum() > 2 * 96 * n
        W = api.affinity(pts, tarl, dino, device=cuda_device, **kw)
        check_affinity(W, A)
        packed = api.PackedChunks([pts], [tarl], None if dino is None else [dino], theta=cfg["theta"], gamma=cfg["gamma"])
        lab = host_and_device_labels(api, packed, device=cuda_device, T=cfg["T"], **kw).labels[0]
        with R.pinned_eigsh():
            g = R.normalized_cut_ref(sp.csr_matrix(A), n, np.arange(n), T=cfg["T"])
        assert R.same_partition(lab, R.labels_from_groups(g, n)), name


def test_level_trace(cuda_device):
    api = _api()
    cfg = CONFIGS["tarl_spatial"]
    chunks = [make_chunk(500 + i, n_target=2000, features="tarl") for i in range(2)]
    packed = api.PackedChunks([c.points for c in chunks], [c.tarl for c in chunks], None, theta=cfg["theta"])
    devc = packed.to_device(cuda_device)
    hd = api.Handle.get(cuda_device)
    for dense in (1, 0):
        hd.set_option(MATVEC, dense)
        hd.set_stage_timing(2)
        try:
            res = api.segment_packed(packed, dev_chunks=devc, alpha=cfg["alpha"], theta=cfg["theta"], T=cfg["T"], want_stats=True)
            lv = hd.levels()
            acc = hd.accounting()
            sa = hd.sparse_accounting()
        finally:
            hd.set_stage_timing(0)
            hd.set_option(MATVEC, 0)
        assert len(lv) >= 1 and all(l["ms"] > 0 for l in lv)
        assert sum(sum(l["bins"]) + l["big"] for l in lv) == len(res.stats)
        assert abs(sum(l["ms"] for l in lv) - acc["matvec"]["ms"]) < 1e-3 * max(acc["matvec"]["ms"], 1.0) + 1e-3
        n = res.stats["n"].astype(np.float64)
        k = res.stats["steps"].astype(np.float64)
        if dense:      # algorithmic bytes of the dense form: every block once per Lanczos step (SURVEY.md §8d)
            assert acc["matvec"]["bytes"] == pytest.approx(float((k * (4 * n * n + 8 * n)).sum()), rel=1e-12)
            assert sa["entries"] == 0
        else:          # shared-memory form: every block read once, then steps x stored entries from shared memory
            assert acc["matvec"]["bytes"] == pytest.approx(float((4 * n * n).sum()), rel=1e-12)
            assert 3 * n.sum() <= sa["entries"] <= (n * n).sum() and sa["entry_steps"] >= sa["entries"]
