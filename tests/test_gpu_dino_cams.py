"""GPU tests of the DINOv2 term over several cameras (the reference's CAM_IDS product, ncuts_utils.py:125-133): the stage
entry and its overflow fallback against the oracle, the exact identity "two identical cameras at gamma = one camera at
2 gamma" through every entry, the _cams entry points at one camera against the old ones, oracle labels, the drop-in, and
the argument checks."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp

from autoinst_b200.synthetic import CONFIGS, make_chunk
from oracle import ncut_ref as R
from oracle.affinity_ref import affinity_ref

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

CFG = CONFIGS["tarl_spatial_dino"]
KW = dict(alpha=CFG["alpha"], theta=CFG["theta"], gamma=CFG["gamma"])


def _api():
    from autoinst_b200 import api
    return api


def check_affinity(W, A):
    W = W.double().cpu().numpy()
    assert np.array_equal(W != 0, A != 0)
    rel = np.abs(W - A)[A != 0] / A[A != 0]
    assert rel.max() <= 1e-5, rel.max()
    assert np.array_equal(W, W.T)


def three_cameras(ch, seed=9):
    """The two synthetic cameras of a "tarl_dino2" chunk and a third: camera 1 with its own noise and unseen rows."""
    rng = np.random.default_rng(seed)
    g0, g1 = ch.dino
    g2 = (g1 + 0.3 * rng.normal(size=g1.shape)).astype(np.float32)
    g2[rng.random(ch.n) < 0.3] = 0.0
    return [g0, g1, g2.astype(np.float64)]


def overflow_inputs():
    """One dense 1 m blob (almost every pair in the mask) and a second one far away: more than 96 in-mask pairs per point,
    so the pair queue overflows and the one-kernel form takes over (as in test_pair_queue_overflow_falls_back)."""
    rng = np.random.default_rng(5)
    n = 900
    pts = (rng.normal(size=(n, 3)) * 0.2).astype(np.float32).astype(np.float64)
    pts[n // 2:] += 7.0
    tarl = rng.normal(size=(n, 96)).astype(np.float32)
    dino = rng.normal(size=(n, 384)).astype(np.float32)
    return pts, tarl, dino


@pytest.mark.parametrize("cams", [2, 3])
def test_stage_affinity_matches_the_oracle(cuda_device, cams):
    api = _api()
    ch = make_chunk(41, n_target=2500, features="tarl_dino2")
    assert ch.n % 64 != 0
    dino = three_cameras(ch)[:cams]
    # hand rows: point 0's neighbours -- one unseen by camera 1 only, one with point 0's rows in every camera
    d0 = np.linalg.norm(ch.points - ch.points[0], axis=1)
    nb = np.flatnonzero((d0 > 0) & (d0 <= 0.9))
    assert len(nb) >= 2
    dino = [g.copy() for g in dino]
    if not dino[0][nb[0]].any():
        dino[0][nb[0]] = 1.0
    dino[1][nb[0]] = 0.0
    for g in dino:
        g[nb[1]] = g[0]
    A = affinity_ref(ch.points, ch.tarl, dino, **KW)
    W = api.affinity(ch.points, ch.tarl, dino, device=cuda_device, **KW)
    check_affinity(W, A)
    # the (n, cams, D) form is the same input
    W3 = api.affinity(ch.points, ch.tarl, np.stack(dino, axis=1), device=cuda_device, **KW)
    assert torch.equal(W, W3)
    # identical rows in every camera: only the spatial and TARL terms remain
    only_st = affinity_ref(ch.points, ch.tarl, None, alpha=KW["alpha"], theta=KW["theta"])
    assert abs(float(W[0, nb[1]]) - only_st[0, nb[1]]) <= 1e-5 * only_st[0, nb[1]]


def test_overflow_fallback_matches_the_oracle(cuda_device):
    api = _api()
    pts, tarl, dino = overflow_inputs()
    rng = np.random.default_rng(6)
    cams = [dino, (dino + 0.5 * rng.normal(size=dino.shape)).astype(np.float32)]
    A = affinity_ref(pts, tarl.astype(np.float64), [c.astype(np.float64) for c in cams], **KW)
    assert (A != 0).sum() > 2 * 96 * len(pts)
    check_affinity(api.affinity(pts, tarl, cams, device=cuda_device, **KW), A)


def segment_all_entries(api, packed, device, **kw):
    """Labels of the host entry, the device entry and segment_stream for one packed batch (concatenated)."""
    host = np.concatenate(api.segment_packed(packed, device=device, **kw).labels)
    dev = packed.to_device(device)
    api.segment_packed(packed, dev_chunks=dev, **kw)
    stream = np.concatenate(next(iter(api.segment_stream([packed], device=device, **kw))).labels)
    return host, dev.labels.cpu().numpy(), stream


def test_two_identical_cameras_equal_one_camera_at_twice_gamma(cuda_device):
    """S = dd + dd = 2 dd exactly, so gamma * S = (2 gamma) * dd: W and labels are bit-identical."""
    api = _api()
    two_g = dict(KW, gamma=2 * KW["gamma"])
    ch = make_chunk(43, n_target=2500, features="tarl_dino")
    g = ch.dino
    W2 = api.affinity(ch.points, ch.tarl, [g, g], device=cuda_device, **KW)
    W1 = api.affinity(ch.points, ch.tarl, g, device=cuda_device, **two_g)
    assert torch.equal(W1, W2)
    pts, tarl, dino = overflow_inputs()                                  # the one-kernel fallback of the stage entry
    assert torch.equal(api.affinity(pts, tarl, [dino, dino], device=cuda_device, **KW),
                       api.affinity(pts, tarl, dino, device=cuda_device, **two_g))
    chunks = [make_chunk(44 + i, n_target=1500 + 400 * i, features="tarl_dino") for i in range(3)]
    batches = [([c.points for c in chunks], [c.tarl for c in chunks], [c.dino for c in chunks]),
               ([pts], [tarl], [dino])]                                  # the segment call's overflow fallback
    for P, T_, D in batches:
        seg = dict(T=CFG["T"], alpha=KW["alpha"], theta=KW["theta"])
        one = api.PackedChunks(P, T_, D, theta=KW["theta"], gamma=1.0)
        two = api.PackedChunks(P, T_, [[d, d] for d in D], theta=KW["theta"], gamma=1.0)
        assert two.dino_cams == 2 and one.dino_cams == 1
        a = segment_all_entries(api, one, cuda_device, gamma=two_g["gamma"], **seg)
        b = segment_all_entries(api, two, cuda_device, gamma=KW["gamma"], **seg)
        for x in a + b:
            assert np.array_equal(x, a[0])


def _raw_affinity(api, dev, ch, cams_entry):
    hd = api.Handle.get(dev)
    pts = torch.as_tensor(ch.points, device=dev)
    t = torch.as_tensor(ch.tarl, dtype=torch.float32, device=dev)
    g = torch.as_tensor(ch.dino, dtype=torch.float32, device=dev)
    p = api.make_params(T=0.0, tarl_dim=96, dino_dim=384, **KW)
    buf, view = api.alloc_matrix(ch.n, dev)
    args = (hd.h, ch.n, api._ptr(pts), api._ptr(t), api._ptr(g))
    tail = (C.byref(p), api._ptr(buf), buf.stride(0), None, api._stream(dev))
    rc = hd.lib.ancuts_affinity_cams_f32(*args, 1, *tail) if cams_entry else hd.lib.ancuts_affinity_f32(*args, *tail)
    assert rc == 0
    return view.clone()


def _raw_segment(api, dev, packed, cams_entry, host):
    hd = api.Handle.get(dev)
    p = api.make_params(T=CFG["T"], tarl_dim=packed.tarl_dim, dino_dim=packed.dino_dim, **KW)
    off = np.ascontiguousarray(packed.off, dtype=np.int64)
    nseg = np.zeros(len(packed.sizes), dtype=np.int32)
    nst = C.c_int32(0)
    pi64, pi32 = off.ctypes.data_as(C.POINTER(C.c_int64)), nseg.ctypes.data_as(C.POINTER(C.c_int32))
    src = packed if host else packed.to_device(dev)
    head = (hd.h, len(packed.sizes), pi64, api._ptr(src.points), api._ptr(src.tarl), api._ptr(src.dino))
    tail = (C.byref(p), api._ptr(src.labels), pi32, None, 0, C.byref(nst), api._stream(dev))
    if host:
        rc = hd.lib.ancuts_segment_chunks_cams_host(*head, 1, *tail) if cams_entry else hd.lib.ancuts_segment_chunks_host(*head, *tail)
    else:
        rc = hd.lib.ancuts_segment_chunks_cams(*head, 1, *tail) if cams_entry else hd.lib.ancuts_segment_chunks(*head, *tail)
    assert rc == 0
    torch.cuda.synchronize(dev)
    return src.labels.cpu().numpy().copy()


def test_one_camera_through_the_new_entry_points_is_unchanged(cuda_device):
    api = _api()
    ch = make_chunk(45, n_target=2500, features="tarl_dino")
    assert torch.equal(_raw_affinity(api, cuda_device, ch, False), _raw_affinity(api, cuda_device, ch, True))
    chunks = [make_chunk(46 + i, n_target=1500 + 300 * i, features="tarl_dino") for i in range(3)]
    packed = api.PackedChunks([c.points for c in chunks], [c.tarl for c in chunks], [c.dino for c in chunks],
                              theta=KW["theta"], gamma=KW["gamma"])
    for host in (True, False):
        assert np.array_equal(_raw_segment(api, cuda_device, packed, False, host),
                              _raw_segment(api, cuda_device, packed, True, host))


def oracle_labels(ch, v0="ones", seed=0):
    A = affinity_ref(ch.points, ch.tarl, ch.dino, **KW)
    with R.pinned_eigsh(v0, seed):
        g = R.normalized_cut_ref(sp.csr_matrix(A), ch.n, np.arange(ch.n), T=CFG["T"], split_lim=0.01)
    return R.labels_from_groups(g, ch.n)


def test_two_camera_batch_gives_the_oracle_labels(cuda_device):
    """Every oracle-stable chunk of a two-camera batch matches (the rule of test_labels_match_oracle_batched); the host entry
    and the device entry give bit-identical labels."""
    api = _api()
    chunks = [make_chunk(100 + i, n_target=1200 + 300 * i, features="tarl_dino2") for i in range(4)]
    res = api.segment_chunks([c.points for c in chunks], [c.tarl for c in chunks], [c.dino for c in chunks],
                             T=CFG["T"], device=cuda_device, want_stats=True, **KW)
    assert res.unconverged == 0 and res.stats["converged"].all()
    stable = matched = 0
    for ch, lab, ns in zip(chunks, res.labels, res.num_segments):
        assert lab.shape == (ch.n,) and lab.min() == 0 and lab.max() + 1 == ns
        ref = oracle_labels(ch)
        if not R.same_partition(ref, oracle_labels(ch, "random", 5)):
            continue
        stable += 1
        matched += R.same_partition(lab, ref)
    assert stable >= 3 and matched == stable
    packed = api.PackedChunks([c.points for c in chunks], [c.tarl for c in chunks], [c.dino for c in chunks],
                              theta=KW["theta"], gamma=KW["gamma"])
    dev = packed.to_device(cuda_device)
    api.segment_packed(packed, dev_chunks=dev, T=CFG["T"], **KW)
    assert np.array_equal(dev.labels.cpu().numpy(), np.concatenate(res.labels))


def test_drop_in_with_two_cameras(cuda_device, monkeypatch):
    import ncuts.ncuts_utils as nu
    from test_gpu_dropin import FakeCloud, install_fake_reference_modules
    from autoinst_b200.synthetic import make_scans
    from oracle.pool_ref import pool_features_ref
    cfg = dict(CFG, name="tarl_spatial_dino", out_folder="x/", gt=True)
    ch = make_chunk(31, n_target=1500, features="tarl_dino2")
    # the array-level core
    groups = nu.segment_major_points(ch.points, ch.tarl, ch.dino, config=cfg)
    ref = oracle_labels(ch)
    assert R.same_partition(R.labels_from_groups(groups, ch.n), ref)
    # ncuts_chunk: dinov2_mean_per_patch returns one array per camera
    install_fake_reference_modules(monkeypatch, ch)
    import autoinst_b200.dino as dino_mod
    monkeypatch.setattr(dino_mod, "dinov2_mean_per_patch", lambda *a, **k: list(ch.dino))
    monkeypatch.setattr(nu, "CONFIG", cfg)
    rng = np.random.default_rng(0)
    minor = ch.points[rng.integers(0, ch.n, size=6000)] + rng.normal(0, 0.03, size=(6000, 3))
    ground = np.stack([rng.uniform(-12, 12, 500), rng.uniform(-12, 12, 500), rng.normal(-12.4, 0.05, 500)], 1)
    d = {"center_ids": [5], "center_positions": [np.zeros(3)], "indices": [np.arange(len(minor))],
         "pcd_nonground_chunks": [FakeCloud(minor)], "pcd_ground_chunks": [FakeCloud(ground)],
         "pcd_nonground_chunks_major_downsampling": [FakeCloud(ch.points)],
         "kitti_labels": {"ground": {"instance": [np.zeros(500, int)], "semantic": [np.full(500, 40)]}}}
    scans = dict(zip((4, 5, 6), make_scans(ch, n_scans=3, pts_per_major=2.0)))
    none = (np.zeros((0, 3)), np.zeros((0, 96), dtype=np.float32))

    class FakeDataset:
        def get_pose(self, i): return np.eye(4)
        def get_point_cloud(self, i): return scans.get(i, none)[0]
        def get_tarl_features(self, i): return scans.get(i, none)[1]
    _, pcd_chunk, _, _, _ = nu.ncuts_chunk(FakeDataset(), d, None, np.eye(4), list(range(40)), sequence=0,
                                           patchwise_indices=[[5]])
    tarl_ref = pool_features_ref(ch.points, [scans[i] for i in (4, 5, 6)], np.zeros(3))
    A = affinity_ref(ch.points, tarl_ref, ch.dino, **KW)
    with R.pinned_eigsh():
        g = R.normalized_cut_ref(sp.csr_matrix(A), ch.n, np.arange(ch.n), T=CFG["T"])
    ref_major = R.labels_from_groups(g, ch.n)
    from scipy.spatial import cKDTree
    _, nn = cKDTree(ch.points).query(minor, k=1)
    _, got = np.unique(np.asarray(pcd_chunk.colors), axis=0, return_inverse=True)
    assert R.same_partition(got.reshape(-1), ref_major[nn])


def test_argument_errors(cuda_device):
    api = _api()
    from autoinst_b200._lib import AncutsError
    ch = make_chunk(47, n_target=1200, features="tarl_dino2")
    with pytest.raises(AncutsError, match="one DINOv2 camera"):                  # tensor-core form, two cameras
        api.affinity(ch.points, ch.tarl, ch.dino, device=cuda_device, impl=1, **KW)
    packed = api.PackedChunks([ch.points], [ch.tarl], [ch.dino], theta=KW["theta"], gamma=KW["gamma"])
    with pytest.raises(AncutsError, match="one DINOv2 camera"):
        api.segment_packed(packed, device=cuda_device, affinity_impl=1, T=CFG["T"], **KW)
    with pytest.raises(AncutsError, match="multiples of 4"):                    # per-camera width 6 (row width 12)
        api.affinity(ch.points, ch.tarl, [g[:, :6] for g in ch.dino], device=cuda_device, **KW)
    with pytest.raises(ValueError):                                              # mismatched camera shapes
        api.affinity(ch.points, ch.tarl, [ch.dino[0], ch.dino[1][:, :380]], device=cuda_device, **KW)
    with pytest.raises(ValueError, match="The length should be longer than 0!"):
        api.affinity(ch.points, ch.tarl, [], device=cuda_device, **KW)
    # dino_cams = 0 through the ABI
    hd = api.Handle.get(cuda_device)
    pts = torch.as_tensor(ch.points, device=cuda_device)
    t = torch.as_tensor(ch.tarl, dtype=torch.float32, device=cuda_device)
    g = torch.as_tensor(ch.dino[0], dtype=torch.float32, device=cuda_device)
    p = api.make_params(T=0.0, tarl_dim=96, dino_dim=384, **KW)
    buf, _ = api.alloc_matrix(ch.n, cuda_device)
    rc = hd.lib.ancuts_affinity_cams_f32(hd.h, ch.n, api._ptr(pts), api._ptr(t), api._ptr(g), 0, C.byref(p), api._ptr(buf),
                                         buf.stride(0), None, api._stream(cuda_device))
    assert rc == -1 and b"dino_cams" in hd.lib.ancuts_last_error()
    off = np.array([0, ch.n], dtype=np.int64)
    nseg = np.zeros(1, dtype=np.int32)
    lab = torch.empty(ch.n, dtype=torch.int32, device=cuda_device)
    for fn in (hd.lib.ancuts_segment_chunks_cams, hd.lib.ancuts_segment_chunks_cams_host):
        host = fn is hd.lib.ancuts_segment_chunks_cams_host
        P, Tt, G = (packed.points, packed.tarl, packed.dino) if host else (pts, t, g)
        rc = fn(hd.h, 1, off.ctypes.data_as(C.POINTER(C.c_int64)), api._ptr(P), api._ptr(Tt), api._ptr(G), 0, C.byref(p),
                api._ptr(packed.labels if host else lab), nseg.ctypes.data_as(C.POINTER(C.c_int32)), None, 0,
                C.byref(C.c_int32(0)), api._stream(cuda_device))
        assert rc == -1 and b"dino_cams" in hd.lib.ancuts_last_error()
