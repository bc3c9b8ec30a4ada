"""Array-level Python API over the C ABI (SURVEY.md §8b item 2).

PyTorch is used only for device memory and streams; every computation happens in
libautoinst_ncuts.so.  The reference-facing call surface (`ncuts.ncuts_utils.ncuts_chunk`,
`ncuts.normalized_cut.normalized_cut`) is in the top-level `ncuts` package and calls into here.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np
import torch

import warnings

from . import _lib
from ._lib import AncutsNoConvergence, NodeStat, Params, check

STAGES = ("affinity", "degree", "matvec", "reorth", "scan", "partition")


def _ptr(t):
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


def _stream(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


class Handle:
    """One library handle (device workspace, counters) per CUDA device."""
    _cache: dict = {}

    def __init__(self, device: int):
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise RuntimeError("autoinst_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.device = int(device)
        self.h = C.c_void_p()
        check(self.lib.ancuts_create(self.device, C.byref(self.h)))

    @classmethod
    def get(cls, device=None, lane: int = 0) -> "Handle":
        """Handle of `device`; `lane` > 0 gives further independent handles (own workspace) for concurrent calls."""
        if device is None:
            device = torch.cuda.current_device() if torch.cuda.is_available() else 0
        if isinstance(device, torch.device):
            device = device.index if device.index is not None else torch.cuda.current_device()
        key = (int(device), int(lane))
        if key not in cls._cache:
            cls._cache[key] = Handle(int(device))
        return cls._cache[key]

    def set_option(self, option: int, value: int):
        """Alternative implementations behind the same results (`ancuts_set_option`): _lib.OPT_PAIR_SEARCH
        (0 cell-sorted sweep, 1 shuffled sweep), OPT_MATVEC (0 slices compressed into shared memory, 1 dense blocks
        from HBM), OPT_CLUSTER_MAP (tuning), OPT_FUSED_CUT (0 the cut decision inside the sparse-form eigensolver kernel,
        1 as its own kernels), OPT_NODE_FORM (0 recursion nodes as CSR, dense blocks only where a kernel reads them,
        1 every node as a dense block).  Option 0 is retired and raises."""
        check(self.lib.ancuts_set_option(self.h, int(option), int(value)))

    def sparse_accounting(self) -> dict:
        """Shared-memory sparse matvec form, last segment call: sum of steps x stored entries, stored entries."""
        b = (C.c_double * 2)()
        check(self.lib.ancuts_last_sparse_accounting(self.h, b))
        return {"entry_steps": b[0], "entries": b[1]}

    def reorth_accounting(self) -> dict:
        """Persistent Lanczos kernel, last segment call: Lanczos steps, and steps that took the full Gram-Schmidt pass."""
        b = (C.c_double * 2)()
        check(self.lib.ancuts_last_reorth_accounting(self.h, b))
        return {"steps": int(b[0]), "full_passes": int(b[1])}

    def last_unconverged(self) -> int:
        return int(self.lib.ancuts_last_unconverged(self.h))

    def launch_count(self, reset=False) -> int:
        return int(self.lib.ancuts_launch_count(self.h, 1 if reset else 0))

    def set_stage_timing(self, mode: int):
        """0 = off, 1 = CUDA events around every launch, 2 = around the matvec launches only."""
        check(self.lib.ancuts_set_stage_timing(self.h, int(mode)))

    def accounting(self) -> dict:
        b = (C.c_double * 6)()
        m = (C.c_double * 6)()
        l = (C.c_int64 * 6)()
        check(self.lib.ancuts_last_accounting(self.h, b, m, l))
        return {s: dict(bytes=b[i], ms=m[i], launches=int(l[i])) for i, s in enumerate(STAGES)}

    def debug_phases(self, reset=True) -> dict:
        """Cycles per phase of the persistent Lanczos kernel (needs ANCUTS_PHASES=1 before the handle is created)."""
        buf = (C.c_double * 32)()
        check(self.lib.ancuts_debug_phases(self.h, buf, 1 if reset else 0))
        names = ["basis", "matvec", "alpha_3term_norm", "check_multisection", "full_pass_dots", "full_pass_update_norm",
                 "norm_exchange_omega", "check_rest"]
        return {c: {nm: buf[8 * i + j] for j, nm in enumerate(names)} for i, c in enumerate((1, 2, 4, 8))}

    def levels(self, cap: int = 256) -> list:
        """Per-level trace of the last segment call made in timing mode 2 (ancuts_last_levels)."""
        buf = (C.c_double * (16 * cap))()
        n = min(int(self.lib.ancuts_last_levels(self.h, buf, cap)), cap)
        return [dict(active=int(buf[16 * i]), big=int(buf[16 * i + 1]), ms=buf[16 * i + 2],
                     bins=[int(buf[16 * i + 3 + b]) for b in range(6)],
                     cluster=[int(buf[16 * i + 9 + b]) for b in range(6)]) for i in range(n)]


def make_params(alpha=1.0, theta=0.0, gamma=0.0, T=0.01, proximity=1.0, split_lim=0.01, beta=0.0,
                tarl_dim=0, dino_dim=0, max_steps=0, check_every=0, tol=0.0, affinity_impl=0,
                lanczos_impl=0) -> Params:
    if beta:
        # SAM term, ncuts_utils.py:115-123; beta = 0.0 in every shipped config (config.py:12,23,34,45)
        raise NotImplementedError("beta != 0 (SAM label term) is not supported by the B200 path")
    return Params(float(alpha or 0.0), float(theta or 0.0), float(gamma or 0.0), float(proximity), float(T),
                  float(split_lim), int(tarl_dim), int(dino_dim), int(max_steps), int(check_every),
                  float(tol), int(affinity_impl), int(lanczos_impl))


def _dev(device):
    if device is None:
        return torch.device("cuda", torch.cuda.current_device())
    d = torch.device(device)
    if d.index is None:
        d = torch.device("cuda", torch.cuda.current_device())
    return d


def _as_dev(x, dtype, device):
    if x is None:
        return None
    if isinstance(x, torch.Tensor):
        return x.to(device=device, dtype=dtype).contiguous()
    return torch.as_tensor(np.ascontiguousarray(x), dtype=dtype).to(device)


def _dino_shape(x):
    """(cameras, width) of one chunk's DINOv2 input: an (n, D) array (one camera), a list or tuple of per-camera (n, D)
    arrays (the reference's per-CAM_IDS means, ncuts_utils.py:81-110), or an (n, cams, D) array or tensor."""
    if isinstance(x, (list, tuple)):
        if len(x) == 0:
            raise ValueError("The length should be longer than 0!")       # ncuts_utils.py:126-127
        shapes = {tuple(int(d) for d in np.shape(c)) for c in x}
        if len(shapes) != 1 or len(next(iter(shapes))) != 2:
            raise ValueError(f"the cameras of a chunk need one (n, D) shape each, got {sorted(shapes)}")
        return len(x), next(iter(shapes))[1]
    shape = tuple(int(d) for d in x.shape)
    if len(shape) == 2:
        return 1, shape[1]
    if len(shape) == 3:
        return shape[1], shape[2]
    raise ValueError(f"DINOv2 input must be (n, D), a list of (n, D) or (n, cams, D), got shape {shape}")


def _dino_rows(x, device):
    """One chunk's DINOv2 input on the device as point-major (n, cams * D) float32 rows; returns (rows, cams, D)."""
    cams, width = _dino_shape(x)
    if isinstance(x, (list, tuple)):
        g = torch.stack([_as_dev(c, torch.float32, device) for c in x], dim=1)
    else:
        g = _as_dev(x, torch.float32, device)
    return g.reshape(g.shape[0], cams * width).contiguous(), cams, width


def padded_ld(n: int) -> int:
    return (int(n) + 31) // 32 * 32


def alloc_matrix(n, device):
    """n x ld float32 storage and its n x n view."""
    ld = padded_ld(n)
    buf = torch.empty((n, ld), dtype=torch.float32, device=device)
    return buf, buf[:, :n]


# ------------------------------------------------------------------------------------------------
# stage entry points
# ------------------------------------------------------------------------------------------------
def affinity(points, tarl=None, dino=None, *, alpha=1.0, theta=0.0, gamma=0.0, proximity=1.0, impl=0,
             device=None, return_rowsum=False, lane: int = 0):
    """Stage 1: dense float32 affinity (ncuts_utils.py:60-156).  Returns the n x n view of an n x ld buffer.
    dino: (n, D), a list of per-camera (n, D) arrays or (n, cams, D); several cameras multiply their terms."""
    device = _dev(device)
    hd = Handle.get(device, lane)
    pts = _as_dev(points, torch.float64, device)
    n = pts.shape[0]
    t = _as_dev(tarl, torch.float32, device) if theta else None
    if theta and t is None:
        raise ValueError("theta != 0 needs TARL features")
    if gamma and dino is None:
        raise ValueError("The length should be longer than 0!")       # ncuts_utils.py:126-127
    g, cams, width = _dino_rows(dino, device) if gamma else (None, 1, 0)
    p = make_params(alpha, theta, gamma, 0.0, proximity, tarl_dim=t.shape[1] if t is not None else 0,
                    dino_dim=width, affinity_impl=impl)
    buf, view = alloc_matrix(n, device)
    rs = torch.empty(n, dtype=torch.float64, device=device) if return_rowsum else None
    with torch.cuda.device(device):
        check(hd.lib.ancuts_affinity_cams_f32(hd.h, n, _ptr(pts), _ptr(t), _ptr(g), cams, C.byref(p), _ptr(buf),
                                              buf.stride(0), _ptr(rs), _stream(device)))
    return (view, rs) if return_rowsum else view


def _matrix_args(W):
    if W.dtype != torch.float32 or W.dim() != 2 or W.stride(1) != 1 or W.stride(0) % 4 or W.data_ptr() % 16:
        n = W.shape[0]
        buf, view = alloc_matrix(n, W.device)
        view.copy_(W)
        W = view
    return W, W.stride(0)


def degree_normalize(W, return_normalized=False):
    """Stage 2: d = (w + I).sum(0) in float64; optionally M = D^-1/2 (w+I) D^-1/2 (normalized_cut.py:38-47)."""
    W, ld = _matrix_args(W)
    device = W.device
    hd = Handle.get(device)
    n = W.shape[0]
    deg = torch.empty(n, dtype=torch.float64, device=device)
    Mbuf = Mv = None
    if return_normalized:
        Mbuf, Mv = alloc_matrix(n, device)
    with torch.cuda.device(device):
        check(hd.lib.ancuts_degree_normalize_f32(hd.h, n, _ptr(W), ld, _ptr(deg), _ptr(Mbuf),
                                                 Mbuf.stride(0) if Mbuf is not None else 0, _stream(device)))
    return (deg, Mv) if return_normalized else deg


def _node_arrays(node_off, node_n):
    off = np.ascontiguousarray(node_off, dtype=np.int32)
    nn = np.ascontiguousarray(node_n, dtype=np.int32)
    return off, nn, off.ctypes.data_as(C.POINTER(C.c_int32)), nn.ctypes.data_as(C.POINTER(C.c_int32))


def lanczos_fiedler(W, node_off, node_n, *, max_steps=0, check_every=0, tol=0.0, lanczos_impl=0):
    """Stage 3: Fiedler vector of every diagonal block (normalized_cut.py:49-53).
    Returns (ev float64 [n_total] on device, lambda2, steps, converged)."""
    W, ld = _matrix_args(W)
    device = W.device
    hd = Handle.get(device)
    n = W.shape[0]
    off, nn, poff, pn = _node_arrays(node_off, node_n)
    k = len(off)
    ev = torch.zeros(n, dtype=torch.float64, device=device)
    lam = np.zeros(k)
    steps = np.zeros(k, dtype=np.int32)
    conv = np.zeros(k, dtype=np.int32)
    p = make_params(T=0.0, max_steps=max_steps, check_every=check_every, tol=tol, lanczos_impl=lanczos_impl)
    with torch.cuda.device(device):
        check(hd.lib.ancuts_lanczos_fiedler_batched(
            hd.h, n, _ptr(W), ld, k, poff, pn, C.byref(p), _ptr(ev), lam.ctypes.data_as(C.POINTER(C.c_double)),
            steps.ctypes.data_as(C.POINTER(C.c_int32)), conv.ctypes.data_as(C.POINTER(C.c_int32)), _stream(device)))
    return ev, lam, steps, conv


def ncut_scan(W, node_off, node_n, ev):
    """Stage 4a: best of the ten threshold cuts per node (normalized_cut.py:13-34).
    Returns (best_k, mcut, costs [k,10], mask uint8 [n_total] on device; 1 where ev > threshold)."""
    W, ld = _matrix_args(W)
    device = W.device
    hd = Handle.get(device)
    n = W.shape[0]
    off, nn, poff, pn = _node_arrays(node_off, node_n)
    k = len(off)
    evd = _as_dev(ev, torch.float64, device)
    best = np.zeros(k, dtype=np.int32)
    mcut = np.zeros(k)
    costs = np.zeros((k, _lib.NUM_CUTS))
    side = torch.zeros(n, dtype=torch.uint8, device=device)
    with torch.cuda.device(device):
        check(hd.lib.ancuts_ncut_scan_batched(
            hd.h, n, _ptr(W), ld, k, poff, pn, _ptr(evd), best.ctypes.data_as(C.POINTER(C.c_int32)),
            mcut.ctypes.data_as(C.POINTER(C.c_double)), costs.ctypes.data_as(C.POINTER(C.c_double)), _ptr(side),
            _stream(device)))
    return best, mcut, costs, side


def partition(W, node_off, node_n, mask, split_components=True):
    """Stage 4b: stable partition (mask side first) + connected components + block gather
    (normalized_cut.py:57-58).  Returns (W_out view, perm [new]->old on device, child_off, child_n)."""
    W, ld = _matrix_args(W)
    device = W.device
    hd = Handle.get(device)
    n = W.shape[0]
    off, nn, poff, pn = _node_arrays(node_off, node_n)
    k = len(off)
    m = _as_dev(mask, torch.uint8, device)
    obuf = torch.zeros((n, ld), dtype=torch.float32, device=device)
    perm = torch.zeros(n, dtype=torch.int32, device=device)
    cnt = C.c_int32(0)
    coff = np.zeros(n, dtype=np.int32)
    cn = np.zeros(n, dtype=np.int32)
    with torch.cuda.device(device):
        check(hd.lib.ancuts_partition_batched(
            hd.h, n, _ptr(W), _ptr(obuf), ld, k, poff, pn, _ptr(m), 1 if split_components else 0, _ptr(perm),
            C.byref(cnt), coff.ctypes.data_as(C.POINTER(C.c_int32)), cn.ctypes.data_as(C.POINTER(C.c_int32)),
            _stream(device)))
    c = cnt.value
    return obuf[:, :n], perm, coff[:c].copy(), cn[:c].copy()


def nn_reproject(query_points, source_points, source_labels=None, max_radius=None, no_label=-1, device=None):
    """Label of the nearest source point for every query point (point_cloud_utils.py:144-174).
    Returns (labels int32 [nq], index int32 [nq]) on the device."""
    device = _dev(device)
    hd = Handle.get(device)
    q = _as_dev(query_points, torch.float64, device)
    s = _as_dev(source_points, torch.float64, device)
    lab = _as_dev(source_labels, torch.int32, device) if source_labels is not None else None
    out = torch.empty(q.shape[0], dtype=torch.int32, device=device)
    idx = torch.empty(q.shape[0], dtype=torch.int32, device=device)
    with torch.cuda.device(device):
        check(hd.lib.ancuts_nn_reproject(hd.h, q.shape[0], _ptr(q), s.shape[0], _ptr(s), _ptr(lab),
                                         float(max_radius) if max_radius else 0.0, int(no_label), _ptr(out), _ptr(idx),
                                         _stream(device)))
    return out, idx


def feature_pool(major_points, scan_points, scan_features, radius, box_min, box_max, *, normalise=False,
                 return_count=False, device=None):
    """Mean of the feature rows of the scan points strictly closer than `radius` to every major point
    (`tarl_features_per_patch`, chunk_generation.py:205-258; C ABI `ancuts_feature_pool`).  Scan points outside
    the open box (box_min, box_max) are ignored (:233-236).  Returns float64 [n_major, F] on the device
    (zero rows where nothing is in range) and, with return_count, the int32 neighbour counts."""
    device = _dev(device)
    hd = Handle.get(device)
    q = _as_dev(major_points, torch.float64, device).reshape(-1, 3)
    sp = _as_dev(scan_points, torch.float64, device).reshape(-1, 3)
    ft = _as_dev(scan_features, torch.float32, device)
    m = int(sp.shape[0])
    ft = ft.reshape(m, -1) if m else ft.reshape(0, ft.shape[-1] if ft.dim() > 1 else 1)
    fdim = int(ft.shape[1])
    out = torch.empty((q.shape[0], fdim), dtype=torch.float64, device=device)
    cnt = torch.empty(q.shape[0], dtype=torch.int32, device=device)
    wsb = int(hd.lib.ancuts_feature_pool_workspace_bytes(m))
    ws = torch.empty(max(wsb, 256), dtype=torch.uint8, device=device)
    lo = (C.c_double * 3)(*[float(v) for v in np.asarray(box_min, dtype=np.float64).ravel()[:3]])
    hi = (C.c_double * 3)(*[float(v) for v in np.asarray(box_max, dtype=np.float64).ravel()[:3]])
    with torch.cuda.device(device):
        check(hd.lib.ancuts_feature_pool(hd.h, q.shape[0], _ptr(q), m, _ptr(sp) if m else None, _ptr(ft) if m else None,
                                         fdim, float(radius), lo, hi, 1 if normalise else 0, _ptr(out), _ptr(cnt),
                                         _ptr(ws), wsb, _stream(device)))
    return (out, cnt) if return_count else out


def dino_mean_views(major_points, views, max_dist, *, feat_dim=384, device=None, return_count=False):
    """DINOv2 features of the major points averaged over the views that see them (`image_based_features_per_patch`
    behind its visibility bookkeeping + `dinov2_mean`, image_utils.py:264-346,363-371; C ABI `ancuts_dino_view_pixels`,
    `ancuts_dino_mean`).  views: list of None (a view the reference skips) or dicts with T_pcd2cam (4 x 4), visible_cam
    ((M, 3) float64: the view's visible chunk points in the camera frame), K (3 x 3), img_hw (h, w), feature_map
    ((Hp, Wp, F) float32, numpy or a CUDA tensor).  Returns (N, F) float64 on the device."""
    device = _dev(device)
    hd = Handle.get(device)
    major = np.ascontiguousarray(major_points, dtype=np.float64)
    n = major.shape[0]
    V = len(views)
    pix = torch.full((max(V, 1), n), -1, dtype=torch.int32, device=device)
    maps, keep = [], []
    hom = np.concatenate([major, np.ones((n, 1))], axis=1)
    with torch.cuda.device(device):
        for v, view in enumerate(views):
            if view is None:
                maps.append(None)
                continue
            fm = view["feature_map"]
            fm = fm.to(device=device, dtype=torch.float32).contiguous() if isinstance(fm, torch.Tensor) else \
                torch.as_tensor(np.ascontiguousarray(fm, dtype=np.float32)).to(device)
            if fm.shape[2] != feat_dim:
                raise ValueError("feature map depth differs from feat_dim")
            keep.append(fm)
            maps.append(fm)
            T = np.asarray(view["T_pcd2cam"], dtype=np.float64)
            cam = hom @ T.T                                        # Open3D PointCloud.transform (:264): homogeneous product,
            cam = np.ascontiguousarray(cam[:, :3] / cam[:, 3:4])  # division by w
            d_cam = torch.as_tensor(cam).to(device)
            vis = _as_dev(view["visible_cam"], torch.float64, device).reshape(-1, 3)
            K = np.ascontiguousarray(view["K"], dtype=np.float64).reshape(9)
            h_img, w_img = int(view["img_hw"][0]), int(view["img_hw"][1])
            check(hd.lib.ancuts_dino_view_pixels(hd.h, n, _ptr(d_cam), int(vis.shape[0]), _ptr(vis) if vis.shape[0] else None,
                                                 float(max_dist), K.ctypes.data_as(C.POINTER(C.c_double)), h_img, w_img,
                                                 int(fm.shape[0]), int(fm.shape[1]), _ptr(pix[v]), _stream(device)))
            keep.extend([d_cam, vis])
        out = torch.empty((n, feat_dim), dtype=torch.float64, device=device)
        cnt = torch.empty(n, dtype=torch.int32, device=device)
        ptrs = (C.c_void_p * max(V, 1))(*[(m.data_ptr() if m is not None else (keep[0].data_ptr() if keep else 0)) for m in maps] or [0])
        check(hd.lib.ancuts_dino_mean(hd.h, n, V, _ptr(pix), ptrs, int(feat_dim), _ptr(out), _ptr(cnt), _stream(device)))
        torch.cuda.current_stream(device).synchronize()           # `keep` may go away
    return (out, cnt) if return_count else out


# ------------------------------------------------------------------------------------------------
# map level: merge (N2), remove_semantics, instance metrics (N4)
# ------------------------------------------------------------------------------------------------
METRIC_KEYS = ("p", "r", "f1", "ap", "ap0.25", "ap0.5", "S_assoc")     # sequence_stats, metrics_class.py:262-269


def _as_i32_labels(x, device):
    if isinstance(x, torch.Tensor):
        return x.to(device=device, dtype=torch.int32).contiguous()
    a = np.asarray(x)
    if a.size and (a.min() < -2 ** 31 or a.max() >= 2 ** 31):
        raise ValueError("labels must fit int32")
    return torch.as_tensor(np.ascontiguousarray(a, dtype=np.int32)).to(device)


def merge_chunks(chunks, *, crop_side=40.0, min_iou=0.01, device=None, return_device=False):
    """merge_chunks_unite_instances2 (point_cloud_utils.py:387-491) on the device (C ABI `ancuts_merge_chunks`).
    chunks: list of (points (n,3) float64, labels (n,) int, 0 = background) in file-name order.
    Returns (merged points, merged labels) as numpy arrays (or device tensors with return_device)."""
    device = _dev(device)
    hd = Handle.get(device)
    sizes = [int(np.asarray(p).shape[0]) if not isinstance(p, torch.Tensor) else int(p.shape[0]) for p, _ in chunks]
    off = np.zeros(len(sizes) + 1, dtype=np.int64)
    off[1:] = np.cumsum(sizes)
    # chunk centres with the reference's own expression (column means of the chunk's points, :397-403)
    centers = np.stack([np.array([np.asarray(p)[:, 0].mean(), np.asarray(p)[:, 1].mean(), np.asarray(p)[:, 2].mean()])
                        if not isinstance(p, torch.Tensor) else p.double().cpu().numpy().mean(axis=0) for p, _ in chunks])
    pts = torch.cat([_as_dev(p, torch.float64, device).reshape(-1, 3) for p, _ in chunks])
    lab = torch.cat([_as_i32_labels(l, device).reshape(-1) for _, l in chunks])
    out_lab, idx, kept = _merge_device(hd, off, pts, lab, centers, crop_side / 2.0, min_iou, device)
    mp, ml = pts[idx[:kept]], out_lab[idx[:kept]]
    if return_device:
        return mp, ml
    return mp.cpu().numpy(), ml.cpu().numpy().astype(np.int64)


def _merge_device(hd, off, pts, lab, centers, half_side, min_iou, device):
    P = int(off[-1])
    out_lab = torch.empty(P, dtype=torch.int32, device=device)
    idx = torch.empty(P, dtype=torch.int64, device=device)
    kept = C.c_int64(0)
    off = np.ascontiguousarray(off, dtype=np.int64)
    centers = np.ascontiguousarray(centers, dtype=np.float64)
    with torch.cuda.device(device):
        check(hd.lib.ancuts_merge_chunks(hd.h, len(off) - 1, off.ctypes.data_as(C.POINTER(C.c_int64)), _ptr(pts), _ptr(lab),
                                         centers.ctypes.data_as(C.POINTER(C.c_double)), float(half_side), float(min_iou),
                                         _ptr(out_lab), _ptr(idx), C.byref(kept), _stream(device)))
    return out_lab, idx, int(kept.value)


def remove_semantics(gt_labels, pred_labels, threshold=0.8, device=None, return_device=False):
    """remove_semantics (point_cloud_utils.py:253-287): predicted labels with more than `threshold` of their points on
    GT background become 0 (C ABI `ancuts_remove_semantics`)."""
    device = _dev(device)
    hd = Handle.get(device)
    gt = _as_i32_labels(gt_labels, device)
    pr = _as_i32_labels(pred_labels, device)
    out = torch.empty_like(pr)
    with torch.cuda.device(device):
        check(hd.lib.ancuts_remove_semantics(hd.h, int(pr.numel()), _ptr(gt), _ptr(pr), float(threshold), _ptr(out),
                                             _stream(device)))
    return out if return_device else out.cpu().numpy().astype(np.int64)


def instance_metrics(all_labels, pred_labels, gt_labels, min_points=200, device=None, full=False):
    """Metrics(...).update_stats(all_labels, pred_labels, gt_labels) for a fresh Metrics object
    (metrics_class.py:137-179; C ABI `ancuts_instance_metrics`).  Returns the dict of sequence_stats' keys."""
    device = _dev(device)
    hd = Handle.get(device)
    a = _as_i32_labels(all_labels, device)
    p = _as_i32_labels(pred_labels, device)
    g = _as_i32_labels(gt_labels, device)
    out = (C.c_double * 21)()
    with torch.cuda.device(device):
        check(hd.lib.ancuts_instance_metrics(hd.h, int(p.numel()), _ptr(a), _ptr(p), _ptr(g), int(min_points), out,
                                             _stream(device)))
    if out[8] == 0 or out[9] == 0:
        raise ZeroDivisionError("no predicted or no ground-truth instances (metrics_class.py:325-326)")
    res = {k: float(out[i]) for i, k in enumerate(METRIC_KEYS)}
    if full:
        res.update(tp=int(out[7]), n_pred=int(out[8]), n_gt=int(out[9]), ap_per_overlap=[float(out[10 + t]) for t in range(11)])
    return res


class MapPost:
    """Everything after the per-chunk cuts of one map, on the device (run_pipeline.py:197-238): labels of all chunks ->
    globally unique instance ids -> merge (N2) -> remove_semantics -> metrics (N4).  Set up once per map (points, GT
    and the chunk table go to the device, the GT map is the de-duplicated concatenation, `merge_unite_gt`,
    point_cloud_utils.py:320-329), then `merge_and_score` per labeling."""

    def __init__(self, chunks, device=None, min_points=200, crop_side=40.0, min_iou=0.01, threshold=0.8):
        self.device = _dev(device)
        self.hd = Handle.get(self.device)
        self.sizes = [int(c.n) for c in chunks]
        self.off = np.zeros(len(chunks) + 1, dtype=np.int64)
        self.off[1:] = np.cumsum(self.sizes)
        self.centers = np.stack([np.array([c.points[:, 0].mean(), c.points[:, 1].mean(), c.points[:, 2].mean()]) for c in chunks])
        self.pts = torch.as_tensor(np.concatenate([c.points for c in chunks]), dtype=torch.float64).to(self.device)
        self.gt_all = _as_i32_labels(np.concatenate([c.instance for c in chunks]), self.device)
        self.min_points, self.half, self.min_iou, self.threshold = int(min_points), crop_side / 2.0, float(min_iou), float(threshold)
        self.keep = None

    def global_labels(self, seg_flat):
        """Per-chunk segment ids (concatenated, chunk order) -> ids unique across the map; segments are numbered by first
        occurrence in point order inside every chunk, like oracle.merge_ref.canonical_labels + globally_unique (the
        reference draws a random colour per segment; the greedy rules downstream depend on the order of the values).
        C ABI `ancuts_map_labels`."""
        seg = _as_i32_labels(seg_flat, self.device)
        out = torch.empty_like(seg)
        with torch.cuda.device(self.device):
            check(self.hd.lib.ancuts_map_labels(self.hd.h, len(self.sizes), self.off.ctypes.data_as(C.POINTER(C.c_int64)),
                                                _ptr(seg), 20, _ptr(out), _stream(self.device)))
        return out

    def merge(self, seg_flat):
        lab = self.global_labels(seg_flat)
        out_lab, idx, kept = _merge_device(self.hd, self.off, self.pts, lab, self.centers, self.half, self.min_iou, self.device)
        keep = idx[:kept]
        if self.keep is None:
            self.keep = keep
            self.gt = self.gt_all[keep].contiguous()
        return out_lab[keep].contiguous()

    def merge_and_score(self, seg_flat):
        """seg_flat: int32 segment ids of all chunks concatenated in chunk order (device or host).  Returns the metrics."""
        merged = self.merge(seg_flat)
        with torch.cuda.device(self.device):
            inst = torch.empty_like(merged)
            check(self.hd.lib.ancuts_remove_semantics(self.hd.h, int(merged.numel()), _ptr(self.gt), _ptr(merged),
                                                      self.threshold, _ptr(inst), _stream(self.device)))
        return instance_metrics(merged, inst, self.gt, min_points=self.min_points, device=self.device)


# ------------------------------------------------------------------------------------------------
# whole path
# ------------------------------------------------------------------------------------------------
@dataclass
class SegmentResult:
    labels: list            # one int32 numpy array per chunk
    num_segments: np.ndarray
    stats: np.ndarray | None   # structured array of ancuts_node_stat rows (all chunks of the call)
    unconverged: int = 0       # eigensolver nodes that stopped at max_steps (their cut used an unconverged vector)


def _report_unconverged(hd, strict: bool) -> int:
    """Non-convergence is never silent: the drop-in callers raise (as the reference's eigsh would), the array
    level warns unless `strict`."""
    cnt = hd.last_unconverged()
    if cnt > 0:
        if strict:
            raise AncutsNoConvergence(cnt)
        warnings.warn(f"Lanczos eigensolver: {cnt} recursion node(s) stopped at the step limit without converging; "
                      "their cuts used the unconverged Ritz vector (raise max_steps)", RuntimeWarning, stacklevel=3)
    return cnt


_STAT_DTYPE = np.dtype([("chunk", "<i4"), ("n", "<i4"), ("steps", "<i4"), ("converged", "<i4"), ("best_k", "<i4"),
                        ("split", "<i4"), ("level", "<i4"), ("n_side", "<i4"), ("lambda2", "<f8"), ("mcut", "<f8")])


def workspace_bytes(sizes, max_steps=0) -> int:
    lib = _lib.load()
    arr = np.ascontiguousarray(sizes, dtype=np.int32)
    return int(lib.ancuts_segment_workspace_bytes(len(arr), arr.ctypes.data_as(C.POINTER(C.c_int32)), int(max_steps)))


def plan_batches(sizes, budget_bytes, max_steps=0):
    """Greedy split of chunk indices (in order) into batches whose workspace fits the budget."""
    batches, cur = [], []
    for i, n in enumerate(sizes):
        trial = cur + [i]
        if cur and workspace_bytes([sizes[j] for j in trial], max_steps) > budget_bytes:
            batches.append(cur)
            cur = [i]
        else:
            cur = trial
    if cur:
        batches.append(cur)
    return batches


class _PinnedPool:
    """Grow-only pinned host buffers reused across calls (cudaHostAlloc of hundreds of MB costs more than the copy)."""
    _bufs: dict = {}

    @classmethod
    def take(cls, name, shape, dtype, pin):
        if not pin:
            return torch.empty(shape, dtype=dtype)
        need = int(np.prod(shape))
        key = (name, dtype)
        buf = cls._bufs.get(key)
        if buf is None or buf.numel() < need:
            buf = torch.empty(max(need, 1), dtype=dtype).pin_memory()
            cls._bufs[key] = buf
        return buf[:need].view(shape)


def _pack_host(points_list, tarl_list, dino_list, use_t, use_d, pin=True, reuse=False):
    """Concatenate the chunks into (pinned) host buffers: float64 coordinates, float32 features.  The float64 -> float32
    conversion of the features (the reference hands float64 means, chunk_generation.py:252) goes straight into the buffer,
    chunks in parallel on a few threads (numpy releases the GIL).  The DINOv2 buffer is point-major (P, cams * D): a
    point's row holds camera 0's D values, then camera 1's, ...  Returns (sizes, off, points, tarl, dino, cams)."""
    sizes = [int(np.asarray(p).shape[0]) for p in points_list]
    off = np.zeros(len(sizes) + 1, dtype=np.int64)
    off[1:] = np.cumsum(sizes)
    total = int(off[-1])
    cams, width = 1, 0
    if use_d:
        shapes = [_dino_shape(g) for g in dino_list]
        if len(set(shapes)) != 1:
            raise ValueError(f"every chunk of a call needs the same DINOv2 cameras and width, got {sorted(set(shapes))}")
        cams, width = shapes[0]

    def mk(name, shape, dtype):
        if reuse:
            return _PinnedPool.take(name, shape, dtype, pin)
        t = torch.empty(shape, dtype=dtype)
        return t.pin_memory() if pin else t
    hp = mk("points", (total, 3), torch.float64)
    ht = mk("tarl", (total, np.asarray(tarl_list[0]).shape[1]), torch.float32) if use_t else None
    hd_ = mk("dino", (total, cams * width), torch.float32) if use_d else None
    hp_n = hp.numpy()
    ht_n = ht.numpy() if use_t else None
    hd_n = hd_.numpy() if use_d else None

    def put(c):
        a, b = int(off[c]), int(off[c + 1])
        np.copyto(hp_n[a:b], np.asarray(points_list[c]), casting="same_kind")
        if use_t:
            np.copyto(ht_n[a:b], np.asarray(tarl_list[c]), casting="same_kind")
        if use_d:
            g = dino_list[c]
            if isinstance(g, (list, tuple)):
                rows = hd_n[a:b].reshape(b - a, cams, width)
                for k, cam in enumerate(g):
                    np.copyto(rows[:, k], np.asarray(cam), casting="same_kind")
            else:
                np.copyto(hd_n[a:b].reshape(np.shape(g)), np.asarray(g), casting="same_kind")
    if len(sizes) >= 4 and total * (3 + (ht_n.shape[1] if use_t else 0) + (hd_n.shape[1] if use_d else 0)) > (1 << 22):
        from concurrent.futures import ThreadPoolExecutor
        import os as _os
        with ThreadPoolExecutor(max_workers=min(8, len(sizes), _os.cpu_count() or 1)) as ex:
            list(ex.map(put, range(len(sizes))))
    else:
        for c in range(len(sizes)):
            put(c)
    return sizes, off, hp, ht, hd_, cams


class PackedChunks:
    """Inputs of a batch of chunks packed once into pinned host buffers (what a data loader hands over).  A chunk's DINOv2
    input is an (n, D) array (one camera), a list or tuple of per-camera (n, D) arrays, or an (n, cams, D) array; every
    chunk of a batch has the same cameras and width.  `dino` is (P, dino_cams * dino_dim), dino_dim the width of one
    camera."""

    def __init__(self, points_list, tarl_list=None, dino_list=None, *, theta=0.0, gamma=0.0, pin=True, reuse=False):
        self.use_t = bool(theta) and tarl_list is not None
        self.use_d = bool(gamma) and dino_list is not None
        if theta and tarl_list is None:
            raise ValueError("theta != 0 needs TARL features")
        if gamma and dino_list is None:
            raise ValueError("The length should be longer than 0!")
        self.sizes, self.off, self.points, self.tarl, self.dino, self.dino_cams = _pack_host(
            points_list, tarl_list, dino_list, self.use_t, self.use_d, pin, reuse)
        if reuse:      # buffers of the module-level pool: valid until the next PackedChunks(reuse=True)
            self.labels = _PinnedPool.take("labels", (int(self.off[-1]),), torch.int32, pin)
        else:
            self.labels = torch.empty(int(self.off[-1]), dtype=torch.int32)
            if pin:
                self.labels = self.labels.pin_memory()
        self.tarl_dim = self.tarl.shape[1] if self.use_t else 0
        self.dino_dim = self.dino.shape[1] // self.dino_cams if self.use_d else 0

    def h2d_bytes(self):
        b = self.points.numel() * 8
        if self.use_t:
            b += self.tarl.numel() * 4
        if self.use_d:
            b += self.dino.numel() * 4
        return b

    def d2h_bytes(self):
        return self.labels.numel() * 4

    def to_device(self, device, labels=None):
        """Inputs resident in HBM.  `labels`: optional int32 device tensor the segment call writes into (e.g. the send
        buffer of sharding.LabelGather, so that the gather needs no copy)."""
        device = _dev(device)
        return DeviceChunks(self, device, labels)


class DeviceChunks:
    def __init__(self, packed: PackedChunks, device, labels=None):
        self.packed = packed
        self.device = device
        self.points = packed.points.to(device, non_blocking=True)
        self.tarl = packed.tarl.to(device, non_blocking=True) if packed.use_t else None
        self.dino = packed.dino.to(device, non_blocking=True) if packed.use_d else None
        total = int(packed.off[-1])
        if labels is not None:
            assert labels.dtype == torch.int32 and labels.is_contiguous() and labels.numel() >= total
            self.labels = labels
        else:
            self.labels = torch.empty(total, dtype=torch.int32, device=device)


def _run_segment(hd, fn_host, packed, dev_chunks, p, want_stats, device):
    B = len(packed.sizes)
    off = np.ascontiguousarray(packed.off, dtype=np.int64)
    nseg = np.zeros(B, dtype=np.int32)
    cap = 128 * B + 64 if want_stats else 0
    stats = np.zeros(max(cap, 1), dtype=_STAT_DTYPE)
    nstats = C.c_int32(0)
    sp = stats.ctypes.data_as(C.POINTER(NodeStat)) if want_stats else None
    with torch.cuda.device(device):
        if fn_host:
            check(hd.lib.ancuts_segment_chunks_cams_host(
                hd.h, B, off.ctypes.data_as(C.POINTER(C.c_int64)), _ptr(packed.points), _ptr(packed.tarl),
                _ptr(packed.dino), packed.dino_cams, C.byref(p), _ptr(packed.labels), nseg.ctypes.data_as(C.POINTER(C.c_int32)),
                sp, cap, C.byref(nstats), _stream(device)))
        else:
            check(hd.lib.ancuts_segment_chunks_cams(
                hd.h, B, off.ctypes.data_as(C.POINTER(C.c_int64)), _ptr(dev_chunks.points), _ptr(dev_chunks.tarl),
                _ptr(dev_chunks.dino), packed.dino_cams, C.byref(p), _ptr(dev_chunks.labels), nseg.ctypes.data_as(C.POINTER(C.c_int32)),
                sp, cap, C.byref(nstats), _stream(device)))
    return nseg, (stats[:nstats.value].copy() if want_stats else None)


def segment_packed(packed: PackedChunks, *, alpha=1.0, theta=0.0, gamma=0.0, T=0.01, proximity=1.0, split_lim=0.01,
                   device=None, dev_chunks: DeviceChunks | None = None, want_stats=False, max_steps=0,
                   check_every=0, tol=0.0, affinity_impl=0, lanczos_impl=0, lane: int = 0,
                   strict: bool = False) -> SegmentResult:
    """Segment a packed batch.  With `dev_chunks` the inputs are already resident in HBM (labels stay on
    the device in dev_chunks.labels); otherwise host buffers go through ancuts_segment_chunks_host."""
    device = _dev(device if dev_chunks is None else dev_chunks.device)
    hd = Handle.get(device, lane)
    p = make_params(alpha, theta if packed.use_t else 0.0, gamma if packed.use_d else 0.0, T, proximity, split_lim,
                    tarl_dim=packed.tarl_dim, dino_dim=packed.dino_dim, max_steps=max_steps, check_every=check_every,
                    tol=tol, affinity_impl=affinity_impl, lanczos_impl=lanczos_impl)
    nseg, stats = _run_segment(hd, dev_chunks is None, packed, dev_chunks, p, want_stats, device)
    unconv = _report_unconverged(hd, strict)
    src = packed.labels if dev_chunks is None else dev_chunks.labels
    labels = None
    if dev_chunks is None:
        arr = src.numpy()
        labels = [arr[a:b].copy() for a, b in zip(packed.off[:-1], packed.off[1:])]
    return SegmentResult(labels=labels, num_segments=nseg, stats=stats, unconverged=unconv)


class SegmentStream:
    """Batches through host buffers with the upload of the NEXT batch overlapping the cut of the current one.

    `segment_packed(packed)` on host buffers is one synchronous C call: upload, cut, labels back.  A caller that has a
    sequence of batches (the chunks of successive maps) loses the upload time of every batch (0.44 GB per 128 chunks with
    TARL features, 8 ms of PCIe) unless the next upload runs while the GPU works.  Here two sets of device input buffers
    alternate: `submit(packed)` starts the upload on a side stream, `result()` cuts the oldest submitted batch with the
    device entry point (`ancuts_segment_chunks`) as soon as its upload event has fired, copies the labels into the
    batch's pinned `packed.labels` and returns them.  Depth 2: at most one batch uploads while one is cut.
    """

    def __init__(self, device=None, lane: int = 0, strict: bool = False, **kw):
        self.device = _dev(device)
        self.lane, self.strict, self.kw = lane, strict, kw
        self.copy_stream = torch.cuda.Stream(device=self.device)
        self.slots = [dict(points=None, tarl=None, dino=None, labels=None, ev=None) for _ in range(2)]
        self.queue = []                 # (slot index, packed) in submission order
        self.next_slot = 0

    @staticmethod
    def _fit(t, src, device):
        if src is None:
            return None
        if t is None or t.numel() < src.numel() or t.dtype != src.dtype:
            t = torch.empty(src.numel(), dtype=src.dtype, device=device)
        return t

    def submit(self, packed: "PackedChunks", labels=None):
        """Start the upload of `packed`.  `labels`: optional int32 device tensor the batch's labels are written into (e.g.
        `sharding.LabelGather.send_view()`, so that the gather needs no copy) instead of the slot's own buffer."""
        if len(self.queue) >= 2:
            raise RuntimeError("SegmentStream: two batches are already in flight; call result() first")
        i = self.next_slot
        self.next_slot ^= 1
        sl = self.slots[i]
        cur = torch.cuda.current_stream(self.device)
        with torch.cuda.device(self.device):
            # buffers are allocated (and later read by the kernels) on the caller's stream; only the copies run aside
            sl["points"] = self._fit(sl["points"], packed.points, self.device)
            sl["tarl"] = self._fit(sl["tarl"], packed.tarl if packed.use_t else None, self.device)
            sl["dino"] = self._fit(sl["dino"], packed.dino if packed.use_d else None, self.device)
            if labels is not None:
                assert labels.dtype == torch.int32 and labels.is_contiguous() and labels.numel() >= int(packed.off[-1])
                sl["labels_ext"] = labels
            else:
                sl["labels_ext"] = None
                sl["labels"] = self._fit(sl["labels"], packed.labels, self.device)
            self.copy_stream.wait_stream(cur)          # the slot's previous batch has been cut (stream order)
            with torch.cuda.stream(self.copy_stream):
                for key, src in (("points", packed.points), ("tarl", packed.tarl if packed.use_t else None),
                                 ("dino", packed.dino if packed.use_d else None)):
                    if src is not None:
                        sl[key][:src.numel()].view(src.shape).copy_(src, non_blocking=True)
                sl["ev"] = torch.cuda.Event()
                sl["ev"].record(self.copy_stream)
        self.queue.append((i, packed))

    def result(self, want_stats: bool = False) -> "SegmentResult":
        if not self.queue:
            raise RuntimeError("SegmentStream: nothing submitted")
        i, packed = self.queue.pop(0)
        sl = self.slots[i]
        total = int(packed.off[-1])
        torch.cuda.current_stream(self.device).wait_event(sl["ev"])
        dc = DeviceChunks.__new__(DeviceChunks)
        dc.packed, dc.device = packed, self.device
        dc.points = sl["points"][:packed.points.numel()].view(packed.points.shape)
        dc.tarl = sl["tarl"][:packed.tarl.numel()].view(packed.tarl.shape) if packed.use_t else None
        dc.dino = sl["dino"][:packed.dino.numel()].view(packed.dino.shape) if packed.use_d else None
        dc.labels = (sl["labels_ext"] if sl.get("labels_ext") is not None else sl["labels"])[:total]
        res = segment_packed(packed, dev_chunks=dc, want_stats=want_stats, lane=self.lane, strict=self.strict, **self.kw)
        packed.labels[:total].copy_(dc.labels, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        arr = packed.labels.numpy()
        res.labels = [arr[a:b].copy() for a, b in zip(packed.off[:-1], packed.off[1:])]
        return res


def segment_stream(batches, *, device=None, lane: int = 0, strict: bool = False, **kw):
    """Generator over `SegmentResult`s of an iterable of PackedChunks (see SegmentStream): batch k+1 uploads while batch k
    is cut.  `kw`: the parameters of `segment_packed` (alpha, theta, gamma, T, ...)."""
    ss = SegmentStream(device=device, lane=lane, strict=strict, **kw)
    it = iter(batches)
    first = next(it, None)
    if first is None:
        return
    ss.submit(first)
    for nxt in it:
        ss.submit(nxt)
        yield ss.result()
    yield ss.result()


def segment_packed_lanes(packed_lanes, dev_lanes=None, **kw):
    """Run several packed batches CONCURRENTLY on one device, one host thread + CUDA stream + library handle
    per batch ("lane").  The recursion of one batch is level-synchronous and its later levels leave most SMs
    idle (few, long-running nodes); a second batch fills them.  ctypes releases the GIL during the calls."""
    import threading
    n = len(packed_lanes)
    device = _dev(kw.pop("device", None) if dev_lanes is None else dev_lanes[0].device)
    out = [None] * n
    err = [None] * n
    streams = [torch.cuda.Stream(device=device) for _ in range(n)]
    cur = torch.cuda.current_stream(device)

    def work(i):
        try:
            with torch.cuda.device(device), torch.cuda.stream(streams[i]):
                streams[i].wait_stream(cur)
                out[i] = segment_packed(packed_lanes[i], device=device, dev_chunks=None if dev_lanes is None else dev_lanes[i],
                                        lane=i, **kw)
        except Exception as ex:          # re-raised in the caller
            err[i] = ex
    threads = [threading.Thread(target=work, args=(i,)) for i in range(n)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for s in streams:
        cur.wait_stream(s)
    for ex in err:
        if ex is not None:
            raise ex
    return out


def segment_chunks(points_list, tarl_list=None, dino_list=None, *, alpha=1.0, theta=0.0, gamma=0.0, T=0.01,
                   proximity=1.0, split_lim=0.01, device=None, want_stats=False, memory_budget=None,
                   **kw) -> SegmentResult:
    """Segment a list of chunks (host arrays in, host labels out), batched to fit device memory.  A chunk's DINOv2 input
    takes any form PackedChunks takes (several cameras: a list of per-camera arrays or an (n, cams, D) array)."""
    device = _dev(device)
    sizes = [int(np.asarray(p).shape[0]) for p in points_list]
    if memory_budget is None:
        free, _total = torch.cuda.mem_get_info(device)
        memory_budget = int(free * 0.7)
    batches = plan_batches(sizes, memory_budget, kw.get("max_steps", 0))
    labels = [None] * len(sizes)
    nseg = np.zeros(len(sizes), dtype=np.int32)
    stats_all = []
    unconv = 0
    for batch in batches:
        pk = PackedChunks([points_list[i] for i in batch],
                          [tarl_list[i] for i in batch] if tarl_list is not None else None,
                          [dino_list[i] for i in batch] if dino_list is not None else None,
                          theta=theta, gamma=gamma, pin=True, reuse=True)      # pooled pinned buffers; labels are copied out below
        res = segment_packed(pk, alpha=alpha, theta=theta, gamma=gamma, T=T, proximity=proximity,
                             split_lim=split_lim, device=device, want_stats=want_stats, **kw)
        unconv += res.unconverged
        for j, i in enumerate(batch):
            labels[i] = res.labels[j]
            nseg[i] = res.num_segments[j]
        if want_stats and res.stats is not None:
            st = res.stats.copy()
            st["chunk"] = np.asarray(batch, dtype=np.int32)[st["chunk"]]
            stats_all.append(st)
    stats = np.concatenate(stats_all) if stats_all else None
    return SegmentResult(labels=labels, num_segments=nseg, stats=stats, unconverged=unconv)


def segment_chunk(points, tarl=None, dino=None, **kw):
    """One chunk: int32 label per point (ncuts_utils.py:56-183 without the Open3D glue)."""
    res = segment_chunks([points], [tarl] if tarl is not None else None, [dino] if dino is not None else None, **kw)
    return res.labels[0]


def segment_dense(W, num_points_orig=None, *, T=0.01, split_lim=0.01, want_stats=False, max_steps=0, tol=0.0,
                  strict: bool = False):
    """normalized_cut(w, num_points_orig, labels, T, split_lim) (normalized_cut.py:37) for a dense float32
    copy of w on the device.  Returns int32 labels (numpy), and stats if requested."""
    W, ld = _matrix_args(W)
    device = W.device
    hd = Handle.get(device)
    n = W.shape[0]
    p = make_params(T=T, split_lim=split_lim, max_steps=max_steps, tol=tol)
    labels = torch.empty(n, dtype=torch.int32, device=device)
    nseg = np.zeros(1, dtype=np.int32)
    cap = 4096 if want_stats else 0
    stats = np.zeros(max(cap, 1), dtype=_STAT_DTYPE)
    nstats = C.c_int32(0)
    with torch.cuda.device(device):
        check(hd.lib.ancuts_segment_dense_f32(
            hd.h, n, _ptr(W), ld, int(num_points_orig if num_points_orig is not None else n), C.byref(p), _ptr(labels),
            nseg.ctypes.data_as(C.POINTER(C.c_int32)), stats.ctypes.data_as(C.POINTER(NodeStat)) if want_stats else None,
            cap, C.byref(nstats), _stream(device)))
    _report_unconverged(hd, strict)
    out = labels.cpu().numpy()
    return (out, stats[:nstats.value].copy()) if want_stats else out


# ------------------------------------------------------------------------------------------------
# caller-supplied sparse affinity graphs (ancuts_segment_csr_f32)
# ------------------------------------------------------------------------------------------------
@dataclass
class PackedGraphs:
    """A batch of graphs as one CSR: global int64 row pointers (P + 1), int32 columns local to each graph, float32 values."""
    sizes: list
    off: np.ndarray         # int64 [B + 1] first row of every graph
    row_ptr: torch.Tensor
    col: torch.Tensor
    val: torch.Tensor

    @property
    def nnz(self) -> int:
        return int(self.col.numel())

    def to(self, device) -> "PackedGraphs":
        return PackedGraphs(self.sizes, self.off, self.row_ptr.to(device), self.col.to(device), self.val.to(device))


def _graph_shape(g):
    shape = tuple(int(s) for s in g.shape)
    if len(shape) != 2 or shape[0] != shape[1]:
        raise ValueError(f"a graph must be a square matrix, got shape {shape}")
    if shape[0] == 0:
        raise ValueError("a graph must have at least one point")
    return shape[0]


def pack_graphs(graphs) -> PackedGraphs:
    """Concatenate sparse affinity graphs into the CSR layout of ancuts_segment_csr_f32; needs no GPU.

    scipy sparse input is made canonical the way `toarray()` reads it: duplicates are summed in the input dtype, then the
    values are rounded to float32 (what `toarray().astype(np.float32)` holds); explicit zeros stay (a stored 0 is no edge).
    torch sparse-CSR input is taken as it is (the library validates it) and stays on its device: the row pointers are offset
    and the columns narrowed there, without a round trip through the host.  Non-square and empty graphs raise ValueError."""
    graphs = list(graphs)
    if not graphs:
        raise ValueError("no graphs")
    sizes = [_graph_shape(g) for g in graphs]
    parts = []
    dev = None
    for g in graphs:
        if isinstance(g, torch.Tensor):
            if g.layout != torch.sparse_csr:
                raise TypeError("torch graphs must be sparse-CSR tensors (Tensor.to_sparse_csr())")
            if g.is_cuda:
                dev = dev or g.device
            parts.append((g.crow_indices().to(torch.int64), g.col_indices().to(torch.int32), g.values().to(torch.float32)))
        elif hasattr(g, "tocsr"):
            m = g.tocsr(copy=True)
            m.sum_duplicates()
            parts.append((torch.from_numpy(np.asarray(m.indptr, dtype=np.int64)),
                          torch.from_numpy(np.asarray(m.indices, dtype=np.int32)),
                          torch.from_numpy(np.asarray(m.data).astype(np.float32))))
        else:
            raise TypeError("graphs must be scipy sparse matrices or torch sparse-CSR tensors")
    dev = dev or torch.device("cpu")
    rows, cols, vals = [], [], []
    e0 = 0
    for rp, cl, vl in parts:
        rp, cl, vl = rp.to(dev), cl.to(dev), vl.to(dev)
        rows.append(rp[:-1] + e0)
        cols.append(cl)
        vals.append(vl)
        e0 += int(cl.numel())
    rows.append(torch.full((1,), e0, dtype=torch.int64, device=dev))
    off = np.zeros(len(sizes) + 1, dtype=np.int64)
    off[1:] = np.cumsum(sizes)
    return PackedGraphs(sizes, off, torch.cat(rows).contiguous(), torch.cat(cols).contiguous(), torch.cat(vals).contiguous())


def _run_graphs(hd, pk: PackedGraphs, norig, p, want_stats, device):
    B = len(pk.sizes)
    off = np.ascontiguousarray(pk.off, dtype=np.int64)
    nseg = np.zeros(B, dtype=np.int32)
    cap = 128 * B + 64 if want_stats else 0
    stats = np.zeros(max(cap, 1), dtype=_STAT_DTYPE)
    nstats = C.c_int32(0)
    labels = torch.empty(int(off[-1]), dtype=torch.int32, device=device)
    no = None if norig is None else np.ascontiguousarray(norig, dtype=np.int32)
    with torch.cuda.device(device):
        check(hd.lib.ancuts_segment_csr_f32(
            hd.h, B, off.ctypes.data_as(C.POINTER(C.c_int64)), _ptr(pk.row_ptr), _ptr(pk.col), _ptr(pk.val), pk.nnz,
            no.ctypes.data_as(C.POINTER(C.c_int32)) if no is not None else None, C.byref(p), _ptr(labels),
            nseg.ctypes.data_as(C.POINTER(C.c_int32)), stats.ctypes.data_as(C.POINTER(NodeStat)) if want_stats else None,
            cap, C.byref(nstats), _stream(device)))
    arr = labels.cpu().numpy()
    return [arr[a:b].copy() for a, b in zip(off[:-1], off[1:])], nseg, (stats[:nstats.value].copy() if want_stats else None)


def segment_graphs(graphs, *, num_points_orig=None, T=0.01, split_lim=0.01, device=None, want_stats=False, max_steps=0,
                   tol=0.0, strict: bool = False, memory_budget=None, lane: int = 0) -> SegmentResult:
    """normalized_cut(w, num_points_orig, labels, T, split_lim) (normalized_cut.py:37-63) for a list of sparse affinity
    graphs (scipy sparse matrices or torch sparse-CSR tensors, host or device), batched to fit device memory like
    `segment_chunks`.  Every graph must be symmetric with a unit diagonal (stored diagonal entries exactly 1, absent ones
    taken as 1) and finite; a violation raises naming the graph and the row.  The labels equal `segment_dense` on the
    densified graph.  num_points_orig: None (each graph's own size), one int for all graphs, or one per graph."""
    device = _dev(device)
    hd = Handle.get(device, lane)
    graphs = list(graphs)
    sizes = [_graph_shape(g) for g in graphs]
    if num_points_orig is None:
        norig = None
    elif np.ndim(num_points_orig) == 0:
        norig = [int(num_points_orig)] * len(graphs)
    else:
        norig = [int(x) for x in num_points_orig]
        if len(norig) != len(graphs):
            raise ValueError("num_points_orig needs one value per graph")
    if memory_budget is None:
        free, _total = torch.cuda.mem_get_info(device)
        memory_budget = int(free * 0.7)
    p = make_params(T=T, split_lim=split_lim, max_steps=max_steps, tol=tol)
    labels = [None] * len(sizes)
    nseg = np.zeros(len(sizes), dtype=np.int32)
    stats_all = []
    unconv = 0
    for batch in plan_batches(sizes, memory_budget, max_steps):
        pk = pack_graphs([graphs[i] for i in batch]).to(device)
        lab, ns, st = _run_graphs(hd, pk, None if norig is None else [norig[i] for i in batch], p, want_stats, device)
        unconv += _report_unconverged(hd, strict)
        for j, i in enumerate(batch):
            labels[i] = lab[j]
            nseg[i] = ns[j]
        if want_stats and st is not None:
            st = st.copy()
            st["chunk"] = np.asarray(batch, dtype=np.int32)[st["chunk"]]
            stats_all.append(st)
    stats = np.concatenate(stats_all) if stats_all else None
    return SegmentResult(labels=labels, num_segments=nseg, stats=stats, unconverged=unconv)
