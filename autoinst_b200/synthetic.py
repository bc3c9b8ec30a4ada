"""Synthetic SemanticKITTI-shaped chunks and maps (SURVEY.md §8d).

The reference never ships data; its hot loop (`pipeline/run_pipeline.py:160-195`) consumes
25 m map chunks voxelised at 0.35 m (`pipeline/config.py:55-57`, `dataset_utils.py:534`).
This module fabricates inputs of that shape, seeded and deterministic, for the parity tests and
for `bench.py`.  numpy/scipy only: it runs on the GPU box as well as in the build container.

Nothing here is on the product compute path; it only makes inputs.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np
from scipy.spatial import cKDTree
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components

MAJOR_VOXEL = 0.35          # config.py:56
CHUNK_EDGE = 25.0           # config.py:57
PROXIMITY = 1.0             # config.py:65

# gains / thresholds exactly as config.py:6-37
CONFIGS = {
    "spatial": dict(alpha=1.0, theta=0.0, gamma=0.0, beta=0.0, T=0.075),
    "tarl_spatial": dict(alpha=1.0, theta=0.5, gamma=0.0, beta=0.0, T=0.03),
    "tarl_spatial_dino": dict(alpha=1.0, theta=0.5, gamma=0.1, beta=0.0, T=0.005),
}


@dataclass
class Chunk:
    """One chunk at the 0.35 m ("major") resolution, the N points NCuts sees."""
    chunk_id: int
    points: np.ndarray                  # (N,3) float64, float32-representable
    instance: np.ndarray                # (N,) int32 ground-truth instance id (>=1)
    tarl: np.ndarray | None = None      # (N,96) float64 from float32, 5 % zero rows
    dino: np.ndarray | list | None = None   # (N,384) float64 from float32, 30 % zero rows ("dino2": one per camera)
    center: np.ndarray = field(default_factory=lambda: np.zeros(3))

    @property
    def n(self) -> int:
        return int(self.points.shape[0])


def voxel_centroid_downsample(points: np.ndarray, voxel: float, payload: np.ndarray | None = None):
    """Centroid per occupied voxel, like Open3D `voxel_down_sample` used at
    `dataset_utils.py:534`.  Returns centroids (and the payload of the first point per voxel)."""
    origin = points.min(axis=0) - 0.5 * voxel
    key = np.floor((points - origin) / voxel).astype(np.int64)
    _, inv, cnt = np.unique(key, axis=0, return_inverse=True, return_counts=True)
    inv = inv.reshape(-1)
    cent = np.zeros((cnt.shape[0], 3))
    np.add.at(cent, inv, points)
    cent /= cnt[:, None]
    if payload is None:
        return cent
    first = np.full(cnt.shape[0], -1, dtype=np.int64)
    order = np.arange(points.shape[0])[::-1]
    first[inv[order]] = order           # smallest source index wins
    return cent, payload[first]


def _box_surface(rng, size, n):
    """n points on the faces of an axis-aligned box of the given size, centred at 0."""
    sx, sy, sz = size
    areas = np.array([sy * sz, sy * sz, sx * sz, sx * sz, sx * sy, sx * sy])
    face = rng.choice(6, size=n, p=areas / areas.sum())
    u = rng.uniform(-0.5, 0.5, size=(n, 3)) * np.array(size)
    axis = face // 2
    sign = np.where(face % 2 == 0, -0.5, 0.5)
    u[np.arange(n), axis] = sign * np.array(size)[axis]
    return u


def _rotz(rng):
    a = rng.uniform(0, 2 * np.pi)
    c, s = np.cos(a), np.sin(a)
    return np.array([[c, -s, 0], [s, c, 0], [0, 0, 1.0]])


def _make_object(rng, kind):
    n = int(rng.integers(3000, 8000))
    if kind == "facade":
        w, h = rng.uniform(10, 25), rng.uniform(4, 8)
        p = np.stack([rng.uniform(-w / 2, w / 2, n), rng.normal(0, 0.03, n),
                      rng.uniform(0, h, n)], axis=1)
    elif kind == "car":
        p = _box_surface(rng, (4.0, 1.8, 1.5), n) + np.array([0, 0, 0.75])
    elif kind == "pole":
        p = _box_surface(rng, (0.3, 0.3, 6.0), n) + np.array([0, 0, 3.0])
    else:  # vegetation blob
        p = rng.normal(0, 1.0, size=(n, 3)) * np.array([0.65, 0.65, 0.55]) + np.array([0, 0, 1.5])
    return p @ _rotz(rng).T


def _components(points, radius):
    tree = cKDTree(points)
    pairs = tree.query_pairs(radius, output_type="ndarray")
    n = points.shape[0]
    g = coo_matrix((np.ones(len(pairs)), (pairs[:, 0], pairs[:, 1])), shape=(n, n))
    return connected_components(g, directed=False)


def _aabb_gap(lo_a, hi_a, lo_b, hi_b):
    """Euclidean distance between two axis-aligned boxes (0 if they intersect)."""
    d = np.maximum(0.0, np.maximum(lo_a - hi_b, lo_b - hi_a))
    return float(np.sqrt((d * d).sum()))


def make_chunk(chunk_id: int = 0, n_target: int = 8192, features: str = "tarl_dino",
               clutter: int = 0, min_component_frac: float = 0.0125, attach_prob: float = 0.25,
               center=(0.0, 0.0, 0.0), seed_base: int = 1234) -> Chunk:
    """Seeded chunk with about `n_target` major points (SURVEY.md §8d).

    Objects are dropped into the 25 m cube with their (inflated) bounding boxes kept apart, except
    that a fraction `attach_prob` is parked 0.5–0.9 m from an earlier object so the proximity
    graph gets weak links that NCuts has to cut.
    clutter == 0: every connected component of the 1 m proximity graph holds more than
    `min_component_frac`·N points, so the reference's 1 % `split_lim` rule
    (`normalized_cut.py:39-40`) never meets a disconnected leaf and the unpinned reference agrees
    with itself (SURVEY.md §7.3 item 1).  clutter > 0 adds that many 2–12 voxel fragments.
    """
    rng = np.random.default_rng(seed_base + chunk_id)
    half = CHUNK_EDGE / 2
    kinds = ["facade", "car", "car", "veg", "car", "veg", "pole", "car"]
    per_kind = {"facade": 900.0, "car": 285.0, "veg": 520.0, "pole": 72.0}   # mean major voxels
    pts, inst, boxes = [], [], []
    total_est, o = 0.0, 0
    while total_est < 0.85 * n_target and o < 4096:
        kind = kinds[o % len(kinds)]
        o += 1
        p = _make_object(rng, kind)
        lo0, hi0 = p.min(0), p.max(0)
        placed = False
        attach = bool(boxes) and rng.random() < attach_prob
        for _ in range(60):
            if attach:
                hl, hh = boxes[int(rng.integers(len(boxes)))]
                ax = int(rng.integers(2))
                gap = rng.uniform(0.5, 0.9)
                shift = np.zeros(3)
                side = rng.random() < 0.5
                shift[ax] = (hh[ax] + gap - lo0[ax]) if side else (hl[ax] - gap - hi0[ax])
                oa = 1 - ax
                a, b = hl[oa] - hi0[oa] + 0.5, hh[oa] - lo0[oa] - 0.5
                shift[oa] = rng.uniform(min(a, b), max(a, b))
                shift[2] = hl[2] - lo0[2]
            else:
                shift = rng.uniform(-half + 0.5, half - 0.5, size=3) - (lo0 + hi0) / 2
                shift[2] = rng.uniform(-half + 0.3, half - 0.3 - (hi0[2] - lo0[2])) - lo0[2]
            lo, hi = lo0 + shift, hi0 + shift
            if np.any(lo < -half) or np.any(hi > half):
                continue
            gaps = [_aabb_gap(lo, hi, bl, bh) for bl, bh in boxes]
            if attach:
                ok = sum(g < 1.3 for g in gaps) == 1 and min(gaps) >= 0.45
            else:
                ok = all(g > 1.3 for g in gaps)
            if ok:
                placed = True
                break
        if not placed:
            continue
        boxes.append((lo, hi))
        pts.append(p + shift)
        inst.append(np.full(p.shape[0], len(boxes), dtype=np.int32))
        total_est += per_kind[kind]
    pts = np.concatenate(pts)
    inst = np.concatenate(inst)
    pm, im = voxel_centroid_downsample(pts, MAJOR_VOXEL, inst)

    if clutter == 0:
        while True:                                            # drop small components
            ncomp, lab = _components(pm, PROXIMITY)
            size = np.bincount(lab, minlength=ncomp)
            keep = size[lab] > min_component_frac * pm.shape[0]
            if keep.all():
                break
            pm, im = pm[keep], im[keep]
    else:
        frag_pts, frag_inst = [], []
        next_id = int(im.max()) + 1
        for f in range(clutter):
            k = int(rng.integers(2, 13))
            c = rng.uniform(-half + 1, half - 1, size=3)
            q = c + rng.uniform(-0.5, 0.5, size=(k, 3))
            frag_pts.append(q)
            frag_inst.append(np.full(k, next_id + f, dtype=np.int32))
        pm = np.concatenate([pm] + frag_pts)
        im = np.concatenate([im] + frag_inst)

    # shuffle so that index order carries no spatial structure (Open3D's voxel hash order is arbitrary)
    perm = rng.permutation(pm.shape[0])
    pm, im = pm[perm], im[perm]
    # float32-representable coordinates, stored as float64 (the oracle reads float64)
    pm = (pm + np.asarray(center, dtype=np.float64)).astype(np.float32).astype(np.float64)
    ch = Chunk(chunk_id=chunk_id, points=pm, instance=im, center=np.asarray(center, dtype=np.float64))
    n = ch.n
    n_inst = int(im.max()) + 1
    if "tarl" in features:
        proto = rng.normal(0, 1, size=(n_inst, 96))
        t = (proto[im] + 0.3 * rng.normal(0, 1, size=(n, 96))).astype(np.float32)
        t[rng.random(n) < 0.05] = 0.0                          # no scan point within 0.175 m
        ch.tarl = t.astype(np.float64)
    if "dino" in features:
        proto = rng.normal(0, 1, size=(n_inst, 384))
        g = (proto[im] + 0.3 * rng.normal(0, 1, size=(n, 384))).astype(np.float32)
        g[rng.random(n) < 0.30] = 0.0                          # never visible in camera 0
        ch.dino = g.astype(np.float64)
        if "dino2" in features:
            # a second camera (CAM_IDS = [0, 1]): same prototypes, its own noise and unseen rows; drawn after every other
            # draw, so that the other feature strings keep their chunks byte for byte.  ch.dino = [camera 0, camera 1]
            g2 = (proto[im] + 0.3 * rng.normal(0, 1, size=(n, 384))).astype(np.float32)
            g2[rng.random(n) < 0.30] = 0.0
            ch.dino = [ch.dino, g2.astype(np.float64)]
    return ch


def make_map(n_chunks: int = 8, n_per_chunk=4096, features: str = "tarl", seed: int = 77,
             background_facades: bool = True, attach_prob: float = 0.4, feature_noise: float = 0.5) -> list[Chunk]:
    """Synthetic "first map": ONE scene along a straight 25 m wide corridor, voxelised once at 0.35 m, then
    cut into 25 m cubes every 22 m (`chunk_generation.py:123-137`, OVERLAP = 3 m, `config.py:58`), so that
    neighbouring chunks share instances and, in the 3 m overlap, exactly the same points — what the
    reference's merge relies on (`point_cloud_utils.py:387-491`).
    `n_per_chunk`: target major points per chunk, or a (lo, hi) pair: the object density then varies along the
    corridor so that the chunk sizes spread over about [lo, hi] (BASELINE.json config 4: N in [3 k, 12 k]).
    Facades are "stuff": their GT instance id is 0 (background) when background_facades is set, like
    buildings in SemanticKITTI; they exercise `remove_semantics`.
    Chunk.instance holds the map-level GT instance id (0 = background)."""
    rng = np.random.default_rng(seed)
    half = CHUNK_EDGE / 2
    length = 22.0 * (n_chunks - 1) + CHUNK_EDGE
    kinds = ["facade", "car", "car", "veg", "car", "veg", "car", "car"]
    per_kind = {"facade": 900.0, "car": 285.0, "veg": 520.0}
    varying = isinstance(n_per_chunk, (tuple, list))
    if varying:
        n_lo, n_hi = float(n_per_chunk[0]), float(n_per_chunk[1])
        want = rng.uniform(n_lo, n_hi, size=n_chunks)               # target size of every chunk
        edges = np.concatenate(([0.0], 22.0 * np.arange(1, n_chunks), [length]))
        mass = want / CHUNK_EDGE * np.diff(edges)                   # expected points per 22 m stride cell
        n_per_chunk = n_lo
    else:
        edges = np.array([0.0, length])
        mass = np.array([n_per_chunk * length / CHUNK_EDGE])
    target = float(mass.sum())
    cell_p = mass / mass.sum()

    def draw_x():
        if not varying:
            return rng.uniform(0.5, length - 0.5)                   # (same random stream as the committed fixtures)
        c = int(rng.choice(len(cell_p), p=cell_p))
        return rng.uniform(max(edges[c], 0.5), min(edges[c + 1], length - 0.5))
    pts, inst, boxes, is_bg, obj_kind = [], [], [], [], []
    total, o = 0.0, 0
    while total < 0.9 * target and o < 100000:
        kind = kinds[o % len(kinds)]
        o += 1
        p = _make_object(rng, kind)
        lo0, hi0 = p.min(0), p.max(0)
        attach = bool(boxes) and rng.random() < attach_prob
        for _ in range(40):
            if attach:                                  # parked 0.5-0.9 m from an earlier object: a weak link to cut
                hl, hh = boxes[int(rng.integers(len(boxes)))]
                ax = int(rng.integers(2))
                gap = rng.uniform(0.5, 0.9)
                shift = np.zeros(3)
                shift[ax] = (hh[ax] + gap - lo0[ax]) if rng.random() < 0.5 else (hl[ax] - gap - hi0[ax])
                oa = 1 - ax
                a_, b_ = hl[oa] - hi0[oa] + 0.5, hh[oa] - lo0[oa] - 0.5
                shift[oa] = rng.uniform(min(a_, b_), max(a_, b_))
                shift[2] = hl[2] - lo0[2]
            else:
                shift = np.array([draw_x(), rng.uniform(-half + 0.5, half - 0.5),
                                  rng.uniform(-half + 0.3, half - 0.3)]) - (lo0 + hi0) / 2
                shift[2] = rng.uniform(-half + 0.3, half - 0.3 - (hi0[2] - lo0[2])) - lo0[2]
            lo, hi = lo0 + shift, hi0 + shift
            if lo[0] < 0 or hi[0] > length or lo[1] < -half or hi[1] > half or lo[2] < -half or hi[2] > half:
                continue
            gaps = [_aabb_gap(lo, hi, bl, bh) for bl, bh in boxes]
            if (attach and sum(g < 1.3 for g in gaps) == 1 and min(gaps) >= 0.45) or \
                    (not attach and all(g > 1.3 for g in gaps)):
                boxes.append((lo, hi))
                pts.append(p + shift)
                inst.append(np.full(p.shape[0], len(boxes), dtype=np.int32))
                is_bg.append(kind == "facade" and background_facades)
                obj_kind.append(kind)
                total += per_kind[kind]
                break
    pts = np.concatenate(pts)
    inst = np.concatenate(inst)
    pm, im = voxel_centroid_downsample(pts, MAJOR_VOXEL, inst)
    while True:                                                 # every component well above the 1 % size limit
        ncomp, lab = _components(pm, PROXIMITY)
        size = np.bincount(lab, minlength=ncomp)
        keep = size[lab] > 0.03 * n_per_chunk
        if keep.all():
            break
        pm, im = pm[keep], im[keep]
    pm = pm.astype(np.float32).astype(np.float64)
    gt = im.copy()
    for k, bg in enumerate(is_bg):
        if bg:
            gt[im == k + 1] = 0
    n_inst = int(im.max()) + 1
    # TARL-like features are class-driven: a prototype per object kind plus a smaller per-instance offset, so that
    # neighbouring objects of one kind are hard to tell apart (the metrics are not trivially perfect)
    kind_proto = {k: rng.normal(0, 1, size=96) for k in ("facade", "car", "veg")}
    proto_t = np.zeros((n_inst, 96))
    for k, kd in enumerate(obj_kind):
        proto_t[k + 1] = kind_proto[kd] + 0.35 * rng.normal(0, 1, size=96)
    tarl_all = (proto_t[im] + feature_noise * rng.normal(0, 1, size=(pm.shape[0], 96))).astype(np.float32)
    tarl_all[rng.random(pm.shape[0]) < 0.05] = 0.0
    dino_all = None
    if "dino" in features:
        proto_d = rng.normal(0, 1, size=(n_inst, 384))
        dino_all = (proto_d[im] + 0.3 * rng.normal(0, 1, size=(pm.shape[0], 384))).astype(np.float32)
        dino_all[rng.random(pm.shape[0]) < 0.30] = 0.0
    chunks = []
    for c in range(n_chunks):
        cx = half + 22.0 * c
        sel = np.where((pm[:, 0] > cx - half) & (pm[:, 0] < cx + half))[0]      # strictly inside (:131-137)
        while True:                                             # objects sliced by the cube faces leave fragments:
            ncomp, lab = _components(pm[sel], PROXIMITY)        # keep the chunk free of components near the 1 % limit
            size = np.bincount(lab, minlength=ncomp)
            keep = size[lab] > 0.02 * sel.shape[0]
            if keep.all():
                break
            sel = sel[keep]
        sel = sel[rng.permutation(sel.shape[0])]
        ch = Chunk(chunk_id=c, points=pm[sel], instance=gt[sel], center=np.array([cx, 0.0, 0.0]))
        ch.tarl = tarl_all[sel].astype(np.float64) if "tarl" in features else None
        ch.dino = dino_all[sel].astype(np.float64) if dino_all is not None else None
        chunks.append(ch)
    return chunks


def small_chunk(seed: int, n_obj: int = 4, pts_per_obj: int = 400, features: str = "tarl_dino"):
    """Small chunk (N in the hundreds) of box-surface objects: golden fixtures and smoke tests."""
    rng = np.random.default_rng(seed)
    pts, inst = [], []
    for o in range(n_obj):
        size = rng.uniform([0.8, 0.8, 0.6], [4.0, 4.0, 2.5])
        p = _box_surface(rng, size, pts_per_obj) @ _rotz(rng).T + rng.uniform(-4.5, 4.5, size=3)
        pts.append(p)
        inst.append(np.full(pts_per_obj, o + 1, dtype=np.int32))
    pm, im = voxel_centroid_downsample(np.concatenate(pts), MAJOR_VOXEL, np.concatenate(inst))
    pm = pm.astype(np.float32).astype(np.float64)
    ch = Chunk(chunk_id=seed, points=pm, instance=im)
    n, n_inst = ch.n, int(im.max()) + 1
    if "tarl" in features:
        t = (rng.normal(0, 1, (n_inst, 96))[im] + 0.3 * rng.normal(0, 1, (n, 96))).astype(np.float32)
        t[rng.random(n) < 0.05] = 0.0
        ch.tarl = t.astype(np.float64)
    if "dino" in features:
        g = (rng.normal(0, 1, (n_inst, 384))[im] + 0.3 * rng.normal(0, 1, (n, 384))).astype(np.float32)
        g[rng.random(n) < 0.30] = 0.0
        ch.dino = g.astype(np.float64)
    return ch


def make_scans(chunk: Chunk, n_scans: int = 21, pts_per_major: float = 3.0, seed: int = 0, fdim: int = 96,
               outside_frac: float = 0.15, empty_frac: float = 0.05):
    """Synthetic per-scan TARL inputs of one chunk for the feature-pooling row (SURVEY.md §8f N3;
    `chunk_generation.py:205-258`): `n_scans` scans (ADJACENT_FRAMES_TARL = (10, 10) -> 21, config.py:69), each a list
    entry (coords (m,3) float64 already in the chunk frame, feats (m,fdim) float32).  Scan points are the
    major points jittered by up to 0.3 m (so some fall outside the 0.175 m radius), `empty_frac` of the major
    points get no scan point at all (zero TARL rows, `:255-256`), and `outside_frac` extra points lie outside
    the 25 m cube (cropped away, `:233-236`).  Features = instance prototype + noise, float32."""
    rng = np.random.default_rng(9000 + 131 * chunk.chunk_id + seed)
    n = chunk.n
    n_inst = int(chunk.instance.max()) + 1
    proto = rng.normal(0, 1, size=(n_inst, fdim))
    covered = rng.random(n) >= empty_frac
    src = np.flatnonzero(covered)
    half = CHUNK_EDGE / 2
    scans = []
    per_scan = max(1, int(round(n * pts_per_major)))
    for s in range(n_scans):
        pick = src[rng.integers(0, src.shape[0], size=per_scan)]
        p = chunk.points[pick] + rng.uniform(-0.3, 0.3, size=(per_scan, 3)) * rng.random((per_scan, 1))
        f = (proto[chunk.instance[pick]] + 0.3 * rng.normal(0, 1, size=(per_scan, fdim))).astype(np.float32)
        n_out = int(per_scan * outside_frac)
        po = chunk.center + rng.uniform(half, half + 5.0, size=(n_out, 3)) * rng.choice([-1.0, 1.0], size=(n_out, 3))
        fo = rng.normal(0, 1, size=(n_out, fdim)).astype(np.float32)
        order = rng.permutation(per_scan + n_out)
        scans.append((np.concatenate((p, po))[order], np.concatenate((f, fo))[order]))
    return scans


def make_camera_scene(seed: int = 31, n_views: int = 5, minor_per_major: int = 6, visible_frac: float = 0.10,
                      map_hw=(7, 23), fdim: int = 384):
    """Synthetic inputs of the DINOv2 half of the feature row (SURVEY.md §8f N3; `image_utils.py:91-371`): a small chunk
    ~12 m in front of a forward-moving KITTI-like camera, a 5 cm "minor" map cloud (jittered copies of the major points
    plus points elsewhere in the map), per-view visibility masks over the map cloud (what hidden point removal would
    give; view 3 sees nothing), poses, calibration and random feature maps with 15 % feature-less pixels.
    Returns a dict of plain arrays and a `dataset` object with the getters the reference calls."""
    rng = np.random.default_rng(seed)
    ch = small_chunk(seed + 2, n_obj=3, pts_per_obj=260, features="tarl")
    major = ch.points + np.array([12.0, 0.0, 0.0])
    n = major.shape[0]
    minor_chunk = np.repeat(major, minor_per_major, axis=0) + rng.uniform(-0.12, 0.12, size=(minor_per_major * n, 3))
    elsewhere = rng.uniform([-30, -30, -2], [-10, 30, 4], size=(400, 3))
    pcd_pts = np.concatenate([elsewhere[:200], minor_chunk, elsewhere[200:]])
    chunk_indices = np.arange(200, 200 + minor_chunk.shape[0])

    def pose(i):                                               # lidar pose of frame i in the world (x forward, z up)
        a = 0.06 * i
        T = np.eye(4)
        T[:3, :3] = [[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]]
        T[:3, 3] = [1.2 * i, 0.15 * i, 0.0]
        return T
    T_lidar2cam = np.array([[0.0, -1.0, 0.0, 0.05], [0.0, 0.0, -1.0, -0.08], [1.0, 0.0, 0.0, -0.27], [0, 0, 0, 1.0]])
    K = np.array([[718.856, 0.0, 607.1928], [0.0, 718.856, 185.2157], [0.0, 0.0, 1.0]])
    img_w, img_h = 1241, 376
    fmaps = []
    for _ in range(n_views):
        f = rng.normal(size=(map_hw[0], map_hw[1], fdim)).astype(np.float32)
        f[rng.random(map_hw) < 0.15] = 0.0
        fmaps.append(f)
    hpr_masks = rng.random((n_views, pcd_pts.shape[0])) < visible_frac
    if n_views > 3:
        hpr_masks[3] = False

    class Image:
        size = (img_w, img_h)

    class Dataset:
        def get_image(self, cam, i): return Image()
        def get_pose(self, i): return pose(i)
        def get_calibration_matrices(self, cam): return T_lidar2cam, K
        def get_dinov2_features(self, cam, i): return fmaps[i]
    return dict(major=major, pcd_points=pcd_pts, chunk_indices=chunk_indices, T_pcd2world=np.eye(4), cam_indices=list(range(n_views)),
                hpr_masks=hpr_masks, K=K, T_lidar2cam=T_lidar2cam, img_hw=(img_h, img_w), feature_maps=fmaps, pose=pose,
                dataset=Dataset())
