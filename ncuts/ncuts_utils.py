"""`ncuts_chunk` / `get_merge_pcds` with the reference's signatures (`pipeline/ncuts/ncuts_utils.py:28,207`).

The affinity build and the recursive cut (`ncuts_utils.py:56-174`) run on the GPU through
`autoinst_b200.api` (C ABI: `ancuts_segment_chunks_host`).  Everything around them — feature
fetching from the dataset, colour coding, ground handling — stays the reference's own helper code under
`utils/` (the TARL radius-mean pooling and the 1-NN re-projection to the 5 cm cloud also run on the GPU,
`ancuts_feature_pool` / `ancuts_nn_reproject`), imported lazily so that this module also
loads where Open3D is absent (the array-level entry `segment_major_points` needs none of it).

Configuration is read the way the reference reads it: module globals star-imported from `config`
(`ncuts_utils.py:25`); tests switch configs by assigning `ncuts.ncuts_utils.CONFIG`.
"""
import os

import numpy as np

import warnings

try:                                            # cwd = pipeline/ in the reference layout (config.py:79)
    from config import *                        # noqa: F401,F403  CONFIG, PROXIMITY_THRESHOLD, SPLIT_LIM, ...
except ModuleNotFoundError as _e:               # stand-alone use ONLY (no `config` module at all): the shipped defaults
    if _e.name != "config":                     # (config.py:17-26,55-73); a config.py that fails for any other reason
        raise                                   # (e.g. wrong cwd for its yaml, config.py:79) must not be papered over
    warnings.warn("ncuts.ncuts_utils: no `config` module on sys.path; using the shipped config_tarl_spatial defaults",
                  RuntimeWarning)
    CONFIG = {"name": "spatial_1.0_tarl_0.5_t_0.03", "out_folder": "ncuts_data_tarl_spatial/", "gamma": 0.0,
              "alpha": 1.0, "theta": 0.5, "beta": 0.0, "T": 0.03, "gt": True}
    PROXIMITY_THRESHOLD = 1.0
    SPLIT_LIM = 0.01
    MEAN_HEIGHT = 0.6
    ADJACENT_FRAMES_CAM = (16, 13)
    ADJACENT_FRAMES_TARL = (10, 10)


def segment_major_points(points_major, tarl_features=None, dino_features=None, config=None,
                         proximity=None, split_lim=None, return_labels=False):
    """Array-level core of `ncuts_chunk`: N x 3 points (+ N x 96 TARL, + per-camera N x 384 DINOv2 means)
    -> the `grouped_labels` list the reference gets from `normalized_cut` (`ncuts_utils.py:168-174`)."""
    from autoinst_b200 import api
    cfg = CONFIG if config is None else config
    if cfg.get("beta"):
        raise NotImplementedError("beta != 0 (SAM label term, ncuts_utils.py:115-123) is not supported")
    dino = None
    if cfg["gamma"]:
        cams = dino_features if isinstance(dino_features, (list, tuple)) else ([dino_features] if dino_features is not None else [])
        if len(cams) == 0:
            raise ValueError("The length should be longer than 0!")          # ncuts_utils.py:126-127
        dino = list(cams)                    # one term per camera (CAM_IDS), multiplied as at ncuts_utils.py:129-133
    if cfg["theta"] and tarl_features is None:
        raise ValueError("theta != 0 needs TARL features")
    seg = api.segment_chunk(points_major, tarl_features if cfg["theta"] else None, dino,
                            alpha=cfg["alpha"], theta=cfg["theta"], gamma=cfg["gamma"], T=cfg["T"],
                            proximity=PROXIMITY_THRESHOLD if proximity is None else proximity,
                            split_lim=SPLIT_LIM if split_lim is None else split_lim,
                            strict=True)        # non-convergence raises, as the reference's eigsh would
    if return_labels:
        return seg
    order = np.argsort(seg, kind="stable")
    return np.split(order, np.flatnonzero(np.diff(seg[order])) + 1)


def ncuts_chunk(dataset, chunk_downsample_dict, pcd_nonground_minor, T_pcd, sampled_indices_global,
                sequence=None, patchwise_indices=None):
    """Same contract as the reference (`ncuts_utils.py:28-204`): returns
    (merged_chunk, pcd_chunk, cut_hight, inst_ground, seg_ground)."""
    import open3d as o3d
    from utils.point_cloud.point_cloud_utils import get_subpcd, get_statistical_inlier_indices
    from autoinst_b200 import api
    from utils.visualization_utils import generate_random_colors
    from autoinst_b200.dino import dinov2_mean_per_patch          # per-view look-up and mean on the GPU (ancuts_dino_*)
    from utils.point_cloud.chunk_generation import get_indices_feature_reprojection
    from autoinst_b200.pooling import tarl_features_per_patch      # radius-mean pooling on the GPU (ancuts_feature_pool)

    d = chunk_downsample_dict
    print("Start of sequence", sequence)
    center_id = d["center_ids"][sequence]
    cam_ids, _ = get_indices_feature_reprojection(sampled_indices_global, patchwise_indices[sequence][0],
                                                  adjacent_frames=ADJACENT_FRAMES_CAM)
    tarl_ids, _ = get_indices_feature_reprojection(sampled_indices_global, center_id,
                                                   adjacent_frames=ADJACENT_FRAMES_TARL)
    pcd_chunk = d["pcd_nonground_chunks"][sequence]
    ground = d["pcd_ground_chunks"][sequence]
    major = d["pcd_nonground_chunks_major_downsampling"][sequence]
    pts = np.asarray(major.points)
    print(pts.shape[0], "points in downsampled chunk (major)")

    # feature producers stay the reference's (out of scope, SURVEY.md §2 rows 4-5)
    dino_list = None
    if CONFIG["gamma"]:
        # image_based_features_per_patch(..., sam=False, dino=True) + dinov2_mean per camera (ncuts_utils.py:81-110)
        dino_list = dinov2_mean_per_patch(dataset, pcd_nonground_minor, d["indices"][sequence], major, T_pcd, cam_ids)
    tarl = None
    if CONFIG["theta"]:
        tarl = tarl_features_per_patch(dataset, major, T_pcd, d["center_positions"][sequence], tarl_ids)

    # remove_isolated_points (ncuts_utils.py:159) never drops anything: A_ii = 1 (SURVEY §8a a6)
    print("Start of normalized Cuts")
    groups = segment_major_points(pts, tarl, dino_list)

    palette = generate_random_colors(max(600, len(groups)))
    colour_major = np.zeros((pts.shape[0], 3))
    for s, idx in enumerate(groups):
        colour_major[idx] = np.array(palette[s]) / 255
    # kDTree_1NN_feature_reprojection (point_cloud_utils.py:144-174): every 5 cm point takes the colour of its
    # nearest 0.35 m point; the nearest-neighbour search runs on the GPU (C ABI ancuts_nn_reproject)
    _, nearest = api.nn_reproject(np.asarray(pcd_chunk.points), pts)
    pcd_chunk.colors = o3d.utility.Vector3dVector(colour_major[nearest.cpu().numpy()])

    inl = get_statistical_inlier_indices(ground)
    g_in = get_subpcd(ground, inl)
    z = np.asarray(g_in.points)[:, 2]
    low = np.where(z < (np.mean(z) + MEAN_HEIGHT))[0]
    cut_hight = get_subpcd(g_in, low)
    cut_hight.paint_uniform_color([0, 0, 0])
    lab_g = d["kitti_labels"]["ground"]
    return (pcd_chunk + cut_hight, pcd_chunk, cut_hight,
            lab_g["instance"][sequence][inl][low], lab_g["semantic"][sequence][inl][low])


def get_merge_pcds(out_folder_ncuts):
    """All .pcd files of a folder in sorted name order (`ncuts_utils.py:207-223`)."""
    import open3d as o3d
    names = sorted(f for f in os.listdir(out_folder_ncuts) if f.endswith(".pcd"))
    print(names)
    return [o3d.io.read_point_cloud(os.path.join(out_folder_ncuts, f)) for f in names]
