"""ctypes binding of libautoinst_ncuts.so (C ABI: include/autoinst_ncuts.h).

There is no CPU fallback: if the shared library is missing, or no sm_100a device is present,
every compute entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ANCUTS_LIB_PATH") or os.path.join(_HERE, "lib", "libautoinst_ncuts.so")   # override: A/B builds
CSRC = os.path.join(_HERE, "csrc")

NUM_CUTS = 10
EINVAL = -1         # ANCUTS_EINVAL: bad argument (also a caller graph that breaks the contract of ancuts_segment_csr_f32)

# every symbol include/autoinst_ncuts.h declares
EXPORTS = [
    "ancuts_version", "ancuts_last_error", "ancuts_create", "ancuts_destroy",
    "ancuts_segment_workspace_bytes", "ancuts_affinity_f32", "ancuts_degree_normalize_f32",
    "ancuts_lanczos_fiedler_batched", "ancuts_ncut_scan_batched", "ancuts_partition_batched",
    "ancuts_segment_chunks", "ancuts_segment_chunks_host", "ancuts_segment_dense_f32",
    "ancuts_launch_count", "ancuts_last_accounting", "ancuts_set_stage_timing", "ancuts_nn_reproject",
    "ancuts_last_levels", "ancuts_debug_phases", "ancuts_feature_pool_workspace_bytes", "ancuts_feature_pool",
    "ancuts_last_unconverged", "ancuts_set_option",
    "ancuts_merge_chunks", "ancuts_remove_semantics", "ancuts_instance_metrics", "ancuts_map_labels",
    "ancuts_last_sparse_accounting", "ancuts_dino_view_pixels", "ancuts_dino_mean",
    "ancuts_last_reorth_accounting", "ancuts_segment_csr_f32",
    "ancuts_affinity_cams_f32", "ancuts_segment_chunks_cams", "ancuts_segment_chunks_cams_host",
]

# ancuts_set_option (include/autoinst_ncuts.h; option 0 is retired)
OPT_PAIR_SEARCH, OPT_MATVEC, OPT_CLUSTER_MAP, OPT_FUSED_CUT, OPT_NODE_FORM = 1, 2, 3, 4, 5
PAIRS_SORTED, PAIRS_SHUFFLED = 0, 1
MATVEC_SPARSE, MATVEC_DENSE = 0, 1


class Params(C.Structure):
    _fields_ = [
        ("alpha", C.c_double), ("theta", C.c_double), ("gamma", C.c_double),
        ("proximity", C.c_double), ("T", C.c_double), ("split_lim", C.c_double),
        ("tarl_dim", C.c_int), ("dino_dim", C.c_int),
        ("lanczos_max_steps", C.c_int), ("lanczos_check_every", C.c_int),
        ("lanczos_tol", C.c_double), ("affinity_impl", C.c_int), ("lanczos_impl", C.c_int),
    ]


class NodeStat(C.Structure):
    _fields_ = [
        ("chunk", C.c_int32), ("n", C.c_int32), ("steps", C.c_int32), ("converged", C.c_int32),
        ("best_k", C.c_int32), ("split", C.c_int32), ("level", C.c_int32), ("n_side", C.c_int32),
        ("lambda2", C.c_double), ("mcut", C.c_double),
    ]


class AncutsError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libautoinst_ncuts error {code}: {msg}")
        self.code = code


class AncutsNoConvergence(RuntimeError):
    """The Lanczos eigensolver stopped at its step limit on `count` recursion nodes (the reference's eigsh raises
    ArpackNoConvergence there, normalized_cut.py:49)."""
    def __init__(self, count):
        super().__init__(f"Lanczos eigensolver: {count} node(s) stopped at lanczos_max_steps without converging")
        self.count = int(count)


_lib = None


def build(verbose: bool = False) -> str:
    """Compile the CUDA sources for sm_100a into autoinst_b200/lib (nvcc cross-compiles without a GPU)."""
    r = subprocess.run(["make", "-j", "4", "-C", CSRC], capture_output=True, text=True)
    if verbose or r.returncode != 0:
        print(r.stdout)
        print(r.stderr)
    if r.returncode != 0:
        raise RuntimeError("building libautoinst_ncuts.so failed:\n" + r.stdout + r.stderr)
    return LIB_PATH


def load():
    """Load the shared library and declare the prototypes.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C autoinst_b200/csrc`). There is no CPU fallback for the NCuts path.")
    lib = C.CDLL(LIB_PATH)
    vp, i32p, i64p, dp = C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int64), C.POINTER(C.c_double)
    pp = C.POINTER(Params)
    sp = C.POINTER(NodeStat)
    lib.ancuts_version.restype = C.c_int
    lib.ancuts_last_error.restype = C.c_char_p
    lib.ancuts_create.argtypes = [C.c_int, C.POINTER(vp)]
    lib.ancuts_destroy.argtypes = [vp]
    lib.ancuts_segment_workspace_bytes.argtypes = [C.c_int, i32p, C.c_int]
    lib.ancuts_segment_workspace_bytes.restype = C.c_int64
    lib.ancuts_affinity_f32.argtypes = [vp, C.c_int, vp, vp, vp, pp, vp, C.c_int64, vp, vp]
    lib.ancuts_affinity_cams_f32.argtypes = [vp, C.c_int, vp, vp, vp, C.c_int, pp, vp, C.c_int64, vp, vp]
    lib.ancuts_degree_normalize_f32.argtypes = [vp, C.c_int, vp, C.c_int64, vp, vp, C.c_int64, vp]
    lib.ancuts_lanczos_fiedler_batched.argtypes = [vp, C.c_int, vp, C.c_int64, C.c_int, i32p, i32p, pp,
                                                   vp, dp, i32p, i32p, vp]
    lib.ancuts_ncut_scan_batched.argtypes = [vp, C.c_int, vp, C.c_int64, C.c_int, i32p, i32p, vp,
                                             i32p, dp, dp, vp, vp]
    lib.ancuts_partition_batched.argtypes = [vp, C.c_int, vp, vp, C.c_int64, C.c_int, i32p, i32p, vp,
                                             C.c_int, vp, i32p, i32p, i32p, vp]
    lib.ancuts_segment_chunks.argtypes = [vp, C.c_int, i64p, vp, vp, vp, pp, vp, i32p, sp, C.c_int32,
                                          i32p, vp]
    lib.ancuts_segment_chunks_host.argtypes = [vp, C.c_int, i64p, vp, vp, vp, pp, vp, i32p, sp,
                                               C.c_int32, i32p, vp]
    lib.ancuts_segment_chunks_cams.argtypes = [vp, C.c_int, i64p, vp, vp, vp, C.c_int, pp, vp, i32p, sp, C.c_int32,
                                               i32p, vp]
    lib.ancuts_segment_chunks_cams_host.argtypes = [vp, C.c_int, i64p, vp, vp, vp, C.c_int, pp, vp, i32p, sp,
                                                    C.c_int32, i32p, vp]
    lib.ancuts_segment_dense_f32.argtypes = [vp, C.c_int, vp, C.c_int64, C.c_int, pp, vp, i32p, sp,
                                             C.c_int32, i32p, vp]
    lib.ancuts_segment_csr_f32.argtypes = [vp, C.c_int, i64p, vp, vp, vp, C.c_int64, i32p, pp, vp, i32p, sp,
                                           C.c_int32, i32p, vp]
    lib.ancuts_nn_reproject.argtypes = [vp, C.c_int, vp, C.c_int, vp, vp, C.c_double, C.c_int32, vp, vp, vp]
    lib.ancuts_feature_pool_workspace_bytes.argtypes = [C.c_int]
    lib.ancuts_feature_pool_workspace_bytes.restype = C.c_int64
    lib.ancuts_feature_pool.argtypes = [vp, C.c_int, vp, C.c_int, vp, vp, C.c_int, C.c_double, dp, dp, C.c_int, vp, vp, vp,
                                        C.c_int64, vp]
    lib.ancuts_launch_count.argtypes = [vp, C.c_int]
    lib.ancuts_launch_count.restype = C.c_int64
    lib.ancuts_last_accounting.argtypes = [vp, dp, dp, i64p]
    lib.ancuts_set_stage_timing.argtypes = [vp, C.c_int]
    lib.ancuts_last_levels.argtypes = [vp, dp, C.c_int]
    lib.ancuts_debug_phases.argtypes = [vp, dp, C.c_int]
    lib.ancuts_last_unconverged.argtypes = [vp]
    lib.ancuts_set_option.argtypes = [vp, C.c_int, C.c_int]
    lib.ancuts_merge_chunks.argtypes = [vp, C.c_int, i64p, vp, vp, dp, C.c_double, C.c_double, vp, vp, i64p, vp]
    lib.ancuts_last_sparse_accounting.argtypes = [vp, dp]
    lib.ancuts_last_reorth_accounting.argtypes = [vp, dp]
    lib.ancuts_dino_view_pixels.argtypes = [vp, C.c_int, vp, C.c_int, vp, C.c_double, dp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp]
    lib.ancuts_dino_mean.argtypes = [vp, C.c_int, C.c_int, vp, C.POINTER(vp), C.c_int, vp, vp, vp]
    lib.ancuts_map_labels.argtypes = [vp, C.c_int, i64p, vp, C.c_int, vp, vp]
    lib.ancuts_remove_semantics.argtypes = [vp, C.c_int64, vp, vp, C.c_double, vp, vp]
    lib.ancuts_instance_metrics.argtypes = [vp, C.c_int64, vp, vp, vp, C.c_int, dp, vp]
    for name in EXPORTS:
        fn = getattr(lib, name)
        if fn.restype is C.c_int and name not in ("ancuts_version",):
            fn.restype = C.c_int
    _lib = lib
    return lib


def check(rc: int):
    if rc != 0:
        raise AncutsError(rc, load().ancuts_last_error().decode("utf-8", "replace"))
