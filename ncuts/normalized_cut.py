"""`normalized_cut` with the reference's signature (`pipeline/ncuts/normalized_cut.py:37`), computed on a B200.

    normalized_cut(w, num_points_orig, labels, T=0.01, split_lim=0.01) -> list[np.ndarray]

`w` may be a scipy sparse matrix (what `ncuts_utils.py:167-174` passes), a dense numpy array or a
CUDA tensor; it must be symmetric with a unit diagonal, as the reference's affinity is.  A scipy sparse
`w` is checked for that on the device and a violation raises ValueError naming the row.  The result
is the same partition of `labels` the reference returns; the ORDER of the groups differs (the
reference emits them depth first, mask side first; here they come out in device layout order), which
only changes which random colour a segment gets downstream (`ncuts_utils.py:177-183`).

Everything is computed by libautoinst_ncuts.so: a scipy sparse `w` goes to the device as CSR
(`ancuts_segment_csr_f32`, no n x n host matrix), dense input through `ancuts_segment_dense_f32`; there
is no CPU path.
"""
import numpy as np


def _to_device_matrix(w):
    import torch
    from autoinst_b200 import api
    if isinstance(w, torch.Tensor):
        if not w.is_cuda:
            w = w.cuda()
        return w.to(torch.float32)
    if hasattr(w, "toarray"):                    # scipy sparse
        dense = np.asarray(w.toarray(), dtype=np.float32)
    else:
        dense = np.asarray(w, dtype=np.float32)
    n = dense.shape[0]
    buf, view = api.alloc_matrix(n, torch.device("cuda", torch.cuda.current_device()))
    view.copy_(torch.from_numpy(dense), non_blocking=False)
    return view


def normalized_cut(w, num_points_orig, labels, T=0.01, split_lim=0.01):
    from autoinst_b200 import api
    from autoinst_b200._lib import EINVAL, AncutsError
    labels = np.asarray(labels)
    n = int(w.shape[0])
    if n != labels.shape[0]:
        raise ValueError("w and labels disagree on the number of points")
    if n == 0:
        return [labels]
    if hasattr(w, "tocsr"):                      # scipy sparse: the CSR front end, no densified copy
        try:
            res = api.segment_graphs([w], num_points_orig=int(num_points_orig), T=float(T), split_lim=float(split_lim),
                                     strict=True)
        except AncutsError as ex:
            if ex.code == EINVAL:         # w breaks the contract above (symmetric, unit diagonal, finite)
                raise ValueError(str(ex)) from ex
            raise
        return _groups(res.labels[0], labels)
    seg = api.segment_dense(_to_device_matrix(w), num_points_orig=int(num_points_orig), T=float(T),
                            split_lim=float(split_lim), strict=True)      # raises AncutsNoConvergence like eigsh
    return _groups(seg, labels)


def _groups(seg, labels):
    order = np.argsort(seg, kind="stable")
    bounds = np.flatnonzero(np.diff(seg[order])) + 1
    return [labels[idx] for idx in np.split(order, bounds)]
