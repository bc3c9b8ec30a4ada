"""CPU tests of the CSR packer behind `api.segment_graphs` (no GPU needed): the global row pointers / local columns /
float32 values of ancuts_segment_csr_f32, canonical form as `toarray()` reads it, torch sparse-CSR input, bad shapes."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

from autoinst_b200.api import pack_graphs


def _sym(n, seed, density=0.3):
    rng = np.random.default_rng(seed)
    a = rng.random((n, n)) * (rng.random((n, n)) < density)
    a = np.triu(a, 1)
    a = a + a.T + np.eye(n)
    return sp.csr_matrix(a)


def _unpack(pk, c):
    """graph c of a packed batch, densified from the packed arrays"""
    rp, col, val = pk.row_ptr.numpy(), pk.col.numpy(), pk.val.numpy()
    a, b = int(pk.off[c]), int(pk.off[c + 1])
    out = np.zeros((b - a, b - a), dtype=np.float32)
    for i in range(b - a):
        for q in range(rp[a + i], rp[a + i + 1]):
            out[i, col[q]] += val[q]
    return out


def test_layout_of_a_batch():
    gs = [_sym(5, 1), _sym(1, 2), _sym(7, 3)]
    pk = pack_graphs(gs)
    assert pk.sizes == [5, 1, 7]
    assert pk.off.tolist() == [0, 5, 6, 13]
    assert pk.row_ptr.dtype == torch.int64 and pk.col.dtype == torch.int32 and pk.val.dtype == torch.float32
    assert pk.row_ptr.numel() == 14 and int(pk.row_ptr[0]) == 0 and int(pk.row_ptr[-1]) == pk.nnz
    e0 = 0
    for c, g in enumerate(gs):
        a, b = int(pk.off[c]), int(pk.off[c + 1])
        assert np.array_equal(pk.row_ptr[a:b + 1].numpy(), g.indptr + e0)
        assert np.array_equal(pk.col[e0:e0 + g.nnz].numpy(), g.indices)             # local columns
        assert np.array_equal(pk.val[e0:e0 + g.nnz].numpy(), g.data.astype(np.float32))
        e0 += g.nnz


def test_non_canonical_input_becomes_what_toarray_holds():
    # unsorted columns, duplicates (summed in float64 before the rounding to float32), an explicit zero, COO input
    rows = np.array([0, 0, 0, 1, 1, 1, 2, 2, 2, 2])
    cols = np.array([2, 0, 2, 1, 0, 0, 0, 2, 1, 1])
    vals = np.array([0.1, 1.0, 0.2 + 1e-9, 1.0, 0.25, 0.0, 0.3 + 1e-9, 1.0, 0.0, 0.0])
    w = sp.csr_matrix((vals, cols, np.array([0, 3, 6, 10])), shape=(3, 3))          # stored as given
    assert w.nnz == 10 and not w.has_canonical_format
    coo = sp.coo_matrix((vals, (rows, cols)), shape=(3, 3))
    for g in (w, coo):
        pk = pack_graphs([g])
        assert np.array_equal(_unpack(pk, 0), g.toarray().astype(np.float32))
        rp, col = pk.row_ptr.numpy(), pk.col.numpy()
        for i in range(3):
            assert np.all(np.diff(col[rp[i]:rp[i + 1]]) > 0)                          # sorted, no duplicates
    # the caller's matrix is left as it was
    assert w.nnz == 10


def test_torch_sparse_csr_packs_like_scipy():
    gs = [_sym(6, 4), _sym(3, 5)]
    a = pack_graphs(gs)
    b = pack_graphs([torch.as_tensor(g.toarray(), dtype=torch.float32).to_sparse_csr() for g in gs])
    c = pack_graphs([gs[0], torch.as_tensor(gs[1].toarray(), dtype=torch.float64).to_sparse_csr()])
    for x in (b, c):
        assert x.off.tolist() == a.off.tolist()
        assert torch.equal(x.row_ptr, a.row_ptr) and torch.equal(x.col, a.col) and torch.equal(x.val, a.val)


def test_bad_shapes_raise_value_error():
    with pytest.raises(ValueError):
        pack_graphs([sp.csr_matrix((3, 4))])
    with pytest.raises(ValueError):
        pack_graphs([_sym(3, 1), sp.csr_matrix((0, 0))])
    with pytest.raises(ValueError):
        pack_graphs([torch.zeros((2, 3)).to_sparse_csr()])
    with pytest.raises(ValueError):
        pack_graphs([])
    with pytest.raises(TypeError):
        pack_graphs([np.eye(3)])
