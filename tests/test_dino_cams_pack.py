"""CPU tests of the DINOv2 input over several cameras: the host packer's point-major (P, cams * D) layout for the three
input forms, the rejection of inconsistent camera shapes, and the synthetic second camera ("tarl_dino2"), which must leave
the chunks of every existing feature string unchanged."""
import hashlib

import numpy as np
import pytest

from autoinst_b200 import api
from autoinst_b200.synthetic import make_chunk


def _chunks(sizes, cams, width, seed=0):
    rng = np.random.default_rng(seed)
    pts = [rng.normal(size=(n, 3)) for n in sizes]
    dino = [[rng.normal(size=(n, width)) for _ in range(cams)] for n in sizes]
    return pts, dino


def _expect(dino, off, cams, width):
    """Point-major rows: camera 0's width values, then camera 1's, ..."""
    out = np.zeros((int(off[-1]), cams * width), dtype=np.float32)
    for c, per_cam in enumerate(dino):
        for k, g in enumerate(per_cam):
            out[off[c]:off[c + 1], k * width:(k + 1) * width] = g.astype(np.float32)
    return out


@pytest.mark.parametrize("form", ["list", "tuple", "array3", "tensor3"])
@pytest.mark.parametrize("cams", [1, 2, 3])
def test_pack_layout(form, cams):
    import torch
    sizes, width = [5, 9, 1, 4], 8
    pts, dino = _chunks(sizes, cams, width)
    if form == "list":
        arg = dino
    elif form == "tuple":
        arg = [tuple(d) for d in dino]
    elif form == "array3":
        arg = [np.stack(d, axis=1) for d in dino]
    else:
        arg = [torch.as_tensor(np.stack(d, axis=1)) for d in dino]
    pk = api.PackedChunks(pts, None, arg, gamma=0.1, pin=False)
    assert pk.sizes == sizes and list(pk.off) == [0, 5, 14, 15, 19]
    assert pk.dino_cams == cams and pk.dino_dim == width
    assert tuple(pk.dino.shape) == (19, cams * width) and pk.dino.dtype == torch.float32
    assert np.array_equal(pk.dino.numpy(), _expect(dino, pk.off, cams, width))
    assert pk.h2d_bytes() == 19 * 3 * 8 + 19 * cams * width * 4


def test_pack_one_camera_as_before():
    """An (n, D) array per chunk is one camera, packed as (P, D)."""
    sizes, width = [6, 3], 12
    pts, dino = _chunks(sizes, 1, width, seed=1)
    pk = api.PackedChunks(pts, None, [d[0] for d in dino], gamma=0.1, pin=False)
    assert pk.dino_cams == 1 and pk.dino_dim == width and tuple(pk.dino.shape) == (9, width)
    assert np.array_equal(pk.dino.numpy(), np.concatenate([d[0] for d in dino]).astype(np.float32))


def test_pack_without_dino_term():
    sizes = [4, 4]
    pts, dino = _chunks(sizes, 2, 8)
    pk = api.PackedChunks(pts, None, dino, gamma=0.0, pin=False)
    assert not pk.use_d and pk.dino is None and pk.dino_cams == 1 and pk.dino_dim == 0


def test_pack_rejects_inconsistent_cameras():
    pts, two = _chunks([5, 6], 2, 8)
    _, one = _chunks([5, 6], 1, 8)
    with pytest.raises(ValueError, match="same DINOv2 cameras"):
        api.PackedChunks(pts, None, [two[0], one[1]], gamma=0.1, pin=False)          # 2 cameras, then 1
    with pytest.raises(ValueError, match="same DINOv2 cameras"):
        api.PackedChunks(pts, None, [two[0], [g[:, :4] for g in two[1]]], gamma=0.1, pin=False)   # width 8, then 4
    with pytest.raises(ValueError, match="one \\(n, D\\) shape"):
        api.PackedChunks(pts, None, [[two[0][0], two[0][1][:, :4]], two[1]], gamma=0.1, pin=False)
    with pytest.raises(ValueError, match="one \\(n, D\\) shape"):
        api.PackedChunks(pts, None, [[two[0][0], two[0][1][:3]], two[1]], gamma=0.1, pin=False)
    with pytest.raises(ValueError, match="The length should be longer than 0!"):
        api.PackedChunks(pts, None, [[], []], gamma=0.1, pin=False)
    with pytest.raises(ValueError, match="The length should be longer than 0!"):
        api.PackedChunks(pts, None, None, gamma=0.1, pin=False)


def _digest(ch):
    h = hashlib.sha256()
    for a in (ch.points, ch.instance, ch.tarl, ch.dino):
        if a is not None:
            h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()[:32]


# digests of make_chunk before the second camera was added (golden files, parity fixtures and bench.py use these chunks)
@pytest.mark.parametrize("args,digest", [
    ((7, 1500, "tarl"), "1ca958662acbbb0d88c99f6a862b54dc"),
    ((41, 2500, "tarl_dino"), "24bf039eeab90604405e550f08eee872"),
    ((1000, 1200, ""), "f8dd1f02cefe1aae7d39617f96aaac1f"),
    ((1003, 2000, "tarl_dino"), "509bc736619dc186bf6b6ce2592a74d8"),
])
def test_make_chunk_unchanged(args, digest):
    cid, n, features = args
    assert _digest(make_chunk(cid, n_target=n, features=features)) == digest


def test_make_chunk_second_camera():
    one = make_chunk(41, n_target=2500, features="tarl_dino")
    two = make_chunk(41, n_target=2500, features="tarl_dino2")
    assert np.array_equal(one.points, two.points) and np.array_equal(one.tarl, two.tarl)
    assert isinstance(two.dino, list) and len(two.dino) == 2
    assert np.array_equal(two.dino[0], one.dino)
    g0, g1 = two.dino
    assert g1.shape == g0.shape and g1.dtype == np.float64
    assert np.array_equal(g1, g1.astype(np.float32).astype(np.float64))
    z0, z1 = ~g0.any(axis=1), ~g1.any(axis=1)
    assert 0.25 < z1.mean() < 0.35 and not np.array_equal(z0, z1)
    both = ~(z0 | z1)
    assert not np.array_equal(g0[both], g1[both])
