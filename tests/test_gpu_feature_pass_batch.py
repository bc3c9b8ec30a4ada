"""GPU test of the deferred feature pass in its two launch forms: with inputs resident on the device it runs every chunk of
the batch in one launch, through the host entry it runs one launch per chunk as the chunk's features arrive.  Both give
every affinity the same float32 value, so every node record of the recursion is bit-identical, eigenvalues and N-cut
values included, for each feature configuration and both pair searches (cell-sorted ranks, input indices)."""
import numpy as np
import pytest

from autoinst_b200.synthetic import CONFIGS, make_chunk

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

PAIRS = 1       # include/autoinst_ncuts.h: ANCUTS_OPT_PAIR_SEARCH (0 cell-sorted sweep, 1 shuffled sweep)


@pytest.mark.parametrize("pairs", [0, 1])
@pytest.mark.parametrize("config", ["spatial", "tarl_spatial", "tarl_spatial_dino"])
def test_one_launch_feature_pass_matches_per_chunk_passes(cuda_device, config, pairs):
    from autoinst_b200 import api
    lane = 40 + pairs
    api.Handle.get(cuda_device, lane).set_option(PAIRS, pairs)
    cfg = CONFIGS[config]
    feats = "tarl_dino" if cfg["gamma"] else "tarl"
    chunks = [make_chunk(510 + i, n_target=1200 + 900 * i, features=feats) for i in range(4)]
    packed = api.PackedChunks([c.points for c in chunks], [c.tarl for c in chunks],
                              [c.dino for c in chunks] if cfg["gamma"] else None, theta=cfg["theta"], gamma=cfg["gamma"])
    kw = dict(lane=lane, alpha=cfg["alpha"], theta=cfg["theta"], gamma=cfg["gamma"], T=cfg["T"], want_stats=True)
    host = api.segment_packed(packed, device=cuda_device, **kw)
    dev = packed.to_device(cuda_device)
    resident = api.segment_packed(packed, dev_chunks=dev, **kw)
    labels = dev.labels.cpu().numpy()
    for c, lab in enumerate(host.labels):
        assert np.array_equal(lab, labels[packed.off[c]:packed.off[c + 1]]), c
    # records are appended in the order nodes finish: compare them sorted on every field
    a, b = (np.sort(st, order=list(st.dtype.names)) for st in (host.stats, resident.stats))
    assert len(a) == len(b) > len(chunks)
    assert a.tobytes() == b.tobytes()
