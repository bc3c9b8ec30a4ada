"""GPU test of the two node forms of the segment path (ANCUTS_OPT_NODE_FORM): recursion nodes kept as CSR (built from the
pair queue, children compacted from their parents, dense blocks written only for the nodes that read dense W) and every
node as a dense block.  The CSR rows hold exactly the entries the shared-memory slices kept from the dense blocks, and the
degrees are summed in the dense order, so labels and every node record (steps, lambda2, N-cut value, split) are
bit-identical.  Covered: the three feature configs, the host and resident entries, both pair searches, a queue overflow,
and each node that needs a dense block in the CSR form (slices that do not fit, more than 4096 points, the grid-wide
Lanczos path); the options that select the dense form for a whole call (separate cut kernels, dense matvec) too."""
import numpy as np
import pytest

from autoinst_b200.synthetic import CONFIGS, make_chunk

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

PAIRS, MATVEC, CMAP, FUSED_CUT, NODE_FORM = 1, 2, 3, 4, 5      # include/autoinst_ncuts.h: ANCUTS_OPT_*


def _sorted(st):
    return np.sort(st, order=list(st.dtype.names))


def _run(api, device, packed, lane, opts, form, resident, **kw):
    hd = api.Handle.get(device, lane)
    for k, v in opts.items():
        hd.set_option(k, v)
    hd.set_option(NODE_FORM, form)
    if resident:
        dev = packed.to_device(device)
        res = api.segment_packed(packed, dev_chunks=dev, lane=lane, want_stats=True, **kw)
        labels = dev.labels.cpu().numpy()
        return [labels[packed.off[c]:packed.off[c + 1]] for c in range(len(packed.off) - 1)], res.stats
    res = api.segment_packed(packed, device=device, lane=lane, want_stats=True, **kw)
    return list(res.labels), res.stats


def _same(api, device, packed, lane, opts=None, resident=(False, True), **kw):
    for rs in resident:
        la, sa = _run(api, device, packed, lane, opts or {}, 0, rs, **kw)
        lb, sb = _run(api, device, packed, lane, opts or {}, 1, rs, **kw)
        for c, (x, y) in enumerate(zip(la, lb)):
            assert np.array_equal(x, y), (rs, c)
        a, b = _sorted(sa), _sorted(sb)
        assert len(a) == len(b) > 0
        assert a.tobytes() == b.tobytes(), rs
    api.Handle.get(device, lane).set_option(NODE_FORM, 0)


def _kw(cfg):
    return dict(alpha=cfg["alpha"], theta=cfg["theta"], gamma=cfg["gamma"], T=cfg["T"])


@pytest.mark.parametrize("pairs", [0, 1])
@pytest.mark.parametrize("config", ["spatial", "tarl_spatial", "tarl_spatial_dino"])
def test_node_forms_give_identical_records(cuda_device, config, pairs):
    from autoinst_b200 import api
    cfg = CONFIGS[config]
    feats = "tarl_dino" if cfg["gamma"] else "tarl"
    chunks = [make_chunk(610 + i, n_target=1500 + 2400 * i, features=feats) for i in range(4)]
    packed = api.PackedChunks([c.points for c in chunks], [c.tarl for c in chunks],
                              [c.dino for c in chunks] if cfg["gamma"] else None, theta=cfg["theta"], gamma=cfg["gamma"])
    _same(api, cuda_device, packed, 70 + pairs, {PAIRS: pairs}, **_kw(cfg))
    api.Handle.get(cuda_device, 70 + pairs).set_option(PAIRS, 0)


def test_node_forms_on_a_cluttered_16k_chunk(cuda_device):
    """A 16 k chunk: root components above 4096 points take the grid-wide path with dense blocks written on demand."""
    from autoinst_b200 import api
    cfg = CONFIGS["tarl_spatial"]
    ch = make_chunk(620, n_target=16384, features="tarl")
    packed = api.PackedChunks([ch.points], [ch.tarl], None, theta=cfg["theta"])
    _same(api, cuda_device, packed, 72, **_kw(cfg))


def test_node_forms_on_nodes_whose_slices_do_not_fit(cuda_device):
    """A dense blob (hundreds of entries per row): its slices do not fit shared memory at one CTA per node, so the CSR form
    writes its dense block before the cluster kernel streams it; at eight CTAs per node they fit."""
    from autoinst_b200 import api
    rng = np.random.default_rng(11)
    n = 1000
    pts = (rng.normal(size=(n, 3)) * 0.45).astype(np.float32).astype(np.float64)
    pts[n // 2:] += 9.0
    tarl = rng.normal(size=(n, 96)).astype(np.float32)
    cfg = CONFIGS["tarl_spatial"]
    packed = api.PackedChunks([pts], [tarl], None, theta=cfg["theta"])
    for cmap in (111111, 888888):
        _same(api, cuda_device, packed, 73, {CMAP: cmap}, **_kw(cfg))
    api.Handle.get(cuda_device, 73).set_option(CMAP, 0)


def test_node_forms_past_the_cluster_step_limit(cuda_device):
    """lanczos_check_every = 300, above the cluster kernel's 256-step limit: nodes that are not done there go to the
    grid-wide path (dense blocks of the whole level, then the separate cut kernels)."""
    from autoinst_b200 import api
    cfg = CONFIGS["tarl_spatial"]
    ch = make_chunk(630, n_target=3000, features="tarl")
    packed = api.PackedChunks([ch.points], [ch.tarl], None, theta=cfg["theta"])
    _same(api, cuda_device, packed, 74, resident=(True,), check_every=300, **_kw(cfg))


@pytest.mark.parametrize("opt", [FUSED_CUT, MATVEC])
def test_call_level_dense_forms(cuda_device, opt):
    from autoinst_b200 import api
    cfg = CONFIGS["tarl_spatial"]
    chunks = [make_chunk(640 + i, n_target=2500, features="tarl") for i in range(2)]
    packed = api.PackedChunks([c.points for c in chunks], [c.tarl for c in chunks], None, theta=cfg["theta"])
    lane = 75 + opt
    _same(api, cuda_device, packed, lane, {opt: 1}, **_kw(cfg))
    api.Handle.get(cuda_device, lane).set_option(opt, 0)


def test_node_forms_after_a_queue_overflow(cuda_device):
    from autoinst_b200 import api
    rng = np.random.default_rng(5)
    n = 900
    pts = (rng.normal(size=(n, 3)) * 0.2).astype(np.float32).astype(np.float64)
    pts[n // 2:] += 7.0
    tarl = rng.normal(size=(n, 96)).astype(np.float32)
    cfg = CONFIGS["tarl_spatial"]
    packed = api.PackedChunks([pts], [tarl], None, theta=cfg["theta"])
    _same(api, cuda_device, packed, 79, **_kw(cfg))
