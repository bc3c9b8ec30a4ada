"""CPU checks (numpy model) of partial re-orthogonalisation in the persistent eigensolver kernel, csrc/kernels_cluster.cuh.

Each Lanczos step there is the three-term recurrence; the classical Gram-Schmidt pass against u1 = D^1/2 1 and the whole
basis runs only when Simon's omega recurrence estimates a loss of orthogonality above sqrt(eps), and on the step after.
`lanczos_fiedler_device` below is that step in numpy, with the kernel's start, check schedule and stopping rule
(`oracle.device_model.lanczos_fiedler`, which re-orthogonalises twice on every step, stays the model of the grid-wide
path).  It is checked here

* against the reference, through `oracle.device_model.segment_model`, on the golden chunks and at the benchmarked size;
* against the same step with the pass on every step (the kernel before partial re-orthogonalisation): same step counts,
  same Ritz vector, a semi-orthogonal basis, and the pass on a small share of the steps.
"""
import os

import numpy as np
import pytest
import scipy.sparse as sp
from scipy.sparse.csgraph import connected_components

from conftest import CONFIG_NAMES, GOLDEN, GOLDEN_SEEDS, load_golden
from autoinst_b200.synthetic import CONFIGS, make_chunk
from oracle import device_model as M
from oracle import ncut_ref as R
from oracle.affinity_ref import affinity_ref

EPS = np.finfo(np.float64).eps
REORTH_TOL = np.sqrt(EPS)                               # csrc CL_REORTH_TOL


def lanczos_fiedler_device(Wb32, d, *, reorth="partial", tol=1e-10, kmax=256, stats=None, v0=None, trace=None):
    """Fiedler vector as the cluster kernel computes it (same signature and result as `M.lanczos_fiedler`).

    reorth = "partial": the full pass when the omega estimates call for it; "full": on every step.
    trace (dict, optional) receives the basis (rows: u1, v_0 .. v_k), the step count and the number of full passes."""
    n = Wb32.shape[0]
    s = 1.0 / np.sqrt(d)
    u1 = np.sqrt(d)
    u1 /= np.linalg.norm(u1)
    Wd = Wb32.astype(np.float64)

    def matvec(x):
        z = s * x
        return s * (Wd @ z + z)

    kcap = min(kmax, n - 1)
    V = np.zeros((kcap + 2, n))                         # row 0 = u1, row j + 1 = Lanczos vector v_j (device basis)
    V[0] = u1
    alpha = np.zeros(kcap)
    beta = np.zeros(kcap)
    v = M.start_vector(n) if v0 is None else np.array(v0, dtype=np.float64)
    v -= u1 * (u1 @ v)
    V[1] = v / np.linalg.norm(v)
    om = np.zeros(kcap + 2, dtype=np.float32)           # omega_{k, i} = estimated v_k . v_i (float32 as in the kernel)
    om_p = np.zeros(kcap + 2, dtype=np.float32)         # omega_{k-1, i}
    om[0] = 1.0
    ou, ou_p = EPS, EPS                                 # u1 against v_k, v_{k-1}
    force = False
    nfull = 0
    k = 0
    converged = False
    th1 = th2 = 0.0
    y = None
    next_check = M.CHECK_FIRST
    prev_k, prev_res = 0, 1.0
    while k < kcap:
        vk = V[k + 1]
        w = matvec(vk)
        a1 = vk @ w
        bk = beta[k - 1] if k > 0 else 0.0
        w = (w - a1 * vk) - bk * V[k]                   # V[0] = u1 when k = 0, with bk = 0
        bn = np.linalg.norm(w)
        full = reorth == "full"
        if reorth == "partial":
            on = np.zeros_like(om)
            i = np.arange(k)
            t = (beta[:k] * om[1:k + 1].astype(np.float64) + (alpha[:k] - a1) * om[:k].astype(np.float64)
                 - bk * om_p[:k].astype(np.float64))
            if k > 1:
                t[1:] += beta[:k - 1] * om[:k - 1].astype(np.float64)
            noise = 0.6 * EPS * (np.abs(beta[:k]) + bn)
            t = (t + np.where(t < 0.0, -noise, noise)) / bn
            on[i] = t
            on[k] = EPS * 0.5 * n
            on[k + 1] = 1.0
            tu = (1.0 - a1) * ou - bk * ou_p
            tu = (tu + (-2.0 if tu < 0.0 else 2.0) * EPS * bn) / bn
            ou_p, ou = ou, tu
            full = bool(force or np.any(~(np.abs(t) <= REORTH_TOL)) or not abs(ou) <= REORTH_TOL)
            if full:
                on[:k + 1] = EPS
                ou = EPS
                force = not force
            om_p, om = om, on
        if full:
            nfull += 1
            h = V[:k + 2] @ w                           # one classical Gram-Schmidt pass against u1 and v_0 .. v_k
            w -= V[:k + 2].T @ h
            a1 += h[k + 1]
        b = np.linalg.norm(w)
        alpha[k] = a1
        beta[k] = b
        k += 1
        breakdown = b < 1e-13
        if not breakdown:
            V[k + 1] = w / b
        if breakdown or k == kcap or k == next_check:
            th1, th2, y = M.tridiag_top2(alpha[:k], beta[:k])
            res = abs(b * y[-1])
            gap = max(th1 - th2, 1e-300)
            if breakdown or k == kcap or k >= n - 1 or res <= tol * gap:
                converged = breakdown or (k >= n - 1) or res <= tol * gap
                break
            adv = M.CHECK_HI
            if 0.0 < res < prev_res:
                rate = np.log(res / prev_res) / (k - prev_k)
                need = M.CHECK_SAFETY * np.log(tol * gap / res) / rate
                adv = int(min(M.CHECK_HI, max(M.CHECK_LO, np.ceil(need))))
            prev_k, prev_res = k, res
            next_check = k + adv
    ev = V[1:k + 1].T @ y
    ev /= np.linalg.norm(ev)
    if ev.sum() < 0:
        ev = -ev
    if stats is not None:
        stats.append(dict(n=n, k=k, lam2=1.0 - th1, lam3=1.0 - th2, converged=converged, full=nfull))
    if trace is not None:
        trace.update(V=V[:k + 1].copy(), k=k, full=nfull)
    return ev, 1.0 - th1


@pytest.fixture
def partial_model(monkeypatch):
    """segment_model with the kernel's eigensolver step (partial re-orthogonalisation) in place of the twice-CGS one."""
    monkeypatch.setattr(M, "lanczos_fiedler", lambda *a, **kw: lanczos_fiedler_device(*a, reorth="partial", **kw))
    return M.segment_model


@pytest.mark.parametrize("seed", GOLDEN_SEEDS)
@pytest.mark.parametrize("name", CONFIG_NAMES)
def test_partial_model_matches_reference_on_golden(partial_model, seed, name):
    inp, out, A = load_golden(seed, name)
    lab = partial_model(A.toarray().astype(np.float32), float(out["T"]))
    assert R.same_partition(lab, out["labels"])


def test_partial_model_matches_oracle_on_a_chunk(partial_model):
    ch = make_chunk(3, n_target=1500, features="tarl")
    cfg = CONFIGS["tarl_spatial"]
    A = affinity_ref(ch.points, ch.tarl, alpha=cfg["alpha"], theta=cfg["theta"])
    with R.pinned_eigsh():
        g = R.normalized_cut_ref(sp.csr_matrix(A), ch.n, np.arange(ch.n), T=cfg["T"])
    lab = partial_model(A.astype(np.float32), cfg["T"])
    assert R.same_partition(lab, R.labels_from_groups(g, ch.n))


def test_partial_model_matches_oracle_at_bench_size(partial_model):
    """One oracle-stable chunk of the benchmarked workload (config_tarl_spatial, 8192 points) against the oracle labels
    of tests/golden/parity_bench_size.npz."""
    fix = np.load(os.path.join(GOLDEN, "parity_bench_size.npz"))
    cfg = CONFIGS["tarl_spatial"]
    seed = next(s for s in range(7000, 7006) if bool(fix[f"stable_tarl_spatial_8192_{s}"]))
    ch = make_chunk(seed, n_target=8192, features="tarl")
    A = affinity_ref(ch.points, ch.tarl, None, alpha=cfg["alpha"], theta=cfg["theta"])
    stats = []
    lab = partial_model(A.astype(np.float32), cfg["T"], stats=stats)
    ref = fix[f"labels_tarl_spatial_8192_{seed}"].astype(np.int32)
    assert ref.shape == lab.shape and R.same_partition(lab, ref)
    steps = sum(s["k"] for s in stats)
    assert all(s["converged"] for s in stats) and sum(s["full"] for s in stats) < 0.15 * steps


@pytest.fixture(scope="module")
def node():
    """The connected block of tests/test_design_choices.py: largest component of a 2000-point tarl_spatial chunk."""
    cfg = CONFIGS["tarl_spatial"]
    ch = make_chunk(1000, n_target=2000, features="tarl")
    A = affinity_ref(ch.points, ch.tarl, None, alpha=cfg["alpha"], theta=cfg["theta"])
    W = A.astype(np.float32).astype(np.float64)
    nc, lab = connected_components(sp.csr_matrix(W != 0), directed=False)
    big = np.argmax(np.bincount(lab))
    idx = np.nonzero(lab == big)[0]
    Wb = W[np.ix_(idx, idx)]
    return Wb.astype(np.float32), Wb.sum(1) + 1.0


def test_partial_reorth_stays_semi_orthogonal_and_rarely_takes_the_full_pass(node):
    Wb, d = node
    tp, tf = {}, {}
    ev_p, lam_p = lanczos_fiedler_device(Wb, d, reorth="partial", trace=tp)
    ev_f, lam_f = lanczos_fiedler_device(Wb, d, reorth="full", trace=tf)
    G = tp["V"] @ tp["V"].T                             # u1 and every Lanczos vector
    assert np.abs(G - np.eye(len(G))).max() < REORTH_TOL
    assert tp["k"] > 40 and tp["full"] < 0.15 * tp["k"]
    assert tf["full"] == tf["k"]
    assert tp["k"] == tf["k"]
    assert abs(lam_p - lam_f) < 1e-9
    assert np.abs(ev_p - ev_f).max() < 1e-9
    assert abs(np.linalg.norm(ev_p) - 1.0) < 1e-12
