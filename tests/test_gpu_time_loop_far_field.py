"""GPU tests of the far-field convection in the device time loop (LUDVM(..., far_field_order=p), fast mode).  The clouds
are at least the library's all-pairs / far-field crossover (SIM_FAR_FIELD_MIN_WAKE), so every step takes the far-field
step, except in the test of a run that crosses it; far_field_info confirms it."""
import ctypes

import numpy as np
import pytest

from conftest import biteq

pytestmark = pytest.mark.gpu

NF = 1 << 16   # >= SIM_FAR_FIELD_MIN_WAKE = 65536: every step's wake bound is NF + 2 i + 2
KW = dict(t0=0, tf=0.3, dt=5e-2, chord=1, rho=1.225, Uinf=1, Npoints=81, Ncoeffs=30, LESPcrit=0.2, Naca="0012")
E_STATE, E_UNSUPPORTED = -4, -5


def gust(nf, seed=5):
    rng = np.random.default_rng(seed)
    xy = np.stack([rng.uniform(-6.0, -0.5, nf), rng.uniform(-1.0, 1.0, nf)])
    return dict(circulation_freevort=rng.standard_normal(nf) * 1e-3, xy_freevort=xy)


@pytest.fixture(scope="module")
def runs():
    from ludvm_b200 import LUDVM
    kw = dict(KW, **gust(NF), verbose=False, mode="fast")
    return kw, LUDVM(**kw), LUDVM(**kw, far_field_order=18)


def _all_far_field(s):
    info = s.far_field_info
    assert info["far_field_steps"] == s.nt - 1 and info["fallback_steps"] == 0, info
    assert info["order"] == 18 and info["leaf_level"] >= 2, info


def test_far_field_tracks_all_pairs(runs):
    _, a, f = runs
    _all_far_field(f)
    for k in ("L", "D", "M"):
        ref = getattr(a, k)
        assert np.max(np.abs(getattr(f, k) - ref)) <= 1e-10 * np.max(np.abs(ref)), k
    assert np.max(np.abs(f.LESP - a.LESP)) <= 1e-10
    assert biteq(f.LEV_shed, a.LEV_shed)
    assert np.max(np.abs(f.path["FREE"] - a.path["FREE"])) <= 1e-12
    assert np.max(np.abs(f.path["TEV"] - a.path["TEV"])) <= 1e-12


def test_first_far_field_step_within_bound_of_the_sum(runs):
    """Step 1 convects FREE (the whole old wake) through the tree.  Everything else in the step is the all-pairs run's
    arithmetic on the same state, so the new positions differ by the tree's error only: at most
    dt * 1e-13 * sum_j |Gamma_j K_ij| per vortex (the tree's own error at order 18 is ~1e-15 of that sum)."""
    kw, a, f = runs
    g = np.asarray(kw["circulation_freevort"], dtype=np.float64)
    x0, z0 = a.path["FREE"][0]
    assert biteq(f.path["FREE"][0], a.path["FREE"][0])
    import torch
    vc4 = a.v_core ** 4
    t = lambda v: torch.tensor(np.ascontiguousarray(v), dtype=torch.float64, device="cuda")
    tx, tz, tg = t(x0), t(z0), t(np.abs(g))
    bound = np.empty(NF)
    for r in range(0, NF, 2048):   # sum_j |Gamma_j| |K_ij|, |K| = r / (2 pi sqrt(r^4 + vc^4))
        r2 = (tx[r:r + 2048, None] - tx[None, :]) ** 2 + (tz[r:r + 2048, None] - tz[None, :]) ** 2
        bound[r:r + 2048] = (tg[None, :] * torch.sqrt(r2) / (2 * np.pi * torch.sqrt(r2 * r2 + vc4))).sum(1).cpu().numpy()
    d = np.hypot(*(f.path["FREE"][1] - a.path["FREE"][1]))
    assert np.all(d <= a.dt * 1e-13 * bound), float(np.max(d / (a.dt * bound)))


def test_far_field_reproducible_and_chunking_independent(runs):
    from ludvm_b200 import LUDVM
    kw, _, f = runs
    kw = dict(kw, tf=0.6)
    b = LUDVM(**kw, far_field_order=18)
    c = LUDVM(**kw, far_field_order=18)
    d = LUDVM(**dict(kw, verbose=True), far_field_order=18, steps_per_graph=7, run=False)
    d.time_loop(print_dt=3)   # ludvm_sim_run in chunks of 7 steps
    _all_far_field(b)
    _all_far_field(d)
    for s in (c, d):
        for k in ("L", "D", "M", "LESP", "LEV_shed", "fourier"):
            assert biteq(getattr(s, k), getattr(b, k)), k
        for k in ("FREE", "TEV", "LEV"):
            assert biteq(s.path[k], b.path[k]), k
    for k in ("L", "M"):   # the first 6 steps are the fixture's run
        assert biteq(getattr(b, k)[:f.nt], getattr(f, k)), k


def test_far_field_composes_with_pressure_and_strided_history(runs):
    from ludvm_b200 import LUDVM
    kw, a, f = runs
    ap = LUDVM(**kw, pressure=True)
    fp = LUDVM(**kw, pressure=True, far_field_order=18)
    _all_far_field(fp)
    assert np.max(np.abs(ap.dp)) > 0
    assert np.max(np.abs(fp.dp - ap.dp)) <= 1e-10 * np.max(np.abs(ap.dp))
    assert biteq(fp.L, f.L) and biteq(fp.path["FREE"], f.path["FREE"])   # pressure changes nothing else
    h = LUDVM(**kw, store_history=5, far_field_order=18)
    _all_far_field(h)
    assert biteq(h.path["TEV"], f.path["TEV"][::5]) and biteq(h.path["LEV"], f.path["LEV"][::5])
    assert biteq(h.path["FREE"], f.path["FREE"]) and biteq(h.L, f.L)


def test_clustered_cloud_falls_back_to_all_pairs():
    """More than 65 536 vortices in a 1e-4 square, plus 16 spread over the gust's box so that the tree's bounding box is
    the box (and not the square) from the first step on: the leaf that holds the square is over the tree's limit, so each
    step runs the all-pairs kernels of the run without the far field -- bit for bit."""
    from ludvm_b200 import LUDVM
    rng = np.random.default_rng(8)
    nc, ns = 70000, 16
    xy = np.concatenate([np.stack([-3.0 + rng.uniform(0, 1e-4, nc), rng.uniform(0, 1e-4, nc)]),
                         np.stack([rng.uniform(-6.0, -0.5, ns), rng.uniform(-1.0, 1.0, ns)])], axis=1)
    kw = dict(KW, circulation_freevort=rng.standard_normal(nc + ns) * 1e-6, xy_freevort=xy, verbose=False, mode="fast")
    a = LUDVM(**kw)
    f = LUDVM(**kw, far_field_order=18)
    assert f.far_field_info["fallback_steps"] == f.nt - 1 and f.far_field_info["far_field_steps"] == 0
    for k in ("L", "D", "M", "LESP", "LEV_shed"):
        assert biteq(getattr(f, k), getattr(a, k)), k
    for k in ("FREE", "TEV", "LEV"):
        assert biteq(f.path[k], a.path[k]), k


def test_enable_far_field_state_checks():
    from ludvm_b200 import LUDVM, _lib
    L = _lib.load()
    s = LUDVM(**KW, verbose=False, mode="fast", run=False)
    s.time_loop(nsteps=1)
    assert L.ludvm_sim_enable_far_field(s._sim, 18) == E_STATE
    info = (ctypes.c_int64 * 4)()
    assert L.ludvm_sim_far_field_info(s._sim, info) == 0 and list(info) == [0, 0, 0, 0]
    e = LUDVM(**KW, verbose=False, mode="exact", run=False)
    e.time_loop(nsteps=0)
    assert L.ludvm_sim_enable_far_field(e._sim, 18) == E_UNSUPPORTED
    assert L.ludvm_sim_enable_far_field(s._sim, 0) == E_STATE
    s.close()
    e.close()


def _sum_abs_terms(g, x, z, vc4):
    """sum_j |Gamma_j| |K_ij| over the cloud at each of its points, |K| = r / (2 pi sqrt(r^4 + vc^4)), on the GPU."""
    import torch
    t = lambda v: torch.tensor(np.ascontiguousarray(v), dtype=torch.float64, device="cuda")
    tx, tz, tg = t(x), t(z), t(np.abs(g))
    out = np.empty(len(x))
    for r in range(0, len(x), 2048):
        r2 = (tx[r:r + 2048, None] - tx[None, :]) ** 2 + (tz[r:r + 2048, None] - tz[None, :]) ** 2
        out[r:r + 2048] = (tg[None, :] * torch.sqrt(r2) / (2 * np.pi * torch.sqrt(r2 * r2 + vc4))).sum(1).cpu().numpy()
    return out


@pytest.mark.parametrize("order", [5, 20, 24])
def test_one_far_field_step_matches_the_model(order):
    """A one-step loop at orders other than 18.  Step 1 convects FREE alone through the tree and everything else in it
    is the all-pairs run's arithmetic on the same state, so (FREE_ff[1] - FREE_ap[1]) / dt is the tree's velocity minus
    the all-pairs velocity: it must equal oracle/tree_model.py's minus the exact all-pairs sum, to the tree's rounding
    (test_gpu_tree_orders.TOL of sum |terms|) plus the rounding of the positions."""
    from ludvm_b200 import LUDVM, ops
    from oracle import tree_model
    from test_gpu_tree_orders import TOL
    kw = dict(KW, tf=KW["dt"], **gust(NF), verbose=False, mode="fast")
    a = LUDVM(**kw)
    f = LUDVM(**kw, far_field_order=order)
    info = f.far_field_info
    assert info["far_field_steps"] == 1 and info["fallback_steps"] == 0 and info["order"] == order, info
    g = np.asarray(kw["circulation_freevort"], dtype=np.float64)
    x0, z0 = a.path["FREE"][0]
    assert biteq(f.path["FREE"][0], a.path["FREE"][0])
    vc4 = a.v_core ** 4
    um, wm, st = tree_model.tree_velocity(g, x0, z0, x0, z0, vc4, order=order)
    assert st["L"] == info["leaf_level"]
    ua, wa = ops.induced_velocity(g, x0, z0, x0, z0, a.v_core, mode="exact")
    d = (f.path["FREE"][1] - a.path["FREE"][1]) / a.dt
    den = _sum_abs_terms(g, x0, z0, vc4)
    pos = 4 * np.spacing(np.abs(a.path["FREE"][1])) / a.dt
    err = np.abs(d - np.stack([um - ua, wm - wa]))
    assert np.all(err <= TOL * den + pos), float(np.max((err - pos) / den))


def test_far_field_from_the_step_whose_wake_crosses_the_threshold():
    """nfree = 65526: the wake bounds of steps 0-2 (65530, 65532, 65534) are below SIM_FAR_FIELD_MIN_WAKE, steps 3-5 take
    the far field.  The first three steps are the run without the option bit for bit, and graph chunks of 2 or 7 steps,
    which ludvm_sim_run cuts at the first far-field step, change nothing."""
    from ludvm_b200 import LUDVM
    kw = dict(KW, **gust(65526), verbose=False, mode="fast")
    a = LUDVM(**kw)
    f = LUDVM(**kw, far_field_order=20)
    assert f.nt == 7
    assert f.far_field_info["far_field_steps"] == 3 and f.far_field_info["fallback_steps"] == 0, f.far_field_info
    for k in ("L", "D", "M", "LESP", "LEV_shed", "fourier"):
        assert biteq(getattr(f, k)[:4], getattr(a, k)[:4]), k
    for k in ("FREE", "TEV", "LEV"):
        assert biteq(f.path[k][:4], a.path[k][:4]), k
    assert not biteq(f.path["FREE"][4], a.path["FREE"][4])
    for K in (2, 7):
        c = LUDVM(**kw, far_field_order=20, steps_per_graph=K)
        assert c.far_field_info == f.far_field_info
        for k in ("L", "D", "M", "LESP", "LEV_shed", "fourier"):
            assert biteq(getattr(c, k), getattr(f, k)), (K, k)
        for k in ("FREE", "TEV", "LEV"):
            assert biteq(c.path[k], f.path[k]), (K, k)
