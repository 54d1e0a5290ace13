"""method='Ramesh' on the single-simulation drivers (single cluster, cooperative grid, CUDA graphs): exact mode bit-equal
to the oracle and the reference's golden run, fast mode within the fast-mode envelope of exact mode.  The Newton
evaluations re-evaluate only the phase-1 tree nodes that hold the step's TEV and LEV (exact) or add the two new vortices
to the old wake's sums (fast); these tests pin both against the oracle's full re-summation."""
import ctypes as C

import numpy as np
import pytest

from conftest import biteq, golden_tables, load_golden
from test_pressure_oracle import pressure_jump

pytestmark = pytest.mark.gpu

README = dict(t0=0, tf=20, dt=5e-2, chord=1, rho=1.225, Uinf=1, Npoints=81, Ncoeffs=30, LESPcrit=0.2, Naca="0012")
SHED = dict(README, tf=4, LESPcrit=0.1, method="Ramesh")   # LEVs shed from the first steps: the 2-D Newton runs
HIST = ("Fn", "Fs", "L", "D", "T", "M", "LESP", "LESP_prev", "LEV_shed", "fourier")
DRIVERS = {"cluster_then_coop": {}, "coop": {"LUDVM_NO_CLUSTER": "1"},
           "graph": {"LUDVM_NO_CLUSTER": "1", "LUDVM_NO_COOP": "1"}}


def _gust(nf, seed):
    rng = np.random.default_rng(seed)
    xy = np.stack([rng.uniform(-6.0, -0.5, nf), rng.uniform(-1.0, 1.0, nf)])
    return dict(circulation_freevort=rng.standard_normal(nf) * 1e-3, xy_freevort=xy)


def _run(kw, drv, monkeypatch, **extra):
    from ludvm_b200 import LUDVM
    with monkeypatch.context() as m:
        for k, v in DRIVERS[drv].items():
            m.setenv(k, v)
        return LUDVM(**kw, verbose=False, **extra)


def _assert_bit_equal(s, o):
    for k in HIST + ("Cl", "Cd", "Cm"):
        assert biteq(getattr(s, k), getattr(o, k)), k
    for k in ("TEV", "LEV", "FREE"):
        assert biteq(s.path[k], o.path[k]), k
    for k in ("TEV", "LEV", "bound", "airfoil", "gamma_airfoil", "Gamma_airfoil"):
        assert biteq(s.circulation[k], o.circulation[k]), k
    assert (s.itev, s.ilev) == (o.itev, o.ilev)


@pytest.mark.parametrize("drv", list(DRIVERS))
def test_exact_shedding_bit_equal_to_oracle(oracle, drv, monkeypatch):
    s, o = _run(SHED, drv, monkeypatch), oracle.OracleLUDVM(**SHED)
    assert o.ilev > 10
    _assert_bit_equal(s, o)


@pytest.mark.parametrize("drv", list(DRIVERS))
def test_golden_ramesh_tf2_on_every_driver(drv, monkeypatch):
    from ludvm_b200 import LUDVM
    g = load_golden("ramesh_tf2")
    tb = golden_tables(g)
    tb["sum_free"] = float(np.sum(tb["free_g"]))
    with monkeypatch.context() as m:
        for k, v in DRIVERS[drv].items():
            m.setenv(k, v)
        s = LUDVM(**g["kw"], verbose=False, run=False)
        s.time_loop(tables=tb)
    s.compute_coefficients()
    for k in ("Fn", "Fs", "L", "D", "M", "LESP", "LESP_prev", "LEV_shed", "fourier", "Cl", "Cd", "Cm"):
        assert biteq(getattr(s, k), g[k]), k
    for k in ("TEV", "LEV", "bound"):
        assert biteq(s.circulation[k], g["circ_" + k]), k
    for k in ("TEV", "LEV", "FREE"):
        assert biteq(s.path[k][g["path_rows"]], g["path_" + k + "_rows"]), k
    assert [s.itev, s.ilev] == list(g["itev_ilev"])


def test_exact_tiled_graph_step(oracle, monkeypatch):
    """8400 free vortices: the graph path's k_conv_partials_exact_tiled under Ramesh."""
    kw = dict(README, tf=0.2, method="Ramesh", **_gust(8400, 11))
    s, o = _run(kw, "cluster_then_coop", monkeypatch), oracle.OracleLUDVM(**kw)
    _assert_bit_equal(s, o)


def test_many_chord_stations(oracle, monkeypatch):
    kw = dict(README, tf=0.6, Npoints=401, Ncoeffs=40, LESPcrit=0.05, alpha_max=30, k=3, method="Ramesh")
    o = oracle.OracleLUDVM(**kw)
    assert o.ilev > 0
    for drv in ("cluster_then_coop", "graph"):
        _assert_bit_equal(_run(kw, drv, monkeypatch), o)


@pytest.mark.parametrize("drv", ["coop", "graph"])
def test_outside_the_range_proof(oracle, drv, monkeypatch):
    """Free vortices at z = +-1e-300 and a subnormal x: the flagged pair arithmetic, in phase 1 and in the dirty nodes."""
    xy = np.array([[-1.0, -2.0, -1e-310, -3.0], [0.3, 1e-300, -0.2, -1e-300]])
    gam = np.array([0.01, -0.02, 0.015, 0.005])
    kw = dict(README, tf=1.5, method="Ramesh", circulation_freevort=gam, xy_freevort=xy)
    s, o = _run(kw, drv, monkeypatch), oracle.OracleLUDVM(**kw)
    assert not s.range_proof_held
    _assert_bit_equal(s, o)


def test_outside_the_range_proof_sweep(oracle):
    """The one-CTA sweep driver's flagged path (k_sim_cta, Faure and Ramesh) with the same out-of-window free vortices."""
    from ludvm_b200 import sweep
    xy = np.array([[-1.0, -2.0, -1e-310, -3.0], [0.3, 1e-300, -0.2, -1e-300]])
    gam = np.array([0.01, -0.02, 0.015, 0.005])
    for method in ("Ramesh", "Faure"):
        cases = [dict(README, tf=1.5, method=method, LESPcrit=lc, circulation_freevort=gam, xy_freevort=xy)
                 for lc in (0.1, 0.2)]
        res = sweep.run_sweep(cases, mode="exact")
        for a, kw in enumerate(cases):
            o = oracle.OracleLUDVM(**kw)
            for k in ("Cl", "Cd", "Cm", "LESP", "LEV_shed", "L", "M"):
                assert biteq(res[k][a], getattr(o, k)), (method, a, k)
            assert biteq(res["circulation_TEV"][a][:-1], o.circulation["TEV"])


@pytest.mark.parametrize("drv", list(DRIVERS))
def test_pressure_bit_equal_to_oracle(oracle, drv, monkeypatch):
    kw = dict(SHED, tf=2)
    s, o = _run(kw, drv, monkeypatch, pressure=True), oracle.OracleLUDVM(**kw)
    _assert_bit_equal(s, o)
    assert biteq(s.dp, pressure_jump(o))


def _pw_left(n):
    n2 = n // 2
    return n2 - n2 % 8


def _node(n, d, e):
    """(node, first element of the node) of logical element e at cut depth d (sim.cu pw_node_of)."""
    b, off = 0, 0
    for lvl in range(d - 1, -1, -1):
        n2 = _pw_left(n)
        if e - off >= n2:
            b |= 1 << lvl
            off += n2
            n -= n2
        else:
            n = n2
    return b, off


def _depth(n):
    d = 0
    while n > 128:
        n = _pw_left(n)
        d += 1
    return min(d, 6)   # graph driver: the phase-1 cut is capped at SIM_WOF_MAX_DEPTH


@pytest.mark.parametrize("nfree,tf", [(1, 1.0), (120, 0.6), (250, 0.6), (1, 12.0)])
def test_dirty_node_edges(oracle, nfree, tf, monkeypatch):
    """Graph driver, exact: Newton wakes of n = itev + ilev + 2 + nfree crossing 8, 128 (cut depth 0 -> 1), 256 and a
    pw_left split, with the TEV and the LEV slot in one node, in two nodes, and first in a node."""
    rng = np.random.default_rng(nfree)
    fv = dict(circulation_freevort=rng.standard_normal(nfree) * 1e-3,
              xy_freevort=np.stack([rng.uniform(-4.0, -0.5, nfree), rng.uniform(-1.0, 1.0, nfree)]))
    kw = dict(README, tf=tf, LESPcrit=0.1, method="Ramesh", **fv)
    s, o = _run(kw, "graph", monkeypatch), oracle.OracleLUDVM(**kw)
    _assert_bit_equal(s, o)
    # which cases the run covered (ilev at the start of step i from LEV_shed)
    seen = set()
    ilev = 0
    for i in range(1, s.nt):
        itev = i - 1
        n = itev + ilev + 2 + nfree
        d = _depth(n)
        (b0, o0), (b1, o1) = _node(n, d, itev), _node(n, d, itev + 1 + ilev)
        if d > 0:
            seen.add("same" if b0 == b1 else "split")
            if o1 == itev + 1 + ilev or o0 == itev:
                seen.add("first")
        for edge in (8, 128, 256):
            if n == edge or n == edge + 1:
                seen.add(edge)
        if s.LEV_shed[i] != -1:
            ilev += 1
    if nfree == 1 and tf < 2:
        assert 8 in seen
    if nfree == 120:
        assert 128 in seen
    if nfree == 250:
        assert {256, "first"} <= seen
    if tf > 2:
        assert {128, 256, "same", "split"} <= seen


@pytest.mark.parametrize("drv", ["graph", "coop", "cluster_then_coop"])
def test_fast_tracks_exact(drv, monkeypatch):
    """Fast mode (the overlapped step on the graph path with 9000 free vortices; the single cluster, then the
    cooperative grid, or the cooperative grid alone on the README case): L, D, M within 1e-10 of max|.| of exact Ramesh before chaos, LEV_shed equal, and dp consistent with Fn."""
    from test_gpu_pressure import _fn_identity
    kw = dict(README, tf=0.3, method="Ramesh", **_gust(9000, 9)) if drv == "graph" else dict(SHED, tf=3)
    e = _run(kw, drv, monkeypatch)
    f = _run(kw, drv, monkeypatch, mode="fast", pressure=True)
    for k in ("L", "D", "M"):
        ref = getattr(e, k)
        assert np.max(np.abs(getattr(f, k)[:60] - ref[:60])) <= 1e-10 * np.max(np.abs(ref)), k
    assert np.array_equal(f.LEV_shed[:60], e.LEV_shed[:60])
    assert _fn_identity(f) <= 1e-12 * np.max(np.abs(f.Fn))


def test_profile_steps_and_launch_counts(monkeypatch):
    """ludvm_sim_profile_steps times the four phases of a Ramesh step; the graph path launches per-step kernels."""
    from ludvm_b200 import LUDVM, _lib
    L = _lib.load()
    kw = dict(SHED, tf=1)
    with monkeypatch.context() as m:
        for k, v in DRIVERS["graph"].items():
            m.setenv(k, v)
        s = LUDVM(**kw, verbose=False, run=False, steps_per_graph=5)
        s.time_loop(nsteps=0)
        ms = (C.c_double * 5)()
        assert L.ludvm_sim_profile_steps(s._sim, 3, ms) == 0
        assert all(ms[q] > 0 for q in range(4)) and ms[4] > 0
        l0 = s.ctx.launch_count()
        _lib.check(L.ludvm_sim_run(s._sim, 10))
        s.ctx.synchronize()
    assert s.ctx.launch_count() - l0 == 2 * (4 * 5 + 1)   # two graphs of 5 steps: 4 kernels a step + k_advance
