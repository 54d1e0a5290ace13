"""The chordwise pressure jump dp (LUDVM(..., pressure=True)) on every step driver: exact mode bit-equal to the
restatement in test_pressure_oracle.py, fast mode consistent with its own normal force, and no other output moved by
switching it on."""
import functools

import numpy as np
import pytest

from conftest import biteq
from test_pressure_oracle import README, pressure_jump

pytestmark = pytest.mark.gpu

HIST = ("Fn", "Fs", "L", "D", "T", "M", "LESP", "LESP_prev", "LEV_shed", "fourier")


def _gust(nf, seed):
    rng = np.random.default_rng(seed)
    xy = np.stack([rng.uniform(-6.0, -0.5, nf), rng.uniform(-1.0, 1.0, nf)])
    return dict(circulation_freevort=rng.standard_normal(nf) * 1e-3, xy_freevort=xy)


SHORT = dict(README, tf=0.2)
CASES = {   # name -> (constructor kwargs, environment)
    "cluster_then_coop": (README, {}),
    "coop": (README, {"LUDVM_NO_CLUSTER": "1"}),
    "graph": (README, {"LUDVM_NO_CLUSTER": "1", "LUDVM_NO_COOP": "1"}),
    "ramesh_cta": (dict(README, tf=3, method="Ramesh"), {}),
    # 8400 free vortices: exact-mode graph path with the tiled convection (k_conv_partials_exact_tiled)
    "exact_tiled": (dict(SHORT, **_gust(8400, 11)), {}),
    "npoints_1025": (dict(README, tf=0.6, Npoints=1025, Ncoeffs=12, LESPcrit=0.05, alpha_max=30, k=3), {}),
}
FAST_CASES = {
    "cluster_then_coop": (README, {}),
    "graph": (README, {"LUDVM_NO_CLUSTER": "1", "LUDVM_NO_COOP": "1"}),
    "ramesh_cta": (dict(README, tf=3, method="Ramesh"), {}),
    # 9000 free vortices: the overlapped fast step (k_conv_old_tiled beside the solve, then k_finish_ov)
    "overlapped": (dict(README, tf=0.3, **_gust(9000, 9)), {}),
}


def _run(kw, env, monkeypatch, **extra):
    from ludvm_b200 import LUDVM
    with monkeypatch.context() as m:
        for k, v in env.items():
            m.setenv(k, v)
        return LUDVM(**kw, verbose=False, **extra)


@functools.lru_cache(maxsize=None)
def _oracle_dp(name):
    from oracle import ludvm_oracle
    ludvm_oracle.build()
    o = ludvm_oracle.OracleLUDVM(**CASES[name][0])
    return o, pressure_jump(o)


def _same_except_dp(a, b):
    """Every output of two runs of one case other than dp / Cp is bit-identical."""
    for k in HIST + ("Cl", "Cd", "Cm", "Cn", "Cs", "Ct"):
        assert biteq(getattr(a, k), getattr(b, k)), k
    for k in ("TEV", "LEV", "bound", "airfoil", "gamma_airfoil", "Gamma_airfoil"):
        assert biteq(a.circulation[k], b.circulation[k]), k
    for k in ("TEV", "LEV", "FREE", "TEV_last", "LEV_last", "FREE_last"):
        assert (k in a.path) == (k in b.path) and (k not in a.path or biteq(a.path[k], b.path[k])), k
    assert (a.itev, a.ilev, a.steps_done) == (b.itev, b.ilev, b.steps_done)


def _check_on_off(on, off):
    _same_except_dp(on, off)
    assert off.dp.shape == on.dp.shape == (on.nt, on.Npoints - 1)
    assert not np.any(off.dp) and not np.any(off.Cp)
    assert not np.any(on.dp[0]) and np.all(np.isfinite(on.dp)) and np.any(on.dp[1:])
    assert biteq(on.Cp, on.dp / (0.5 * on.rho * on.Uinf ** 2))


@pytest.mark.parametrize("name", list(CASES))
def test_exact_pressure_bit_equal_to_oracle(name, monkeypatch):
    kw, env = CASES[name]
    on = _run(kw, env, monkeypatch, pressure=True)
    off = _run(kw, env, monkeypatch)
    _check_on_off(on, off)
    o, dp = _oracle_dp(name)
    assert biteq(on.L, o.L) and biteq(on.circulation["Gamma_airfoil"], o.circulation["Gamma_airfoil"])
    assert biteq(on.dp, dp)


def _fn_identity(s):
    """trapz(dp/rho - dGamma/dt - vrel gamma, x_p) against (Fn - rho pi c U [vrel (A0 + A1/2) + c (3/4 A0' + 1/4 A1'
    + 1/8 A2')]) / rho, step by step: both are trapz(u gamma, x_p) of the same u and gamma."""
    rho, U, c, dt = s.rho, s.Uinf, s.chord, s.dt
    x = s.airfoil["x_panel"]
    gam, Gam = s.circulation["gamma_airfoil"], s.circulation["Gamma_airfoil"]
    vrel = U * np.cos(s.alpha) + s.h_dot * np.sin(s.alpha)
    err = 0.0
    for i in range(1, s.nt):
        itev = i - 1
        dG = Gam[itev] - (Gam[itev - 1] if itev >= 1 else 0.0)
        lhs = np.trapezoid(s.dp[i] / rho - dG / dt - vrel[i] * gam[itev], x)
        A, Ad = s.fourier[i, 0], s.fourier[i, 1]
        rhs = (s.Fn[i] - rho * np.pi * c * U * (vrel[i] * (A[0] + A[1] / 2) + c * (0.75 * Ad[0] + 0.25 * Ad[1] + 0.125 * Ad[2]))) / rho
        err = max(err, abs(lhs - rhs))
    return err


@pytest.mark.parametrize("name", list(FAST_CASES))
def test_fast_pressure_consistent_with_normal_force(name, monkeypatch):
    """A dp formed from a half-written Gamma row, or from another wake velocity than the loads', breaks the identity."""
    kw, env = FAST_CASES[name]
    on = _run(kw, env, monkeypatch, pressure=True, mode="fast")
    off = _run(kw, env, monkeypatch, mode="fast")
    _check_on_off(on, off)
    assert _fn_identity(on) <= 1e-12 * np.max(np.abs(on.Fn))


def test_fast_pressure_tracks_oracle_before_chaos(monkeypatch):
    """README case, fast arithmetic: within 1e-9 of max|dp| of the exact restatement over the first 100 steps."""
    on = _run(README, {}, monkeypatch, pressure=True, mode="fast")
    _, dp = _oracle_dp("cluster_then_coop")
    assert np.max(np.abs(on.dp[:101] - dp[:101])) <= 1e-9 * np.max(np.abs(dp))


def test_enable_and_fetch_states(monkeypatch):
    """ludvm_sim_enable_pressure only before the first step; fetching DP of a run without it is refused."""
    from ludvm_b200 import LUDVM, _lib
    L = _lib.load()
    s = LUDVM(**dict(README, tf=1), verbose=False, run=False)
    s.time_loop(nsteps=5)
    buf = np.empty((s.nt, s.Npoints - 1))
    assert L.ludvm_sim_fetch(s._sim, _lib.FIELDS["DP"], buf.ctypes.data, buf.nbytes) == -4     # LUDVM_E_STATE
    assert L.ludvm_sim_enable_pressure(s._sim) == -4
    assert not np.any(s.dp)


@pytest.mark.parametrize("store_history", [0, 5])
def test_pressure_with_reduced_history(store_history, monkeypatch):
    kw = dict(README, tf=6)
    full = _run(kw, {}, monkeypatch, pressure=True)
    part = _run(kw, {}, monkeypatch, pressure=True, store_history=store_history)
    assert biteq(part.dp, full.dp) and biteq(part.L, full.L)


def test_pressure_nsteps_prefix(monkeypatch):
    """time_loop(nsteps=n): rows 1..n equal the full run's, the rows of steps not run stay zero."""
    from ludvm_b200 import LUDVM
    kw = dict(README, tf=6)
    full = _run(kw, {}, monkeypatch, pressure=True)
    s = LUDVM(**kw, verbose=False, run=False, pressure=True)
    s.time_loop(nsteps=73)
    assert s.steps_done == 73
    assert biteq(s.dp[:74], full.dp[:74]) and not np.any(s.dp[74:])
