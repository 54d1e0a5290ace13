"""The chordwise pressure jump of batched parameter sweeps (sweep.run_sweep over cases with pressure=True) on every
instantiation of the one-CTA-per-case driver: exact mode bit-equal to the restatement in test_pressure_oracle.py and
to single runs, fast mode close to exact before chaos, and no other output moved by switching it on."""
import functools

import numpy as np
import pytest

from conftest import biteq
from test_pressure_oracle import README, pressure_jump

pytestmark = pytest.mark.gpu

COMBOS = [(0.1, 0.1), (0.1, 1.0), (0.4, 0.1), (0.4, 1.0), (0.25, 0.55)]   # test_sweep_matches_reference_golden_...
GRID = dict(lespcrits=np.linspace(0.1, 0.4, 3), ks=np.linspace(0.1, 1.0, 4), tf=5)


def _with_pressure(cases):
    return [dict(kw, pressure=True) for kw in cases]


@functools.lru_cache(maxsize=None)
def _oracle_dp(items):
    from oracle import ludvm_oracle
    ludvm_oracle.build()
    return pressure_jump(ludvm_oracle.OracleLUDVM(**dict(items)))


def oracle_dp(kw):
    return _oracle_dp(tuple(sorted(kw.items())))


def _grid():
    from ludvm_b200 import sweep
    g = GRID
    return sweep.lespcrit_k_grid(g["lespcrits"], g["ks"], **dict(README, tf=g["tf"]))


def _close(a, ref):
    return np.max(np.abs(a - ref)) <= 1e-9 * np.max(np.abs(ref))


def test_exact_sweep_pressure_bit_equal_to_oracle_and_single_runs():
    """Five corner/interior cases of the LESPcrit x k grid, 128-thread exact driver."""
    from ludvm_b200 import LUDVM, sweep
    cases = [dict(README, LESPcrit=lc, k=k) for lc, k in COMBOS]
    res = sweep.run_sweep(_with_pressure(cases), mode="exact")
    assert res["dp"].shape == res["Cp"].shape == (len(cases), res["nt"], README["Npoints"] - 1)
    for a, kw in enumerate(cases):
        assert biteq(res["dp"][a], oracle_dp(kw)), a
        assert biteq(res["Cp"][a], LUDVM(**kw, verbose=False, pressure=True).Cp), a


@pytest.mark.parametrize("mode", ["exact", "fast"])
def test_sweep_pressure_leaves_other_outputs_unchanged(mode):
    from ludvm_b200 import sweep
    cases = _grid()
    off = sweep.run_sweep(cases, mode=mode)
    on = sweep.run_sweep(_with_pressure(cases), mode=mode)
    assert "dp" not in off and "Cp" not in off
    for k in sweep.SW_FIELDS + ("Cl", "Cd", "Ct", "Cn", "Cs", "Cm"):
        assert biteq(on[k], off[k]), k
    assert not np.any(on["dp"][:, 0]) and np.all(np.isfinite(on["dp"])) and np.all(np.any(on["dp"][:, 1:], axis=(1, 2)))


def test_ramesh_sweep_pressure_bit_equal_to_oracle():
    """method='Ramesh': the 256-thread Ramesh sweep driver."""
    from ludvm_b200 import sweep
    cases = [dict(README, tf=3, method="Ramesh", LESPcrit=lc) for lc in (0.1, 0.2, 0.3)]
    res = sweep.run_sweep(_with_pressure(cases), mode="exact")
    for a, kw in enumerate(cases):
        assert biteq(res["dp"][a], oracle_dp(kw)), a


def test_sweep_pressure_with_many_free_vortices():
    """700 free vortices (base of test_sweep_with_many_free_vortices_covers_the_wide_shared_memory_tiles): the wide
    shared-memory tiles; exact bit-equal to the oracle, the fast 256-thread driver close to exact."""
    from oracle import ludvm_oracle
    from ludvm_b200 import sweep
    rng = np.random.default_rng(13)
    nf = 700
    xy = np.stack([rng.uniform(-4.0, -0.5, nf), rng.uniform(-0.6, 0.6, nf)])
    gam = rng.standard_normal(nf) * 2e-3
    base = dict(README, tf=1, circulation_freevort=gam, xy_freevort=xy)
    cases = [dict(base, LESPcrit=0.15), dict(base, LESPcrit=0.3, k=0.5)]
    ex = sweep.run_sweep(_with_pressure(cases), mode="exact")
    fa = sweep.run_sweep(_with_pressure(cases), mode="fast")
    ludvm_oracle.build()
    assert biteq(ex["dp"][1], pressure_jump(ludvm_oracle.OracleLUDVM(**cases[1])))
    assert _close(fa["dp"], ex["dp"]), np.max(np.abs(fa["dp"] - ex["dp"])) / np.max(np.abs(ex["dp"]))


def test_fast_sweep_pressure_tracks_exact_and_single_fast_runs_before_chaos():
    """README-size cases, first 100 steps: the fast sweep within 1e-9 of max|dp| of the exact sweep and of
    LUDVM(..., mode='fast', pressure=True)."""
    from ludvm_b200 import LUDVM, sweep
    cases = [README, dict(README, LESPcrit=0.1, k=0.1), dict(README, LESPcrit=0.4, k=0.1)]
    ex = sweep.run_sweep(_with_pressure(cases), mode="exact")["dp"][:, :101]
    fa = sweep.run_sweep(_with_pressure(cases), mode="fast")["dp"][:, :101]
    assert _close(fa, ex), np.max(np.abs(fa - ex)) / np.max(np.abs(ex))
    for a, kw in enumerate(cases):
        single = LUDVM(**kw, verbose=False, mode="fast", pressure=True).dp[:101]
        assert _close(fa[a], single), (a, np.max(np.abs(fa[a] - single)) / np.max(np.abs(single)))


def test_sweep_pressure_npoints_1025():
    """1024 panels: the solve needs more than 48 KB of dynamic shared memory in the DP instantiations too."""
    from ludvm_b200 import sweep
    base = dict(README, tf=0.6, Npoints=1025, Ncoeffs=12, alpha_max=30, k=3)
    cases = [dict(base, LESPcrit=0.05), dict(base, LESPcrit=0.1)]
    res = sweep.run_sweep(_with_pressure(cases), mode="exact")
    for a, kw in enumerate(cases):
        assert biteq(res["dp"][a], oracle_dp(kw)), a


def test_split_sweep_pressure_equals_full_sweep():
    from ludvm_b200 import sweep
    cases = _with_pressure(_grid())
    full = sweep.run_sweep(cases, mode="exact")
    lo = sweep.run_sweep(cases, mode="exact", case_slice=slice(0, 7))
    hi = sweep.run_sweep(cases, mode="exact", case_slice=slice(7, None))
    assert biteq(np.concatenate([lo["dp"], hi["dp"]]), full["dp"])
    assert biteq(np.concatenate([lo["Cp"], hi["Cp"]]), full["Cp"])
