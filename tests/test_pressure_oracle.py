"""The chordwise pressure jump dp (LUDVM(..., pressure=True)) pinned on the CPU oracle: `pressure_jump` restates the
definition the device evaluates, and the physics checks below tie that definition to thin-aerofoil theory and to the
normal force the time loop already computes.  The device is compared with `pressure_jump` in test_gpu_pressure.py."""
import numpy as np
import pytest

README = dict(t0=0, tf=20, dt=5e-2, chord=1, rho=1.225, Uinf=1, Npoints=81, Ncoeffs=30, LESPcrit=0.2, Naca="0012")


def pressure_jump(o):
    """dp [nt, P] of a finished OracleLUDVM run.  For step i >= 1, itev = i - 1, in this operation order:
        vrel  = Uinf*cos_a[i] + h_dot[i]*sin_a[i]
        u     = u1*cos_a[i] - w1*sin_a[i]
        dp[i] = rho * ((vrel + u) * gamma_airfoil[itev] + (Gamma_airfoil[itev] - Gamma_airfoil[itev-1]) / dt)
    with Gamma_airfoil[itev-1] = 0 at itev = 0 and (u1, w1) the velocity the wake TEV[:itev+1] ++ LEV[:ilev+1] ++ FREE
    induces at the gamma points before the step's convection (LUDVM.py:1049-1057), i.e. the tangential velocity whose
    product with gamma the normal force integrates.  cos_a / sin_a are the array evaluations the step tables hold.
    dp[0] = 0."""
    nt, P = o.nt, o.Npoints - 1
    dp = np.zeros([nt, P])
    ca, sa = np.cos(o.alpha), np.sin(o.alpha)
    gam, Gam = o.circulation['gamma_airfoil'], o.circulation['Gamma_airfoil']
    gpts = o.path['airfoil_gamma_points']
    ilev = 0
    for i in range(1, nt):
        itev = i - 1
        g, xw, zw = o._wake_before_convection(i, ilev)
        u1, w1 = o.induced_velocity(g, xw, zw, gpts[i, 0, :], gpts[i, 1, :])
        u = u1 * ca[i] - w1 * sa[i]
        vrel = o.Uinf * ca[i] + o.h_dot[i] * sa[i]
        Gprev = Gam[itev - 1] if itev >= 1 else 0.0
        dp[i] = o.rho * ((vrel + u) * gam[itev] + (Gam[itev] - Gprev) / o.dt)
        if o.LEV_shed[i] != -1:
            ilev += 1
    return dp


def test_steady_flat_plate_matches_thin_aerofoil_theory(oracle):
    """A plate held at 5 degrees (k -> 0, no plunge, no LEV): Delta Cp -> 4 alpha sqrt((c - x) / x).  The run's lift is
    still 5 % below 2 pi alpha at t* = 20 (Wagner), so the shape is compared after dividing by the run's own
    Cl / (2 pi alpha).  Panels aft of mid-chord are left out: there the 30-term Fourier series rings."""
    o = oracle.OracleLUDVM(**dict(README, alpha_max=5, phi=0, k=1e-4, h_max=0, LESPcrit=10))
    assert np.all(o.LEV_shed == -1)
    dp = pressure_jump(o)
    q = 0.5 * o.rho * o.Uinf ** 2
    c, x = o.chord, o.airfoil['x_panel']
    fore = x < 0.5 * c
    for i in (200, 400):
        lag = o.L[i] / (q * c) / (2 * np.pi * o.alpha[i])
        ratio = dp[i] / q / (4 * o.alpha[i] * np.sqrt((c - x) / x)) / lag
        assert np.all(np.abs(ratio[fore] - 1) <= 0.03), (i, ratio[fore].min(), ratio[fore].max())


def test_readme_pressure_integrates_to_the_normal_force(oracle):
    """trapz(dp, x_p) is the normal force Fn on steps that shed no LEV (same wake term rho trapz(u gamma, x_p); the
    rest differs only by the trapezoidal rule against the Fourier closed form).  Shedding steps are left out: there Fn
    keeps the Fourier rates of before the shedding iteration (SURVEY.md B.5)."""
    o = oracle.OracleLUDVM(**README)
    dp = pressure_jump(o)
    x = o.airfoil['x_panel']
    Fi = np.array([np.trapezoid(dp[i], x) for i in range(o.nt)])
    steps = np.arange(2, o.nt)
    calm = steps[o.LEV_shed[steps] == -1]
    assert len(calm) > 100 and (o.LEV_shed != -1).any()
    assert np.max(np.abs(Fi[calm] - o.Fn[calm])) <= 2e-2 * np.max(np.abs(o.Fn))
    assert not np.any(dp[0]) and np.all(o.dp == 0)     # the oracle's own dp stays the reference's zeros


def test_pressure_is_keyword_only_and_off_by_default():
    import inspect
    from ludvm_b200 import LUDVM
    p = inspect.signature(LUDVM.__init__).parameters["pressure"]
    assert p.kind is inspect.Parameter.KEYWORD_ONLY and p.default is False


def test_sweep_rejects_pressure():
    """Sweep cases keep no bound-vortex history, so a case asking for the pressure jump is refused before any device
    work instead of being run without it."""
    from ludvm_b200 import sweep
    cases = sweep.lespcrit_k_grid((0.1, 0.2), (0.2,), tf=1, dt=5e-2, Npoints=81, Naca="0012")
    cases[1]["pressure"] = True
    with pytest.raises(ValueError, match="pressure"):
        sweep.run_sweep(cases)
