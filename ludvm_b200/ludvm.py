"""Drop-in `LUDVM` class: the reference's constructor, attributes and method surface (LUDVM.py:132-1372) with the
per-timestep vortex-velocity path executed by libludvm_b200.so on a B200.

What stays on the host (one-off O(nt*Npoints) set-up, evaluated with numpy exactly as the reference does so
that the device consumes bit-identical tables): `airfoil_generation` (LUDVM.py:299), `motion_sinusoidal`
(LUDVM.py:382), `motion_plunge` (LUDVM.py:459), `compute_coefficients` (LUDVM.py:1173).
What runs on the GPU through the C ABI: `induced_velocity` (LUDVM.py:549), `airfoil_downwash` (LUDVM.py:572),
`time_loop` (LUDVM.py:597), `flowfield` (LUDVM.py:1186).

Extra keyword-only arguments (not in the reference): `mode` ('exact' bit-reproduces numpy, 'fast' uses FMA
arithmetic), `device`, `store_history`, `motion`, `run`, `steps_per_graph`, `pressure` (True: `time_loop` fills the
chordwise pressure jump `dp` [nt, Npoints-1] and so `Cp`, which the reference allocates but leaves zero; see
`time_loop`), `far_field_order` (fast mode: convect large wakes through the treecode far field; see `time_loop`).
"""
import ctypes as C
import timeit

import numpy as np

from . import _lib, ops
from ._lib import FIELDS, SimParams, SimTables, TABLE_FIELDS, check, f64, load

__all__ = ["LUDVM"]


def _naca4_camber(naca, x):
    """Analytic NACA 4-digit mean line on x/c in [0,1].  The reference obtains it from the un-vendored PyPI
    package `airfoils` (LUDVM.py:328-335; no version pinned) -- identical (zero) for symmetric 00xx sections,
    parity unpinned for cambered ones."""
    m, p = int(naca[0]) / 100.0, int(naca[1]) / 10.0
    x = np.asarray(x, dtype=np.float64)
    if m == 0.0 or p == 0.0:
        return np.zeros_like(x)
    fore = m / p ** 2 * (2 * p * x - x ** 2)
    aft = m / (1 - p) ** 2 * ((1 - 2 * p) + 2 * p * x - x ** 2)
    return np.where(x < p, fore, aft)


def _read_uiuc(filename):
    """Upper/lower surfaces of a Selig-format UIUC .dat file (replaces airfoils.fileio.import_airfoil_data)."""
    pts = []
    with open(filename) as fh:
        for line in fh:
            parts = line.replace(",", " ").split()
            if len(parts) == 2:
                try:
                    pts.append((float(parts[0]), float(parts[1])))
                except ValueError:
                    pass
    pts = np.array(pts)
    ile = int(np.argmin(pts[:, 0]))
    upper, lower = pts[:ile + 1][::-1], pts[ile:]
    return upper.T, lower.T


class LUDVM:
    """LESP-modulated unsteady discrete-vortex method; see the reference docstring (LUDVM.py:133-230)."""

    def __init__(self, t0=0, tf=12, dt=1.5e-2, chord=1, rho=1.225, Uinf=1, Npoints=80, Ncoeffs=30,
                 LESPcrit=0.2, Naca='0012', foil_filename=None, G=1, T=2, alpha_m=0, alpha_max=10,
                 k=0.2 * np.pi, phi=90, h_max=1, verbose=True, method='Faure',
                 circulation_freevort=None, xy_freevort=None, *, mode='exact', device=0, store_history=True,
                 motion='cos', run=True, steps_per_graph=0, ctx=None, pressure=False, far_field_order=None):
        # LUDVM.py:237-260
        self.t0, self.tf, self.dt = t0, tf, dt
        self.chord, self.rho, self.Uinf = chord, rho, Uinf
        self.Npoints, self.Ncoeffs = Npoints, Ncoeffs
        self.piv = 0.25 * chord
        self.LESPcrit = LESPcrit
        self.maxerror, self.maxiter, self.epsilon = 1e-10, 50, 1e-4
        self.xgamma = 0.25
        self.method = method
        self.t = np.arange(t0, tf + dt, dt)
        self.nt = len(self.t)
        self.verbose = verbose
        self.dt_star = dt * Uinf / chord
        self.v_core = 1.3 * self.dt_star * chord
        self.ilev2 = 0
        self.alpha_m = alpha_m
        if circulation_freevort is not None and xy_freevort is not None:   # LUDVM.py:268-277
            self.n_freevort = len(circulation_freevort)
            self.circulation_freevort = circulation_freevort
            self.xy_freevort = xy_freevort
        else:
            self.n_freevort = 1
            self.circulation_freevort = np.array([0])
            self.xy_freevort = np.array([0, 0])[:, np.newaxis]
        # device options
        if mode not in ("exact", "fast"):
            raise ValueError("mode must be 'exact' or 'fast'")
        # store_history: True / 1 = the reference's full [nt,2,nt-1] vortex paths; False / 0 = latest positions only;
        # k > 1 = strided snapshots (rows of steps i % k == 0), the O(nt^2) history is the memory wall at dt=2e-3, tf=40
        self.mode, self.device, self.store_history = mode, device, int(store_history)
        if self.store_history < 0:
            raise ValueError('store_history must be >= 0')
        self.steps_per_graph = int(steps_per_graph)
        self.pressure = bool(pressure)
        # far_field_order=p (2..24, 18 documented): time_loop convects large wakes through the treecode (see time_loop)
        if far_field_order is not None:
            if mode == 'exact':
                raise ValueError("far_field_order needs mode='fast': exact mode reproduces numpy's sums bit for bit")
            if method == 'Ramesh':
                raise ValueError("far_field_order is available for method='Faure' only (the far-field step is built on Faure's solve)")
            if Npoints > 257:
                raise ValueError("far_field_order supports Npoints <= 257 (the overlapped step needs at most 256 panels)")
            if isinstance(far_field_order, bool) or int(far_field_order) != far_field_order or not 2 <= far_field_order <= 24:
                raise ValueError("far_field_order must be an integer in 2..24 (18: the all-pairs fast kernel's accuracy)")
            far_field_order = int(far_field_order)
        self.far_field_order = far_field_order
        self.far_field_info = None
        self._ctx = ctx
        self._sim = None

        self.start_time = timeit.default_timer()
        if Naca is not None:
            self.airfoil_generation(Naca=Naca)
        else:
            self.airfoil_generation(Naca=None, filename=foil_filename)
        self.motion_sinusoidal(alpha_m=alpha_m, alpha_max=alpha_max, h_max=h_max, k=k, phi=phi, h0=0, x0=0,
                               motion=motion)
        if run:
            self.time_loop()
            self.compute_coefficients()
            if verbose:
                print('Elapsed time:', timeit.default_timer() - self.start_time)

    # ------------------------------------------------------------------------------------------------
    # host-side set-up
    # ------------------------------------------------------------------------------------------------
    @property
    def ctx(self):
        if self._ctx is None:
            self._ctx = _lib.default_context(self.device)
        return self._ctx

    def airfoil_generation(self, Naca='0012', filename=None, Npoints=None, uniform_spacing='theta'):
        """Camber line, cosine-spaced stations, gamma points at 25% of each panel (LUDVM.py:299-380)."""
        if Npoints is None:
            Npoints = self.Npoints
        c = self.chord
        if Naca is None and filename is not None:
            from scipy.interpolate import interp1d
            upper, lower = _read_uiuc(filename)
            yu = interp1d(upper[0], upper[1], kind='cubic', bounds_error=False, fill_value="extrapolate")
            yl = interp1d(lower[0], lower[1], kind='cubic', bounds_error=False, fill_value="extrapolate")
            xs = np.linspace(0, 1, int(np.floor(Npoints / 2)))      # LUDVM.py:321 (float count fixed)
            xa = c * 0.5 * (xs + xs)
            etaa = c * 0.5 * (yu(xs) + yl(xs))
        elif Naca is not None:
            xs = np.linspace(0, 1, Npoints)
            xa = c * 0.5 * (xs + xs)
            etaa = c * _naca4_camber(Naca, xs)
        else:
            raise ValueError('Please introduce a valid foil_filename file')
        if uniform_spacing == 'theta':
            theta = np.linspace(0, np.pi, self.Npoints)
            x = c / 2 * (1 - np.cos(theta))
            eta = np.interp(x, xa, etaa)
        else:
            x, eta = xa, etaa
            theta = np.arccos(1 - 2 * x / c)
        x_panel = x[:-1] + self.xgamma * (x[1:] - x[:-1])
        eta_panel = np.interp(x_panel, x, eta)
        theta_panel = np.arccos(1 - 2 * x_panel / c)

        def fd(y, s):   # forward / centred / backward differences, LUDVM.py:353-372
            d = np.zeros(len(y))
            d[0] = (y[1] - y[0]) / (s[1] - s[0])
            d[-1] = (y[-1] - y[-2]) / (s[-1] - s[-2])
            d[1:-1] = (y[2:] - y[:-2]) / (2 * (s[2:] - s[:-2]))
            return d

        self.Npoints = len(eta)
        self.airfoil = {'x': x, 'theta': theta, 'eta': eta, 'detadx': fd(eta, x), 'detadtheta': fd(eta, theta),
                        'x_panel': x_panel, 'theta_panel': theta_panel, 'eta_panel': eta_panel,
                        'detadx_panel': fd(eta_panel, x_panel), 'detadtheta_panel': fd(eta_panel, theta_panel)}
        return None

    def _rigid_body_path(self, alpha, hpiv, xpiv):
        """Path of the Npoints nodes and of the gamma points under pitch/plunge (LUDVM.py:431-448)."""
        ca, sa = np.cos(-alpha), np.sin(-alpha)
        pa = np.zeros([self.nt, 2, self.Npoints])
        pa[:, 0, 0] = xpiv - self.piv * ca
        pa[:, 1, 0] = hpiv + self.piv * sa
        ax, ae = self.airfoil['x'][1:], self.airfoil['eta'][1:]
        pa[:, 0, 1:] = pa[:, 0, :1] + ca[:, None] * ax[None, :] - sa[:, None] * ae[None, :]
        pa[:, 1, 1:] = pa[:, 1, :1] + sa[:, None] * ax[None, :] + ca[:, None] * ae[None, :]
        gp = pa[:, :, :-1] + self.xgamma * (pa[:, :, 1:] - pa[:, :, :-1])
        self.path = {'airfoil': pa, 'airfoil_gamma_points': gp}

    def motion_sinusoidal(self, alpha_m=0, alpha_max=10, h_max=1, k=0.2 * np.pi, phi=90, h0=0, x0=0.25,
                          motion='cos'):
        """Pitch/heave tables alpha(t), h(t), x(t) (LUDVM.py:382-457)."""
        pi, U, t = np.pi, self.Uinf, self.t
        f = k * U / (2 * pi * self.chord)
        self.f = f
        alpha_m, alpha_max, phi = alpha_m * pi / 180, alpha_max * pi / 180, phi * pi / 180
        wt = 2 * pi * f * t
        if motion == 'cos':
            alpha = alpha_m + alpha_max * np.cos(wt + phi)
            alpha_dot = - alpha_max * 2 * pi * f * np.sin(wt + phi)
            h = h0 + h_max * np.cos(wt)
            h_dot = - h_max * 2 * pi * f * np.sin(wt)
        elif motion == 'sin':
            alpha = alpha_m + alpha_max * np.sin(wt + phi)
            alpha_dot = alpha_max * 2 * pi * f * np.cos(wt + phi)
            h = h0 + h_max * np.sin(wt)
            h_dot = - h_max * 2 * pi * f * np.cos(wt)
        else:
            raise ValueError("motion must be 'cos' or 'sin'")
        x = x0 - U * t
        self.phi, self.h_max = phi, h_max
        self.alpha, self.alpha_dot = alpha, alpha_dot
        self.alpha_e = alpha - np.arctan2(h_dot, U)
        self.hpiv, self.h_dot = h, h_dot
        self.xpiv, self.x_dot = x, -U * np.ones(self.nt)
        self._rigid_body_path(alpha, h, x)
        return None

    def motion_plunge(self, G=1, T=2, alpha_m=0, h0=0, x0=0.25):
        """sin^2 plunge manoeuvre (LUDVM.py:459-547); the one-argument arctan2 of LUDVM.py:520 is fixed."""
        pi, U, t = np.pi, self.Uinf, self.t
        alpha_m = alpha_m * pi / 180
        Vmax = G * U
        T = T * self.chord / U
        self.G, self.T = G, T
        alpha, alpha_dot = alpha_m * np.ones(self.nt), np.zeros(self.nt)
        during = t <= T
        h = np.where(during, h0 - Vmax * t / 2 + Vmax * T / (4 * pi) * np.sin(2 * pi * t / T), 0.0)
        h_dot = np.where(during, - Vmax * np.sin(pi * t / T) ** 2, 0.0)
        if not during.all():   # after the manoeuvre the height is frozen (LUDVM.py:513)
            h[~during] = h[during][-1] if during.any() else h0
        x = x0 - U * t
        self.alpha, self.alpha_dot = alpha, alpha_dot
        self.alpha_e = alpha - np.arctan2(h_dot, U)
        self.hpiv, self.h_dot = h, h_dot
        self.xpiv, self.x_dot = x, -U * np.ones(self.nt)
        self._rigid_body_path(alpha, h, x)
        return None

    # ------------------------------------------------------------------------------------------------
    # GPU path
    # ------------------------------------------------------------------------------------------------
    def induced_velocity(self, circulation, xw, zw, xp, zp, viscous=True):
        """All-pairs Vatistas-core Biot-Savart sum on the GPU (LUDVM.py:549-570)."""
        return ops.induced_velocity(circulation, xw, zw, xp, zp, self.v_core, viscous, mode=self.mode, ctx=self.ctx)

    def airfoil_downwash(self, circulation, xw, zw, i):
        """Normal downwash W(x,t) at the gamma points of step i (LUDVM.py:572-595)."""
        alpha, alpha_dot, h_dot = self.alpha[i], self.alpha_dot[i], self.h_dot[i]
        gp = self.path['airfoil_gamma_points'][i]
        u1, w1 = self.induced_velocity(circulation, xw, zw, gp[0], gp[1])
        u = u1 * np.cos(alpha) - w1 * np.sin(alpha)
        w = u1 * np.sin(alpha) + w1 * np.cos(alpha)
        af = self.airfoil
        return af['detadx_panel'] * (self.Uinf * np.cos(alpha) + h_dot * np.sin(alpha) + u
                                     - alpha_dot * af['eta_panel']) \
            - self.Uinf * np.sin(alpha) - alpha_dot * (af['x_panel'] - self.piv) + h_dot * np.cos(alpha) - w

    def step_tables(self):
        """Every host-evaluated table the device step consumes (SURVEY.md A.4), with numpy as the reference."""
        af, P, Nc = self.airfoil, self.Npoints - 1, self.Ncoeffs
        tp = af['theta_panel']
        A0 = np.sin(self.alpha_m)                        # alpha_m in degrees, as LUDVM.py:645 does
        free_g = f64(self.circulation_freevort)
        sum_free = float(np.sum(self.circulation_freevort))
        ic = np.sum(self.circulation_freevort) + self.Uinf * self.chord * np.pi * (A0 + 0 / 2)   # LUDVM.py:646-649
        nvec = np.arange(Nc)[:, None]
        return dict(
            nt=self.nt, P=P, Nc=Nc, nfree=self.n_freevort, method=1 if self.method == 'Ramesh' else 0,
            dt=float(self.dt), Uinf=float(self.Uinf), chord=float(self.chord), rho=float(self.rho),
            piv=float(self.piv), lespcrit=float(self.LESPcrit), vc4=float(self.v_core ** 4), ic=float(ic),
            sum_free=sum_free, a0_init=float(A0), a1_init=0.0,
            maxerror=self.maxerror, epsilon=self.epsilon, maxiter=self.maxiter,
            cos_a=f64(np.cos(self.alpha)), sin_a=f64(np.sin(self.alpha)),
            alpha_dot=f64(self.alpha_dot), h_dot=f64(self.h_dot),
            gp=f64(self.path['airfoil_gamma_points']),
            le=f64(self.path['airfoil'][:, :, 0]), te=f64(self.path['airfoil'][:, :, -1]),
            detadx_p=f64(af['detadx_panel']), eta_p=f64(af['eta_panel']), x_p=f64(af['x_panel']), theta_p=f64(tp),
            dtheta=f64(af['theta'][1:] - af['theta'][:-1]), cos_tp=f64(np.cos(tp)), sin_tp=f64(np.sin(tp)),
            cosn=f64(np.cos(nvec * tp[None, :])), sinn=f64(np.sin(nvec * tp[None, :])),
            free_g=free_g, free_xz=f64(self.xy_freevort))

    def time_loop(self, print_dt=50, BCcheck=False, tables=None, nsteps=None):
        """The time integrator (LUDVM.py:597-1171) on the device: CUDA-graph replay of the 4-kernel step.

        With `pressure=True` the device also fills dp[i, j], the pressure jump at gamma point j of step i (row 0 and the
        rows of steps not run stay zero):
            dp[i] = rho * ((Uinf*cos(alpha[i]) + h_dot[i]*sin(alpha[i]) + u) * gamma_airfoil[i-1]
                           + (Gamma_airfoil[i-1] - Gamma_airfoil[i-2]) / dt)
        where u is the tangential wake velocity at the gamma points that the normal force integrates
        (LUDVM.py:1049-1057); at i = 1 the Gamma_airfoil[i-2] term is 0.

        With `far_field_order=p` the steps whose wake bound 2*i + 2 + n_freevort reaches the library's all-pairs /
        far-field crossover (DESIGN.md 4b) convect the old wake through the treecode of `ops.induced_velocity_tree` at
        order p instead of all pairs (about 1e-15 of sum|terms| at p = 18); a cloud too clustered for the tree falls back
        to all pairs for that step.  The run is bitwise reproducible but not bit-equal to the all-pairs run.  Afterwards
        `self.far_field_info` = dict(far_field_steps, fallback_steps, order, leaf_level) (leaf level of the last tree)."""
        if BCcheck and not (self.store_history == 1 and nsteps is None):
            raise ValueError("BCcheck=True is evaluated from the full vortex-path history (store_history=True, whole run)")
        tb = tables if tables is not None else self.step_tables()
        if tb['P'] > 1024:
            raise ValueError("Npoints = %d: the device step supports at most 1025 chord stations (18 doubles of shared "
                             "memory per panel in the solve kernel)" % (tb['P'] + 1))
        self._tables = tb
        nt, P, Nc, nf = tb['nt'], tb['P'], tb['Nc'], tb['nfree']
        nv = nt - 1
        L = load()
        p = SimParams()
        for name, _ in SimParams._fields_:
            if name in tb:
                setattr(p, name, tb[name])
        p.mode = _lib.MODES[self.mode]
        p.store_history = self.store_history
        p.steps_per_graph = self.steps_per_graph
        t = SimTables()
        keep = []
        for name in TABLE_FIELDS:
            a = f64(tb[name])
            keep.append(a)
            setattr(t, name, a.ctypes.data_as(_lib.c_dp))
        if self._sim is not None:
            L.ludvm_sim_destroy(self._sim)
        sim = _lib.c_vp()
        check(L.ludvm_sim_create(self.ctx.handle, C.byref(p), C.byref(t), C.byref(sim)))
        self._sim = sim
        if self.pressure:
            check(L.ludvm_sim_enable_pressure(sim))
        if self.far_field_order is not None:
            check(L.ludvm_sim_enable_far_field(sim, self.far_field_order))
        total = nv if nsteps is None else min(int(nsteps), nv)
        K = self.steps_per_graph if self.steps_per_graph > 0 else 50
        chunk = max(K, (max(print_dt, 1) // K) * K) if self.verbose else total
        done = 0
        while done < total:
            n = min(chunk, total - done)
            check(L.ludvm_sim_run(sim, n))
            done += n
            if self.verbose:
                self.ctx.synchronize()
                print('Step {} out of {}. Elapsed time {}'.format(done, nv, timeit.default_timer() - self.start_time))
        self._fetch_results(nt, P, Nc, nf, nv)
        if self.far_field_order is not None:
            info = (C.c_int64 * 4)()
            check(L.ludvm_sim_far_field_info(sim, info))
            self.far_field_info = dict(far_field_steps=info[0], fallback_steps=info[1], order=info[2], leaf_level=info[3])
        if BCcheck:
            self.BC = self._bc_check()
        return None

    def _wake_before_convection(self, i, ilev):
        """(circulation, xw, zw) of the wake TEV[:itev+1] ++ LEV[:ilev+1] ++ FREE as it stood at step i BEFORE that step's
        convection (LUDVM.py:1095-1100): row i-1 of the stored paths plus the vortices placed in step i
        (LUDVM.py:672-681, :784-800).  Needs the full history."""
        itev = i - 1
        pa = self.path['airfoil']
        TEV, LEV, FREE = self.path['TEV'], self.path['LEV'], self.path['FREE']
        xT, zT = TEV[i - 1, 0, :itev + 1].copy(), TEV[i - 1, 1, :itev + 1].copy()
        if itev == 0:
            xT[0], zT[0] = pa[0, :, -1] + [0.5 * self.Uinf * self.dt, 0]
        else:
            xT[itev], zT[itev] = pa[i, :, -1] + 1 / 3 * (TEV[i - 1, :, itev - 1] - pa[i, :, -1])
        xL, zL = LEV[i - 1, 0, :ilev + 1].copy(), LEV[i - 1, 1, :ilev + 1].copy()
        cL = self.circulation['LEV'][:ilev + 1].copy()
        if self.LEV_shed[i] != -1:
            if ilev > 0 and self.LEV_shed[i - 1] != -1:
                xL[ilev], zL[ilev] = pa[i, :, 0] + 1 / 3 * (LEV[i - 1, :, ilev - 1] - pa[i, :, 0])
            else:
                xL[ilev], zL[ilev] = pa[i, :, 0]
        else:           # idle slot of row i: zero circulation at the origin (SURVEY.md B.3)
            xL[ilev], zL[ilev], cL[ilev] = 0.0, 0.0, 0.0
        ap = np.append
        return (ap(ap(self.circulation['TEV'][:itev + 1], cL), self.circulation['FREE']),
                ap(ap(xT, xL), FREE[i - 1, 0, :]), ap(ap(zT, zL), FREE[i - 1, 1, :]))

    def _bc_check(self):
        """Boundary-condition residual of LUDVM.py:1144-1161 (BCcheck=True), evaluated after the run from the stored
        history.  The reference raises there (it mixes `airfoil['x']`, length Npoints, with length-(Npoints-1) arrays
        at LUDVM.py:1153 and assigns Npoints-1 values to a row of Npoints at :1161); with `airfoil['x_panel']` in the
        first place, BC[itev, :Npoints-1] = BCnx + BCnz is the no-penetration residual, zero up to rounding; the last
        column keeps the reference's allocation (LUDVM.py:625) and stays zero."""
        nt, P = self.nt, self.Npoints - 1
        BC = np.zeros([nt - 1, self.Npoints])
        af, gpts = self.airfoil, self.path['airfoil_gamma_points']
        ilev = 0
        for i in range(1, nt):
            g, xw, zw = self._wake_before_convection(i, ilev)
            alpha, alpha_dot, h_dot = self.alpha[i], self.alpha_dot[i], self.h_dot[i]
            u1, w1 = self.induced_velocity(g, xw, zw, gpts[i, 0, :], gpts[i, 1, :])
            u = u1 * np.cos(alpha) - w1 * np.sin(alpha)
            w = u1 * np.sin(alpha) + w1 * np.cos(alpha)
            W = af['detadx_panel'] * (self.Uinf * np.cos(alpha) + h_dot * np.sin(alpha) + u
                                      - alpha_dot * af['eta_panel']) \
                - self.Uinf * np.sin(alpha) - alpha_dot * (af['x_panel'] - self.piv) \
                + h_dot * np.cos(alpha) - w
            BCnx = af['detadx_panel'] * (- u - self.Uinf * np.cos(alpha)
                                         - h_dot * np.sin(alpha) + alpha_dot * af['eta_panel'])
            BCnz = W + w + self.Uinf * np.sin(alpha) - h_dot * np.cos(alpha) \
                + alpha_dot * (af['x_panel'] - self.piv)
            BC[i - 1, :P] = BCnx + BCnz
            if self.LEV_shed[i] != -1:
                ilev += 1
        return BC

    def _fetch_results(self, nt, P, Nc, nf, nv):
        # every result field in ONE C call (one stream synchronisation instead of one per field)
        want = [('G_TEV', nv), ('G_LEV', nv), ('G_BOUND', nv), ('G_AIRFOIL', (nv, P)), ('GAMMA_AIRFOIL', (nv, P)),
                ('GAMMA_INT_AIRFOIL', (nv, P)), ('FOURIER', (nt, 2, Nc)), ('LESP', nt), ('LESP_PREV', nt), ('LEV_SHED', nt),
                ('FN', nt), ('FS', nt), ('L', nt), ('D', nt), ('T', nt), ('M', nt)]
        if self.store_history:
            hrows = (nt - 1) // self.store_history + 1
            want += [('PATH_TEV', (hrows, 2, nv)), ('PATH_LEV', (hrows, 2, nv)), ('PATH_FREE', (nt, 2, nf))]
        else:   # only the latest positions exist (the O(nt^2) history is the memory wall at dt=2e-3, tf=40)
            want += [('CUR_TEV', (2, nv)), ('CUR_LEV', (2, nv)), ('CUR_FREE', (2, nf))]
        if self.pressure:
            want.append(('DP', (nt, P)))
        got = {name: np.empty(shape) for name, shape in want}
        got['COUNTERS'], got['RANGE_BAD'] = np.empty(4, dtype=np.int64), np.empty(1, dtype=np.int32)
        n = len(got)
        fields = (C.c_int * n)(*[FIELDS[k] for k in got])
        dsts = (_lib.c_vp * n)(*[a.ctypes.data for a in got.values()])
        sizes = (C.c_size_t * n)(*[a.nbytes for a in got.values()])
        check(load().ludvm_sim_fetch_many(self._sim, n, fields, dsts, sizes))
        self.circulation = {'TEV': got['G_TEV'], 'LEV': got['G_LEV'], 'FREE': self.circulation_freevort,
                            'bound': got['G_BOUND'], 'airfoil': got['G_AIRFOIL'], 'gamma_airfoil': got['GAMMA_AIRFOIL'],
                            'Gamma_airfoil': got['GAMMA_INT_AIRFOIL'], 'IC': self._tables['ic']}
        if self.store_history:
            self.path['TEV'], self.path['LEV'], self.path['FREE'] = got['PATH_TEV'], got['PATH_LEV'], got['PATH_FREE']
            self.history_steps = np.arange(hrows) * self.store_history   # time index of each TEV/LEV path row
        else:
            self.path['TEV_last'], self.path['LEV_last'], self.path['FREE_last'] = got['CUR_TEV'], got['CUR_LEV'], got['CUR_FREE']
        self.fourier = got['FOURIER']
        self.LESP, self.LESP_prev, self.LEV_shed = got['LESP'], got['LESP_PREV'], got['LEV_SHED']
        self.Fn, self.Fs, self.L, self.D, self.T, self.M = (got[k] for k in ('FN', 'FS', 'L', 'D', 'T', 'M'))
        # never assigned by the reference (LUDVM.py:1059-1064): zero unless pressure=True
        self.dp = got['DP'] if self.pressure else np.zeros([nt, P])
        self.BC = np.zeros([nv, self.Npoints])
        cnt = got['COUNTERS']
        self.steps_done, self.itev, self.ilev = int(cnt[0]), int(cnt[1]), int(cnt[2])
        self.range_proof_held = not bool(got['RANGE_BAD'][0])   # exact mode: flag-free arithmetic ran
        if cnt[3] != 0:
            raise _lib.LudvmError("device time loop reported error flags %d (grid barrier timed out)" % int(cnt[3]))

    def compute_coefficients(self):
        """Force and moment coefficients (LUDVM.py:1173-1184)."""
        q = 0.5 * self.rho * self.Uinf ** 2
        qc = q * self.chord
        self.Cp = self.dp / q
        self.Cn, self.Cs = self.Fn / qc, self.Fs / qc
        self.Cl, self.Cd, self.Ct = self.L / qc, self.D / qc, self.T / qc
        self.Cm = self.M / (qc * self.chord)
        return None

    def flowfield(self, xmin=-10, xmax=0, zmin=-4, zmax=4, dr=0.02, tsteps=[0, 1, 2], rows=None, far_field_order=None):
        """Velocity and vorticity on a uniform grid for the chosen steps (LUDVM.py:1186-1298), GPU kernels.

        `far_field_order=p` (e.g. 18) evaluates the velocity through the hierarchical far field of csrc/tree.cu instead of
        all pairs (wake and bound vortices as one source set): the same sum to about 1e-15 of sum|terms| at p = 18,
        4e-13 at p = 14, at a small fraction of the cost on large grids; the vorticity stencil is unchanged.

        `rows=(row0, nrows)` restricts the evaluation to a slab of x-rows (multi-GPU sharding, see
        `sharded.grid_slab`): `x_ff, z_ff, u_ff, w_ff, ome_ff` then hold only those rows.  The vorticity stencil of a
        slab's first / last row is one-sided (LUDVM.py:1222-1292 applied to the slab), so a caller that shards a grid
        includes one halo row per interior side and drops it afterwards."""
        if not self.store_history:
            raise RuntimeError("flowfield needs the vortex path history (store_history=True)")
        x1, z1 = np.arange(xmin, xmax, dr), np.arange(zmin, zmax, dr)
        row0, nrows = (0, len(x1)) if rows is None else (int(rows[0]), int(rows[1]))
        if row0 < 0 or nrows < 2 or row0 + nrows > len(x1):
            raise ValueError("rows=(row0, nrows) must select at least two rows of the %d-row grid" % len(x1))
        xs = x1[row0:row0 + nrows]
        x, z = np.meshgrid(xs, z1, indexing='ij')
        ns = len(tsteps)
        u, w, ome = (np.zeros([ns, nrows, len(z1)]) for _ in range(3))
        vc4 = float(self.v_core ** 4)
        ap = np.append
        def ff(ga, xa, za, gb, xb, zb):
            if far_field_order is None:
                return ops.flowfield(ga, xa, za, gb, xb, zb, vc4, x1, z1, row0=row0, nrows=nrows, mode=self.mode, ctx=self.ctx)
            if gb is not None:
                ga, xa, za = ap(ga, gb), ap(xa, xb), ap(za, zb)
            uu, ww = ops.flowfield_velocity_tree(ga, xa, za, vc4, x1, z1, row0=row0, nrows=nrows, order=far_field_order,
                                                 ctx=self.ctx)
            return uu, ww, ops.flowfield_vorticity(xs, z1, uu[None], ww[None], ctx=self.ctx)[0]
        for ii, itev in enumerate(tsteps):
            if self.verbose:
                print('Flowfield tstep =', itev)
            if far_field_order is not None and itev == 0:
                u[ii], w[ii], ome[ii] = ff(self.circulation['FREE'], self.path['FREE'][0, 0], self.path['FREE'][0, 1],
                                           None, None, None)
            elif itev == 0:     # only the free vortices exist (LUDVM.py:1202-1207)
                u[ii], w[ii], ome[ii] = ops.flowfield(self.circulation['FREE'], self.path['FREE'][0, 0],
                                                      self.path['FREE'][0, 1], None, None, None, vc4, x1, z1,
                                                      row0=row0, nrows=nrows, mode=self.mode, ctx=self.ctx)
            else:             # index conventions of LUDVM.py:1209-1217 kept (SURVEY.md B.8)
                if (itev - 1) % self.store_history:
                    raise ValueError("flowfield step %d needs path row %d, which the strided history (every %d steps) "
                                     "does not hold" % (itev, itev - 1, self.store_history))
                hrow = (itev - 1) // self.store_history
                ilev = int(self.LEV_shed[itev])
                g = ap(ap(self.circulation['TEV'][:itev + 1], self.circulation['LEV'][:ilev + 1]),
                       self.circulation['FREE'])
                xw = ap(ap(self.path['TEV'][hrow, 0, :itev + 1], self.path['LEV'][hrow, 0, :ilev + 1]),
                        self.path['FREE'][itev, 0])
                zw = ap(ap(self.path['TEV'][hrow, 1, :itev + 1], self.path['LEV'][hrow, 1, :ilev + 1]),
                        self.path['FREE'][itev, 1])
                gp = self.path['airfoil_gamma_points'][itev - 1]
                u[ii], w[ii], ome[ii] = ff(g, xw, zw, self.circulation['airfoil'][itev - 1], gp[0], gp[1])
        self.x_ff, self.z_ff = x, z
        self.u_ff, self.w_ff = u, w
        self.ome_ff = ome        # velocity and stencil of a snapshot in one call: the fields cross the bus once
        return None

    def animation(self, step=1, ani_interval=10):
        raise NotImplementedError("animation (LUDVM.py:1301-1351) is matplotlib GUI code outside the GPU path; "
                                  "the history it plots is in self.path")

    def propulsive_efficiency(self, T=None):
        """Period-averaged Ct/Cp (LUDVM.py:1353-1372; the undefined `Uinf` of LUDVM.py:1367 is fixed)."""
        if T is None:
            T = 1 / self.f
        tt = self.t / T
        Nt = int(np.floor(tt[-1]))
        Ctm, Cpm = np.zeros([Nt]), np.zeros([Nt])
        for ii in range(Nt):
            indt = np.where(np.logical_and(tt >= ii - 1, tt < ii))
            Ctm[ii] = np.mean(self.Ct[indt])
            Cpi = abs(self.h_dot[indt] / self.Uinf * self.Cl[indt]) + \
                abs(self.alpha_dot[indt] * self.Cm[indt] * self.chord / self.Uinf)
            Cpm[ii] = np.mean(Cpi)
        self.tt = tt
        self.etap = Ctm / Cpm
        return None

    def close(self):
        if self._sim is not None:
            load().ludvm_sim_destroy(self._sim)
            self._sim = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
