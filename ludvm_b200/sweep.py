"""Batched parameter sweeps (BASELINE.json configs[3]): many independent LUDVM cases in one launch, one persistent
CTA per case (C ABI `ludvm_sweep_run`), no collective.  Cases are constructor-kwarg dicts of `ludvm_b200.LUDVM`;
cases that differ only in `LESPcrit` share one set of host tables (geometry + kinematics are computed once).

A sweep whose cases all pass `pressure=True` also returns the chordwise pressure jump `dp` and `Cp = dp / q` of every
case (C ABI `ludvm_sweep_run_pressure`), the same values as `LUDVM(..., pressure=True)`.  Every case asks for it or
none does."""
import ctypes as C
import hashlib
import inspect

import numpy as np

from . import _lib
from ._lib import SimParams, SimTables, TABLE_FIELDS, check, f64, load
from .ludvm import LUDVM

SW_FIELDS = ("Fn", "Fs", "L", "D", "T", "M", "LESP", "LESP_prev", "LEV_shed", "circulation_TEV", "circulation_LEV",
             "circulation_bound")


_LESPCRIT_DEFAULT = inspect.signature(LUDVM.__init__).parameters["LESPcrit"].default


def _key_of(v):
    """Hashable identity of a constructor argument for table sharing: arrays by their bytes (repr() elides long ones)."""
    if isinstance(v, (np.ndarray, list, tuple)):
        a = np.asarray(v)
        return ("array", a.shape, str(a.dtype), hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest())
    return repr(v)


def lespcrit_k_grid(lespcrits, ks, **base):
    """The 2-D sweep of BASELINE.json: LESPcrit x reduced frequency, everything else from `base`."""
    return [dict(base, LESPcrit=float(lc), k=float(k)) for lc in lespcrits for k in ks]


def run_sweep(cases, mode="exact", ctx=None, device=0, case_slice=None):
    """Run every case of `cases` (or `cases[case_slice]`, for splitting a sweep over GPUs/ranks) and return a dict
    of [ncases, nt] arrays: the load histories, coefficients (LUDVM.py:1173-1184), LESP, LEV_shed, circulations.

    If every case of `cases` passes `pressure=True`, the dict also holds `dp` and `Cp`, [ncases, nt, Npoints-1] each
    (row 0 of each case zero).  dp takes ncases * nt * (Npoints-1) * 8 bytes on the device and again on the host, and
    Cp as much on the host: about 1.05 GB each for configs[3] (4096 cases, 401 steps, 80 panels); `case_slice` bounds
    it.  The choice is made over all of `cases`, so every slice of one sweep agrees; a list in which some cases ask
    for pressure and others do not raises ValueError."""
    import time
    t_host = time.perf_counter()
    asks = {bool(kw.get("pressure")) for kw in cases}
    if len(asks) > 1:
        raise ValueError("run_sweep computes the pressure jump for every case or for none: pass pressure=True to "
                         "all cases or to none")
    pressure = asks == {True}
    sel = list(cases[case_slice] if case_slice is not None else cases)
    if not sel:
        raise ValueError("empty sweep")
    ctx = ctx or _lib.default_context(device)
    # The host tables and the parameter / table structs depend on everything but LESPcrit: built once per distinct
    # motion, copied per case (filling 4096 structs field by field cost more than the fast-mode kernel's launch).
    shared, params, tables, objs = {}, [], [], []
    for kw in sel:
        key = tuple(sorted((k, _key_of(v)) for k, v in kw.items() if k != "LESPcrit"))
        if key not in shared:
            s = LUDVM(**dict(kw, verbose=False, run=False))
            tb = s.step_tables()
            arrs = {n: f64(tb[n]) for n in TABLE_FIELDS}          # kept alive by `shared` until the call returns
            p0 = SimParams()
            for name, _ in SimParams._fields_:
                if name in tb:
                    setattr(p0, name, tb[name])
            p0.mode = _lib.MODES[mode]
            p0.store_history = 0
            t0 = SimTables()
            for n in TABLE_FIELDS:
                setattr(t0, n, arrs[n].ctypes.data_as(_lib.c_dp))
            shared[key] = (s, arrs, p0, t0)
        s, arrs, p0, t0 = shared[key]
        p = SimParams.from_buffer_copy(p0)
        p.lespcrit = float(kw.get("LESPcrit", _LESPCRIT_DEFAULT))
        params.append(p)
        tables.append(t0)
        objs.append(s)
    n, nt, npan = len(sel), params[0].nt, params[0].P
    P = (SimParams * n)(*params)
    T = (SimTables * n)(*tables)
    out = np.empty((n, len(SW_FIELDS), nt))
    t_dev = time.perf_counter()
    if pressure:
        dp = np.empty((n, nt, npan))
        check(load().ludvm_sweep_run_pressure(ctx.handle, n, P, T, out.ctypes.data, len(SW_FIELDS) * nt,
                                              dp.ctypes.data, nt * npan))
    else:
        check(load().ludvm_sweep_run(ctx.handle, n, P, T, out.ctypes.data, len(SW_FIELDS) * nt))
    t_end = time.perf_counter()
    res = {name: out[:, i, :] for i, name in enumerate(SW_FIELDS)}
    rho = np.array([o.rho for o in objs], dtype=float)[:, None]
    U = np.array([o.Uinf for o in objs], dtype=float)[:, None]
    c = np.array([o.chord for o in objs], dtype=float)[:, None]
    q = 0.5 * rho * U ** 2
    qc = q * c                                                     # LUDVM.py:1175-1177
    res["Cl"], res["Cd"], res["Ct"] = res["L"] / qc, res["D"] / qc, res["T"] / qc
    res["Cn"], res["Cs"], res["Cm"] = res["Fn"] / qc, res["Fs"] / qc, res["M"] / (qc * c)
    if pressure:
        res["dp"], res["Cp"] = dp, dp / q[:, :, None]              # as LUDVM.compute_coefficients
    res["nt"] = nt
    res["timing"] = {"host_tables_s": t_dev - t_host, "ludvm_sweep_run_s": t_end - t_dev}
    return res
