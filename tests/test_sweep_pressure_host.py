"""CPU tests of the host side of a sweep with the pressure jump (sweep.run_sweep over cases with pressure=True): which
C entry point it calls with which arguments, how it forms Cp, and which case lists it refuses.  The C entry points are
replaced by a recorder (no device work); one test calls the library's own argument checks, which come first."""
import types

import numpy as np
import pytest

from conftest import biteq

BASE = dict(t0=0, tf=1, dt=5e-2, chord=1, rho=1.225, Uinf=1, Npoints=81, Ncoeffs=30, Naca="0012")


class FakeLib:
    """Records what run_sweep passes; fills `dp` with a per-case, per-element pattern."""

    def __init__(self):
        self.calls = []

    @staticmethod
    def _structs(n, P, T):
        """Each case's parameter struct as bytes and the first and last value of each of its tables (the table
        pointers of two run_sweep calls differ)."""
        from ludvm_b200._lib import TABLE_FIELDS
        nt, npan, nc, nf = P[0].nt, P[0].P, P[0].Nc, P[0].nfree
        size = dict(cos_a=nt, sin_a=nt, alpha_dot=nt, h_dot=nt, gp=nt * 2 * npan, le=nt * 2, te=nt * 2,
                    cosn=nc * npan, sinn=nc * npan, free_g=nf, free_xz=2 * nf)
        return ([bytes(P[i]) for i in range(n)],
                [tuple((getattr(T[i], f)[0], getattr(T[i], f)[size.get(f, npan) - 1]) for f in TABLE_FIELDS)
                 for i in range(n)])

    def ludvm_sweep_run(self, ctx, n, P, T, out, stride):
        self.calls.append(dict(fn="ludvm_sweep_run", n=n, stride=stride, structs=self._structs(n, P, T)))
        return 0

    def ludvm_sweep_run_pressure(self, ctx, n, P, T, out, stride, dp, dp_stride):
        nt, npan = P[0].nt, P[0].P
        buf = np.ctypeslib.as_array((np.ctypeslib.ctypes.c_double * (n * dp_stride)).from_address(dp))
        buf[:] = np.arange(1, n * dp_stride + 1, dtype=float) * 1e-3
        self.calls.append(dict(fn="ludvm_sweep_run_pressure", n=n, stride=stride, dp_stride=dp_stride, nt=nt,
                               npan=npan, dp_len=buf.size, structs=self._structs(n, P, T)))
        return 0


def _run(monkeypatch, cases, **kw):
    from ludvm_b200 import sweep
    fake = FakeLib()
    monkeypatch.setattr(sweep, "load", lambda: fake)
    res = sweep.run_sweep(cases, mode="fast", ctx=types.SimpleNamespace(handle=None), **kw)
    return fake, res


def test_pressure_sweep_calls_the_pressure_entry_point_with_the_same_structs(monkeypatch):
    from ludvm_b200 import sweep
    cases = sweep.lespcrit_k_grid((0.1, 0.3), (0.2, 0.9), **BASE)
    f_off, off = _run(monkeypatch, cases)
    f_on, on = _run(monkeypatch, [dict(kw, pressure=True) for kw in cases])
    a, b = f_off.calls[-1], f_on.calls[-1]
    assert a["fn"] == "ludvm_sweep_run" and b["fn"] == "ludvm_sweep_run_pressure"
    assert "dp" not in off and "Cp" not in off
    assert (b["n"], b["stride"]) == (a["n"], a["stride"]) == (4, len(sweep.SW_FIELDS) * on["nt"])
    assert a["structs"][0] == b["structs"][0], "parameter structs differ"
    assert a["structs"][1] == b["structs"][1], "table structs differ"
    nt, npan = on["nt"], 80
    assert (b["nt"], b["npan"]) == (nt, npan)
    assert b["dp_stride"] == nt * npan and b["dp_len"] == 4 * nt * npan
    assert on["dp"].shape == on["Cp"].shape == (4, nt, npan)
    assert biteq(on["dp"].ravel(), np.arange(1, 4 * nt * npan + 1, dtype=float) * 1e-3)


def test_pressure_sweep_cp_uses_each_cases_dynamic_pressure(monkeypatch):
    cases = [dict(BASE, pressure=True, LESPcrit=0.2), dict(BASE, pressure=True, rho=1.0, Uinf=1.7),
             dict(BASE, pressure=True, rho=0.8, Uinf=0.6, k=0.5)]
    _, res = _run(monkeypatch, cases)
    for a, kw in enumerate(cases):
        q = 0.5 * kw["rho"] * kw["Uinf"] ** 2                  # LUDVM.compute_coefficients
        assert biteq(res["Cp"][a], res["dp"][a] / q), a


def test_pressure_entry_point_checks_its_buffer_before_any_device_work(monkeypatch):
    """ludvm_sweep_run_pressure refuses a null dp and a dp_doubles_per_case other than nt * P with LUDVM_E_ARG; the
    checks come before the context is used (a zeroed stand-in is passed), so they hold without a GPU."""
    import ctypes as C
    import __graft_entry__ as ge
    from ludvm_b200 import _lib, sweep
    ge.build()
    kept = {}

    class Keep(FakeLib):   # keeps the structs run_sweep built (the table pointers are only checked for null)
        def ludvm_sweep_run_pressure(self, ctx, n, P, T, out, stride, dp, dp_stride):
            kept.update(n=n, P=P, T=T, stride=stride, dp_stride=dp_stride)
            return super().ludvm_sweep_run_pressure(ctx, n, P, T, out, stride, dp, dp_stride)

    monkeypatch.setattr(sweep, "load", lambda: Keep())
    sweep.run_sweep([dict(BASE, pressure=True)], ctx=types.SimpleNamespace(handle=None))
    L, ctx = _lib.load(), C.create_string_buffer(4096)
    out = np.empty(kept["stride"])
    dp = np.empty(kept["dp_stride"] + 1)
    args = (C.addressof(ctx), kept["n"], kept["P"], kept["T"], out.ctypes.data, kept["stride"])
    assert L.ludvm_sweep_run_pressure(*args, None, kept["dp_stride"]) == -1
    assert L.ludvm_sweep_run_pressure(*args, dp.ctypes.data, kept["dp_stride"] + 1) == -1
    assert "dp_doubles_per_case" in L.ludvm_last_error().decode()


def test_pressure_must_be_asked_by_every_case_of_the_whole_list(monkeypatch):
    """The choice is made over all of `cases`, before `case_slice`, so every slice of one sweep makes the same one."""
    from ludvm_b200 import sweep
    cases = sweep.lespcrit_k_grid((0.1, 0.2, 0.3, 0.4), (0.2,), **BASE)
    for kw in cases[:2]:
        kw["pressure"] = True
    fake = FakeLib()
    monkeypatch.setattr(sweep, "load", lambda: fake)
    for sl in (slice(0, 2), slice(2, None), None):
        with pytest.raises(ValueError, match="pressure"):
            sweep.run_sweep(cases, ctx=types.SimpleNamespace(handle=None), case_slice=sl)
    assert not fake.calls
