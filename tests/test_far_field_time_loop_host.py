"""CPU tests of LUDVM(..., far_field_order=): the constructor refuses what the far-field step cannot do before any device
work, the option leaves the host tables alone, and the two C entry points are declared and bound."""
import ctypes
import os
import re

import numpy as np
import pytest

from conftest import ROOT, biteq

KW = dict(t0=0, tf=0.3, dt=5e-2, chord=1, rho=1.225, Uinf=1, Npoints=81, Ncoeffs=30, LESPcrit=0.2, Naca="0012",
          verbose=False, run=False)


@pytest.mark.parametrize("extra", [dict(mode="exact"), dict(mode="fast", method="Ramesh"),
                                   dict(mode="fast", Npoints=301), dict(mode="fast", far_field_order=1),
                                   dict(mode="fast", far_field_order=25), dict(mode="fast", far_field_order=18.5)])
def test_constructor_refuses(extra):
    from ludvm_b200 import LUDVM
    kw = dict(KW, far_field_order=18)
    kw.update(extra)
    with pytest.raises(ValueError):
        LUDVM(**kw)


def test_far_field_order_leaves_step_tables_unchanged():
    from ludvm_b200 import LUDVM
    rng = np.random.default_rng(3)
    kw = dict(KW, mode="fast", circulation_freevort=rng.standard_normal(50) * 1e-3,
              xy_freevort=np.stack([rng.uniform(-6, -0.5, 50), rng.uniform(-1, 1, 50)]))
    a = LUDVM(**kw).step_tables()
    for ff in (None, 18):
        s = LUDVM(**kw, far_field_order=ff)
        assert s.far_field_order == ff and s.far_field_info is None
        b = s.step_tables()
        assert a.keys() == b.keys()
        for k in a:
            assert biteq(a[k], b[k]) if isinstance(a[k], np.ndarray) else a[k] == b[k], k


def test_far_field_symbols_declared_and_bound():
    from ludvm_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "ludvm_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    for name in ("ludvm_sim_enable_far_field", "ludvm_sim_far_field_info"):
        assert re.search(r"\b%s\s*\(" % name, hdr), name
        assert name in _lib.SIGNATURES, name
    assert _lib.SIGNATURES["ludvm_sim_enable_far_field"] == (ctypes.c_int, [_lib.c_vp, ctypes.c_int])
    assert _lib.SIGNATURES["ludvm_sim_far_field_info"] == (ctypes.c_int, [_lib.c_vp, ctypes.POINTER(ctypes.c_int64)])
    if os.path.isfile(_lib.LIB_PATH):
        L = ctypes.CDLL(_lib.LIB_PATH)
        assert hasattr(L, "ludvm_sim_enable_far_field") and hasattr(L, "ludvm_sim_far_field_info")
