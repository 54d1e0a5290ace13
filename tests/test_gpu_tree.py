"""O(N log N) far field (csrc/tree.cu, SURVEY.md section 8(f)-4) against the all-pairs oracle.

The reference has no treecode, so there is nothing to be bit-equal to: the checker is the oracle's all-pairs sum
(LUDVM.py:549-570) and the bound is the one SURVEY.md 8(d)-3 states for fast mode -- |error_i| <= 1e-12 * sum_j |term_ij|
at the default order -- plus the looser bounds of the lower orders, reproducibility, and shard independence."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

VC = 0.065


def _cloud(n, seed, sheet=False):
    rng = np.random.default_rng(seed)
    g = rng.standard_normal(n) * 1e-2
    if sheet:   # a rolled-up wake: thin, strongly non-uniform
        s = np.sort(rng.uniform(0, 1, n))
        x = -20 * s + 0.05 * rng.standard_normal(n)
        z = 0.8 * np.sin(9 * s) * s + 0.02 * rng.standard_normal(n)
    else:
        x, z = rng.uniform(-20, 0, n), rng.uniform(-4, 4, n)
    return g, x, z


def _sum_abs_terms(g, xw, zw, xp, zp, vc4):
    out = np.empty(len(xp))
    for i in range(len(xp)):
        dx, dz = xp[i] - xw, zp[i] - zw
        out[i] = np.sum(np.abs(g) * np.hypot(dx, dz) / np.sqrt((dx * dx + dz * dz) ** 2 + vc4)) / (2 * np.pi)
    return out


def _check(g, x, z, xp, zp, order, leaf, tol, level=None, monkeypatch=None):
    from ludvm_b200 import ops
    from oracle import ludvm_oracle as oracle
    if level is not None:
        monkeypatch.setenv("LUDVM_TREE_LEVEL", str(level))
    u, w, st = ops.induced_velocity_tree(g, x, z, xp, zp, VC, order=order, leaf=leaf, return_stats=True)
    rng = np.random.default_rng(7)
    sel = rng.choice(len(xp), min(len(xp), 600), replace=False)
    uo, wo = oracle.induced_velocity(g, x, z, xp[sel], zp[sel], VC)
    den = _sum_abs_terms(g, x, z, xp[sel], zp[sel], VC ** 4)
    err = np.max(np.hypot(u[sel] - uo, w[sel] - wo) / den)
    assert err <= tol, (err, st)
    return st, err


@pytest.mark.parametrize("order,tol", [(18, 1e-12), (16, 5e-12), (12, 2e-9), (6, 1e-4)])
def test_tree_self_evaluation_vs_oracle(order, tol, monkeypatch):
    g, x, z = _cloud(60000, 1)
    st, err = _check(g, x, z, x, z, order, 48, tol, level=6, monkeypatch=monkeypatch)   # deep tree: 5 far-field levels
    assert st["leaf_level"] == 6 and st["pair_evaluations"] < 0.8 * st["all_pairs"]


@pytest.mark.parametrize("level,leaf", [(5, 0), (7, 0)])
def test_tree_at_forced_levels_vs_oracle(level, leaf, monkeypatch):
    """A shallow and a deep leaf level forced on the same cloud: the local fields (M2L / L2L / L2P) of either tree stay
    within the default order's bound of the oracle."""
    g, x, z = _cloud(120000, 8)
    _check(g, x, z, x, z, 18, leaf, 1e-12, level=level, monkeypatch=monkeypatch)


def test_tree_default_parameters_and_separate_targets():
    g, x, z = _cloud(150000, 2)
    rng = np.random.default_rng(3)
    xp, zp = rng.uniform(-25, 5, 30000), rng.uniform(-6, 6, 30000)     # targets beyond the sources' box
    st, err = _check(g, x, z, xp, zp, 18, 0, 1e-12)
    assert st["pair_evaluations"] < 0.5 * st["all_pairs"]


def test_tree_nonuniform_sheet():
    g, x, z = _cloud(80000, 4, sheet=True)
    _check(g, x, z, x, z, 18, 64, 1e-12)


def test_tree_small_and_degenerate_inputs():
    from ludvm_b200 import ops
    from oracle import ludvm_oracle as oracle
    for n in (1, 2, 37, 500):
        g, x, z = _cloud(n, 10 + n)
        u, w = ops.induced_velocity_tree(g, x, z, x, z, VC)
        uo, wo = oracle.induced_velocity(g, x, z, x, z, VC)
        den = _sum_abs_terms(g, x, z, x, z, VC ** 4) + 1e-300
        assert np.max(np.hypot(u - uo, w - wo) / den) <= 1e-12
    g = np.ones(300) * 1e-2                                              # every vortex at one point: a single crowded leaf
    u, w = ops.induced_velocity_tree(g, np.full(300, -1.0), np.full(300, 0.5), np.array([0.0, -1.0]), np.array([0.0, 0.5]), VC)
    uo, wo = oracle.induced_velocity(g, np.full(300, -1.0), np.full(300, 0.5), np.array([0.0, -1.0]), np.array([0.0, 0.5]), VC)
    assert np.allclose(u, uo, rtol=1e-12, atol=1e-15) and np.allclose(w, wo, rtol=1e-12, atol=1e-15)
    u, w = ops.induced_velocity_tree(np.zeros(0), np.zeros(0), np.zeros(0), np.array([1.0]), np.array([2.0]), VC)
    assert u[0] == 0.0 and w[0] == 0.0
    g, x, z = _cloud(5000, 77)
    a, b = ops.induced_velocity(g, x, z, x, z, VC, mode="tree"), ops.induced_velocity_tree(g, x, z, x, z, VC)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def test_tree_bitwise_reproducible_and_shard_independent():
    import torch
    from ludvm_b200 import _lib, ops
    g, x, z = _cloud(100000, 5)
    a = ops.induced_velocity_tree(g, x, z, x, z, VC, order=12, leaf=64)
    for _ in range(3):
        b = ops.induced_velocity_tree(g, x, z, x, z, VC, order=12, leaf=64)
        assert np.array_equal(a[0].view(np.uint64), b[0].view(np.uint64)) and np.array_equal(a[1].view(np.uint64), b[1].view(np.uint64))
    # the Euler step on row shards: the tree is built over sources + the shard's targets, whose bounding box is the
    # sources' (targets are a subset), so every shard sees the same cells and the same sums
    dev = torch.device("cuda", 0)
    ctx = _lib.Context(0, torch.cuda.current_stream(dev).cuda_stream)
    tg, tx, tz = (torch.from_numpy(v).to(dev) for v in (g, x, z))
    full_x, full_z = torch.empty_like(tx), torch.empty_like(tz)
    ops.selfconv_step_tree(ctx, tg, tx, tz, VC ** 4, 0.05, full_x, full_z, order=12, leaf=64)
    sh_x, sh_z = torch.empty_like(tx), torch.empty_like(tz)
    n = len(g)
    for r0, r1 in ((0, 30000), (30000, 30001), (30001, n)):
        ops.selfconv_step_tree(ctx, tg, tx, tz, VC ** 4, 0.05, sh_x, sh_z, row0=r0, nrows=r1 - r0, order=12, leaf=64)
    torch.cuda.synchronize()
    assert torch.equal(full_x, sh_x) and torch.equal(full_z, sh_z)
    assert np.array_equal(full_x.cpu().numpy(), x + 0.05 * a[0])
    assert ctx.last_plan()["kernel"] == "tree"
    ctx.close()


def test_tree_refuses_a_cloud_that_is_one_point_and_handles_crowded_leaves():
    from ludvm_b200 import _lib, ops
    from oracle import ludvm_oracle as oracle
    n = 70000
    g = np.full(n + 2, 1e-3)
    x, z = np.full(n + 2, -1.0), np.full(n + 2, 0.25)
    x[-2:], z[-2:] = (-20.0, 0.0), (-4.0, 4.0)
    with pytest.raises(_lib.LudvmError, match="too clustered"):
        ops.induced_velocity_tree(g, x, z, x[-2:], z[-2:], VC)
    # a tight Gaussian blob inside a sparse background: leaves with thousands of vortices, many passes per leaf
    rng = np.random.default_rng(12)
    gb, xb, zb = _cloud(40000, 13)
    xc, zc = -7.0 + 0.01 * rng.standard_normal(20000), 1.0 + 0.01 * rng.standard_normal(20000)
    g2, x2, z2 = np.concatenate([gb, 1e-3 * rng.standard_normal(20000)]), np.concatenate([xb, xc]), np.concatenate([zb, zc])
    u, w, st = ops.induced_velocity_tree(g2, x2, z2, x2, z2, VC, return_stats=True)
    sel = np.concatenate([rng.choice(40000, 150, replace=False), 40000 + rng.choice(20000, 150, replace=False)])
    uo, wo = oracle.induced_velocity(g2, x2, z2, x2[sel], z2[sel], VC)
    den = _sum_abs_terms(g2, x2, z2, x2[sel], z2[sel], VC ** 4)
    assert np.max(np.hypot(u[sel] - uo, w[sel] - wo) / den) <= 1e-12, st


def test_flowfield_grid_through_the_far_field_vs_oracle_and_slabs():
    """Grid targets: cells holding more than (order+1)^2 grid points carry a local field even away from the sources; the
    density comes from the full grid, so row slabs reproduce the full-grid values bit for bit."""
    from ludvm_b200 import ops
    from oracle import ludvm_oracle as oracle
    g, x, z = _cloud(60000, 21)
    x1, z1 = np.arange(-22.0, 2.0, 0.03), np.arange(-9.0, 9.0, 0.03)          # 800 x 600, extends far beyond the sources
    u, w, st = ops.flowfield_velocity_tree(g, x, z, VC ** 4, x1, z1, return_stats=True)
    assert u.shape == (len(x1), len(z1)) and st["pair_evaluations"] < 0.1 * st["all_pairs"]
    rng = np.random.default_rng(5)
    ii, jj = rng.integers(0, len(x1), 500), rng.integers(0, len(z1), 500)
    uo, wo = oracle.induced_velocity(g, x, z, x1[ii], z1[jj], VC)
    den = _sum_abs_terms(g, x, z, x1[ii], z1[jj], VC ** 4)
    assert np.max(np.hypot(u[ii, jj] - uo, w[ii, jj] - wo) / den) <= 1e-12
    for r0, nr in ((0, 300), (299, 2), (301, len(x1) - 301)):
        us, ws = ops.flowfield_velocity_tree(g, x, z, VC ** 4, x1, z1, row0=r0, nrows=nr)
        assert np.array_equal(us.view(np.uint64), u[r0:r0 + nr].view(np.uint64))
        assert np.array_equal(ws.view(np.uint64), w[r0:r0 + nr].view(np.uint64))


def test_class_flowfield_far_field_order():
    from ludvm_b200 import LUDVM
    kw = dict(t0=0, tf=3, dt=5e-2, chord=1, rho=1.225, Uinf=1, Npoints=81, Ncoeffs=30, LESPcrit=0.2, Naca="0012")
    s = LUDVM(**kw, verbose=False, mode="fast")
    s.flowfield(xmin=-3.0, xmax=0.5, zmin=-1.0, zmax=1.0, dr=0.02, tsteps=[0, 30, 59])
    ua, wa, oa = s.u_ff.copy(), s.w_ff.copy(), s.ome_ff.copy()
    s.flowfield(xmin=-3.0, xmax=0.5, zmin=-1.0, zmax=1.0, dr=0.02, tsteps=[0, 30, 59], far_field_order=18)
    scale = np.max(np.abs(ua))
    assert np.max(np.abs(s.u_ff - ua)) <= 1e-11 * scale and np.max(np.abs(s.w_ff - wa)) <= 1e-11 * scale
    assert np.max(np.abs(s.ome_ff - oa)) <= 1e-8 * np.max(np.abs(oa))
