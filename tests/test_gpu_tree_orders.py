"""The far field (csrc/tree.cu) at every interpolation order against oracle/tree_model.py, the float64 model of the same
algorithm: same tree, lists, proxies and local fields, so the GPU must agree with it to rounding at every order, however
large that order's truncation error against the all-pairs sum.

The order selects different code: the leaf level of the upward pass runs k_tree_up_leaf_mma up to order 23 and the scalar
k_tree_up at 24; L2P runs k_tree_l2p_mma up to order 19 and the scalar k_tree_l2p from 20; k_tree_m2l_dmma's 64-row tiles
and 16-wide k-slices of P2 = (order + 1)^2 are exact at orders 3, 7, 11, 15, 19, 23 and padded elsewhere; only even orders
have a Chebyshev node at a cell's centre.  The tests run all of them."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

VC = 0.065
VC4 = VC ** 4
ORDERS = list(range(2, 25))
# |GPU - model| <= TOL * sum_j |term_ij| per target.  The model's own rounding noise (its sources permuted, so that every
# sum runs in another order) is about 8e-17 of that sum at any order (test_tree_model.py::test_model_rounding_noise); the
# GPU measured at most 3.8e-16 over these tests (B200), at every order.
TOL = 2e-15


def mixed_cloud(seed=31):
    """30 000 vortices whose density falls by orders of magnitude from x = 0 to x = -20, and a tight Gaussian blob of
    6 000: at every order the leaf level has cells above and below the proxy threshold, at least two levels carry local
    fields, and some targets take their local field from above the leaf level."""
    rng = np.random.default_rng(seed)
    nu, nb = 30000, 6000
    x = np.concatenate([-20.0 * rng.uniform(0, 1, nu) ** 4, -7.0 + 0.03 * rng.standard_normal(nb)])
    z = np.concatenate([rng.uniform(-4, 4, nu), 1.0 + 0.03 * rng.standard_normal(nb)])
    g = np.concatenate([rng.standard_normal(nu) * 1e-2, rng.standard_normal(nb) * 1e-3])
    return g, x, z


def outside_targets(seed=32, n=4000):
    """Targets over a box larger than the sources' on every side."""
    rng = np.random.default_rng(seed)
    return rng.uniform(-26, 4, n), rng.uniform(-9, 9, n)


def grid_case():
    """Sources: the mixed cloud plus two weak corner vortices that fix the root square at [-22, -22 + side) x [-12, ...).
    Grid: spacing side / 2^10 from that corner, so grid lines run exactly through the centres of the cells of every level
    up to 9 (for even orders the node p/2 of the cell), over a window of the cloud that holds part of the blob."""
    from oracle import tree_model
    g, x, z = mixed_cloud()
    g = np.concatenate([g, [1e-4, -1e-4]])
    x = np.concatenate([x, [-22.0, 2.0]])
    z = np.concatenate([z, [-12.0, 12.0]])
    side = tree_model.Geom(x, z, x[:0], z[:0], 2).side
    sp = side / 1024
    x1 = -22.0 + np.arange(560, 760) * sp
    z1 = -12.0 + np.arange(480, 620) * sp
    return g, x, z, x1, z1


def sum_abs_terms(g, xw, zw, xp, zp):
    """sum_j |Gamma_j| r_ij / (2 pi sqrt(r_ij^4 + vc^4)) per target, on the GPU."""
    import torch
    t = lambda v: torch.tensor(np.ascontiguousarray(v, dtype=np.float64), device="cuda")
    tg, tx, tz, px, pz = t(np.abs(g)), t(xw), t(zw), t(xp), t(zp)
    out = np.empty(len(xp))
    for r in range(0, len(xp), 2048):
        r2 = (px[r:r + 2048, None] - tx[None, :]) ** 2 + (pz[r:r + 2048, None] - tz[None, :]) ** 2
        out[r:r + 2048] = (tg[None, :] * torch.sqrt(r2) / (2 * np.pi * torch.sqrt(r2 * r2 + VC4))).sum(1).cpu().numpy()
    return out


def _ratio(u, w, um, wm, den):
    return float(np.max(np.hypot(u - um, w - wm) / den))


@pytest.fixture(scope="module")
def cloud():
    g, x, z = mixed_cloud()
    return g, x, z, sum_abs_terms(g, x, z, x, z)


@pytest.mark.parametrize("order", ORDERS)
def test_every_order_matches_the_model(cloud, order):
    from ludvm_b200 import ops
    from oracle import tree_model
    g, x, z, den = cloud
    u, w, st = ops.induced_velocity_tree(g, x, z, x, z, VC, order=order, return_stats=True)
    um, wm, info = tree_model.tree_velocity(g, x, z, x, z, VC4, order=order)
    L = info["L"]
    assert st["leaf_level"] == L
    assert st["pair_evaluations"] == info["pairs"]
    assert info["proxy_cells"][L] > 0 and info["plain_cells"][L] > 0, info      # both leaf paths of the upward pass
    assert sum(n > 0 for n in info["local_cells"].values()) >= 2, info
    assert info["targets_below_leaf_level"] > 0, info
    r = _ratio(u, w, um, wm, den)
    print("order %d: L %d, max |GPU - model| / sum|terms| = %.3e" % (order, L, r))
    assert r <= TOL, r


@pytest.mark.parametrize("order", [3, 7, 19, 20, 23, 24])
def test_separate_targets_match_the_model(order):
    from ludvm_b200 import ops
    from oracle import tree_model
    g, x, z = mixed_cloud()
    xp, zp = outside_targets()
    u, w, st = ops.induced_velocity_tree(g, x, z, xp, zp, VC, order=order, return_stats=True)
    um, wm, info = tree_model.tree_velocity(g, x, z, xp, zp, VC4, order=order)
    assert st["leaf_level"] == info["L"] and st["pair_evaluations"] == info["pairs"]
    r = _ratio(u, w, um, wm, sum_abs_terms(g, x, z, xp, zp))
    print("order %d, separate targets: max |GPU - model| / sum|terms| = %.3e" % (order, r))
    assert r <= TOL, r


@pytest.mark.parametrize("order", [2, 7, 19, 20, 24])
def test_grid_targets_match_the_model_and_slabs(order):
    from ludvm_b200 import ops
    from oracle import tree_model
    g, x, z, x1, z1 = grid_case()
    u, w, st = ops.flowfield_velocity_tree(g, x, z, VC4, x1, z1, order=order, return_stats=True)
    um, wm, info = tree_model.flowfield_velocity(g, x, z, VC4, x1, z1, order=order)
    assert st["leaf_level"] == info["L"] and st["pair_evaluations"] == info["pairs"]
    G = tree_model.Geom(x, z, x1[[0, -1]], z1[[0, -1]], order, tdens=tree_model.grid_density(x1, z1))
    cx, cz = G.centre(info["L"], np.arange(1 << (2 * info["L"])))
    assert np.isin(x1, cx).any() and np.isin(z1, cz).any()           # grid points on cell centres
    X, Z = np.meshgrid(x1, z1, indexing="ij")
    r = _ratio(u.ravel(), w.ravel(), um.ravel(), wm.ravel(), sum_abs_terms(g, x, z, X.ravel(), Z.ravel()))
    print("order %d, grid: max |GPU - model| / sum|terms| = %.3e" % (order, r))
    assert r <= TOL, r
    us, ws = ops.flowfield_velocity_tree(g, x, z, VC4, x1, z1, row0=57, nrows=31, order=order)
    assert np.array_equal(us.view(np.uint64), u[57:88].view(np.uint64))
    assert np.array_equal(ws.view(np.uint64), w[57:88].view(np.uint64))


@pytest.mark.parametrize("order", [7, 20, 24])
def test_bitwise_reproducible(order):
    from ludvm_b200 import ops
    g, x, z = mixed_cloud()
    a = ops.induced_velocity_tree(g, x, z, x, z, VC, order=order)
    b = ops.induced_velocity_tree(g, x, z, x, z, VC, order=order)
    assert np.array_equal(a[0].view(np.uint64), b[0].view(np.uint64))
    assert np.array_equal(a[1].view(np.uint64), b[1].view(np.uint64))
