"""oracle/tree_model.py, the float64 model of the far field of csrc/tree.cu, on the CPU: its truncation error against
direct summation, its exactness when nothing is represented by proxies, its own rounding noise (which sets the tolerance
of the GPU comparison in test_gpu_tree_orders.py), and mutations of the algorithm that comparison must be able to see."""
import numpy as np
import pytest

from test_gpu_tree_orders import TOL, VC, VC4, mixed_cloud

NT = 1500        # targets: a fixed sample of the cloud's own points


def sum_abs_terms(g, xw, zw, xp, zp):
    out = np.empty(len(xp))
    for i in range(len(xp)):
        dx, dz = xp[i] - xw, zp[i] - zw
        out[i] = np.sum(np.abs(g) * np.hypot(dx, dz) / np.sqrt((dx * dx + dz * dz) ** 2 + VC4)) / (2 * np.pi)
    return out


def _diff(u, w, ur, wr, den):
    d = np.hypot(u - ur, w - wr) / den
    return float(np.max(np.where(np.isfinite(d), d, np.inf)))


@pytest.fixture(scope="module")
def case():
    g, x, z = mixed_cloud()
    sel = np.sort(np.random.default_rng(4).choice(len(x), NT, replace=False))
    return g, x, z, x[sel], z[sel], sum_abs_terms(g, x, z, x[sel], z[sel])


@pytest.mark.parametrize("order,bound", [(2, 2e-3), (8, 5e-8), (14, 1e-11), (18, 5e-14), (24, 2e-15)])
def test_model_vs_direct_summation(case, oracle, order, bound):
    """The truncation error of each order against the all-pairs sum: these bounds describe the representation, the GPU
    tests do not rely on them."""
    from oracle import tree_model
    g, x, z, xp, zp, den = case
    u, w, info = tree_model.tree_velocity(g, x, z, xp, zp, VC4, order=order)
    assert info["proxy_cells"][info["L"]] > 0
    uo, wo = oracle.induced_velocity(g, x, z, xp, zp, VC)
    assert _diff(u, w, uo, wo, den) <= bound


@pytest.mark.parametrize("order", [2, 11, 24])
def test_model_without_proxies_is_direct_summation(oracle, monkeypatch, order):
    from oracle import tree_model
    rng = np.random.default_rng(order)
    n = 3000
    g, x, z = rng.standard_normal(n) * 1e-2, rng.uniform(-20, 0, n), rng.uniform(-4, 4, n)
    monkeypatch.setattr(tree_model, "_proxy_threshold", lambda P2: n)
    u, w, info = tree_model.tree_velocity(g, x, z, x, z, VC4, order=order, L=4)
    assert sum(info["proxy_cells"].values()) == 0 and sum(info["local_cells"].values()) == 0
    uo, wo = oracle.induced_velocity(g, x, z, x, z, VC)
    assert _diff(u, w, uo, wo, sum_abs_terms(g, x, z, x, z)) <= 1e-15


def test_model_rounding_noise(case):
    """The model on the same cloud with its sources permuted: every cell's sources, and so every sum, run in another
    order.  The largest change is the rounding noise of the algorithm; the GPU tolerance TOL sits above it and no more
    than 100x it."""
    from oracle import tree_model
    g, x, z, xp, zp, den = case
    p = np.random.default_rng(9).permutation(len(x))
    noise = {}
    for order in range(2, 25):
        u, w, _ = tree_model.tree_velocity(g, x, z, xp, zp, VC4, order=order)
        up, wp, _ = tree_model.tree_velocity(g[p], x[p], z[p], xp, zp, VC4, order=order)
        noise[order] = _diff(u, w, up, wp, den)
    print("model rounding noise / sum|terms| per order:", {k: "%.1e" % v for k, v in noise.items()})
    assert max(noise.values()) < TOL <= 100 * max(noise.values()), noise


def _no_snap_basis(s, bw, xi):
    d = np.asarray(xi, np.float64)[:, None] - s[None, :]
    with np.errstate(divide="ignore", invalid="ignore"):
        t = bw[None, :] / d
        return t / t.sum(1)[:, None]


def _mutations(tree_model):
    orig_l2l, orig_mat = tree_model._l2l, tree_model._m2l_matrix

    def skip_l2l(G, l, *a):
        if l != 3:
            orig_l2l(G, l, *a)

    def drop_slice(G, l, dx, dz, vc4):
        Mu, Mw = orig_mat(G, l, dx, dz, vc4)
        if (l, dx, dz) == (2, 2, 0):
            j0 = 16 * ((G.P2 - 1) // 16)
            Mu, Mw = Mu.copy(), Mw.copy()
            Mu[j0:] = Mw[j0:] = 0.0
        return Mu, Mw

    return {"pth = P2": ("_proxy_threshold", lambda P2: P2), "L2L skipped at level 3": ("_l2l", skip_l2l),
            "last k-slice of one M2L matrix dropped": ("_m2l_matrix", drop_slice),
            "node snap disabled": ("basis", _no_snap_basis)}


@pytest.mark.parametrize("order", [3, 12, 24])
def test_mutations_are_visible_to_the_gpu_comparison(case, monkeypatch, order):
    """Each variant of the algorithm differs from the model by at least 100x the GPU tolerance on the GPU tests' cloud,
    so a kernel with that defect cannot pass test_gpu_tree_orders.py.  The one exception is pth = P2 at order 24, where
    proxies reproduce their cells' vortices to rounding: there the lists change, and the GPU tests' exact comparison of
    the pair count sees it."""
    from oracle import tree_model
    g, x, z, xp, zp, den = case
    u, w, info = tree_model.tree_velocity(g, x, z, xp, zp, VC4, order=order)
    assert info["L"] >= 3 and info["local_cells"][3] > 0
    for name, (attr, fn) in _mutations(tree_model).items():
        with monkeypatch.context() as m:
            m.setattr(tree_model, attr, fn)
            um, wm, mi = tree_model.tree_velocity(g, x, z, xp, zp, VC4, order=order)
        margin = _diff(um, wm, u, w, den) / TOL
        print("order %d, %s: %.1e x TOL, pairs %d -> %d" % (order, name, margin, info["pairs"], mi["pairs"]))
        if name == "pth = P2" and order == 24:
            assert mi["pairs"] != info["pairs"]
        else:
            assert margin >= 100, (name, margin)
