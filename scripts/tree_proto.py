"""Command line over oracle/tree_model.py, the float64 numpy model of the far field of csrc/tree.cu: the error of one
order and leaf size against direct summation on a uniform cloud, and the pairs the tree evaluates.
Usage: python scripts/tree_proto.py [N] [order] [leaf]"""
import math
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import tree_model  # noqa: E402
from oracle.tree_model import direct  # noqa: E402,F401  (sum of g / sqrt(r^4 + vc^4) terms, circulations as given)


def tree_velocity(g, xs, zs, xt, zt, vc4, p=18, leaf=256, L=None):
    """The model's velocity at order p on this script's scale, that of direct(..., g, ...): circulations without the
    1 / (2 pi).  Returns u, w and dict(L, pairs, proxy_cells = number of cells with proxies over all levels)."""
    u, w, info = tree_model.tree_velocity(g, xs, zs, xt, zt, vc4, order=p, leaf=leaf, L=L)
    return (2.0 * math.pi) * u, (2.0 * math.pi) * w, dict(L=info["L"], pairs=info["pairs"],
                                                          proxy_cells=sum(info["proxy_cells"].values()))


if __name__ == "__main__":
    N = int(sys.argv[1]) if len(sys.argv) > 1 else 20000
    p = int(sys.argv[2]) if len(sys.argv) > 2 else 18
    leaf = int(sys.argv[3]) if len(sys.argv) > 3 else 64
    rng_ = np.random.default_rng(5)
    g = rng_.standard_normal(N) * 1e-2
    x, z = rng_.uniform(-20, 0, N), rng_.uniform(-4, 4, N)
    vc4 = 0.065 ** 4
    u, w, st = tree_velocity(g, x, z, x, z, vc4, p, leaf)
    sel = rng_.choice(N, 400, replace=False)
    ud, wd = direct(x[sel], z[sel], x, z, g, vc4)
    den = np.zeros(len(sel))
    for k, i in enumerate(sel):
        dx, dz = x[i] - x, z[i] - z
        den[k] = (np.abs(g) * np.hypot(dx, dz) / np.sqrt((dx * dx + dz * dz) ** 2 + vc4)).sum()
    print(st, "pairs/N^2 = %.4f" % (st["pairs"] / N / N))
    print("max |du| / sum|terms| = %.3e   max|du|/max|u| = %.3e" % (np.max(np.hypot(u[sel] - ud, w[sel] - wd) / den),
                                                               np.max(np.abs(u[sel] - ud)) / np.max(np.abs(ud))))
