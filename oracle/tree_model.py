"""float64 numpy model of the far field of ludvm_b200/csrc/tree.cu, written from its kernels.

It is test infrastructure, the far-field counterpart of ludvm_oracle.c: the same bounding box and leaf level, the same
cells, interaction lists and proxy threshold, the same proxies (k_tree_up_leaf_mma / k_tree_up), local fields (the M2L
items of k_tree_eval, k_tree_m2l_dmma, k_tree_l2l), L2P (k_tree_l2p_mma / k_tree_l2p) and leaf items (k_tree_eval).  Only
the order of the floating-point sums differs, so the GPU agrees with it to rounding at every order, whatever that order's
truncation error against the all-pairs sum.  The pair counter counts what the kernels' `pairs` counter counts.

Circulations are scaled by 1 / (2 pi) up front, as k_tree_gather does; every velocity is
u = sum_j g_j dz / sqrt(r^4 + vc^4), w = -sum_j g_j dx / sqrt(r^4 + vc^4) with (dx, dz) = target - source."""
import math

import numpy as np

MAX_ORDER = 24
MAX_LEVEL = 10
_CHUNK = 1 << 22      # pair-matrix elements per block of the direct sums


def fma(a, b, c):
    """a * b + c rounded once (as the kernels' fma), through the 64-bit-mantissa long double."""
    return (np.asarray(a, np.longdouble) * np.asarray(b, np.longdouble) + np.asarray(c, np.longdouble)).astype(np.float64)


def nodes(order):
    """Chebyshev points of the second kind and barycentric weights, as tree_velocity_device builds them."""
    p1 = order + 1
    k = np.arange(p1)
    s = np.sin(np.pi * (order - 2 * k).astype(np.float64) / (2 * order))
    if order % 2 == 0:
        s[order // 2] = 0.0
    for j in range(p1 // 2):
        s[order - j] = -s[j]
    bw = np.where(k & 1, -1.0, 1.0) * np.where((k == 0) | (k == order), 0.5, 1.0)
    return s, bw


def basis(s, bw, xi):
    """Barycentric Lagrange basis l_k(xi) [len(xi), P1]; a point on a node gets that node's unit vector (the snap)."""
    d = np.asarray(xi, np.float64)[:, None] - s[None, :]
    hit = d == 0.0
    d[hit] = 1.0
    t = bw[None, :] / d
    out = t / t.sum(1)[:, None]
    rows = hit.any(1)
    out[rows] = hit[rows]
    return out


def _proxy_threshold(P2):
    """A cell with more than this many source vortices is represented by proxies and carries a local field."""
    return max(1, P2 // 4)


def _spread(v):
    v = np.asarray(v, np.int64) & 0xFFFF
    v = (v | (v << 8)) & 0x00FF00FF
    v = (v | (v << 4)) & 0x0F0F0F0F
    v = (v | (v << 2)) & 0x33333333
    v = (v | (v << 1)) & 0x55555555
    return v


def _compact(v):
    v = np.asarray(v, np.int64) & 0x55555555
    v = (v | (v >> 1)) & 0x33333333
    v = (v | (v >> 2)) & 0x0F0F0F0F
    v = (v | (v >> 4)) & 0x00FF00FF
    v = (v | (v >> 8)) & 0x0000FFFF
    return v


def morton(ix, iz):
    return _spread(ix) | (_spread(iz) << 1)


def level_offset(l):
    return ((1 << (2 * l)) - 16) // 3


def _lround(x):
    f = math.floor(x)
    return int(f) + (1 if x - f >= 0.5 else 0)


class Geom:
    """Host planning of tree_velocity_device: root square, leaf level L, nodes, proxy threshold."""

    def __init__(self, xs, zs, bx, bz, order, leaf=0, tdens=0.0, L=None):
        if not 2 <= order <= MAX_ORDER:
            raise ValueError("order %d outside 2..%d" % (order, MAX_ORDER))
        fin = lambda v: v[np.isfinite(v)]
        xa, za = fin(np.concatenate([xs, bx])), fin(np.concatenate([zs, bz]))
        xlo, xhi, zlo, zhi = xa.min(), xa.max(), za.min(), za.max()
        sxl, sxh, szl, szh = xs.min(), xs.max(), zs.min(), zs.max()
        side = max(xhi - xlo, zhi - zlo)
        side = side * (1.0 + 1e-12) + 1e-300
        P1 = order + 1
        P2 = P1 * P1
        nw = len(xs)
        pop = float(leaf) if leaf > 0 else (64.0 if tdens > 0.0 else 1.0 * P2)
        area = max((sxh - sxl) * (szh - szl), side * side * 1e-12)
        a0 = math.sqrt(pop * area / max(1, nw))
        Lw = _lround(math.log2(max(side / a0, 1.0)))
        lcap = 2
        while lcap < MAX_LEVEL and (1 << (2 * (lcap - 1))) < nw:
            lcap += 1
        Lw = max(2, min(min(MAX_LEVEL, lcap), Lw))
        if L is not None:        # LUDVM_TREE_LEVEL
            Lw = max(2, min(MAX_LEVEL, int(L)))
        self.x0, self.z0, self.side, self.L = xlo, zlo, side, Lw
        self.inv_leaf = float(1 << Lw) / side
        self.order, self.P1, self.P2 = order, P1, P2
        self.tdens = tdens
        self.pth = _proxy_threshold(P2)
        self.s, self.bw = nodes(order)

    def h(self, l):
        return math.ldexp(self.side, -(l + 1))

    def centre(self, l, c):
        """Centres of cells c (Morton index, array) of level l, as the kernels compute them."""
        h = self.h(l)
        c = np.asarray(c, np.int64)
        return self.x0 + (2.0 * _compact(c) + 1.0) * h, self.z0 + (2.0 * _compact(c >> 1) + 1.0) * h

    def keys(self, x, z):
        nc = 1 << self.L
        ix = np.clip(np.trunc((x - self.x0) * self.inv_leaf), 0, nc - 1).astype(np.int64)
        iz = np.clip(np.trunc((z - self.z0) * self.inv_leaf), 0, nc - 1).astype(np.int64)
        return morton(ix, iz)


def direct(xt, zt, xs, zs, gs, vc4):
    """sum_j of the pair velocity over sources (xs, zs, gs) at every target; gs already carries the 1 / (2 pi)."""
    u, w = np.zeros(len(xt)), np.zeros(len(xt))
    if len(xs) == 0 or len(xt) == 0:
        return u, w
    step = max(1, _CHUNK // len(xs))
    for i0 in range(0, len(xt), step):
        dx = xt[i0:i0 + step, None] - xs[None, :]
        dz = zt[i0:i0 + step, None] - zs[None, :]
        q = dx * dx
        q += dz * dz
        q *= q
        q += vc4
        np.sqrt(q, out=q)
        np.divide(1.0, q, out=q)
        dz *= q
        dx *= q
        u[i0:i0 + step] = dz @ gs
        w[i0:i0 + step] = -(dx @ gs)
    return u, w


def _m2l_matrix(G, l, dx, dz, vc4):
    """(Mu, Mw)[j, i]: velocity at node i of a cell of level l from a unit proxy j of the cell at offset (dx, dz)
    (k_tree_m2l_mats, coordinates relative to the target cell's centre)."""
    h, s, P1 = G.h(l), G.s, G.P1
    i1, i2 = np.divmod(np.arange(G.P2), P1)
    xt, zt = h * s[i1], h * s[i2]
    xs, zs = fma(h, s[i1], 2.0 * h * dx), fma(h, s[i2], 2.0 * h * dz)
    ddx = xt[None, :] - xs[:, None]
    ddz = zt[None, :] - zs[:, None]
    r2 = ddx * ddx + ddz * ddz
    q = 1.0 / np.sqrt(r2 * r2 + vc4)
    return q * ddz, -q * ddx


def _l2l(G, l, child, parent, U, W):
    """L2L of level l (k_tree_l2l): the parents' local fields interpolated to the points of the children, added."""
    P1 = G.P1
    for ch in range(4):
        sel = (child & 3) == ch
        if not sel.any():
            continue
        Bx = basis(G.s, G.bw, (G.s + float((ch & 1) * 2 - 1)) * 0.5)
        Bz = basis(G.s, G.bw, (G.s + float((ch >> 1) * 2 - 1)) * 0.5)
        for F, Fp in ((U[l], U[l - 1]), (W[l], W[l - 1])):
            Pm = Fp[parent[sel]].reshape(-1, P1, P1)
            F[child[sel]] += np.einsum("km,cmn,jn->ckj", Bx, Pm, Bz, optimize=True).reshape(-1, G.P2)


class _Tree:
    def __init__(self, G, g, xs, zs, xt, zt, vc4):
        self.G, self.vc4 = G, vc4
        L = G.L
        ks = G.keys(xs, zs)
        ps = np.argsort(ks, kind="stable")          # cells in Morton order, a cell's sources by original index
        self.xs, self.zs, self.gs = xs[ps], zs[ps], g[ps] * (1.0 / (2.0 * math.pi))
        ncell = 1 << (2 * L)
        self.startS = np.searchsorted(ks[ps], np.arange(ncell + 1))
        self.keyT = G.keys(xt, zt)
        cntT = np.bincount(self.keyT, minlength=ncell)
        cntS = np.diff(self.startS)
        self.nS, self.nT = {}, {}
        for l in range(2, L + 1):
            self.nS[l] = cntS.reshape(1 << (2 * l), -1).sum(1)
            self.nT[l] = cntT.reshape(1 << (2 * l), -1).sum(1)
        self.prox = {l: self.nS[l] > G.pth for l in self.nS}
        self.local = {l: self.prox[l] | (G.tdens * math.ldexp(G.side, -l) ** 2 > float(G.P2)) for l in self.nS}
        self.pairs = 0
        self._lists = {}
        self._src = {}

    def srange(self, l, c):
        sh = 2 * (self.G.L - l)
        return int(self.startS[c << sh]), int(self.startS[(c + 1) << sh])

    def far_list(self, l, c):
        """Level-l far list of cell c of level l in slot order: cells of level l, empty ones dropped."""
        key = (l, c)
        if key not in self._lists:
            cx, cz = int(_compact(c)), int(_compact(c >> 1))
            out = []
            for r in range(36):
                pn, ch = r >> 2, r & 3
                qx, qz = (cx >> 1) + pn % 3 - 1, (cz >> 1) + pn // 3 - 1
                if not (0 <= qx < (1 << (l - 1)) and 0 <= qz < (1 << (l - 1))):
                    continue
                jx, jz = 2 * qx + (ch & 1), 2 * qz + (ch >> 1)
                if max(abs(jx - cx), abs(jz - cz)) <= 1:
                    continue
                cc = int(morton(jx, jz))
                if self.nS[l][cc] > 0:
                    out.append(cc)
            self._lists[key] = out
        return self._lists[key]

    def sources(self, l, c):
        """What cell c of level l contributes as a list entry: its proxies, or its vortices."""
        if self.prox[l][c]:
            key = (l, c)
            if key not in self._src:
                G = self.G
                h = G.h(l)
                cx, cz = G.centre(l, c)
                k1, k2 = np.divmod(np.arange(G.P2), G.P1)
                self._src[key] = (fma(h, G.s[k1], cx), fma(h, G.s[k2], cz), self.qhat[l][c])
            return self._src[key]
        b, e = self.srange(l, c)
        return self.xs[b:e], self.zs[b:e], self.gs[b:e]

    def upward(self):
        G, L, P1, P2 = self.G, self.G.L, self.G.P1, self.G.P2
        self.qhat = {l: np.zeros((1 << (2 * l), P2)) for l in range(2, L + 1)}
        Tq = [basis(G.s, G.bw, (G.s + float(2 * v - 1)) * 0.5).T for v in (0, 1)]     # Tq[v][k][m]
        for l in range(L, 1, -1):
            h = G.h(l)
            inv_h = 1.0 / h
            for c in np.nonzero(self.prox[l])[0]:
                c = int(c)
                cx, cz = G.centre(l, c)
                acc = np.zeros((P1, P1))
                if l == L:
                    segs = [self.srange(l, c)]
                else:
                    segs = []
                    for ch in range(4):
                        cc = 4 * c + ch
                        b, e = self.srange(l + 1, cc)
                        if e == b:
                            continue
                        if self.prox[l + 1][cc]:
                            acc += Tq[ch & 1] @ self.qhat[l + 1][cc].reshape(P1, P1) @ Tq[ch >> 1].T
                        else:
                            segs.append((b, e))
                if segs:
                    idx = np.concatenate([np.arange(b, e) for b, e in segs])
                    Lx = basis(G.s, G.bw, (self.xs[idx] - cx) * inv_h)
                    Lz = basis(G.s, G.bw, (self.zs[idx] - cz) * inv_h)
                    acc += (Lx * self.gs[idx][:, None]).T @ Lz
                self.qhat[l][c] = acc.ravel()

    def downward(self):
        """Local fields of every level (M2L items of k_tree_eval + k_tree_m2l_dmma, then k_tree_l2l)."""
        G, L, P1, P2, vc4 = self.G, self.G.L, self.G.P1, self.G.P2, self.vc4
        self.U, self.W = {}, {}
        k1, k2 = np.divmod(np.arange(P2), P1)
        for l in range(2, L + 1):
            U, W = np.zeros((1 << (2 * l), P2)), np.zeros((1 << (2 * l), P2))
            self.U[l], self.W[l] = U, W
            act = np.nonzero(self.local[l] & (self.nT[l] > 0))[0]
            h = G.h(l)
            for c in act:        # plain-vortex cells of the list, at the cell's P2 points
                c = int(c)
                ent = [self.sources(l, b) for b in self.far_list(l, c) if not self.prox[l][b]]
                n = sum(len(e[0]) for e in ent)
                self.pairs += P2 * n
                if n:
                    cx, cz = G.centre(l, c)
                    u, w = direct(fma(h, G.s[k1], cx), fma(h, G.s[k2], cz), *(np.concatenate(v) for v in zip(*ent)), vc4)
                    U[c], W[c] = u, w
            if len(act) == 0:
                continue
            ax, az = _compact(act), _compact(act >> 1)
            nc = 1 << l
            for off in range(49):          # proxy cells of the list: one matrix product per offset
                dx, dz = off % 7 - 3, off // 7 - 3
                if max(abs(dx), abs(dz)) <= 1:
                    continue
                px, pz = ax & 1, az & 1
                bx, bz = ax + dx, az + dz
                ok = (dx >= -2 - px) & (dx <= 3 - px) & (dz >= -2 - pz) & (dz <= 3 - pz)
                ok &= (bx >= 0) & (bz >= 0) & (bx < nc) & (bz < nc)
                bc = morton(np.where(ok, bx, 0), np.where(ok, bz, 0))
                ok &= self.prox[l][bc]
                if not ok.any():
                    continue
                Mu, Mw = _m2l_matrix(G, l, dx, dz, vc4)
                Q = self.qhat[l][bc[ok]]
                U[act[ok]] += Q @ Mu
                W[act[ok]] += Q @ Mw
            if l >= 3:
                _l2l(G, l, act, act >> 2, self.U, self.W)

    def local_level(self, c):
        """tree_local_level: deepest level whose ancestor of leaf c carries a local field, or 1."""
        L = self.G.L
        for l in range(L, 1, -1):
            if self.local[l][c >> (2 * (L - l))]:
                return l
        return 1

    def evaluate(self, xt, zt):
        G, L, vc4 = self.G, self.G.L, self.vc4
        nc = 1 << L
        u, w = np.zeros(len(xt)), np.zeros(len(xt))
        pt = np.argsort(self.keyT, kind="stable")
        startT = np.searchsorted(self.keyT[pt], np.arange((1 << (2 * L)) + 1))
        self.lstar_count = np.zeros(L + 1, np.int64)
        for c in np.nonzero(np.diff(startT))[0]:
            c = int(c)
            ti = pt[startT[c]:startT[c + 1]]
            lstar = self.local_level(c)
            self.lstar_count[lstar] += len(ti)
            cx, cz = int(_compact(c)), int(_compact(c >> 1))
            ent = []
            for s in range(9):      # the 3 x 3 neighbour leaves: their vortices, proxies or not
                jx, jz = cx + s % 3 - 1, cz + s // 3 - 1
                if 0 <= jx < nc and 0 <= jz < nc:
                    b, e = self.srange(L, int(morton(jx, jz)))
                    ent.append((self.xs[b:e], self.zs[b:e], self.gs[b:e]))
            for l in range(lstar + 1, L + 1):
                ent += [self.sources(l, b) for b in self.far_list(l, c >> (2 * (L - l)))]
            sx, sz, sg = (np.concatenate(v) for v in zip(*ent))
            self.pairs += len(ti) * len(sx)
            uu, ww = direct(xt[ti], zt[ti], sx, sz, sg, vc4)
            if lstar >= 2:          # L2P
                a = c >> (2 * (L - lstar))
                h = G.h(lstar)
                acx, acz = G.centre(lstar, a)
                bx = basis(G.s, G.bw, (xt[ti] - acx) * (1.0 / h))
                bz = basis(G.s, G.bw, (zt[ti] - acz) * (1.0 / h))
                Ua, Wa = self.U[lstar][a].reshape(G.P1, G.P1), self.W[lstar][a].reshape(G.P1, G.P1)
                uu = uu + np.einsum("tk,kj,tj->t", bx, Ua, bz)
                ww = ww + np.einsum("tk,kj,tj->t", bx, Wa, bz)
            u[ti], w[ti] = uu, ww
        return u, w

    def info(self):
        L = self.G.L
        lv = range(2, L + 1)
        return dict(
            L=L, pth=self.G.pth, P2=self.G.P2, pairs=int(self.pairs),
            proxy_cells={l: int(self.prox[l].sum()) for l in lv},
            plain_cells={l: int(((self.nS[l] > 0) & ~self.prox[l]).sum()) for l in lv},
            local_cells={l: int((self.local[l] & (self.nT[l] > 0)).sum()) for l in lv},
            targets_by_local_level={l: int(self.lstar_count[l]) for l in range(1, L + 1)},
            targets_below_leaf_level=int(self.lstar_count[:L].sum()))


def _run(g, xs, zs, xt, zt, vc4, G):
    T = _Tree(G, g, xs, zs, xt, zt, vc4)
    T.upward()
    T.downward()
    u, w = T.evaluate(xt, zt)
    return u, w, T.info()


def _f64(a):
    return np.ascontiguousarray(np.atleast_1d(a), dtype=np.float64)


def tree_velocity(g, xs, zs, xt, zt, vc4, order=18, leaf=0, L=None):
    """ludvm_induced_velocity_tree: velocity of sources (g, xs, zs) at targets (xt, zt), core radius vc4 ** 0.25.
    `L` forces the leaf level (LUDVM_TREE_LEVEL).  Returns u, w and a dict of the tree's counters: L, pth, P2, pairs
    (= the kernels' pair_evaluations), per level the cells with proxies, the non-empty cells without, the cells that
    carry a local field for these targets, and the targets per level of the local field they take (1: none)."""
    g, xs, zs, xt, zt = (_f64(a) for a in (g, xs, zs, xt, zt))
    G = Geom(xs, zs, xt, zt, order, leaf, 0.0, L)
    return _run(g, xs, zs, xt, zt, vc4, G)


def grid_density(x1, z1):
    """Points per unit area of the 'ij' mesh x1 x z1 (what ops.flowfield_velocity_tree passes)."""
    dx = (x1[-1] - x1[0]) / max(len(x1) - 1, 1)
    dz = (z1[-1] - z1[0]) / max(len(z1) - 1, 1)
    return 1.0 / (dx * dz) if dx > 0 and dz > 0 else 0.0


def flowfield_velocity(g, xs, zs, vc4, x1, z1, row0=0, nrows=None, order=18, leaf=0, L=None):
    """ludvm_flowfield_velocity_tree: velocity on rows [row0, row0 + nrows) of the 'ij' mesh x1 x z1 -> [nrows, len(z1)];
    the tree is the full grid's (its corners and its density), whatever the rows."""
    g, xs, zs, x1, z1 = (_f64(a) for a in (g, xs, zs, x1, z1))
    nrows = len(x1) - row0 if nrows is None else nrows
    xt = np.repeat(x1[row0:row0 + nrows], len(z1))
    zt = np.tile(z1, nrows)
    G = Geom(xs, zs, np.array([x1[0], x1[-1]]), np.array([z1[0], z1[-1]]), order, leaf, grid_density(x1, z1), L)
    u, w, info = _run(g, xs, zs, xt, zt, vc4, G)
    return u.reshape(nrows, len(z1)), w.reshape(nrows, len(z1)), info
