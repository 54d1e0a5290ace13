"""Array-level entry points over the C ABI (numpy in / numpy out, or torch CUDA tensors in place)."""
import numpy as np

from . import _lib
from ._lib import MODES, PTR_DEVICE, PTR_HOST, check, f64, load, ptr


def _mode(mode):
    return MODES[mode] if isinstance(mode, str) else int(mode)


def induced_velocity(circulation, xw, zw, xp, zp, v_core, viscous=True, mode="exact", ctx=None, vc4_per_source=None):
    """LUDVM.induced_velocity (LUDVM.py:549-570) on the GPU with host (numpy) buffers.

    `v_core` is the core radius (the reference reads `self.v_core`); `viscous=False` uses point vortices.
    `mode="tree"` routes to `induced_velocity_tree` (hierarchical far field, default order)."""
    if mode == "tree":
        if vc4_per_source is not None or np.size(circulation) == 1:
            raise ValueError("mode='tree' needs one circulation per vortex and a single core radius")
        return induced_velocity_tree(circulation, xw, zw, xp, zp, v_core if viscous == True else 0.0, ctx=ctx)  # noqa: E712
    ctx = ctx or _lib.default_context()
    g, xw, zw, xp, zp = (f64(np.atleast_1d(a)) for a in (circulation, xw, zw, xp, zp))
    if xw.size != zw.size or xp.size != zp.size or g.size not in (1, xw.size):
        raise ValueError("shape mismatch: circulation %d, xw %d, zw %d, xp %d, zp %d"
                         % (g.size, xw.size, zw.size, xp.size, zp.size))
    vc4 = float(v_core) ** 4 if viscous == True else 0.0  # noqa: E712 (LUDVM.py:562 compares with ==)
    vcs = f64(vc4_per_source) if vc4_per_source is not None else None
    u, w = np.empty(xp.size), np.empty(xp.size)
    check(load().ludvm_induced_velocity(ctx.handle, _mode(mode), ptr(g), g.size, ptr(xw), ptr(zw), ptr(vcs), vc4,
                                        xw.size, ptr(xp), ptr(zp), xp.size, ptr(u), ptr(w), PTR_HOST))
    return u, w


def induced_velocity_device(ctx, mode, g, xw, zw, xp, zp, vc4, u, w, vc4_per_source=None):
    """Same with torch CUDA float64 tensors (results written into u, w; asynchronous on ctx's stream)."""
    check(load().ludvm_induced_velocity(ctx.handle, _mode(mode), ptr(g), g.numel(), ptr(xw), ptr(zw),
                                        ptr(vc4_per_source), float(vc4), xw.numel(), ptr(xp), ptr(zp), xp.numel(),
                                        ptr(u), ptr(w), PTR_DEVICE))


def induced_velocity_tree(circulation, xw, zw, xp, zp, v_core, order=18, leaf=0, ctx=None, return_stats=False):
    """The sum of `induced_velocity` (LUDVM.py:549-570) through the O(N log N) treecode (csrc/tree.cu), host buffers.

    `order` (2..24) is the Chebyshev interpolation order of the far field: the error against the all-pairs sum,
    relative to sum |terms|, is about 2e-11 at 12, 5e-14 at 16 and 3e-15 at 18.  `leaf`: wanted mean number of vortices
    per leaf cell (0: library default).  The reference has no counterpart; the all-pairs modes are the checker."""
    ctx = ctx or _lib.default_context()
    g, xw, zw, xp, zp = (f64(np.atleast_1d(a)) for a in (circulation, xw, zw, xp, zp))
    if xw.size != zw.size or xp.size != zp.size or g.size != xw.size:
        raise ValueError("shape mismatch: circulation %d, xw %d, zw %d, xp %d, zp %d"
                         % (g.size, xw.size, zw.size, xp.size, zp.size))
    u, w = np.empty(xp.size), np.empty(xp.size)
    stats = np.zeros(8)
    check(load().ludvm_induced_velocity_tree(ctx.handle, ptr(g), ptr(xw), ptr(zw), float(v_core) ** 4, xw.size, ptr(xp),
                                             ptr(zp), xp.size, int(order), int(leaf), ptr(u), ptr(w), PTR_HOST,
                                             stats.ctypes.data_as(_lib.c_dp) if return_stats else None))
    return (u, w, _tree_stats(stats)) if return_stats else (u, w)


def _tree_stats(s):
    return dict(leaf_level=int(s[0]), leaf_side=s[1], pair_evaluations=s[2], all_pairs=s[3], proxies_per_cell=int(s[4]),
                arena_bytes=int(s[5]), build_ms=s[6], eval_ms=s[7])


def induced_velocity_tree_device(ctx, g, xw, zw, xp, zp, vc4, u, w, order=18, leaf=0, return_stats=False):
    """Same with torch CUDA float64 tensors (asynchronous on ctx's stream unless stats are asked for)."""
    stats = np.zeros(8)
    check(load().ludvm_induced_velocity_tree(ctx.handle, ptr(g), ptr(xw), ptr(zw), float(vc4), xw.numel(), ptr(xp), ptr(zp),
                                             xp.numel(), int(order), int(leaf), ptr(u), ptr(w), PTR_DEVICE,
                                             stats.ctypes.data_as(_lib.c_dp) if return_stats else None))
    return _tree_stats(stats) if return_stats else None


def _grid_density(x1, z1):
    dx = (x1[-1] - x1[0]) / max(len(x1) - 1, 1)
    dz = (z1[-1] - z1[0]) / max(len(z1) - 1, 1)
    return 1.0 / (dx * dz) if dx > 0 and dz > 0 else 0.0


def flowfield_velocity_tree(g, xw, zw, vc4, x1, z1, row0=0, nrows=None, order=18, leaf=0, ctx=None, return_stats=False):
    """`flowfield_velocity` for one source set through the hierarchical far field (csrc/tree.cu), host buffers."""
    ctx = ctx or _lib.default_context()
    g, xw, zw, x1, z1 = (f64(a) for a in (g, xw, zw, x1, z1))
    nrows = x1.size - row0 if nrows is None else nrows
    u, w = np.empty((nrows, z1.size)), np.empty((nrows, z1.size))
    stats = np.zeros(8)
    check(load().ludvm_flowfield_velocity_tree(ctx.handle, ptr(g), ptr(xw), ptr(zw), g.size, float(vc4), ptr(x1), x1.size,
                                               ptr(z1), z1.size, int(row0), int(nrows), _grid_density(x1, z1), int(order),
                                               int(leaf), ptr(u), ptr(w), PTR_HOST,
                                               stats.ctypes.data_as(_lib.c_dp) if return_stats else None))
    return (u, w, _tree_stats(stats)) if return_stats else (u, w)


def flowfield_velocity_tree_device(ctx, g, xw, zw, vc4, x1, z1, row0, nrows, u, w, tgt_density, order=18, leaf=0,
                                   return_stats=False):
    """Same with torch CUDA float64 tensors; `tgt_density` = grid points per unit area of the full grid."""
    stats = np.zeros(8)
    check(load().ludvm_flowfield_velocity_tree(ctx.handle, ptr(g), ptr(xw), ptr(zw), g.numel(), float(vc4), ptr(x1),
                                               x1.numel(), ptr(z1), z1.numel(), int(row0), int(nrows), float(tgt_density),
                                               int(order), int(leaf), ptr(u), ptr(w), PTR_DEVICE,
                                               stats.ctypes.data_as(_lib.c_dp) if return_stats else None))
    return _tree_stats(stats) if return_stats else None


def selfconv_step_tree(ctx, g, x, z, vc4, dt, x_out, z_out, row0=0, nrows=None, u_out=None, w_out=None, order=18, leaf=0,
                       return_stats=False):
    """`selfconv_step` through the treecode (torch CUDA float64 tensors)."""
    n = x.numel()
    nrows = n - row0 if nrows is None else nrows
    stats = np.zeros(8)
    check(load().ludvm_selfconv_step_tree(ctx.handle, ptr(g), ptr(x), ptr(z), float(vc4), n, int(row0), int(nrows), float(dt),
                                          int(order), int(leaf), ptr(x_out), ptr(z_out), ptr(u_out), ptr(w_out),
                                          stats.ctypes.data_as(_lib.c_dp) if return_stats else None))
    return _tree_stats(stats) if return_stats else None


def selfconv_step(ctx, mode, g, x, z, vc4, dt, x_out, z_out, row0=0, nrows=None, u_out=None, w_out=None,
                  vc4_per_source=None):
    """One forward-Euler self-convection step of rows [row0, row0+nrows) (torch CUDA float64 tensors)."""
    n = x.numel()
    nrows = n - row0 if nrows is None else nrows
    check(load().ludvm_selfconv_step(ctx.handle, _mode(mode), ptr(g), ptr(x), ptr(z), ptr(vc4_per_source), float(vc4),
                                     n, int(row0), int(nrows), float(dt), ptr(x_out), ptr(z_out), ptr(u_out),
                                     ptr(w_out)))


def selfconv_step_all(ctx, mode, g, x, z, vc4, dt, x_out, z_out, u_out=None, w_out=None, vc4_per_source=None):
    """`selfconv_step` of the whole cloud (all rows), bit for bit; in fast mode with one core radius it evaluates each
    pair of vortices once (kernel fast_sym, see ludvm_selfconv_step_all)."""
    check(load().ludvm_selfconv_step_all(ctx.handle, _mode(mode), ptr(g), ptr(x), ptr(z), ptr(vc4_per_source), float(vc4),
                                         x.numel(), float(dt), ptr(x_out), ptr(z_out), ptr(u_out), ptr(w_out)))


def selfconv_step_p2p(ctx, mode, g, x, z, vc4, dt, x_out_peer_ptrs, z_out_peer_ptrs, row0, nrows):
    """Self-convection step whose epilogue stores the shard's updated rows into every peer's buffers (raw peer-mapped
    device pointers, this rank included) -- the all-gather fused into the kernel over NVLink."""
    import ctypes as C
    n = x.numel()
    npeers = len(x_out_peer_ptrs)
    xs = (_lib.c_vp * npeers)(*[int(p) for p in x_out_peer_ptrs])
    zs = (_lib.c_vp * npeers)(*[int(p) for p in z_out_peer_ptrs])
    check(load().ludvm_selfconv_step_p2p(ctx.handle, _mode(mode), ptr(g), ptr(x), ptr(z), None, float(vc4), n, int(row0),
                                         int(nrows), float(dt), npeers, xs, zs))


def flowfield_velocity(ga, xa, za, gb, xb, zb, vc4, x1, z1, row0=0, nrows=None, mode="exact", ctx=None):
    """Velocity of up to two source sets on the 'ij' mesh x1 x z1 (LUDVM.py:1193-1220), host buffers."""
    ctx = ctx or _lib.default_context()
    ga, xa, za, x1, z1 = (f64(a) for a in (ga, xa, za, x1, z1))
    nb = 0 if gb is None else len(gb)
    if nb:
        gb, xb, zb = (f64(a) for a in (gb, xb, zb))
    nrows = x1.size - row0 if nrows is None else nrows
    u, w = np.empty((nrows, z1.size)), np.empty((nrows, z1.size))
    check(load().ludvm_flowfield_velocity(ctx.handle, _mode(mode), ptr(ga), ptr(xa), ptr(za), ga.size,
                                          ptr(gb) if nb else None, ptr(xb) if nb else None, ptr(zb) if nb else None,
                                          nb, float(vc4), ptr(x1), x1.size, ptr(z1), z1.size, int(row0), int(nrows),
                                          ptr(u), ptr(w), PTR_HOST))
    return u, w


def flowfield(ga, xa, za, gb, xb, zb, vc4, x1, z1, row0=0, nrows=None, mode="exact", ctx=None):
    """Velocity and vorticity of one snapshot on rows [row0, row0+nrows) of the 'ij' mesh x1 x z1 in one call
    (LUDVM.py:1193-1292), host buffers: returns (u, w, ome), each [nrows, len(z1)]."""
    ctx = ctx or _lib.default_context()
    ga, xa, za, x1, z1 = (f64(a) for a in (ga, xa, za, x1, z1))
    nb = 0 if gb is None else len(gb)
    if nb:
        gb, xb, zb = (f64(a) for a in (gb, xb, zb))
    nrows = x1.size - row0 if nrows is None else nrows
    u, w, ome = (np.empty((nrows, z1.size)) for _ in range(3))
    check(load().ludvm_flowfield(ctx.handle, _mode(mode), ptr(ga), ptr(xa), ptr(za), ga.size,
                                 ptr(gb) if nb else None, ptr(xb) if nb else None, ptr(zb) if nb else None, nb,
                                 float(vc4), ptr(x1), x1.size, ptr(z1), z1.size, int(row0), int(nrows), ptr(u), ptr(w),
                                 ptr(ome), PTR_HOST))
    return u, w, ome


def flowfield_velocity_device(ctx, mode, g, xw, zw, vc4, x1, z1, row0, nrows, u, w):
    """Same for one source set with torch CUDA float64 tensors; u, w are [nrows, len(z1)] (asynchronous on ctx's
    stream)."""
    check(load().ludvm_flowfield_velocity(ctx.handle, _mode(mode), ptr(g), ptr(xw), ptr(zw), g.numel(), None, None,
                                          None, 0, float(vc4), ptr(x1), x1.numel(), ptr(z1), z1.numel(), int(row0),
                                          int(nrows), ptr(u), ptr(w), PTR_DEVICE))


def flowfield_vorticity(x1, z1, u, w, ctx=None):
    """Finite-difference vorticity of LUDVM.py:1222-1292 on [ns,nx,nz] fields, host buffers."""
    ctx = ctx or _lib.default_context()
    x1, z1, u, w = (f64(a) for a in (x1, z1, u, w))
    ome = np.empty_like(u)
    check(load().ludvm_flowfield_vorticity(ctx.handle, ptr(x1), x1.size, ptr(z1), z1.size, ptr(u), ptr(w), u.shape[0],
                                           ptr(ome), PTR_HOST))
    return ome
