"""CPU test of the multi-rank path: world_size-2 gloo, the per-row kernel replaced by the oracle (tests may use it).
Checks the row partition, the all-gather assembly and that the 2-rank result equals the 1-rank one bitwise."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

N, STEPS, VC, DT = 512, 3, 0.065, 0.05


def _cloud():
    rng = np.random.default_rng(5)
    return rng.standard_normal(N) * 1e-2, rng.uniform(-20, 0, N), rng.uniform(-4, 4, N)


def _oracle_kernel(g, x, z, vc4, dt, row0, nrows, x_out, z_out):
    from oracle import ludvm_oracle as o
    gn, xn, zn = g.numpy(), x.numpy(), z.numpy()
    u, w = o.induced_velocity(gn, xn, zn, xn[row0:row0 + nrows], zn[row0:row0 + nrows], vc4 ** 0.25, nthreads=1)
    x_out[row0:row0 + nrows] = torch.from_numpy(xn[row0:row0 + nrows] + dt * u)
    z_out[row0:row0 + nrows] = torch.from_numpy(zn[row0:row0 + nrows] + dt * w)


def _serial():
    from ludvm_b200.sharded import ShardedSelfConvection
    g, x, z = (torch.from_numpy(a.copy()) for a in _cloud())
    s = ShardedSelfConvection(g, x, z, VC, DT, kernel=_oracle_kernel)
    for _ in range(STEPS):
        xs, zs = s.step()
    return xs.numpy().copy(), zs.numpy().copy()


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from ludvm_b200.sharded import ShardedSelfConvection, shard_bounds
    g, x, z = (torch.from_numpy(a.copy()) for a in _cloud())
    s = ShardedSelfConvection(g, x, z, VC, DT, kernel=_oracle_kernel)
    assert (s.row0, s.nrows) == shard_bounds(N, world, rank) == (rank * N // world, N // world)
    for _ in range(STEPS):
        xs, zs = s.step()
    q.put((rank, xs.numpy().copy(), zs.numpy().copy()))
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_rows_equal_serial(oracle):
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    xs, zs = _serial()
    for _, x2, z2 in res:
        assert np.array_equal(x2, xs) and np.array_equal(z2, zs)


def test_shard_bounds_rejects_ragged():
    from ludvm_b200.sharded import shard_bounds
    with pytest.raises(ValueError):
        shard_bounds(10, 4, 0)
    assert shard_bounds(16, 4, 3) == (12, 4)


# ---------------------------------------------------------------------------------------------------
# collective-free shardings: parameter sweeps (configs[3]) and flow-field x-row slabs (configs[4])
# ---------------------------------------------------------------------------------------------------
SWEEP_KW = dict(t0=0, tf=0.5, dt=5e-2, chord=1, rho=1.225, Uinf=1, Npoints=81, Ncoeffs=30, Naca="0012")
SWEEP_CASES = [dict(SWEEP_KW, LESPcrit=lc, k=k) for lc in (0.1, 0.2, 0.3) for k in (0.3, 0.8)][:5]   # ragged over 2 ranks
FF_NX, FF_NZ, FF_NSRC = 37, 11, 200


def _ff_inputs():
    rng = np.random.default_rng(21)
    g, xw, zw = rng.standard_normal(FF_NSRC) * 1e-2, rng.uniform(-3, 0, FF_NSRC), rng.uniform(-1, 1, FF_NSRC)
    return g, xw, zw, np.linspace(-3.0, 0.5, FF_NX), np.linspace(-1.0, 1.0, FF_NZ)


def _ff_eval(o, g, xw, zw, x1, z1):
    """velocity + vorticity of the oracle on the 'ij' mesh x1 x z1 -> (u, w, ome), each [len(x1), len(z1)]"""
    X, Z = np.meshgrid(x1, z1, indexing="ij")
    u, w = o.induced_velocity(g, xw, zw, X.ravel(), Z.ravel(), VC, nthreads=1)
    u, w = u.reshape(X.shape), w.reshape(X.shape)
    return u, w, o.vorticity(X, Z, u[None], w[None])[0]


def _worker_nocollective(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from ludvm_b200.sharded import case_slice, grid_slab
    from oracle import ludvm_oracle as o
    sl = case_slice(len(SWEEP_CASES), world, rank)
    cl = [o.OracleLUDVM(**kw).Cl.copy() for kw in SWEEP_CASES[sl]]
    g, xw, zw, x1, z1 = _ff_inputs()
    r0, r1, h0, h1 = grid_slab(FF_NX, world, rank)
    u, w, ome = _ff_eval(o, g, xw, zw, x1[h0:h1], z1)
    keep = slice(r0 - h0, r1 - h0)
    q.put((rank, (sl.start, sl.stop), cl, (r0, r1), u[keep].copy(), w[keep].copy(), ome[keep].copy()))
    dist.barrier()                       # the only collective: nothing travels on the data path
    dist.destroy_process_group()


def test_two_rank_sweep_and_flowfield_slabs_equal_serial(oracle):
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker_nocollective, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=180) for _ in procs], key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    # sweep: the slices tile the case list, every history equals the serial run bitwise
    assert [r[1] for r in res] == [(0, 3), (3, 5)]
    serial_cl = [oracle.OracleLUDVM(**kw).Cl for kw in SWEEP_CASES]
    got = [c for r in res for c in r[2]]
    assert len(got) == len(serial_cl) and all(np.array_equal(a, b, equal_nan=True) for a, b in zip(got, serial_cl))
    # flow field: owned rows tile the grid; velocity AND the halo-fed vorticity stencil equal the whole-grid evaluation
    assert [r[3] for r in res] == [(0, 19), (19, 37)]
    us, ws, oms = _ff_eval(oracle, *_ff_inputs())
    for k, ref in ((4, us), (5, ws), (6, oms)):
        assert np.array_equal(np.concatenate([r[k] for r in res]), ref)


@pytest.mark.parametrize("world", [1, 2, 3, 4, 8])
def test_slab_and_case_partitions(oracle, world):
    """Any rank count: slices tile the range, halos never leave the grid, and the per-slab vorticity of the owned rows
    equals the whole-grid stencil (checked serially, rank by rank)."""
    from ludvm_b200.sharded import case_slice, grid_slab
    for n in (1, 5, 64, 4096):
        sl = [case_slice(n, world, r) for r in range(world)]
        assert sl[0].start == 0 and sl[-1].stop == n and all(a.stop == b.start for a, b in zip(sl, sl[1:]))
    g, xw, zw, x1, z1 = _ff_inputs()
    _, _, oms = _ff_eval(oracle, g, xw, zw, x1, z1)
    rows = []
    for r in range(world):
        r0, r1, h0, h1 = grid_slab(FF_NX, world, r)
        assert 0 <= h0 <= r0 <= r1 <= h1 <= FF_NX and r0 - h0 <= 1 and h1 - r1 <= 1
        rows.append((r0, r1))
        if r1 - r0 >= 1 and h1 - h0 >= 2:
            _, _, ome = _ff_eval(oracle, g, xw, zw, x1[h0:h1], z1)
            assert np.array_equal(ome[r0 - h0:r1 - h0], oms[r0:r1])
    assert rows[0][0] == 0 and rows[-1][1] == FF_NX and all(a[1] == b[0] for a, b in zip(rows, rows[1:]))


def test_morton_order_is_a_permutation_that_makes_row_shards_compact():
    """sharded.morton_order (used to relabel a cloud before a sharded far-field run): a permutation; the first eighth of
    the relabelled cloud covers about an eighth of the area instead of all of it."""
    from ludvm_b200.sharded import morton_order
    rng = np.random.default_rng(3)
    x, z = rng.uniform(-20, 0, 40000), rng.uniform(-4, 4, 40000)
    p = morton_order(x, z)
    assert sorted(p.tolist()) == list(range(40000))
    xs, zs = x[p][:5000], z[p][:5000]
    assert np.ptp(xs) * np.ptp(zs) < 0.3 * 160.0
    assert np.ptp(x[:5000]) * np.ptp(z[:5000]) > 0.9 * 160.0


def test_far_field_model_matches_direct_summation():
    """oracle/tree_model.py is the float64 model of csrc/tree.cu (same tree, lists, nested Chebyshev proxies and local
    fields): against direct summation it must show the orders' accuracy that DESIGN.md section 4b quotes."""
    from oracle import tree_model as tm
    rng = np.random.default_rng(5)
    n = 6000
    g, x, z = rng.standard_normal(n) * 1e-2, rng.uniform(-20, 0, n), rng.uniform(-4, 4, n)
    vc4 = 0.065 ** 4
    sel = rng.choice(n, 200, replace=False)
    ud, wd = tm.direct(x[sel], z[sel], x, z, g / (2 * np.pi), vc4)
    den = np.array([np.sum(np.abs(g) * np.hypot(x[i] - x, z[i] - z) / np.sqrt(((x[i] - x) ** 2 + (z[i] - z) ** 2) ** 2 + vc4))
                    for i in sel]) / (2 * np.pi)
    for order, tol in ((8, 1e-6), (14, 1e-10)):
        u, w, st = tm.tree_velocity(g, x, z, x[sel], z[sel], vc4, order=order, leaf=16, L=5)
        assert sum(st["proxy_cells"].values()) > 0
        assert np.max(np.hypot(u - ud, w - wd) / den) <= tol
