"""GPU tests of the whole-cloud self-convection step `ludvm_selfconv_step_all`: in fast mode with one core radius it
runs k_fast_sym (each unordered pair evaluated once, the shared part of the term applied to both vortices) + k_combine,
and must give exactly the bits of `ludvm_selfconv_step(row0=0, nrows=n)` -- velocities and Euler update alike.  Every
test asserts which kernel ran (`ludvm_ctx_last_plan`)."""
import numpy as np
import pytest

from conftest import biteq

pytestmark = pytest.mark.gpu

SEED, VCORE, DT, N = 20260101, 0.065, 0.05, 1 << 20


@pytest.fixture(scope="module")
def env():
    """bench.py's cloud (make_cloud) on the device, one context on torch's current stream."""
    import torch
    from ludvm_b200 import _lib
    rng = np.random.default_rng(SEED)
    x, z = rng.uniform(-20, 0, N), rng.uniform(-4, 4, N)
    g = rng.standard_normal(N) * 1e-2
    dev = torch.device("cuda", 0)
    ctx = _lib.Context(0, torch.cuda.current_stream().cuda_stream)
    return dict(g=g, x=x, z=z, ctx=ctx, torch=torch, dev=dev)


def _run(env, entry, g, x, z, vc4=VCORE ** 4, mode="fast", vc4_per_source=None):
    """One step of the whole cloud through `entry` ("all" or "rows"); returns (u, w, x_out, z_out, plan) on the host."""
    from ludvm_b200 import ops
    torch = env["torch"]
    t = [torch.as_tensor(a, device=env["dev"]) for a in (g, x, z)]
    vcs = None if vc4_per_source is None else torch.as_tensor(vc4_per_source, device=env["dev"])
    xo, zo = torch.full_like(t[1], float("nan")), torch.full_like(t[2], float("nan"))
    u, w = torch.full_like(t[1], float("nan")), torch.full_like(t[2], float("nan"))
    if entry == "all":
        ops.selfconv_step_all(env["ctx"], mode, *t, vc4, DT, xo, zo, u_out=u, w_out=w, vc4_per_source=vcs)
    else:
        ops.selfconv_step(env["ctx"], mode, *t, vc4, DT, xo, zo, u_out=u, w_out=w, vc4_per_source=vcs)
    env["ctx"].synchronize()
    plan = env["ctx"].last_plan()
    return u.cpu().numpy(), w.cpu().numpy(), xo.cpu().numpy(), zo.cpu().numpy(), plan


def _same_as_rows(env, g, x, z, want, **kw):
    a = _run(env, "all", g, x, z, **kw)
    b = _run(env, "rows", g, x, z, **kw)
    assert a[4]["kernel"] == want, a[4]
    for k, (p, q) in enumerate(zip(a[:4], b[:4])):
        assert biteq(p, q), ("u", "w", "x_out", "z_out")[k]
    return a


def test_bench_cloud_2p20(env):
    """The headline step: N = 2^20, bench.py's cloud."""
    u, w, xo, zo, plan = _same_as_rows(env, env["g"], env["x"], env["z"], "fast_sym")
    assert plan["fold"] == 16 and plan["rows_per_thread"] == 4 and plan["pair_slots"] == 8, plan
    assert np.isfinite(u).all() and np.isfinite(w).all()


@pytest.mark.parametrize("n", [1 << 17, 200001])
def test_sizes_full_and_ragged(env, n):
    """2^17 (the smallest eligible cloud) and a ragged n, where the last chunk and its last row block are partial."""
    _same_as_rows(env, env["g"][:n], env["x"][:n], env["z"][:n], "fast_sym")


def test_duplicated_coordinates(env):
    """Distinct vortices that share x, share z, or sit on the same point: dx or dz is +0 in both directions, the case in
    which the transposed term's sign of zero differs from the direct one."""
    n = 150001
    rng = np.random.default_rng(11)
    g, x, z = env["g"][:n].copy(), env["x"][:n].copy(), env["z"][:n].copy()
    a, b = rng.choice(n, 4000, replace=False), rng.choice(n, 4000, replace=False)
    x[a[:2000]] = x[b[:2000]]
    z[a[2000:]] = z[b[2000:]]
    c, d = rng.choice(n, 500, replace=False), rng.choice(n, 500, replace=False)
    x[c], z[c] = x[d], z[d]
    x[:64], z[100:164] = -3.0, 0.0          # whole row blocks on one line, adjacent blocks sharing them
    _same_as_rows(env, g, x, z, "fast_sym")


def test_ten_steps_through_sharded_selfconvection(env):
    """bench.py's timed loop on one GPU: 10 ShardedSelfConvection steps against 10 ludvm_selfconv_step steps."""
    from ludvm_b200 import ops
    from ludvm_b200.sharded import ShardedSelfConvection
    torch, n = env["torch"], 200001
    g, x, z = (torch.tensor(a[:n], device=env["dev"]) for a in (env["g"], env["x"], env["z"]))
    sc = ShardedSelfConvection(g, x.clone(), z.clone(), VCORE, DT, mode="fast", ctx=env["ctx"])
    for _ in range(10):
        xs, zs = sc.step()
    torch.cuda.synchronize()
    assert env["ctx"].last_plan()["kernel"] == "fast_sym"
    xa, za = x.clone(), z.clone()
    xb, zb = torch.empty_like(xa), torch.empty_like(za)
    for _ in range(10):
        ops.selfconv_step(env["ctx"], "fast", g, xa, za, VCORE ** 4, DT, xb, zb)
        xa, xb, za, zb = xb, xa, zb, za
    torch.cuda.synchronize()
    assert env["ctx"].last_plan()["kernel"] == "fast_fused"
    assert biteq(xs.cpu().numpy(), xa.cpu().numpy()) and biteq(zs.cpu().numpy(), za.cpu().numpy())


def test_repeated_launches_are_bitwise_stable(env):
    """The ticket order, progress counters and chain hand-offs must give the same bits on every launch."""
    n = (1 << 18) + 12345
    g, x, z = env["g"][:n], env["x"][:n], env["z"][:n]
    ref = _run(env, "all", g, x, z)
    assert ref[4]["kernel"] == "fast_sym"
    for _ in range(20):
        got = _run(env, "all", g, x, z)
        assert all(biteq(p, q) for p, q in zip(got[:4], ref[:4]))


def test_fallbacks_select_the_row_kernels(env):
    """Per-source cores, vc^4 = 0, a cloud below 2^17, the 12-slot and exact modes: the whole-cloud entry point runs
    exactly what ludvm_selfconv_step runs."""
    n = 1 << 17
    g, x, z = env["g"][:n], env["x"][:n], env["z"][:n]
    vcs = np.full(n, VCORE ** 4)
    vcs[::7] *= 2.0
    _same_as_rows(env, g, x, z, "fast_tiled", vc4_per_source=vcs)
    _same_as_rows(env, g, x, z, "fast_fused", vc4=0.0)
    _same_as_rows(env, g[:n - 1], x[:n - 1], z[:n - 1], "fast_fused")
    _same_as_rows(env, g, x, z, "fast_fused", mode="fast12")
    _same_as_rows(env, g[:20000], x[:20000], z[:20000], "exact_tiled", mode="exact")
