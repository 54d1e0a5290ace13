"""GPU parity tests of the code bench.py actually times (BASELINE.json configs[2] and [4]): the N = 2^20 self-convection
step through `ludvm_selfconv_step` / `ludvm_selfconv_step_p2p` (LUDVM.py:549-570 inside LUDVM.py:1095-1127), the
16-chunk launches, the fused single-launch kernel, the packed fp32x2 kernel and a flow-field grid large enough for the
4-rows-per-thread instantiations.  Every test asserts WHICH kernel instantiation ran (`ludvm_ctx_last_plan`), so the
parity statement is about the code the benchmark measures."""
import numpy as np
import pytest

from conftest import biteq

pytestmark = pytest.mark.gpu

SEED, VCORE, DT, N = 20260101, 0.065, 0.05, 1 << 20


def cond_bound_rows(g, xw, zw, xp, zp, vc, chunk=16):
    """sum_j |Gamma_j K_ij| for both components (SURVEY.md 8d-3), evaluated in row chunks (the full matrix is TBs)."""
    bu, bw = np.empty(len(xp)), np.empty(len(xp))
    ag = np.abs(g)[None, :]
    for i in range(0, len(xp), chunk):
        dx, dz = xp[i:i + chunk, None] - xw[None, :], zp[i:i + chunk, None] - zw[None, :]
        k = ag / (2 * np.pi * np.sqrt((dx * dx + dz * dz) ** 2 + vc ** 4))
        bu[i:i + chunk], bw[i:i + chunk] = (k * np.abs(dz)).sum(1), (k * np.abs(dx)).sum(1)
    return bu, bw


@pytest.fixture(scope="module")
def cloud():
    """bench.py's cloud (make_cloud) on the device, one context on torch's current stream."""
    import torch
    from ludvm_b200 import _lib
    rng = np.random.default_rng(SEED)
    x, z = rng.uniform(-20, 0, N), rng.uniform(-4, 4, N)
    g = rng.standard_normal(N) * 1e-2
    dev = torch.device("cuda", 0)
    ctx = _lib.Context(0, torch.cuda.current_stream().cuda_stream)
    t = {k: torch.tensor(v, device=dev) for k, v in dict(g=g, x=x, z=z).items()}
    return dict(g=g, x=x, z=z, t=t, ctx=ctx, torch=torch, dev=dev)


def _step(c, mode, row0=0, nrows=None, n=None, want_uw=True):
    """One ludvm_selfconv_step on the first n vortices of the cloud; returns (u, w, x_out, z_out) of the shard's rows."""
    from ludvm_b200 import ops
    torch, t = c["torch"], c["t"]
    n = N if n is None else n
    nrows = n - row0 if nrows is None else nrows
    g, x, z = t["g"][:n], t["x"][:n], t["z"][:n]
    xo, zo = torch.full_like(x, float("nan")), torch.full_like(z, float("nan"))
    u = torch.empty(nrows, dtype=torch.float64, device=c["dev"]) if want_uw else None
    w = torch.empty(nrows, dtype=torch.float64, device=c["dev"]) if want_uw else None
    ops.selfconv_step(c["ctx"], mode, g, x, z, VCORE ** 4, DT, xo, zo, row0=row0, nrows=nrows, u_out=u, w_out=w)
    torch.cuda.synchronize()
    plan = c["ctx"].last_plan()
    sl = slice(row0, row0 + nrows)
    assert torch.isnan(xo[:row0]).all() and torch.isnan(xo[row0 + nrows:]).all()     # only the shard's rows are written
    return (u.cpu().numpy() if want_uw else None, w.cpu().numpy() if want_uw else None,
            xo[sl].cpu().numpy(), zo[sl].cpu().numpy(), plan)


def test_selfconv_step_2p20_fast_vs_oracle(cloud, oracle, monkeypatch):
    """The headline launch: N = 2^20, fast mode.  4096 sampled rows (seed 7) against the oracle, u AND w, with the
    condition-aware bound of SURVEY.md 8(d)-3; the Euler-updated x, z of every row; the fused single-launch kernel
    against the 16-chunk partial-sum kernels (k_fast_tiled_tma<4> + k_combine) bit for bit; a 1/8 row shard (the
    per-rank launch of the 8-GPU run) and the p2p entry point against the full launch bit for bit."""
    g, x, z = cloud["g"], cloud["x"], cloud["z"]
    u, w, xo, zo, plan = _step(cloud, "fast")
    assert plan == dict(kernel="fast_fused", rows_per_thread=4, fold=16, tma=True, cluster=2, variant=4, warps=8, range_bad=0, pair_slots=13), plan
    rows = np.sort(np.random.default_rng(7).choice(N, 4096, replace=False))
    uo, wo = oracle.induced_velocity(g, x, z, x[rows], z[rows], VCORE)
    assert np.max(np.abs(u[rows] - uo)) <= 1e-12 * np.max(np.abs(uo))
    assert np.max(np.abs(w[rows] - wo)) <= 1e-12 * np.max(np.abs(wo))
    sub = rows[:256]
    bu, bw = cond_bound_rows(g, x, z, x[sub], z[sub], VCORE)
    assert np.all(np.abs(u[sub] - uo[:256]) <= 1e-12 * bu) and np.all(np.abs(w[sub] - wo[:256]) <= 1e-12 * bw)
    assert biteq(xo, x + DT * u) and biteq(zo, z + DT * w)                          # LUDVM.py:1108-1109
    # the partial-sum path bench.py timed in round 1
    monkeypatch.setenv("LUDVM_NO_FUSED", "1")
    u2, w2, xo2, zo2, plan2 = _step(cloud, "fast")
    assert plan2 == dict(kernel="fast_tiled_tma", rows_per_thread=4, fold=16, tma=True, cluster=1, variant=0, warps=0, range_bad=0, pair_slots=13), plan2
    assert biteq(u2, u) and biteq(w2, w) and biteq(xo2, xo) and biteq(zo2, zo)
    us, ws, xs, zs, plans = _step(cloud, "fast", row0=3 * (N // 8), nrows=N // 8)
    assert plans["kernel"] == "fast_tiled_tma" and plans["rows_per_thread"] == 4 and plans["fold"] == 16
    monkeypatch.delenv("LUDVM_NO_FUSED")
    # one rank of eight: same sums for its rows whatever the sharding
    uf, wf, xf, zf, planf = _step(cloud, "fast", row0=3 * (N // 8), nrows=N // 8)
    assert planf["kernel"] == "fast_fused" and planf["rows_per_thread"] == 4 and planf["cluster"] == 2
    sl = slice(3 * (N // 8), 4 * (N // 8))
    for a, b in ((uf, u[sl]), (wf, w[sl]), (xf, xo[sl]), (zf, zo[sl]), (us, u[sl]), (xs, xo[sl]), (zs, zo[sl])):
        assert biteq(a, b)
    # fused all-gather entry point with this rank as its only peer, and without velocity outputs
    from ludvm_b200 import ops
    torch, t = cloud["torch"], cloud["t"]
    buf = torch.zeros(2 * N, dtype=torch.float64, device=cloud["dev"])
    ops.selfconv_step_p2p(cloud["ctx"], "fast", t["g"], t["x"], t["z"], VCORE ** 4, DT, [buf.data_ptr()],
                          [buf.data_ptr() + 8 * N], sl.start, N // 8)
    torch.cuda.synchronize()
    assert cloud["ctx"].last_plan()["kernel"] == "fast_fused"
    assert biteq(buf[sl].cpu().numpy(), xo[sl]) and biteq(buf[N + sl.start:N + sl.stop].cpu().numpy(), zo[sl])
    assert float(buf[:sl.start].abs().sum()) == 0.0 and float(buf[sl.stop:N].abs().sum()) == 0.0


def test_fused_kernel_shapes_match_partial_sum_path(cloud, monkeypatch):
    """Every instantiation of the fused kernel (rows per thread 4/2/1 with source-loop unroll 4/4/8, cluster 1/2, ragged
    last stage) against the partial-sum kernels bit for bit."""
    for n, row0, nrows, want in [(N, 0, N // 16, dict(rows_per_thread=2, cluster=2)),
                                 (N, 12345, N // 32 + 77, dict(rows_per_thread=1, cluster=2)),
                                 (1 << 17, 0, 1 << 17, dict(rows_per_thread=4, cluster=2)),
                                 (100000, 0, 100000, dict(rows_per_thread=1, cluster=1)),
                                 (130001, 0, 130001, dict(rows_per_thread=2, cluster=1)),
                                 (200001, 1000, 150000, dict(rows_per_thread=4, cluster=2)),
                                 (60001, 0, 59993, dict(rows_per_thread=1, cluster=1))]:
        u, w, xo, zo, plan = _step(cloud, "fast", row0=row0, nrows=nrows, n=n)
        assert plan["kernel"] == "fast_fused" and all(plan[k] == v for k, v in want.items()), (n, nrows, plan)
        assert plan["variant"] == (8 if plan["rows_per_thread"] == 1 else 4) and plan["warps"] == 8, plan
        monkeypatch.setenv("LUDVM_NO_FUSED", "1")
        u2, w2, xo2, zo2, plan2 = _step(cloud, "fast", row0=row0, nrows=nrows, n=n)
        monkeypatch.delenv("LUDVM_NO_FUSED")
        assert plan2["kernel"] == "fast_tiled_tma" and plan2["fold"] == plan["fold"]
        assert biteq(u2, u) and biteq(w2, w) and biteq(xo2, xo) and biteq(zo2, zo), (n, nrows)


def test_selfconv_step_2p17_exact_all_rows_bit_equal(cloud, oracle):
    """Exact mode at N = 2^17: every row of u, w and of the Euler update bit-equal to the oracle (numpy's summation
    tree over 131072 sources, cut across thread blocks)."""
    n = 1 << 17
    g, x, z = cloud["g"][:n], cloud["x"][:n], cloud["z"][:n]
    u, w, xo, zo, plan = _step(cloud, "exact", n=n)
    assert plan["kernel"] == "exact_tiled" and plan["variant"] == 1 and plan["range_bad"] == 0, plan   # flag-free
    uo, wo = oracle.induced_velocity(g, x, z, x, z, VCORE)
    assert biteq(u, uo) and biteq(w, wo)
    assert biteq(xo, x + DT * uo) and biteq(zo, z + DT * wo)


def test_selfconv_step_2p20_exact_sampled_rows(cloud, oracle):
    """Exact mode at the bench size through a row shard made of sampled-row neighbourhoods: 8 blocks of 512
    consecutive rows against all 2^20 sources, bit-equal to the oracle."""
    g, x, z = cloud["g"], cloud["x"], cloud["z"]
    for row0 in (0, 517 * 1024 + 3, N - 4096):
        u, w, xo, zo, plan = _step(cloud, "exact", row0=row0, nrows=4096)
        assert plan["kernel"] == "exact_tiled", plan
        uo, wo = oracle.induced_velocity(g, x, z, x[row0:row0 + 4096], z[row0:row0 + 4096], VCORE)
        assert biteq(u, uo) and biteq(w, wo), row0


def test_fp32x2_kernel_at_bench_size(cloud, oracle):
    """fp32-fast at N = 2^20 runs the packed fp32x2 kernel (8 rows per thread); reported accuracy vs fp64."""
    g, x, z = cloud["g"], cloud["x"], cloud["z"]
    u, w, xo, zo, plan = _step(cloud, "fp32")
    assert plan["kernel"] == "fast32x2_tiled" and plan["rows_per_thread"] == 8 and plan["fold"] == 16, plan
    rows = np.sort(np.random.default_rng(8).choice(N, 1024, replace=False))
    uo, wo = oracle.induced_velocity(g, x, z, x[rows], z[rows], VCORE)
    err = max(np.max(np.abs(u[rows] - uo)) / np.max(np.abs(uo)), np.max(np.abs(w[rows] - wo)) / np.max(np.abs(wo)))
    assert err < 5e-4, err
    assert biteq(xo, x + DT * u)


def test_flowfield_quarter_million_points(cloud, oracle, monkeypatch):
    """A 512 x 512 grid against 2^17 sources (configs[4] scaled down): >= 2.3e5 points, so the 4-rows-per-thread
    16-chunk launches run.  Sampled points against the oracle in fast and exact mode, x-row slabs (the multi-GPU
    decomposition) against the whole grid bit for bit, fused against partial-sum path bit for bit."""
    from ludvm_b200 import ops
    n = 1 << 17
    g, xw, zw = cloud["g"][:n], cloud["x"][:n], cloud["z"][:n]
    x1, z1 = np.arange(-10.24, 0, 0.02), np.arange(-5.12, 5.12, 0.02)
    assert len(x1) == 512 and len(z1) == 512
    vc4, ctx = VCORE ** 4, cloud["ctx"]
    u, w = ops.flowfield_velocity(g, xw, zw, None, None, None, vc4, x1, z1, mode="fast", ctx=ctx)
    plan = ctx.last_plan()
    assert plan == dict(kernel="fast_fused", rows_per_thread=4, fold=16, tma=True, cluster=2, variant=4, warps=8, range_bad=0, pair_slots=13), plan
    pts = np.sort(np.random.default_rng(3).choice(512 * 512, 2048, replace=False))
    X, Z = np.meshgrid(x1, z1, indexing="ij")
    uo, wo = oracle.induced_velocity(g, xw, zw, X.ravel()[pts], Z.ravel()[pts], VCORE)
    bu, bw = cond_bound_rows(g, xw, zw, X.ravel()[pts[:256]], Z.ravel()[pts[:256]], VCORE)
    assert np.all(np.abs(u.ravel()[pts[:256]] - uo[:256]) <= 1e-12 * bu)
    assert np.all(np.abs(w.ravel()[pts[:256]] - wo[:256]) <= 1e-12 * bw)
    assert np.max(np.abs(u.ravel()[pts] - uo)) <= 1e-12 * np.max(np.abs(uo))
    assert np.max(np.abs(w.ravel()[pts] - wo)) <= 1e-12 * np.max(np.abs(wo))
    parts = [ops.flowfield_velocity(g, xw, zw, None, None, None, vc4, x1, z1, row0=r0, nrows=nr, mode="fast", ctx=ctx)
             for r0, nr in ((0, 200), (200, 57), (257, 255))]
    assert biteq(np.concatenate([p[0] for p in parts]), u) and biteq(np.concatenate([p[1] for p in parts]), w)
    monkeypatch.setenv("LUDVM_NO_FUSED", "1")
    u2, w2 = ops.flowfield_velocity(g, xw, zw, None, None, None, vc4, x1, z1, mode="fast", ctx=ctx)
    monkeypatch.delenv("LUDVM_NO_FUSED")
    plan2 = ctx.last_plan()
    assert plan2 == dict(kernel="fast_tiled_tma", rows_per_thread=4, fold=16, tma=True, cluster=1, variant=0, warps=0, range_bad=0, pair_slots=13), plan2
    assert biteq(u2, u) and biteq(w2, w)
    # with a second (bound-vortex) source set the partial-sum path serves both sets; compare with the sum of two calls
    gb, xb, zb = np.linspace(0.01, 0.02, 80), np.linspace(-1.0, 0.0, 80), np.zeros(80)
    u3, w3 = ops.flowfield_velocity(g, xw, zw, gb, xb, zb, vc4, x1, z1, mode="fast", ctx=ctx)
    ub, wb = ops.flowfield_velocity(gb, xb, zb, None, None, None, vc4, x1, z1, mode="fast", ctx=ctx)
    assert biteq(u3, u + ub) and biteq(w3, w + wb)
    # exact mode on the same grid: sampled points bit-equal to the oracle
    ue, we = ops.flowfield_velocity(g, xw, zw, None, None, None, vc4, x1, z1, mode="exact", ctx=ctx)
    assert ctx.last_plan()["kernel"] == "exact_tiled"
    assert biteq(ue.ravel()[pts], uo) and biteq(we.ravel()[pts], wo)


def test_repeated_launches_are_bitwise_stable(cloud, monkeypatch):
    """Stress stand-in for racecheck (compute-sanitizer is closed on this pool): the double-buffered bulk-copy
    pipelines and the cluster fold must give the same bits on every launch, for several chunkings."""
    n, nrows = 1 << 18, 1 << 16
    for chunks in (None, "8", "16"):
        if chunks:
            monkeypatch.setenv("LUDVM_FAST_CHUNKS", chunks)
        ref = _step(cloud, "fast", n=n, nrows=nrows)
        for _ in range(20):
            got = _step(cloud, "fast", n=n, nrows=nrows)
            assert all(biteq(a, b) for a, b in zip(got[:4], ref[:4]))
        monkeypatch.setenv("LUDVM_NO_FUSED", "1")
        for _ in range(10):
            got = _step(cloud, "fast", n=n, nrows=nrows)
            assert all(biteq(a, b) for a, b in zip(got[:4], ref[:4]))
        monkeypatch.delenv("LUDVM_NO_FUSED")
        if chunks:
            monkeypatch.delenv("LUDVM_FAST_CHUNKS")


def test_fast12_opt_in_mode_within_tolerance(cloud, oracle):
    """LUDVM_FAST12_F64 (opt-in): the 12-slot pair -- one second-order refinement of the centred MUFU seed.  Per-call
    results must stay inside BASELINE.json's 1e-12 (relative to sum |terms|); the measured error is reported."""
    g, x, z = cloud["g"], cloud["x"], cloud["z"]
    u, w, xo, zo, plan = _step(cloud, "fast12", row0=N // 2, nrows=N // 8)
    assert plan["kernel"] == "fast_fused" and plan["pair_slots"] == 12 and plan["rows_per_thread"] == 4, plan
    rows = np.sort(np.random.default_rng(5).choice(N // 8, 1024, replace=False))
    uo, wo = oracle.induced_velocity(g, x, z, x[N // 2 + rows], z[N // 2 + rows], VCORE)
    bu, bw = cond_bound_rows(g, x, z, x[N // 2 + rows[:256]], z[N // 2 + rows[:256]], VCORE)
    eu, ew = np.abs(u[rows[:256]] - uo[:256]) / bu, np.abs(w[rows[:256]] - wo[:256]) / bw
    assert eu.max() <= 5e-13 and ew.max() <= 5e-13, (eu.max(), ew.max())
    assert np.max(np.abs(u[rows] - uo)) <= 1e-12 * np.max(np.abs(uo))
    assert biteq(xo, x[N // 2:N // 2 + N // 8] + DT * u)
    u13 = _step(cloud, "fast", row0=N // 2, nrows=N // 8)[0]
    assert not biteq(u13, u) and np.max(np.abs(u13 - u)) <= 1e-12 * np.max(np.abs(u13))
    # a launch the fused kernel does not take falls back to the 13-slot kernels
    u_s, _, _, _, plan_s = _step(cloud, "fast12", n=20000)
    assert plan_s["kernel"] == "fast_tiled_tma" and plan_s["pair_slots"] == 13
    assert biteq(u_s, _step(cloud, "fast", n=20000)[0])
