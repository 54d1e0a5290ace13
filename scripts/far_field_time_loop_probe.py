"""All-pairs vs far-field convection in the device time loop (LUDVM(..., far_field_order=18)), fast mode.

A seeded uniform random gust ahead of the aerofoil (x in [-6, -0.5], z in [-1, 1], Gamma ~ N(0, 1) * 1e-3, the tests'
distribution) of nfree = 2^14 .. 2^20 vortices, README kinematics, tf = 1.1 (22 steps).  For each size, in one process:
  * device seconds per step, far field off and on alternating, best of REPS after a warm-up round (host clock around
    ludvm_sim_run of every step, ending in a device synchronise; store_history=False);
  * the far field's standalone treecode time on the same cloud (ops.selfconv_step_tree, targets = sources), so that
    what the far-field step spends beyond the tree (branch A, the join, launches and the per-step synchronisations) can
    be stated as a share of the step;
  * accuracy over the whole run (store_history=True): the largest relative difference of L and M (over max|.|) and the
    largest displacement difference of path['FREE'] between the two runs.
`far_field_steps` is what far_field_info reports: sizes below the library's SIM_FAR_FIELD_MIN_WAKE take no far-field
steps, so there "on" and "off" run the same kernels.  One JSON line per measurement, then one summary line per size."""
import ctypes, json, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from ludvm_b200 import LUDVM, _lib, ops
L = _lib.load()
README = dict(t0=0, tf=1.1, dt=5e-2, chord=1, rho=1.225, Uinf=1, Npoints=81, Ncoeffs=30, LESPcrit=0.2, Naca="0012")
REPS = int(os.environ.get("PROBE_REPS", "5"))
SIZES = [int(v) for v in os.environ.get("PROBE_SIZES", "14,15,16,17,18,20").split(",")]
ORDER = 18


def gust(nf, seed=1):
    rng = np.random.default_rng(seed)
    xy = np.stack([rng.uniform(-6.0, -0.5, nf), rng.uniform(-1.0, 1.0, nf)])
    return rng.standard_normal(nf) * 1e-3, xy


def device_seconds(kw, ff):
    s = LUDVM(**kw, verbose=False, run=False, mode="fast", store_history=False, far_field_order=ff)
    s.time_loop(nsteps=0)
    s.ctx.synchronize()
    t = time.perf_counter()
    _lib.check(L.ludvm_sim_run(s._sim, s.nt - 1))
    s.ctx.synchronize()
    sec = time.perf_counter() - t
    info = (ctypes.c_int64 * 4)()
    _lib.check(L.ludvm_sim_far_field_info(s._sim, info))
    n = s.nt - 1
    s.close()
    return sec, n, int(info[0]), int(info[3])


def tree_seconds(g, xy, vc4, reps):
    import torch
    ctx = _lib.default_context(0)
    d = lambda a: torch.tensor(np.ascontiguousarray(a), dtype=torch.float64, device="cuda")
    tg, tx, tz = d(g), d(xy[0]), d(xy[1])
    xo, zo = torch.empty_like(tx), torch.empty_like(tz)
    best = None
    for rep in range(reps + 1):
        ctx.synchronize()
        t = time.perf_counter()
        ops.selfconv_step_tree(ctx, tg, tx, tz, vc4, 5e-2, xo, zo, order=ORDER)
        ctx.synchronize()
        sec = time.perf_counter() - t
        if rep:
            best = sec if best is None else min(best, sec)
    return best


gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
print(json.dumps({"gpu": gpu[0] if gpu else "unknown", "order": ORDER, "steps": 22}), flush=True)
for lg in SIZES:
    nf = 1 << lg
    g, xy = gust(nf)
    kw = dict(README, circulation_freevort=g, xy_freevort=xy)
    times = {False: [], True: []}
    for rep in range(REPS + 1):
        for ff in (False, True):
            sec, n, nff, leaf = device_seconds(kw, ORDER if ff else None)
            if rep:   # the first round warms up modules, graphs and scratch
                times[ff].append(sec)
            print(json.dumps({"nfree": nf, "far_field": ff, "rep": rep, "s": sec, "ms_per_step": sec / n * 1e3,
                              "far_field_steps": nff, "leaf_level": leaf}), flush=True)
    vc4 = float((1.3 * README["dt"]) ** 4)
    tree_s = tree_seconds(g, xy, vc4, REPS)
    a = LUDVM(**kw, verbose=False, mode="fast")
    b = LUDVM(**kw, verbose=False, mode="fast", far_field_order=ORDER)
    rel = lambda p, q: float(np.max(np.abs(p - q)) / np.max(np.abs(p)))
    disp = float(np.max(np.hypot(*(b.path["FREE"] - a.path["FREE"]).transpose(1, 0, 2))))
    off, on = min(times[False]), min(times[True])
    on_ms = on / n * 1e3
    print(json.dumps({"summary": nf, "steps": n, "far_field_steps": b.far_field_info["far_field_steps"],
                      "fallback_steps": b.far_field_info["fallback_steps"], "leaf_level": b.far_field_info["leaf_level"],
                      "off_ms_per_step": off / n * 1e3, "on_ms_per_step": on_ms,
                      "off_spread_ms": (max(times[False]) - off) / n * 1e3, "on_spread_ms": (max(times[True]) - on) / n * 1e3,
                      "speedup": off / on, "tree_alone_ms": tree_s * 1e3,
                      "rest_of_step_share": max(0.0, on_ms - tree_s * 1e3) / on_ms,
                      "L_rel_diff": rel(a.L, b.L), "M_rel_diff": rel(a.M, b.M), "FREE_max_disp_diff": disp}), flush=True)
    a.close()
    b.close()
