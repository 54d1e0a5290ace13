"""Cost of the chordwise pressure jump (LUDVM(..., pressure=True)): device time of the README time loop (us per step,
exact and fast) and of the dt = 2e-3, tf = 40 fast run (s), with pressure off and on alternating in one process.
One JSON line per measurement, then one summary line per configuration (best of the repetitions after the first)."""
import json, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ludvm_b200 import LUDVM, _lib
L = _lib.load()
README = dict(t0=0, tf=20, dt=5e-2, chord=1, rho=1.225, Uinf=1, Npoints=81, Ncoeffs=30, LESPcrit=0.2, Naca="0012")
LONG = dict(README, dt=2e-3, tf=40)
REPS = int(os.environ.get("PROBE_REPS", "5"))


def device_seconds(kw, mode, pressure):
    """Host clock around ludvm_sim_run of every step, ending in a device synchronise (set-up and fetch excluded)."""
    s = LUDVM(**kw, verbose=False, run=False, mode=mode, store_history=False, pressure=pressure)
    s.time_loop(nsteps=0)
    s.ctx.synchronize()
    t = time.perf_counter()
    _lib.check(L.ludvm_sim_run(s._sim, s.nt - 1))
    s.ctx.synchronize()
    dt = time.perf_counter() - t
    nsteps = s.nt - 1
    s.close()
    return dt, nsteps


gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
print(json.dumps({"gpu": gpu[0] if gpu else "unknown"}), flush=True)
runs = {}
for label, kw, mode, reps in [("readme_exact", README, "exact", REPS), ("readme_fast", README, "fast", REPS),
                              ("dt2e-3_tf40_fast", LONG, "fast", max(2, REPS // 2))]:
    for rep in range(reps + 1):
        for pressure in (False, True):
            sec, n = device_seconds(kw, mode, pressure)
            if rep:   # the first round warms up modules and graphs
                runs.setdefault((label, pressure), []).append(sec)
            print(json.dumps({"case": label, "pressure": pressure, "rep": rep, "s": sec, "us_per_step": sec / n * 1e6}),
                  flush=True)
        runs.setdefault((label, "steps"), n)
for label in ("readme_exact", "readme_fast", "dt2e-3_tf40_fast"):
    n = runs[(label, "steps")]
    off, on = runs[(label, False)], runs[(label, True)]
    print(json.dumps({"summary": label, "steps": n, "off_best_s": min(off), "on_best_s": min(on),
                      "off_us_per_step": min(off) / n * 1e6, "on_us_per_step": min(on) / n * 1e6,
                      "off_spread_s": max(off) - min(off), "on_spread_s": max(on) - min(on),
                      "on_over_off": min(on) / min(off)}), flush=True)
