"""method='Ramesh' on the single-simulation drivers against the library it replaces (LUDVM_B200_LIB of the parent build, where
every Ramesh run was one CTA) and against Faure on this build.

Cases (README kinematics unless stated):
  readme_exact / readme_fast   400 steps, us per step;
  gust_2^12 .. gust_2^16       fast, 22 steps, seeded uniform gust of free vortices (the far-field probe's distribution);
  dt2e-3                       fast, the first 5 000 steps of the dt = 2e-3, tf = 40 run.
Both methods run on both libraries, each library in a worker process of its own; the parent alternates the four
(library, method) pairs, one warm-up round then best of REPS.  Time = host clock around ludvm_sim_run of all steps, ending
in a device synchronise (store_history=False, set-up and fetch excluded).

Usage: python scripts/ramesh_probe.py PARENT_LIB, where PARENT_LIB is libludvm_b200.so built from the parent commit, e.g.
  git worktree add /tmp/parent HEAD~1 && (cd /tmp/parent && python -m ludvm_b200.build)
  python scripts/ramesh_probe.py /tmp/parent/ludvm_b200/libludvm_b200.so"""
import json, os, subprocess, sys, time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REPS = int(os.environ.get("PROBE_REPS", "5"))
README = dict(t0=0, tf=20, dt=5e-2, chord=1, rho=1.225, Uinf=1, Npoints=81, Ncoeffs=30, LESPcrit=0.2, Naca="0012")


def cases():
    c = [("readme_exact", dict(README), "exact", None), ("readme_fast", dict(README), "fast", None)]
    c += [("gust_2^%d" % lg, dict(README, tf=1.1), "fast", 1 << lg) for lg in range(12, 17)]
    c += [("dt2e-3", dict(README, dt=2e-3, tf=40), "fast", None)]
    return c


def worker():
    sys.path.insert(0, ROOT)
    import numpy as np
    from ludvm_b200 import LUDVM, _lib
    L = _lib.load()
    for line in sys.stdin:
        name, method = json.loads(line)
        kw, mode, nf = {c[0]: c[1:] for c in cases()}[name]
        kw = dict(kw, method=method)
        if nf:
            rng = np.random.default_rng(1)
            kw.update(xy_freevort=np.stack([rng.uniform(-6.0, -0.5, nf), rng.uniform(-1.0, 1.0, nf)]),
                      circulation_freevort=rng.standard_normal(nf) * 1e-3)
        s = LUDVM(**kw, verbose=False, run=False, mode=mode, store_history=False)
        s.time_loop(nsteps=0)
        s.ctx.synchronize()
        n = min(s.nt - 1, 5000)
        t = time.perf_counter()
        _lib.check(L.ludvm_sim_run(s._sim, n))
        s.ctx.synchronize()
        sec = time.perf_counter() - t
        print(json.dumps({"s": sec, "steps": n}), flush=True)
        s.close()


def main():
    if len(sys.argv) < 2 or not os.path.isfile(sys.argv[1]):
        sys.exit(__doc__)
    parent = sys.argv[1]
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    print(json.dumps({"gpu": gpu[0] if gpu else "unknown", "reps": REPS}), flush=True)
    libs = {"parent": parent, "this": os.path.join(ROOT, "ludvm_b200", "libludvm_b200.so")}
    procs = {}
    for k, lib in libs.items():
        env = dict(os.environ, LUDVM_B200_LIB=lib)
        procs[k] = subprocess.Popen([sys.executable, __file__, "--worker"], stdin=subprocess.PIPE, stdout=subprocess.PIPE,
                                    text=True, env=env)
    runs = [("parent", "Ramesh"), ("this", "Ramesh"), ("parent", "Faure"), ("this", "Faure")]
    try:
        for name, _, _, _ in cases():
            best = {}
            for rep in range(REPS + 1):
                for lib, method in runs:
                    p = procs[lib]
                    p.stdin.write(json.dumps([name, method]) + "\n")
                    p.stdin.flush()
                    r = json.loads(p.stdout.readline())
                    us = r["s"] / r["steps"] * 1e6
                    print(json.dumps({"case": name, "lib": lib, "method": method, "rep": rep, "us_per_step": us}), flush=True)
                    if rep:
                        best[lib + "_" + method] = min(best.get(lib + "_" + method, us), us)
            print(json.dumps({"summary": name, "steps": r["steps"], "best_us_per_step": best,
                              "ramesh_speedup": best["parent_Ramesh"] / best["this_Ramesh"],
                              "faure_this_over_parent": best["this_Faure"] / best["parent_Faure"]}), flush=True)
    finally:
        for p in procs.values():
            p.stdin.close()
            p.wait()


if __name__ == "__main__":
    worker() if "--worker" in sys.argv else main()
