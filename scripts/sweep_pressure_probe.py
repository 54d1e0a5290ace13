"""Cost of the chordwise pressure jump in the batched sweep (BASELINE.json configs[3]: 4096 README-size cases over
LESPcrit x k, as bench.py's sweep): sweep.run_sweep with pressure off and on alternating in one process, exact and fast.

Two sources, one JSON line per measurement and one summary line per (source, mode), best of REPS after a warm-up round:
  "call"   -- timing["ludvm_sweep_run_s"] of run_sweep: the whole C call, including the dp download (~1.05 GB with
              pressure on); "run_sweep_s" adds the host tables and the Cp division.
  "kernel" -- the kernel line of the LUDVM_SWEEP_TIMING breakdown, taken in a child process (the breakdown synchronises
              between the phases of the call), with the resident cases per SM of the launched instantiation.
Usage: python scripts/sweep_pressure_probe.py [--out FILE]   (default profiles/sweep_pressure_probe.txt)"""
import argparse, json, os, re, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np

README = dict(t0=0, tf=20, dt=5e-2, chord=1, rho=1.225, Uinf=1, Npoints=81, Ncoeffs=30, LESPcrit=0.2, Naca="0012")
REPS = int(os.environ.get("PROBE_REPS", "5"))
MODES = ("exact", "fast")
LINE = re.compile(r"ludvm_sweep_run: upload\+alloc\+init ([\d.]+) ms, kernel ([\d.]+) ms, gather\+D2H ([\d.]+) ms, "
                  r"free ([\d.]+) ms \(arena \d+ MB, dp (\d+) MB, (\d+) cases resident per SM\)")


def cases(pressure):
    from ludvm_b200 import sweep
    grid = sweep.lespcrit_k_grid(np.linspace(0.1, 0.4, 64), np.linspace(0.1, 1.0, 64), **README)   # bench.sweep_cases()
    return [dict(kw, pressure=True) for kw in grid] if pressure else grid


def rounds():
    """(mode, rep, pressure) in run order; rep 0 warms up modules, pools and host tables."""
    return [(mode, rep, p) for mode in MODES for rep in range(REPS + 1) for p in (False, True)]


def child():
    """Runs the calls of rounds() with LUDVM_SWEEP_TIMING set, then a small Ramesh sweep off and on (for the resident
    cases per SM of the Ramesh instantiations); the parent pairs the stderr lines with the order printed here."""
    from ludvm_b200 import sweep
    cs = {p: cases(p) for p in (False, True)}
    for mode, rep, p in rounds():
        sweep.run_sweep(cs[p], mode=mode)
        print(json.dumps([mode, rep, p]), flush=True)
    for p in (False, True):
        sweep.run_sweep([dict(kw, tf=1, method="Ramesh") for kw in cs[p][:4]], mode="exact")
        print(json.dumps(["ramesh", 0, p]), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "sweep_pressure_probe.txt"))
    ap.add_argument("--child", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.child:
        return child()
    from ludvm_b200 import sweep
    out = open(args.out, "w")

    def emit(d):
        line = json.dumps(d)
        print(line, flush=True)
        out.write(line + "\n")
        out.flush()

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    emit({"gpu": gpu[0] if gpu else "unknown", "cases": 64 * 64, "steps": 400, "reps": REPS})
    cs = {p: cases(p) for p in (False, True)}
    call, wall = {}, {}
    for mode, rep, p in rounds():
        t = time.perf_counter()
        res = sweep.run_sweep(cs[p], mode=mode)
        w = time.perf_counter() - t
        s = res["timing"]["ludvm_sweep_run_s"]
        del res
        emit({"source": "call", "mode": mode, "pressure": p, "rep": rep, "ludvm_sweep_run_s": s, "run_sweep_s": w})
        if rep:
            call.setdefault((mode, p), []).append(s)
            wall.setdefault((mode, p), []).append(w)
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child"], capture_output=True, text=True,
                       env=dict(os.environ, LUDVM_SWEEP_TIMING="1"))
    if r.returncode:
        sys.stderr.write(r.stdout + r.stderr)
        raise SystemExit("child failed")
    order = [tuple(json.loads(x)) for x in r.stdout.splitlines() if x.startswith("[")]
    lines = [LINE.search(x) for x in r.stderr.splitlines() if x.startswith("ludvm_sweep_run:")]
    assert len(order) == len(lines) == len(rounds()) + 2 and all(lines), (len(order), len(lines))
    kern, per_sm = {}, {}
    for (mode, rep, p), m in zip(order, lines):
        k_ms, d_ms, dp_mb, occ = float(m.group(2)), float(m.group(3)), int(m.group(5)), int(m.group(6))
        emit({"source": "kernel", "mode": mode, "pressure": p, "rep": rep, "kernel_ms": k_ms, "gather_d2h_ms": d_ms,
              "dp_MB": dp_mb, "cases_per_sm": occ})
        per_sm[(mode, p)] = occ
        if rep:
            kern.setdefault((mode, p), []).append((k_ms, d_ms))
    for mode in MODES:
        off, on = call[(mode, False)], call[(mode, True)]
        emit({"summary": "call", "mode": mode, "off_best_s": min(off), "on_best_s": min(on),
              "off_spread_s": max(off) - min(off), "on_spread_s": max(on) - min(on), "on_over_off": min(on) / min(off),
              "off_case_steps_per_s": 4096 * 400 / min(off), "on_case_steps_per_s": 4096 * 400 / min(on),
              "run_sweep_off_best_s": min(wall[(mode, False)]), "run_sweep_on_best_s": min(wall[(mode, True)])})
        koff, kon = [k for k, _ in kern[(mode, False)]], [k for k, _ in kern[(mode, True)]]
        doff, don = [d for _, d in kern[(mode, False)]], [d for _, d in kern[(mode, True)]]
        emit({"summary": "kernel", "mode": mode, "off_best_ms": min(koff), "on_best_ms": min(kon),
              "off_spread_ms": max(koff) - min(koff), "on_spread_ms": max(kon) - min(kon), "on_over_off": min(kon) / min(koff),
              "gather_d2h_off_best_ms": min(doff), "gather_d2h_on_best_ms": min(don),
              "cases_per_sm_off": per_sm[(mode, False)], "cases_per_sm_on": per_sm[(mode, True)]})
    emit({"summary": "cases_per_sm", "exact_128_faure": [per_sm[("exact", p)] for p in (False, True)],
          "fast_256_faure": [per_sm[("fast", p)] for p in (False, True)],
          "ramesh_256": [per_sm[("ramesh", p)] for p in (False, True)], "order": "[pressure off, on]"})
    out.close()


if __name__ == "__main__":
    main()
