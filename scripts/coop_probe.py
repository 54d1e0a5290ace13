"""Device time of the README-size time loop: single-cluster kernel, persistent cooperative grid, CUDA-graph replay."""
import ctypes as C, json, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ludvm_b200 import LUDVM, _lib
L = _lib.load()
TF = float(os.environ.get("PROBE_TF", "20"))
README = dict(t0=0, tf=TF, dt=5e-2, chord=1, rho=1.225, Uinf=1, Npoints=81, Ncoeffs=30, LESPcrit=0.2, Naca="0012")
NS = int(round(TF / 5e-2))
VARIANTS = [("cluster", {}), ("coop", {"LUDVM_NO_CLUSTER": "1"}), ("graph", {"LUDVM_NO_CLUSTER": "1", "LUDVM_NO_COOP": "1"})]
for label, env in VARIANTS:
    for k in ("LUDVM_NO_COOP", "LUDVM_NO_CLUSTER"):
        os.environ.pop(k, None)
    os.environ.update(env)
    for mode in ("exact", "fast"):
        best = 1e9
        for rep in range(4):
            s = LUDVM(**README, verbose=False, run=False, mode=mode, store_history=False, steps_per_graph=400)
            s.time_loop(nsteps=0)
            s.ctx.synchronize()
            t = time.perf_counter(); _lib.check(L.ludvm_sim_run(s._sim, NS)); s.ctx.synchronize(); dt = time.perf_counter() - t
            if rep: best = min(best, dt)
            s.close()
        print(json.dumps({"path": label, "mode": mode, "us_per_step": best / NS * 1e6, "steps_per_s_device": NS / best, "steps": NS}), flush=True)
