"""Time the fused single-launch self-convection kernel against the partial-sum path (1 GPU):
N = 2^20 full launch and the 131072-row shard of one rank of eight, 16 and 8 source chunks."""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ludvm_b200 import _lib, ops  # noqa: E402

N = 1 << 20
rng = np.random.default_rng(20260101)
dev = torch.device("cuda", 0)
x = torch.tensor(rng.uniform(-20, 0, N), device=dev)
z = torch.tensor(rng.uniform(-4, 4, N), device=dev)
g = torch.tensor(rng.standard_normal(N) * 1e-2, device=dev)
xo, zo = torch.empty_like(x), torch.empty_like(z)
ctx = _lib.Context(0, torch.cuda.current_stream().cuda_stream)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)


def timed(nrows, reps=3):
    ops.selfconv_step(ctx, "fast", g, x, z, 0.065 ** 4, 0.05, xo, zo, row0=0, nrows=nrows)
    torch.cuda.synchronize()
    best = 1e9
    for _ in range(reps):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ops.selfconv_step(ctx, "fast", g, x, z, 0.065 ** 4, 0.05, xo, zo, row0=0, nrows=nrows)
        e1.record()
        e1.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return best


dfma = ctx.fp64_fma_rate(300.0)
print("dfma/s %.4g" % dfma)
CONFIGS = [{}, {"LUDVM_NO_FUSED": "1"}, {"LUDVM_FAST_CHUNKS": "8"}]
if os.environ.get("PROBE_FUSED_ONLY"):
    CONFIGS = [c for c in CONFIGS if "LUDVM_NO_FUSED" not in c]
KEYS = ("LUDVM_NO_FUSED", "LUDVM_FAST_CHUNKS")
print("lib", _lib.LIB_PATH)
for nrows in (N, N // 8):
    for env in CONFIGS:
        for k in KEYS:
            os.environ.pop(k, None)
        os.environ.update(env)
        ms = timed(nrows)
        p = ctx.last_plan()
        rate = float(nrows) * N / (ms * 1e-3)
        print("rows %8d  %-62s %-14s R=%d cl=%d w=%d  %9.3f ms  %.4g pairs/s  %.3f of dfma" %
              (nrows, env, p["kernel"], p["rows_per_thread"], p["cluster"], p["warps"], ms, rate, rate * 13 / dfma),
              flush=True)
