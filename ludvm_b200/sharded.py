"""Target-row sharded self-convection of one vortex cloud over the ranks of a torch.distributed group
(BASELINE.json configs[2]; the convection phase LUDVM.py:1095-1127 for a free cloud).

Every rank holds the full source state (32 B/vortex), evaluates the rows [rank*N/G, (rank+1)*N/G) against all N
sources with the CUDA kernel behind `ludvm_selfconv_step`, and every rank must end the step with all N updated
positions (16 B/vortex/step).  Two transports:

  transport="p2p"   the Euler-update kernel stores its rows straight into the next-position buffers of ALL ranks
                    (peer-mapped symmetric memory, NVLink/NVSwitch stores) -- compute and all-gather in one kernel,
                    no NCCL call in the step; consecutive steps are separated by a symmetric-memory barrier.
  transport="nccl"  the kernel writes its rows locally, then one NCCL all-gather per coordinate.

Row sums do not depend on the shard, so the G-rank result is bitwise equal to the 1-rank one.  The per-row kernel is
injectable so the sharding/assembly logic can be exercised on CPU tensors with gloo.
"""
import torch
import torch.distributed as dist

from . import ops


def shard_bounds(n, world, rank):
    """Contiguous, equal row shards (the all-gather needs equal counts)."""
    if n % world:
        raise ValueError("number of vortices (%d) must be a multiple of the number of ranks (%d)" % (n, world))
    per = n // world
    return rank * per, per


def case_slice(ncases, world, rank):
    """Cases of a parameter sweep owned by `rank` (BASELINE.json configs[3]): contiguous, sizes differ by at most one
    block of ceil(ncases / world); no collective is needed, every case is independent."""
    per = (ncases + world - 1) // world
    return slice(min(ncases, rank * per), min(ncases, (rank + 1) * per))


def grid_slab(nx, world, rank):
    """x-rows of a flow-field grid owned by `rank` (BASELINE.json configs[4]): returns (r0, r1, h0, h1) -- the rank
    owns rows [r0, r1) and evaluates [h0, h1), one halo row per interior side, so that the central-difference
    vorticity stencil (LUDVM.py:1222-1292) of every owned row sees its neighbours without any exchange; at the ends of
    the grid the stencil is one-sided in the reference too.  Keep `field[r0 - h0 : r1 - h0]` of what was evaluated."""
    per = (nx + world - 1) // world
    r0, r1 = min(nx, rank * per), min(nx, (rank + 1) * per)
    return r0, r1, max(0, r0 - 1), min(nx, r1 + 1)


def morton_order(x, z, bits=10):
    """Permutation that sorts points (numpy arrays) along the Z-order curve of a 2^bits x 2^bits grid over their bounding
    square.  Row shards of a cloud relabelled this way are compact in space, so in `mode="tree"` a rank's targets live
    under ~1/world of the tree's cells and it evaluates only that share of the cell-to-cell (M2L) work; with a random
    labelling every rank would evaluate all of it.  The relabelling does not change any vortex's velocity."""
    import numpy as np
    x, z = np.asarray(x, dtype=np.float64), np.asarray(z, dtype=np.float64)
    side = max(x.max() - x.min(), z.max() - z.min()) * (1 + 1e-12) + 1e-300
    n = 1 << bits

    def spread(v):
        v = v.astype(np.int64) & 0xFFFF
        v = (v | (v << 8)) & 0x00FF00FF
        v = (v | (v << 4)) & 0x0F0F0F0F
        v = (v | (v << 2)) & 0x33333333
        v = (v | (v << 1)) & 0x55555555
        return v
    ix = np.minimum(((x - x.min()) / side * n).astype(np.int64), n - 1)
    iz = np.minimum(((z - z.min()) / side * n).astype(np.int64), n - 1)
    return np.argsort(spread(ix) | (spread(iz) << 1), kind="stable")


class ShardedSelfConvection:
    def __init__(self, g, x, z, v_core, dt, mode="fast", ctx=None, group=None, kernel=None, transport="auto", order=18,
                 leaf=0):
        """mode: "exact" | "fast" | "fp32" | "fast12" (all-pairs) or "tree" (O(N log N) treecode of csrc/tree.cu with
        interpolation order `order`: every rank builds the same tree over all sources and evaluates its own target
        rows; positions are exchanged with NCCL all_gather)."""
        self.group = group
        self.order, self.leaf = int(order), int(leaf)
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.g = g
        self.n = x.numel()
        # The kernels are enqueued on the context's stream while the collectives / symmetric-memory barriers run on
        # torch's current stream: the two must be the same stream, otherwise nothing orders them.
        if kernel is None and x.is_cuda:
            from . import _lib
            cur = torch.cuda.current_stream(x.device).cuda_stream
            if ctx is None:
                ctx = _lib.Context(x.device.index if x.device.index is not None else torch.cuda.current_device(), cur)
                ctx.stream_handle = cur
            elif getattr(ctx, "stream_handle", None) not in (cur, _lib.Context.CUDA_STREAM_LEGACY if cur == 0 else cur):
                raise ValueError("ShardedSelfConvection: ctx must wrap torch's current CUDA stream "
                                 "(_lib.Context(device, torch.cuda.current_stream().cuda_stream))")
        self.vc4, self.dt, self.mode, self.ctx = float(v_core) ** 4, float(dt), mode, ctx
        self.row0, self.nrows = shard_bounds(self.n, self.world, self.rank)
        self._kernel = kernel or self._cuda_kernel
        self.transport = "none"
        self._hdl = None
        if self.world > 1:
            want = transport
            if mode == "tree" and want == "p2p":
                raise ValueError("ShardedSelfConvection: the treecode step has no fused peer-store epilogue; use transport='nccl'")
            if want == "auto":
                want = "p2p" if (kernel is None and x.is_cuda and mode != "tree") else "nccl"
            if want == "p2p":
                try:
                    self._init_p2p(x, z)
                    self.transport = "p2p"
                except Exception as e:  # symmetric memory unavailable on this system: use the collective instead
                    if transport == "p2p":
                        raise
                    self.transport_note = "p2p unavailable (%s)" % e
                    want = "nccl"
            if want == "nccl":
                self.transport = "nccl"
        if self.transport != "p2p":
            self.x, self.z = x, z
            self._xs, self._zs = torch.empty_like(x), torch.empty_like(z)   # shard rows land here
            self._xn, self._zn = torch.empty_like(x), torch.empty_like(z)   # gathered next state

    # -- p2p transport ---------------------------------------------------------------------------------------
    def _init_p2p(self, x, z):
        import torch.distributed._symmetric_memory as symm_mem
        grp = self.group if self.group is not None else dist.group.WORLD
        n = self.n
        self._bufs, self._hdls = [], []
        for _ in range(2):                      # double buffer: [x | z] per buffer, symmetric across ranks
            t = symm_mem.empty(2 * n, dtype=torch.float64, device=x.device)
            h = symm_mem.rendezvous(t, grp)
            self._bufs.append(t)
            self._hdls.append(h)
        self._bufs[0][:n].copy_(x)
        self._bufs[0][n:].copy_(z)
        self._cur = 0
        self._hdls[0].barrier()
        self.x, self.z = self._bufs[0][:n], self._bufs[0][n:]

    def _step_p2p(self):
        n, cur, nxt = self.n, self._cur, 1 - self._cur
        xin, zin = self._bufs[cur][:n], self._bufs[cur][n:]
        peers = [int(p) for p in self._hdls[nxt].buffer_ptrs]
        ops.selfconv_step_p2p(self.ctx, self.mode, self.g, xin, zin, self.vc4, self.dt,
                              peers, [p + 8 * n for p in peers], self.row0, self.nrows)
        self._hdls[nxt].barrier()               # every rank's stores have landed; nobody still reads `nxt`'s old data
        self._cur = nxt
        self.x, self.z = self._bufs[nxt][:n], self._bufs[nxt][n:]
        return self.x, self.z

    # -- nccl / single-rank ----------------------------------------------------------------------------------
    def _cuda_kernel(self, g, x, z, vc4, dt, row0, nrows, x_out, z_out):
        if self.mode == "tree":
            ops.selfconv_step_tree(self.ctx, g, x, z, vc4, dt, x_out, z_out, row0=row0, nrows=nrows, order=self.order,
                                   leaf=self.leaf)
            return
        if row0 == 0 and nrows == self.n:      # one rank owns every row: the whole-cloud step (same bits)
            ops.selfconv_step_all(self.ctx, self.mode, g, x, z, vc4, dt, x_out, z_out)
            return
        ops.selfconv_step(self.ctx, self.mode, g, x, z, vc4, dt, x_out, z_out, row0=row0, nrows=nrows)

    def step(self):
        """One forward-Euler step of the whole cloud; returns the new (x, z) (full length on every rank)."""
        if self.transport == "p2p":
            return self._step_p2p()
        if self.world == 1:
            self._kernel(self.g, self.x, self.z, self.vc4, self.dt, 0, self.n, self._xn, self._zn)
        else:
            r0, nr = self.row0, self.nrows
            self._kernel(self.g, self.x, self.z, self.vc4, self.dt, r0, nr, self._xs, self._zs)
            dist.all_gather_into_tensor(self._xn, self._xs[r0:r0 + nr], group=self.group)
            dist.all_gather_into_tensor(self._zn, self._zs[r0:r0 + nr], group=self.group)
        self.x, self._xn = self._xn, self.x
        self.z, self._zn = self._zn, self.z
        return self.x, self.z
