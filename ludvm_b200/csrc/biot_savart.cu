// biot_savart.cu -- generic all-pairs entry points: ludvm_induced_velocity (LUDVM.py:549-570),
// ludvm_selfconv_step (LUDVM.py:1095-1127 without the aerofoil), ludvm_flowfield_* (LUDVM.py:1186-1298).
#include <cmath>

#include "biot_savart.cuh"

namespace ludvm {

// ---------------------------------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------------------------------
// Range scan behind the flag-free exact kernels (common.cuh, coord_in_safe_window): *bad |= 1 if any coordinate of the
// four arrays lies outside the window in which the branch-free division / square root need no range test.
__global__ void __launch_bounds__(256) k_range_scan(const double *a, int na, const double *b, int nb, const double *c,
                                                    int nc, const double *d, int nd, int *bad)
{
    const long tot = (long)na + nb + nc + nd;
    bool ok = true;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < tot; i += (long)gridDim.x * blockDim.x) {
        double v;
        if (i < na) v = a[i];
        else if (i < (long)na + nb) v = b[i - na];
        else if (i < (long)na + nb + nc) v = c[i - na - nb];
        else v = d[i - na - nb - nc];
        ok = ok && coord_in_safe_window(v);
    }
    if (!ok) atomicOr(bad, 1);
}

// `bad`: nullptr = always evaluate the range words; otherwise the scan's verdict selects the instantiation (uniform).
template <int R, class Tgt>
__global__ void __launch_bounds__(256) k_exact_rows(SrcView S, Tgt T, int nrows, int d, double *pu, double *pw_,
                                                    const int *bad)
{
    int lane = threadIdx.x & 31;
    long gw = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    long nwarps = (long)gridDim.x * (blockDim.x >> 5);
    long ntasks = (long)((nrows + 4 * R - 1) / (4 * R)) << d;
    if (bad && *bad == 0)
        for (long t = gw; t < ntasks; t += nwarps) exact_rows_warp_task<R, false>(S, T, nrows, d, t, lane, pu, pw_);
    else
        for (long t = gw; t < ntasks; t += nwarps) exact_rows_warp_task<R, true>(S, T, nrows, d, t, lane, pu, pw_);
}

template <class Tgt>
__global__ void __launch_bounds__(ET_THREADS, 3) k_exact_tiled(SrcView S, Tgt T, int nrows, int d, double *pu, double *pw_,
                                                               const int *bad)
{
    __shared__ __align__(16) double2 sxz[ET_TILE], sgv[ET_TILE];
    if (bad && *bad == 0) exact_tiled_block<false>(S, T, nrows, blockIdx.x, d, blockIdx.y, pu, pw_, sxz, sgv);
    else exact_tiled_block<true>(S, T, nrows, blockIdx.x, d, blockIdx.y, pu, pw_, sxz, sgv);
}

template <class Tgt>
__global__ void __launch_bounds__(256) k_fast_rows(SrcView S, Tgt T, int nrows, int nchunks, double *pu, double *pw_)
{
    int lane = threadIdx.x & 31;
    long gw = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    long nwarps = (long)gridDim.x * (blockDim.x >> 5);
    long ntasks = (long)((nrows + 3) >> 2) * nchunks;
    for (long t = gw; t < ntasks; t += nwarps) fast_rows_warp_task(S, T, nrows, nchunks, t, lane, pu, pw_);
}

template <int R, class Tgt>
__global__ void __launch_bounds__(FT_THREADS, 2)
k_fast_tiled(SrcView S, Tgt T, int nrows, int chunk_len, double *pu, double *pw_)
{
    __shared__ double sx[FT_TILE], sz[FT_TILE], sg[FT_TILE], sv[FT_TILE];
    int c0 = blockIdx.y * chunk_len, c1 = min(S.n, c0 + chunk_len);
    size_t po = (size_t)blockIdx.y * nrows;
    fast_tiled_block<R>(S, T, nrows, blockIdx.x, c0, c1, pu + po, pw_ + po, sx, sz, sg, sv);
}

template <int R, class Tgt>
__global__ void __launch_bounds__(FT_THREADS, 2)
k_fast_tiled_tma(SrcView S, Tgt T, int nrows, int chunk_len, double *pu, double *pw_)
{
    __shared__ __align__(128) TmaTiles tiles;
    int c0 = blockIdx.y * chunk_len, c1 = min(S.n, c0 + chunk_len);
    size_t po = (size_t)blockIdx.y * nrows;
    fast_tiled_block_tma<R>(S, T, nrows, blockIdx.x, c0, c1, pu + po, pw_ + po, tiles);
}

template <int R, class Tgt>
__global__ void __launch_bounds__(FT_THREADS, 2)
k_fast32_tiled(SrcView S, Tgt T, int nrows, int chunk_len, double *pu, double *pw_)
{
    __shared__ float4 ssrc[FT_TILE];
    int c0 = blockIdx.y * chunk_len, c1 = min(S.n, c0 + chunk_len);
    size_t po = (size_t)blockIdx.y * nrows;
    fast32_tiled_block<R>(S, T, nrows, blockIdx.x, c0, c1, pu + po, pw_ + po, ssrc);
}

// fp32 with packed fp32x2 arithmetic: 8 rows (4 float2 pairs) per thread; scalar core radius only.
template <class Tgt>
__global__ void __launch_bounds__(FT_THREADS, 2)
k_fast32x2_tiled(SrcView S, Tgt T, int nrows, int chunk_len, double *pu, double *pw_)
{
    __shared__ Src32x2 ssrc[FT_TILE];
    int c0 = blockIdx.y * chunk_len, c1 = min(S.n, c0 + chunk_len);
    size_t po = (size_t)blockIdx.y * nrows;
    fast32x2_tiled_block<4>(S, T, nrows, blockIdx.x, c0, c1, pu + po, pw_ + po, ssrc);
}

// Whole row sums in one launch: warp-private bulk-copy pipelines, chunk partials folded through (distributed) shared
// memory, Euler update and peer stores in the epilogue (biot_savart.cuh, "fast fused").
template <int R, int CL, int V, class Tgt>
__global__ void __launch_bounds__(32 * FW_WARPS, 2)
k_fast_fused(SrcView S, Tgt T, int nrows, int chunk_len, int nchunks, RowOut O)
{
    extern __shared__ __align__(128) unsigned char fw_raw[];
    fast_fused_block<R, CL, V>(S, T, nrows, chunk_len, nchunks, O, *reinterpret_cast<FwSmem *>(fw_raw));
}

// Whole-cloud self-convection with each unordered pair evaluated once (biot_savart.cuh, "fast symmetric"): chain
// states / partial sums [chunk][n] for k_combine.
__global__ void __launch_bounds__(32 * FS_WARPS, 2) k_fast_sym(SymArgs A)
{
    extern __shared__ __align__(128) unsigned char fs_raw[];
    fast_sym_warp(A, reinterpret_cast<FsSmem *>(fs_raw)->w[threadIdx.x >> 5]);
}

// One set of partial row sums.  exact: nfold = tree depth d; fast: nfold = number of chunks.
struct Partials {
    double *u, *w;   // [fold][nrows]; nullptr: no such set
    int nfold;
};

// Fold partials, plus an optional second set (the reference's `u_wake + u_foil`, LUDVM.py:1108, :1219).
struct CombineArgs {
    Partials p, q;
    int exact;
    int nrows;
    RowOut out;
};

__global__ void __launch_bounds__(256) k_combine(CombineArgs a)
{
    int row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= a.nrows) return;
    double u, w;
    if (a.exact) {
        u = exact_combine_row(a.p.u, a.nrows, row, a.p.nfold);
        w = exact_combine_row(a.p.w, a.nrows, row, a.p.nfold);
        if (a.q.u) {
            u = __dadd_rn(u, exact_combine_row(a.q.u, a.nrows, row, a.q.nfold));
            w = __dadd_rn(w, exact_combine_row(a.q.w, a.nrows, row, a.q.nfold));
        }
    } else {
        u = fast_combine_row(a.p.u, a.nrows, row, a.p.nfold);
        w = fast_combine_row(a.p.w, a.nrows, row, a.p.nfold);
        if (a.q.u) {
            u += fast_combine_row(a.q.u, a.nrows, row, a.q.nfold);
            w += fast_combine_row(a.q.w, a.nrows, row, a.q.nfold);
        }
    }
    store_row(a.out, 0, row, u);
    store_row(a.out, 1, row, w);
}

// Vorticity stencil, LUDVM.py:1222-1292: clamped neighbours reproduce the centred / one-sided variants.
__global__ void __launch_bounds__(256) k_vorticity(const double *x1, int nx, const double *z1, int nz, const double *u,
                                                   const double *w, int ns, double *ome)
{
    long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    long per = (long)nx * nz;
    if (idx >= per * ns) return;
    long s = idx / per, r = idx - s * per;
    int i = (int)(r / nz), j = (int)(r - (long)i * nz);
    int ip = min(i + 1, nx - 1), im = max(i - 1, 0), jp = min(j + 1, nz - 1), jm = max(j - 1, 0);
    const double *us = u + s * per, *ws = w + s * per;
    double dx = __dsub_rn(x1[ip], x1[im]);
    double dz = __dsub_rn(z1[jp], z1[jm]);
    double dw = __dsub_rn(ws[(long)ip * nz + j], ws[(long)im * nz + j]);
    double du = __dsub_rn(us[(long)i * nz + jp], us[(long)i * nz + jm]);
    ome[idx] = __dsub_rn(__ddiv_rn(dw, dx), __ddiv_rn(du, dz));
}

// ---------------------------------------------------------------------------------------------------
// host-side planning and launch
// ---------------------------------------------------------------------------------------------------
static int ilog2_ceil(long v)
{
    int l = 0;
    while ((1L << l) < v) l++;
    return l;
}

// Source chunking of the fast tiled kernels.  It depends on the number of SOURCES only, so a row's sum does not depend
// on how the target rows are sharded over GPUs (G-rank results are bitwise equal to 1-rank results).
// 16 chunks from 131072 sources (measured at 2^20 sources: 866 ms against 875 ms with 8 for 2^20 rows, and 109.4 ms
// against 115.5 ms for the 131072 rows of one rank of eight, where 8 chunks force R = 2; 32 chunks: no further gain;
// profiles/r01e_chunks_probe.txt).  LUDVM_FAST_CHUNKS overrides (experiments; same value on every rank).
static void fast_chunking(int n, int *chunk_len, long *chunks)
{
    const char *ce = getenv("LUDVM_FAST_CHUNKS");
    const long cap = ce ? std::max(1L, atol(ce)) : (n >= 131072 ? 16L : 8L);
    long ch = std::max(1L, std::min(cap, (long)n / (FT_TILE * 2)));
    *chunk_len = (int)(((n + ch - 1) / ch + FT_TILE - 1) / FT_TILE * FT_TILE);
    *chunks = ((long)n + *chunk_len - 1) / *chunk_len;
}

static void set_plan(ludvm_ctx *ctx, int kernel, int R, int fold, int tma, int cluster, int variant = 0)
{
    ctx->plan[0] = kernel; ctx->plan[1] = R; ctx->plan[2] = fold; ctx->plan[3] = tma; ctx->plan[4] = cluster;
    ctx->plan[5] = variant; ctx->plan[6] = ctx->plan[7] = 0;
}

// Targets as (up to) two coordinate arrays for the range scan.
static void tgt_arrays(const TgtArray &T, long nrows, const double **a, int *na, const double **b, int *nb)
{
    *a = T.x; *na = (int)nrows; *b = T.z; *nb = (int)nrows;
}
static void tgt_arrays(const TgtGrid &T, long nrows, const double **a, int *na, const double **b, int *nb)
{
    *a = T.x1 + T.row0; *na = (int)((nrows + T.nz - 1) / T.nz); *b = T.z1; *nb = T.nz;
}

// Launch the range scan for an exact-mode evaluation; *flag = device flag for the kernels, or nullptr when the proof
// does not apply (per-source cores, vc^4 outside its window -- e.g. viscous=False --, LUDVM_EXACT_FLAGS=1).
template <class Tgt>
static int prove_exact_ranges(ludvm_ctx *ctx, const SrcView &S, const Tgt &T, long nrows, const int **flag)
{
    *flag = nullptr;
    if (S.vc4 != nullptr || !vc4_in_safe_window(S.vc4s) || S.n0 != S.n || getenv("LUDVM_EXACT_FLAGS")) return LUDVM_OK;
    void *p;
    int rc = scratch_reserve(ctx, SLOT_FLAG, 256, &p);
    if (rc) return rc;
    int *bad = (int *)((char *)p + 128);
    CUDA_TRY(cudaMemsetAsync(bad, 0, sizeof(int), ctx->stream));
    const double *ta, *tb;
    int na, nb;
    tgt_arrays(T, nrows, &ta, &na, &tb, &nb);
    const long tot = 2L * S.n + na + nb;
    const int blocks = (int)std::min<long>((tot + 1023) / 1024, (long)ctx->sm_count * 8);
    k_range_scan<<<blocks, 256, 0, ctx->stream>>>(S.x, S.n, S.z, S.n, ta, na, tb, nb, bad);
    ctx->launches++;
    ctx->range_flag = bad;
    *flag = bad;
    return LUDVM_OK;
}

template <int R, int CL, int V, class Tgt>
static int launch_fused_inst(ludvm_ctx *ctx, const SrcView &S, const Tgt &T, int nrows, int chunk_len, int nchunks,
                             const RowOut &O)
{
    auto kern = k_fast_fused<R, CL, V, Tgt>;
    static bool configured[16] = {};                       // per device; a function attribute is per device
    if (!configured[ctx->device & 15]) {
        CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FwSmem)));
        configured[ctx->device & 15] = true;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)ceil_div(nrows, 32 * R), CL, 1);
    cfg.blockDim = dim3(32 * FW_WARPS, 1, 1);
    cfg.dynamicSmemBytes = sizeof(FwSmem);
    cfg.stream = ctx->stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 1;
    at[0].val.clusterDim.y = CL;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = CL > 1 ? 1 : 0;
    CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, S, T, nrows, chunk_len, nchunks, O));
    ctx->launches++;
    set_plan(ctx, LUDVM_K_FAST_FUSED, R, nchunks, 1, CL, fw_unroll(R));
    ctx->plan[6] = FW_WARPS;
    ctx->plan[7] = V;
    return LUDVM_OK;
}

// The fused single-launch path: fast f64, one contiguous 16-byte aligned source segment with a scalar core, 8 or 16
// source chunks (>= 8192 sources) and enough rows for >= ~6 waves of 2 CTAs/SM.  *launched = false: not eligible, the
// caller takes the partial-sum path.
template <class Tgt>
static int try_launch_fused(ludvm_ctx *ctx, int mode, const SrcView &S, const Tgt &T, long nrows, const RowOut &O,
                            bool *launched)
{
    *launched = false;
    if ((mode != LUDVM_FAST_F64 && mode != LUDVM_FAST12_F64) || getenv("LUDVM_NO_FUSED")) return LUDVM_OK;
    if (S.vc4 != nullptr || S.gstride != 1 || S.n0 != S.n ||
        (((uintptr_t)S.x | (uintptr_t)S.z | (uintptr_t)S.g) & 15) != 0)
        return LUDVM_OK;
    int chunk_len;
    long chunks;
    fast_chunking(S.n, &chunk_len, &chunks);
    if (chunks != 8 && chunks != 16) return LUDVM_OK;
    // 16 chunks: a cluster of two 8-warp CTAs
    const int CL = (int)chunks / FW_WARPS;
    const long want = (long)ctx->sm_count * 2 * 6;
    int R = 4;
    while (R >= 1 && (long)ceil_div(nrows, 32 * R) * (chunks / 8) < want) R >>= 1;
    if (R < 1) return LUDVM_OK;
    int rc;
#define FUSED_CASE(RR, VV)                                                                                          \
    rc = CL == 2 ? launch_fused_inst<RR, 2, VV>(ctx, S, T, (int)nrows, chunk_len, (int)chunks, O)                   \
                 : launch_fused_inst<RR, 1, VV>(ctx, S, T, (int)nrows, chunk_len, (int)chunks, O)
    if (mode == LUDVM_FAST12_F64) {   // opt-in 12-slot pair arithmetic
        if (R == 4) FUSED_CASE(4, 1);
        else if (R == 2) FUSED_CASE(2, 1);
        else FUSED_CASE(1, 1);
    } else if (R == 4) FUSED_CASE(4, 0);
    else if (R == 2) FUSED_CASE(2, 0);
    else FUSED_CASE(1, 0);
#undef FUSED_CASE
    if (rc) return rc;
    CUDA_TRY(cudaGetLastError());
    *launched = true;
    return LUDVM_OK;
}

// Evaluate partial row sums for `nrows` targets against S into scratch slots slot / slot + 1; *P describes what
// k_combine must fold.
template <class Tgt>
static int launch_partials(ludvm_ctx *ctx, int mode, const SrcView &S, const Tgt &T, long nrows, int slot, Partials *P)
{
    const int sm = ctx->sm_count;
    // both partial buffers, `per_row` values per row
    auto reserve = [&](size_t per_row, int nfold) -> int {
        const size_t bytes = sizeof(double) * (size_t)nrows * per_row;
        void *a, *b;
        int rc;
        if ((rc = scratch_reserve(ctx, slot, bytes, &a))) return rc;
        if ((rc = scratch_reserve(ctx, slot + 1, bytes, &b))) return rc;
        *P = {(double *)a, (double *)b, nfold};
        return LUDVM_OK;
    };
    int rc;
    if (mode == LUDVM_FAST12_F64) mode = LUDVM_FAST_F64;   // outside the fused kernel: the (more accurate) 13-slot pair
    if (mode == LUDVM_EXACT_F64) {
        const int *bad;
        if ((rc = prove_exact_ranges(ctx, S, T, nrows, &bad))) return rc;
        if (nrows >= 4096 && (S.n >= 1024 || nrows >= (long)sm * ET_THREADS * 3)) {   // (few sources: only if the rows alone fill the GPU)
            // Many rows: one thread per row, sources staged through shared memory; the tree is cut at depth d so
            // that >= ~6 waves of 4 CTAs/SM are in flight.
            long rblocks = (nrows + ET_THREADS - 1) / ET_THREADS;
            int want = ilog2_ceil(std::max(1L, (long)sm * 24 / rblocks));
            int d = std::min(pw_max_depth(S.n), want);
            if ((rc = reserve((size_t)1 << d, d))) return rc;
            k_exact_tiled<<<dim3((unsigned)rblocks, 1u << d), ET_THREADS, 0, ctx->stream>>>(S, T, (int)nrows, d, P->u, P->w, bad);
            ctx->launches++;
            set_plan(ctx, LUDVM_K_EXACT_TILED, 1, d, 0, 1, bad ? 1 : 0);
            return LUDVM_OK;
        }
        // Few rows (or few rows and few sources): 8 lanes per row, tree nodes spread over warps.
        constexpr int R = 1;
        long nquads = (nrows + 4 * R - 1) / (4 * R);
        int want = ilog2_ceil(std::max(1L, (long)sm * 64 / std::max(1L, nquads)));
        int d = std::min(pw_max_depth(S.n), want);
        if ((rc = reserve((size_t)1 << d, d))) return rc;
        long ntasks = nquads << d;
        int blocks = (int)std::min((ntasks + 7) / 8, (long)sm * 16);
        k_exact_rows<R><<<blocks, 256, 0, ctx->stream>>>(S, T, (int)nrows, d, P->u, P->w, bad);
        ctx->launches++;
        set_plan(ctx, LUDVM_K_EXACT_ROWS, R, d, 0, 1, bad ? 1 : 0);
        return LUDVM_OK;
    }
    const bool f32 = (mode == LUDVM_FAST_F32);
    if (f32 || nrows >= 8192) {
        // source chunking from the number of sources only (fast_chunking); the rows-per-thread factor R adapts to the
        // number of rows to keep >= ~6 waves of 2 CTAs/SM in flight
        int chunk_len;
        long chunks;
        fast_chunking(S.n, &chunk_len, &chunks);
        // fp32: the packed fp32x2 kernel (8 rows per thread) when the core radius is a scalar and there are enough rows
        const bool f32x2 = f32 && S.vc4 == nullptr && (long)ceil_div(nrows, FT_THREADS * 8) * chunks >= (long)sm * 2;
        int R = f32x2 ? 8 : 4;
        if (!f32) {
            while (R > 1 && (long)ceil_div(nrows, FT_THREADS * R) * chunks < (long)sm * 2 * 6) R >>= 1;
        }
        int row_blocks = ceil_div(nrows, FT_THREADS * R);
        if ((rc = reserve((size_t)chunks, (int)chunks))) return rc;
        dim3 grid(row_blocks, (unsigned)chunks);
        // one contiguous, 16-byte aligned source segment with a scalar core: TMA-staged tiles
        const bool tma = !f32 && S.vc4 == nullptr && S.gstride == 1 && S.n0 == S.n &&
                         (((uintptr_t)S.x | (uintptr_t)S.z | (uintptr_t)S.g) & 15) == 0;
        if (f32x2) k_fast32x2_tiled<<<grid, FT_THREADS, 0, ctx->stream>>>(S, T, (int)nrows, chunk_len, P->u, P->w);
        else if (f32) k_fast32_tiled<4><<<grid, FT_THREADS, 0, ctx->stream>>>(S, T, (int)nrows, chunk_len, P->u, P->w);
        else if (tma && R == 4) k_fast_tiled_tma<4><<<grid, FT_THREADS, 0, ctx->stream>>>(S, T, (int)nrows, chunk_len, P->u, P->w);
        else if (tma && R == 2) k_fast_tiled_tma<2><<<grid, FT_THREADS, 0, ctx->stream>>>(S, T, (int)nrows, chunk_len, P->u, P->w);
        else if (tma) k_fast_tiled_tma<1><<<grid, FT_THREADS, 0, ctx->stream>>>(S, T, (int)nrows, chunk_len, P->u, P->w);
        else if (R == 4) k_fast_tiled<4><<<grid, FT_THREADS, 0, ctx->stream>>>(S, T, (int)nrows, chunk_len, P->u, P->w);
        else if (R == 2) k_fast_tiled<2><<<grid, FT_THREADS, 0, ctx->stream>>>(S, T, (int)nrows, chunk_len, P->u, P->w);
        else k_fast_tiled<1><<<grid, FT_THREADS, 0, ctx->stream>>>(S, T, (int)nrows, chunk_len, P->u, P->w);
        ctx->launches++;
        set_plan(ctx, f32x2 ? LUDVM_K_FAST32X2_TILED : f32 ? LUDVM_K_FAST32_TILED : tma ? LUDVM_K_FAST_TILED_TMA : LUDVM_K_FAST_TILED,
                 R, (int)chunks, tma ? 1 : 0, 1);
        return LUDVM_OK;
    }
    long nquads = (nrows + 3) / 4;
    long chunks = std::max(1L, std::min((long)sm * 64 / std::max(1L, nquads), ((long)S.n + 63) / 64));
    if ((rc = reserve((size_t)chunks, (int)chunks))) return rc;
    long ntasks = nquads * chunks;
    int blocks = (int)std::min((ntasks + 7) / 8, (long)sm * 16);
    k_fast_rows<<<blocks, 256, 0, ctx->stream>>>(S, T, (int)nrows, (int)chunks, P->u, P->w);
    ctx->launches++;
    set_plan(ctx, LUDVM_K_FAST_ROWS, 1, (int)chunks, 0, 1);
    return LUDVM_OK;
}

// The all-pairs evaluation of every entry point: the row sums of S (plus those of S2, if given) at the `nrows` targets
// T, stored as O says.  One source set: the fused single launch when eligible.  Otherwise partial sums (S in
// SLOT_PART_A, S2 in SLOT_PART_B) folded by k_combine.
template <class Tgt>
static int eval_rows(ludvm_ctx *ctx, int mode, const SrcView &S, const SrcView *S2, const Tgt &T, long nrows,
                     const RowOut &O)
{
    int rc;
    if (!S2) {
        bool fused;
        if ((rc = try_launch_fused(ctx, mode, S, T, nrows, O, &fused)) || fused) return rc;
    }
    CombineArgs a{};
    if ((rc = launch_partials(ctx, mode, S, T, nrows, SLOT_PART_A, &a.p))) return rc;
    if (S2 && (rc = launch_partials(ctx, mode, *S2, T, nrows, SLOT_PART_B, &a.q))) return rc;
    CUDA_TRY(cudaGetLastError());
    a.exact = (mode == LUDVM_EXACT_F64);
    a.nrows = (int)nrows;
    a.out = O;
    k_combine<<<ceil_div(nrows, 256), 256, 0, ctx->stream>>>(a);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return LUDVM_OK;
}

// Smallest cloud for k_fast_sym: from 2^17 vortices fast_chunking cuts 16 chunks, whose 136 chunk pairs x 128-row blocks
// give ~8700 strips and more for the 2368 warps of the persistent grid.
#define FS_MIN_N (1L << 17)

// The whole-cloud step through k_fast_sym + k_combine when the cloud is eligible: fast f64 with the 13-slot pair, one
// finite core vc^4 > 0 for all sources, 16-byte aligned arrays and n >= FS_MIN_N.  *launched = false otherwise.
static int try_launch_sym(ludvm_ctx *ctx, int mode, const double *gamma, const double *x, const double *z,
                          const double *vc4_per_source, double vc4, long n, const RowOut &O, bool *launched)
{
    *launched = false;
    if (mode != LUDVM_FAST_F64 || vc4_per_source || !(vc4 > 0.0 && std::isfinite(vc4)) || n < FS_MIN_N ||
        (((uintptr_t)x | (uintptr_t)z | (uintptr_t)gamma) & 15) != 0)
        return LUDVM_OK;
    int chunk_len;
    long chunks;
    fast_chunking((int)n, &chunk_len, &chunks);
    SymArgs A;
    A.x = x; A.z = z; A.g = gamma; A.vc4 = vc4;
    A.n = (int)n; A.chunk_len = chunk_len; A.nchunks = (int)chunks;
    A.bpc = chunk_len / FS_ROWS;
    A.blast = ceil_div(n - (chunks - 1) * chunk_len, FS_ROWS);
    A.npairs = (int)(chunks * (chunks + 1) / 2);
    A.nitems = (long)A.blast * A.npairs + (long)(A.bpc - A.blast) * (A.npairs - 1);
    const long nblocks = (long)(chunks - 1) * A.bpc + A.blast;
    int rc;
    void *pa, *pb, *sync;
    const size_t part_bytes = sizeof(double) * (size_t)n * chunks;
    const size_t sync_bytes = 256 + sizeof(unsigned) * (size_t)nblocks * chunks;
    if ((rc = scratch_reserve(ctx, SLOT_PART_A, part_bytes, &pa)) || (rc = scratch_reserve(ctx, SLOT_PART_A + 1, part_bytes, &pb)) ||
        (rc = scratch_reserve(ctx, SLOT_SYM_SYNC, sync_bytes, &sync)))
        return rc;
    if (!ctx->sym_timeout) {
        CUDA_TRY(cudaHostAlloc((void **)&ctx->sym_timeout, sizeof(int), cudaHostAllocMapped));
        *(volatile int *)ctx->sym_timeout = 0;
    }
    int *timeout_dev;
    CUDA_TRY(cudaHostGetDevicePointer((void **)&timeout_dev, ctx->sym_timeout, 0));
    A.pu = (double *)pa;
    A.pw = (double *)pb;
    A.ticket = (unsigned *)sync;
    A.abort = (int *)((char *)sync + 128);
    A.progress = (unsigned *)((char *)sync + 256);
    A.timeout = timeout_dev;
    CUDA_TRY(cudaMemsetAsync(sync, 0, sync_bytes, ctx->stream));
    static bool configured[16] = {};                       // per device; a function attribute is per device
    static int ctas_per_sm[16] = {};
    if (!configured[ctx->device & 15]) {
        CUDA_TRY(cudaFuncSetAttribute(k_fast_sym, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FsSmem)));
        CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas_per_sm[ctx->device & 15], k_fast_sym,
                                                               32 * FS_WARPS, sizeof(FsSmem)));
        configured[ctx->device & 15] = true;
    }
    // persistent: every CTA that fits at once (a waiting warp only waits on a warp that holds an earlier ticket and
    // is therefore running, so co-residency is not needed for progress)
    const int grid = ctx->sm_count * std::max(1, ctas_per_sm[ctx->device & 15]);
    k_fast_sym<<<grid, 32 * FS_WARPS, sizeof(FsSmem), ctx->stream>>>(A);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    CombineArgs ca{};
    ca.p = {A.pu, A.pw, (int)chunks};
    ca.nrows = (int)n;
    ca.out = O;
    k_combine<<<ceil_div(n, 256), 256, 0, ctx->stream>>>(ca);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    set_plan(ctx, LUDVM_K_FAST_SYM, 4, (int)chunks, 1, 1, FS_STAGE);
    ctx->plan[6] = FS_WARPS;
    *launched = true;
    return LUDVM_OK;
}

static int check_mode(int mode)
{
    if (mode != LUDVM_EXACT_F64 && mode != LUDVM_FAST_F64 && mode != LUDVM_FAST_F32 && mode != LUDVM_FAST12_F64)
        return set_error(LUDVM_E_ARG, "unknown arithmetic mode %d", mode);
    return LUDVM_OK;
}

// The self-convection step of rows [row0, row0 + nrows) of one cloud.  O holds the velocity outputs, indexed from the
// first row, and the position outputs, indexed by vortex; the latter are offset to row0 here, and x, z, dt filled in.
static int selfconv_rows(ludvm_ctx *ctx, int mode, const double *gamma, const double *x, const double *z,
                         const double *vc4_per_source, double vc4, long n, long row0, long nrows, double dt, RowOut O)
{
    ARG_CHECK(ctx != nullptr);
    int rc = check_mode(mode);
    if (rc) return rc;
    ARG_CHECK(n > 0 && n < (1L << 30) && row0 >= 0 && nrows >= 0 && row0 + nrows <= n);
    ARG_CHECK(gamma && x && z);
    if (nrows == 0) return LUDVM_OK;
    DeviceGuard g(ctx->device);
    O.x = x + row0;
    O.z = z + row0;
    O.dt = dt;
    if (O.xo) {
        O.xo += row0;
        O.zo += row0;
    }
    for (int p = 0; p < O.npeers; p++) {
        O.xo_peer[p] += row0;
        O.zo_peer[p] += row0;
    }
    SrcView S = make_src(gamma, 1, x, z, vc4_per_source, vc4, (int)n);
    return eval_rows(ctx, mode, S, nullptr, TgtArray{x + row0, z + row0}, nrows, O);
}

}  // namespace ludvm

using namespace ludvm;

LUDVM_API int ludvm_induced_velocity(ludvm_ctx *ctx, int mode, const double *gamma, long ngamma, const double *xw,
                                     const double *zw, const double *vc4_per_source, double vc4, long nw,
                                     const double *xp, const double *zp, long np_, double *u, double *w, int ptr_kind)
{
    ARG_CHECK(ctx != nullptr);
    int rc = check_mode(mode);
    if (rc) return rc;
    ARG_CHECK(nw >= 0 && np_ >= 0 && nw < (1L << 30) && np_ < (1L << 30));
    ARG_CHECK(ngamma == nw || ngamma == 1);
    ARG_CHECK(ptr_kind == LUDVM_PTR_HOST || ptr_kind == LUDVM_PTR_DEVICE);
    if (np_ == 0) return LUDVM_OK;
    ARG_CHECK(u && w && xp && zp);
    ARG_CHECK(nw == 0 || (gamma && xw && zw));
    DeviceGuard g(ctx->device);

    const bool host = ptr_kind == LUDVM_PTR_HOST;
    const double *dg = gamma, *dxw = xw, *dzw = zw, *dvc = vc4_per_source, *dxp = xp, *dzp = zp;
    double *du = u, *dw = w;
    if (host && ((rc = stage_in(ctx, {{gamma, nw ? ngamma : 0, &dg}, {xw, nw, &dxw}, {zw, nw, &dzw},
                                      {vc4_per_source, vc4_per_source ? nw : 0, &dvc}, {xp, np_, &dxp}, {zp, np_, &dzp}})) ||
                 (rc = stage_out(ctx, {{u, np_, &du}, {w, np_, &dw}}))))
        return rc;
    if (nw == 0) {  // np.sum over an empty axis
        CUDA_TRY(cudaMemsetAsync(du, 0, (size_t)np_ * sizeof(double), ctx->stream));
        CUDA_TRY(cudaMemsetAsync(dw, 0, (size_t)np_ * sizeof(double), ctx->stream));
    } else {
        RowOut O{};
        O.u = du;
        O.w = dw;
        SrcView S = make_src(dg, ngamma == nw ? 1 : 0, dxw, dzw, dvc, vc4, (int)nw);
        if ((rc = eval_rows(ctx, mode, S, nullptr, TgtArray{dxp, dzp}, np_, O))) return rc;
    }
    return host ? copy_back(ctx, {{u, np_, &du}, {w, np_, &dw}}) : LUDVM_OK;
}

LUDVM_API int ludvm_selfconv_step(ludvm_ctx *ctx, int mode, const double *gamma, const double *x, const double *z,
                                  const double *vc4_per_source, double vc4, long n, long row0, long nrows, double dt,
                                  double *x_out, double *z_out, double *u_out, double *w_out)
{
    ARG_CHECK(x_out && z_out);
    RowOut O{};
    O.u = u_out;
    O.w = w_out;
    O.xo = x_out;
    O.zo = z_out;
    return selfconv_rows(ctx, mode, gamma, x, z, vc4_per_source, vc4, n, row0, nrows, dt, O);
}

LUDVM_API int ludvm_selfconv_step_all(ludvm_ctx *ctx, int mode, const double *gamma, const double *x, const double *z,
                                      const double *vc4_per_source, double vc4, long n, double dt, double *x_out,
                                      double *z_out, double *u_out, double *w_out)
{
    ARG_CHECK(ctx != nullptr);
    int rc = check_mode(mode);
    if (rc) return rc;
    ARG_CHECK(n > 0 && n < (1L << 30));
    ARG_CHECK(gamma && x && z && x_out && z_out);
    if ((rc = sym_timeout_check(ctx))) return rc;
    DeviceGuard g(ctx->device);
    RowOut O{};
    O.u = u_out;
    O.w = w_out;
    O.x = x;
    O.z = z;
    O.xo = x_out;
    O.zo = z_out;
    O.dt = dt;
    bool sym;
    if ((rc = try_launch_sym(ctx, mode, gamma, x, z, vc4_per_source, vc4, n, O, &sym)) || sym) return rc;
    return ludvm_selfconv_step(ctx, mode, gamma, x, z, vc4_per_source, vc4, n, 0, n, dt, x_out, z_out, u_out, w_out);
}

LUDVM_API int ludvm_selfconv_step_p2p(ludvm_ctx *ctx, int mode, const double *gamma, const double *x, const double *z,
                                      const double *vc4_per_source, double vc4, long n, long row0, long nrows,
                                      double dt, int npeers, double *const *x_out_peers, double *const *z_out_peers)
{
    ARG_CHECK(x_out_peers && z_out_peers && npeers >= 1 && npeers <= LUDVM_MAX_PEERS);
    RowOut O{};
    O.npeers = npeers;
    for (int p = 0; p < npeers; p++) {
        ARG_CHECK(x_out_peers[p] && z_out_peers[p]);
        O.xo_peer[p] = x_out_peers[p];
        O.zo_peer[p] = z_out_peers[p];
    }
    return selfconv_rows(ctx, mode, gamma, x, z, vc4_per_source, vc4, n, row0, nrows, dt, O);
}

LUDVM_API int ludvm_flowfield_velocity(ludvm_ctx *ctx, int mode, const double *ga, const double *xa, const double *za,
                                       long na, const double *gb, const double *xb, const double *zb, long nb,
                                       double vc4, const double *x1, long nx, const double *z1, long nz, long row0,
                                       long nrows, double *u, double *w, int ptr_kind)
{
    ARG_CHECK(ctx != nullptr);
    int rc = check_mode(mode);
    if (rc) return rc;
    ARG_CHECK(na > 0 && nb >= 0 && nx > 0 && nz > 0 && row0 >= 0 && nrows >= 0 && row0 + nrows <= nx);
    ARG_CHECK(na < (1L << 30) && nb < (1L << 30) && nrows * nz < (1L << 31) - 1024);
    ARG_CHECK(ga && xa && za && x1 && z1 && u && w && (nb == 0 || (gb && xb && zb)));
    ARG_CHECK(ptr_kind == LUDVM_PTR_HOST || ptr_kind == LUDVM_PTR_DEVICE);
    if (nrows == 0) return LUDVM_OK;
    DeviceGuard g(ctx->device);
    const long npts = nrows * nz;
    const bool host = ptr_kind == LUDVM_PTR_HOST;
    const double *dga = ga, *dxa = xa, *dza = za, *dgb = gb, *dxb = xb, *dzb = zb, *dx1 = x1, *dz1 = z1;
    double *du = u, *dw = w;
    if (host && ((rc = stage_in(ctx, {{ga, na, &dga}, {xa, na, &dxa}, {za, na, &dza}, {gb, nb, &dgb}, {xb, nb, &dxb},
                                      {zb, nb, &dzb}, {x1, nx, &dx1}, {z1, nz, &dz1}})) ||
                 (rc = stage_out(ctx, {{u, npts, &du}, {w, npts, &dw}}))))
        return rc;
    RowOut O{};
    O.u = du;
    O.w = dw;
    const SrcView SA = make_src(dga, 1, dxa, dza, nullptr, vc4, (int)na);
    const SrcView SB = make_src(dgb, 1, dxb, dzb, nullptr, vc4, (int)nb);
    if ((rc = eval_rows(ctx, mode, SA, nb ? &SB : nullptr, TgtGrid{dx1, dz1, (int)nz, (int)row0}, npts, O))) return rc;
    return host ? copy_back(ctx, {{u, npts, &du}, {w, npts, &dw}}) : LUDVM_OK;
}

// Velocity and vorticity of one snapshot in one call: with host buffers the fields make one trip (u, w, ome out) instead
// of u, w out, back in for the stencil, and ome out.
LUDVM_API int ludvm_flowfield(ludvm_ctx *ctx, int mode, const double *ga, const double *xa, const double *za, long na,
                              const double *gb, const double *xb, const double *zb, long nb, double vc4,
                              const double *x1, long nx, const double *z1, long nz, long row0, long nrows, double *u,
                              double *w, double *ome, int ptr_kind)
{
    ARG_CHECK(ctx && ome && u && w && x1 && z1);
    ARG_CHECK(ptr_kind == LUDVM_PTR_HOST || ptr_kind == LUDVM_PTR_DEVICE);
    ARG_CHECK(nrows >= 2 && nz >= 2 && row0 >= 0 && row0 + nrows <= nx);
    DeviceGuard g(ctx->device);
    const long npts = nrows * nz;
    const bool host = ptr_kind == LUDVM_PTR_HOST;
    const double *dga = ga, *dxa = xa, *dza = za, *dgb = gb, *dxb = xb, *dzb = zb, *dx1 = x1, *dz1 = z1;
    double *du = u, *dw = w, *dome = ome;
    int rc;
    if (host && ((rc = stage_in(ctx, {{ga, na, &dga}, {xa, na, &dxa}, {za, na, &dza}, {gb, nb, &dgb}, {xb, nb, &dxb},
                                      {zb, nb, &dzb}, {x1, nx, &dx1}, {z1, nz, &dz1}})) ||
                 (rc = stage_out(ctx, {{u, npts, &du}, {w, npts, &dw}, {ome, npts, &dome}}))))
        return rc;
    if ((rc = ludvm_flowfield_velocity(ctx, mode, dga, dxa, dza, na, dgb, dxb, dzb, nb, vc4, dx1, nx, dz1, nz, row0, nrows,
                                       du, dw, LUDVM_PTR_DEVICE)) ||
        (rc = ludvm_flowfield_vorticity(ctx, dx1 + row0, nrows, dz1, nz, du, dw, 1, dome, LUDVM_PTR_DEVICE)))
        return rc;
    return host ? copy_back(ctx, {{u, npts, &du}, {w, npts, &dw}, {ome, npts, &dome}}) : LUDVM_OK;
}

LUDVM_API int ludvm_flowfield_vorticity(ludvm_ctx *ctx, const double *x1, long nx, const double *z1, long nz,
                                        const double *u, const double *w, long ns, double *ome, int ptr_kind)
{
    ARG_CHECK(ctx && x1 && z1 && u && w && ome);
    ARG_CHECK(nx >= 2 && nz >= 2 && ns >= 1);
    ARG_CHECK(ptr_kind == LUDVM_PTR_HOST || ptr_kind == LUDVM_PTR_DEVICE);
    DeviceGuard g(ctx->device);
    const long tot = ns * nx * nz;
    const bool host = ptr_kind == LUDVM_PTR_HOST;
    const double *dx1 = x1, *dz1 = z1, *du = u, *dw = w;
    double *dome = ome;
    int rc;
    if (host && ((rc = stage_in(ctx, {{x1, nx, &dx1}, {z1, nz, &dz1}, {u, tot, &du}, {w, tot, &dw}})) ||
                 (rc = stage_out(ctx, {{ome, tot, &dome}}))))
        return rc;
    k_vorticity<<<ceil_div(tot, 256), 256, 0, ctx->stream>>>(dx1, (int)nx, dz1, (int)nz, du, dw, (int)ns, dome);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return host ? copy_back(ctx, {{ome, tot, &dome}}) : LUDVM_OK;
}
