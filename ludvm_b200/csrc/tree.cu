// tree.cu -- O(N log N) far field for vortex clouds with N >> 2^20 (SURVEY.md section 8(f)-4): ludvm_induced_velocity_tree,
// ludvm_selfconv_step_tree.  The reference has no such path (LUDVM.induced_velocity, LUDVM.py:549-570, is all-pairs); the
// checker is therefore the all-pairs oracle, and the error against it is a reported quantity, not a bit-parity claim.
//
// Method: a kernel-independent treecode (barycentric Lagrange interpolation at Chebyshev points, as in Wang, Krasny &
// Tlupova's BLTC) over a complete quadtree in Morton order.  The Vatistas kernel 1 / sqrt(r^4 + vc^4) has no harmonic
// multipole expansion -- its far field is the point vortex plus a series in (vc / r)^4 that is not small at leaf scale
// (vc / a ~ 0.2-0.6) -- so the far field of a cell is represented by (order + 1)^2 PROXY vortices at the tensor Chebyshev
// points of the cell, whose strengths are the anterpolated circulations
//     qhat[k1, k2] = sum_j  l_k1(xi_j) l_k2(zeta_j) Gamma_j
// (children's proxies are anterpolated again for the parent: the nested form).  A proxy is an ordinary vortex, so the
// far-field evaluation is the SAME 13-slot fast pair arithmetic as the all-pairs kernels (pair_fast, common.cuh) and
// runs on the FP64 pipe at the same rate; the only question is how many pairs are left.  Lists are the standard
// one-cell separation: a target leaf sees its 3x3 neighbour leaves directly and, on every level l = 2 .. L, the children
// of its parent's neighbours that are not its own neighbours (<= 27 cells), each through its proxies -- or through its
// own vortices when it holds at most pth = P2 / 4 of them.  On top of that, cells with more than pth vortices carry a local
// field at their own Chebyshev points (M2L / L2L / L2P, see "evaluation" below), so that a far list acts on P2 points per
// cell instead of on every target: the black-box FMM of Fong & Darve with this file's proxies; between two cells that both
// carry proxies that action is a fixed matrix per level and offset, applied on the FP64 tensor cores (k_tree_m2l_dmma).
// Measured error of the representation (oracle/tree_model.py,
// float64 numpy model of this file): order 12 -> 2e-11, 16 -> 5e-14, 18 -> 3e-15 of sum |terms|.
//
// Everything runs on one stream (the context's, or the stream a caller such as the time loop's far-field step passes);
// the host round trips are the bounding box (32 bytes), which fixes the tree depth, and the largest leaf population.  The order of every sum is fixed (cells sorted by original index, lists walked in slot order), so results
// are bitwise reproducible from run to run and independent of how the target rows are sharded over GPUs.
#include "common.cuh"

#include <algorithm>
#include <cmath>

namespace ludvm {

#define TR_MAX_P1 (TR_MAX_ORDER + 1)
#define TR_MAX_LEVEL 10
#define TR_MAX_SLOTS (9 + 36 * (TR_MAX_LEVEL - 1))
#define TE_THREADS 128
#define TE_TILE 128
#define TU_THREADS 256
#define TU_TILE 32
#define TR_MAX_LEAF_POP 65536   // refuse clouds that put more than this into one leaf of the deepest tree
#define TR_SORT_WARP_MAX 96     // cells up to this many vortices are ordered by one warp, larger ones by a whole CTA

struct TreeGeom {
    double x0, z0, side;     // root square [x0, x0 + side) x [z0, z0 + side)
    double inv_leaf;         // 2^L / side
    double vc4;
    double tdens;            // targets per unit area when they are a uniform grid (0: unknown): cells that hold more than P2
                             // grid points carry a local field even where they hold few sources
    int pth;                 // a cell with more than pth source vortices is represented by proxies (and carries a local field)
    int L, P1, P2;
    double s[TR_MAX_P1];     // Chebyshev points of the second kind on [-1, 1], exactly antisymmetric
    double bw[TR_MAX_P1];    // barycentric weights
};

__host__ __device__ __forceinline__ unsigned spread16(unsigned v)
{
    v &= 0xFFFFu;
    v = (v | (v << 8)) & 0x00FF00FFu;
    v = (v | (v << 4)) & 0x0F0F0F0Fu;
    v = (v | (v << 2)) & 0x33333333u;
    v = (v | (v << 1)) & 0x55555555u;
    return v;
}
__host__ __device__ __forceinline__ unsigned compact16(unsigned v)
{
    v &= 0x55555555u;
    v = (v | (v >> 1)) & 0x33333333u;
    v = (v | (v >> 2)) & 0x0F0F0F0Fu;
    v = (v | (v >> 4)) & 0x00FF00FFu;
    v = (v | (v >> 8)) & 0x0000FFFFu;
    return v;
}
__host__ __device__ __forceinline__ int morton2(int ix, int iz) { return (int)(spread16((unsigned)ix) | (spread16((unsigned)iz) << 1)); }
// cells of levels 2 .. l-1 precede level l in the proxy array
__host__ __device__ __forceinline__ long level_offset(int l) { return ((1L << (2 * l)) - 16) / 3; }

// D (8 x 8) += A (8 x 4) B (4 x 8) on the FP64 tensor cores; fragments (PTX ISA, m8n8k4 .f64): A[row = lane >> 2][k = lane & 3],
// B[k = lane & 3][col = lane >> 2], D[row = lane >> 2][col = 2 (lane & 3) + {0, 1}]
__device__ __forceinline__ void dmma_m8n8k4(double &d0, double &d1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

// ---------------------------------------------------------------------------------------------------
// bounding box: order-preserving map double -> uint64, atomicMin / atomicMax
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long dkey(double v)
{
    unsigned long long b = (unsigned long long)__double_as_longlong(v);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
static double dkey_inv(unsigned long long k)
{
    unsigned long long b = (k >> 63) ? (k & 0x7FFFFFFFFFFFFFFFull) : ~k;
    double v;
    memcpy(&v, &b, 8);
    return v;
}

// mm[0..3] = min x, max x, min z, max z over both point sets; mm[4..7] the same over set A (the sources) only
__global__ void __launch_bounds__(256) k_tree_bbox(const double *xa, const double *za, int na, const double *xb,
                                                   const double *zb, int nb, unsigned long long *mm)
{
    unsigned long long lo_x = ~0ull, hi_x = 0, lo_z = ~0ull, hi_z = 0, alo_x = ~0ull, ahi_x = 0, alo_z = ~0ull, ahi_z = 0;
    const long tot = (long)na + nb;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < tot; i += (long)gridDim.x * blockDim.x) {
        const bool a = i < na;
        const double x = a ? xa[i] : xb[i - na], z = a ? za[i] : zb[i - na];
        if (x != x || z != z) continue;
        const unsigned long long kx = dkey(x), kz = dkey(z);
        lo_x = min(lo_x, kx); hi_x = max(hi_x, kx); lo_z = min(lo_z, kz); hi_z = max(hi_z, kz);
        if (a) { alo_x = min(alo_x, kx); ahi_x = max(ahi_x, kx); alo_z = min(alo_z, kz); ahi_z = max(ahi_z, kz); }
    }
    for (int o = 16; o; o >>= 1) {
        lo_x = min(lo_x, __shfl_xor_sync(~0u, lo_x, o)); hi_x = max(hi_x, __shfl_xor_sync(~0u, hi_x, o));
        lo_z = min(lo_z, __shfl_xor_sync(~0u, lo_z, o)); hi_z = max(hi_z, __shfl_xor_sync(~0u, hi_z, o));
        alo_x = min(alo_x, __shfl_xor_sync(~0u, alo_x, o)); ahi_x = max(ahi_x, __shfl_xor_sync(~0u, ahi_x, o));
        alo_z = min(alo_z, __shfl_xor_sync(~0u, alo_z, o)); ahi_z = max(ahi_z, __shfl_xor_sync(~0u, ahi_z, o));
    }
    if ((threadIdx.x & 31) == 0) {
        atomicMin(mm + 0, lo_x); atomicMax(mm + 1, hi_x); atomicMin(mm + 2, lo_z); atomicMax(mm + 3, hi_z);
        atomicMin(mm + 4, alo_x); atomicMax(mm + 5, ahi_x); atomicMin(mm + 6, alo_z); atomicMax(mm + 7, ahi_z);
    }
}

// ---------------------------------------------------------------------------------------------------
// Morton keys, counting sort (deterministic: cells ordered by original index)
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_tree_keys(const __grid_constant__ TreeGeom G, const double *x, const double *z, int n,
                                                   int *key, int *slot, int *cnt)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int nc = 1 << G.L;
    int ix = (int)((x[i] - G.x0) * G.inv_leaf), iz = (int)((z[i] - G.z0) * G.inv_leaf);
    ix = max(0, min(nc - 1, ix));
    iz = max(0, min(nc - 1, iz));
    const int k = morton2(ix, iz);
    key[i] = k;
    // any free slots of the cell (k_tree_cellsort fixes the order of the sources afterwards); lanes of a warp that hit the
    // same cell -- grid targets: all of them -- take their slots with one atomic
    const int lane = threadIdx.x & 31;
    const unsigned peers = __match_any_sync(__activemask(), k);
    const int leader = __ffs(peers) - 1;
    int base = 0;
    if (lane == leader) base = atomicAdd(cnt + k, __popc(peers));
    base = __shfl_sync(peers, base, leader);
    slot[i] = base + __popc(peers & ((1u << lane) - 1u));
}

// exclusive scan of cnt[0 .. n) into start[0 .. n], and the largest count into *maxcnt; one CTA
__global__ void __launch_bounds__(1024) k_tree_scan(const int *cnt, int *start, int n, int *maxcnt)
{
    __shared__ int part[1024];
    const int t = threadIdx.x, chunk = (n + 1023) / 1024, b = min(n, t * chunk), e = min(n, b + chunk);
    int s = 0, mx = 0;
    for (int i = b; i < e; i++) {
        s += cnt[i];
        mx = max(mx, cnt[i]);
    }
    atomicMax(maxcnt, mx);
    part[t] = s;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {
        int v = t >= o ? part[t - o] : 0;
        __syncthreads();
        part[t] += v;
        __syncthreads();
    }
    int run = part[t] - s;
    for (int i = b; i < e; i++) {
        start[i] = run;
        run += cnt[i];
    }
    if (t == 1023) start[n] = part[1023];
}

__global__ void __launch_bounds__(256) k_tree_place(const int *key, const int *slot, const int *start, int n, int *tmp)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) tmp[start[key[i]] + slot[i]] = i;
}

// perm[start[c] .. start[c+1]) = the cell's original indices in ascending order (rank by counting: the entries are distinct)
__global__ void __launch_bounds__(256) k_tree_cellsort(const int *__restrict__ tmp, const int *__restrict__ start, int ncell,
                                                       int *__restrict__ perm)
{
    const int lane = threadIdx.x & 31;
    const long gw = (long)blockIdx.x * 8 + (threadIdx.x >> 5), nw = (long)gridDim.x * 8;
    for (long c = gw; c < ncell; c += nw) {
        const int b = start[c], m = start[c + 1] - b;
        if (m == 0 || m > TR_SORT_WARP_MAX) continue;
        const int *__restrict__ cell = tmp + b;
        for (int i = lane; i < m; i += 64) {          // two entries per lane and trip: the loads of a trip are independent
            const int i2 = min(i + 32, m - 1);
            const int v = cell[i], v2 = cell[i2];
            int r = 0, r2 = 0, j = 0;
            for (; j + 8 <= m; j += 8) {
                int t[8];
#pragma unroll
                for (int q = 0; q < 8; q++) t[q] = cell[j + q];
#pragma unroll
                for (int q = 0; q < 8; q++) { r += t[q] < v; r2 += t[q] < v2; }
            }
            for (; j < m; j++) { const int t = cell[j]; r += t < v; r2 += t < v2; }
            perm[b + r] = v;
            if (i + 32 < m) perm[b + r2] = v2;
        }
    }
}
__global__ void __launch_bounds__(256) k_tree_cellsort_big(const int *__restrict__ tmp, const int *__restrict__ start, int ncell,
                                                           int *__restrict__ perm)
{
    __shared__ int tile[1024];
    for (long c = blockIdx.x; c < ncell; c += gridDim.x) {
        const int b = start[c], m = start[c + 1] - b;
        if (m <= TR_SORT_WARP_MAX) continue;
        for (int i0 = 0; i0 < m; i0 += 512) {          // two entries per thread and trip
            const int i = i0 + threadIdx.x, i2 = i + 256;
            const int v = i < m ? tmp[b + i] : 0, v2 = i2 < m ? tmp[b + i2] : 0;
            int r = 0, r2 = 0;
            for (int j0 = 0; j0 < m; j0 += 1024) {
                __syncthreads();
                for (int j = threadIdx.x; j < 1024; j += 256) tile[j] = j0 + j < m ? tmp[b + j0 + j] : 0x7FFFFFFF;
                __syncthreads();
                const int jn = min(1024, m - j0);
                int j = 0;
                for (; j + 8 <= jn; j += 8) {
#pragma unroll
                    for (int q = 0; q < 8; q++) { const int t = tile[j + q]; r += t < v; r2 += t < v2; }
                }
                for (; j < jn; j++) { const int t = tile[j]; r += t < v; r2 += t < v2; }
            }
            if (i < m) perm[b + r] = v;
            if (i2 < m) perm[b + r2] = v2;
        }
    }
}

// sorted copies of the sources; circulations pre-scaled by 1 / (2 pi) as in every fast kernel
__global__ void __launch_bounds__(256) k_tree_gather(const int *perm, const double *x, const double *z, const double *g, int n,
                                                     double *xs, double *zs, double *gs)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int p = perm[i];
    xs[i] = x[p];
    zs[i] = z[p];
    gs[i] = g[p] * LUDVM_INV_TWO_PI;
}

// barycentric Lagrange basis l_k(xi), k < P1, into row[]
__device__ __forceinline__ void tree_basis(const TreeGeom &G, double xi, double *row)
{
    double sum = 0.0;
    int hit = -1;
    for (int k = 0; k < G.P1; k++) {
        double d = xi - G.s[k];
        if (d == 0.0) { hit = k; d = 1.0; }
        const double t = G.bw[k] / d;
        row[k] = t;
        sum += t;
    }
    const double inv = 1.0 / sum;
    for (int k = 0; k < G.P1; k++) row[k] = hit >= 0 ? (k == hit ? 1.0 : 0.0) : row[k] * inv;
}

// ---------------------------------------------------------------------------------------------------
// upward pass: proxies of every cell of level l that holds more than pth vortices
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(TU_THREADS) k_tree_up(const __grid_constant__ TreeGeom G, int l, const int *startS,
                                                        const double *xs, const double *zs, const double *gs, double *qhat)
{
    const int c = blockIdx.x, sh = 2 * (G.L - l), tid = threadIdx.x;
    const int b = startS[(long)c << sh], e = startS[((long)c + 1) << sh];
    if (e - b <= G.pth) return;
    __shared__ double Lx[TU_TILE][TR_MAX_P1], Lz[TU_TILE][TR_MAX_P1], gt[TU_TILE];
    __shared__ int seg_a[4], seg_pre[5], nseg_s, prox_ch[4], prox_cell[4], nprox_s;
    __shared__ double Tq[2][TR_MAX_P1][TR_MAX_P1], Qc[TR_MAX_P1 * TR_MAX_P1], Tm[TR_MAX_P1 * TR_MAX_P1];
    const int P1 = G.P1, P2 = G.P2;
    const double h = ldexp(G.side, -(l + 1)), inv_h = 1.0 / h;
    const double cx = G.x0 + (2.0 * compact16((unsigned)c) + 1.0) * h, cz = G.z0 + (2.0 * compact16((unsigned)c >> 1) + 1.0) * h;
    // Children that carry proxies are anterpolated with the two fixed (P1 x P1) transfer matrices Tq[v][k][m] =
    // l_k((s_m -+ 1) / 2) -- 2 P1^3 multiply-adds per child instead of P2^2; children (or a leaf's own vortices) that
    // are plain vortices go through the tile loop below.
    if (tid == 0) {
        int ns = 0, run = 0, np = 0;
        if (l == G.L) {
            seg_a[0] = b; seg_pre[0] = 0; run = e - b; ns = 1;
        } else {
            for (int ch = 0; ch < 4; ch++) {
                const long cc = 4L * c + ch;
                const int cb = startS[cc << (sh - 2)], ce = startS[(cc + 1) << (sh - 2)], n = ce - cb;
                if (n == 0) continue;
                if (n > G.pth) { prox_ch[np] = ch; prox_cell[np] = (int)cc; np++; continue; }
                seg_pre[ns] = run; seg_a[ns] = cb; run += n;
                ns++;
            }
        }
        seg_pre[ns] = run;
        nseg_s = ns;
        nprox_s = np;
    }
    if (l < G.L && tid < 2 * P1) {
        const int v = tid / P1, m = tid - v * P1;
        double col[TR_MAX_P1];
        tree_basis(G, (G.s[m] + (double)(2 * v - 1)) * 0.5, col);
        for (int k = 0; k < P1; k++) Tq[v][k][m] = col[k];
    }
    __syncthreads();
    const int nseg = nseg_s, total = seg_pre[nseg];
    const double *qchild = qhat + level_offset(l + 1) * P2;
    double acc[3] = {0.0, 0.0, 0.0};
    for (int pc = 0; pc < nprox_s; pc++) {
        const int vx = prox_ch[pc] & 1, vz = prox_ch[pc] >> 1;
        const double *q = qchild + (long)prox_cell[pc] * P2;
        for (int k = tid; k < P2; k += TU_THREADS) Qc[k] = q[k];
        __syncthreads();
        for (int idx = tid; idx < P2; idx += TU_THREADS) {       // Tm[k1][m2] = sum_m1 Tq[vx][k1][m1] Q[m1][m2]
            const int k1 = idx / P1, m2 = idx - k1 * P1;
            double a = 0.0;
            for (int m1 = 0; m1 < P1; m1++) a = fma(Tq[vx][k1][m1], Qc[m1 * P1 + m2], a);
            Tm[idx] = a;
        }
        __syncthreads();
#pragma unroll
        for (int qq = 0; qq < 3; qq++) {                        // out[k1][k2] += sum_m2 Tm[k1][m2] Tq[vz][k2][m2]
            const int k = tid + qq * TU_THREADS;
            if (k < P2) {
                const int k1 = k / P1, k2 = k - k1 * P1;
                double a = acc[qq];
                for (int m2 = 0; m2 < P1; m2++) a = fma(Tm[k1 * P1 + m2], Tq[vz][k2][m2], a);
                acc[qq] = a;
            }
        }
        __syncthreads();
    }
    for (int t0 = 0; t0 < total; t0 += TU_TILE) {
        {   // barycentric bases of the tile: thread = (pseudo-vortex tt, dimension, quarter of the nodes)
            const int tt = tid >> 3, dim = (tid >> 2) & 1, part = tid & 3, j = t0 + tt;
            double *row = dim ? Lz[tt] : Lx[tt];
            const bool valid = j < total;
            double xi = 0.0, gval = 0.0;
            if (valid) {
                int sg = 0;
                while (sg + 1 < nseg && seg_pre[sg + 1] <= j) sg++;
                const int p = seg_a[sg] + j - seg_pre[sg];
                xi = dim ? (zs[p] - cz) * inv_h : (xs[p] - cx) * inv_h;
                gval = gs[p];
            }
            double sum = 0.0, tk[(TR_MAX_P1 + 3) / 4];
            int hit = -1;
#pragma unroll
            for (int q = 0; q < (TR_MAX_P1 + 3) / 4; q++) {
                const int k = part + 4 * q;
                tk[q] = 0.0;
                if (valid && k < P1) {
                    double d = xi - G.s[k];
                    if (d == 0.0) { hit = k; d = 1.0; }
                    tk[q] = G.bw[k] / d;
                    sum += tk[q];
                }
            }
            sum += __shfl_xor_sync(~0u, sum, 1);      // the four quarters sit in adjacent lanes (every lane takes part)
            sum += __shfl_xor_sync(~0u, sum, 2);
            hit = max(hit, __shfl_xor_sync(~0u, hit, 1));
            hit = max(hit, __shfl_xor_sync(~0u, hit, 2));
            const double inv = valid ? 1.0 / sum : 0.0;
#pragma unroll
            for (int q = 0; q < (TR_MAX_P1 + 3) / 4; q++) {
                const int k = part + 4 * q;
                if (k < P1) row[k] = !valid ? 0.0 : hit >= 0 ? (k == hit ? 1.0 : 0.0) : tk[q] * inv;
            }
            if (dim == 0 && part == 0) gt[tt] = gval;
        }
        __syncthreads();
#pragma unroll
        for (int q = 0; q < 3; q++) {
            const int k = tid + q * TU_THREADS;
            if (k < P2) {
                const int k1 = k / P1, k2 = k - k1 * P1;
                double a = acc[q];
                for (int tt = 0; tt < TU_TILE; tt++) a = fma(Lx[tt][k1] * gt[tt], Lz[tt][k2], a);
                acc[q] = a;
            }
        }
        __syncthreads();
    }
    double *out = qhat + (level_offset(l) + c) * P2;
#pragma unroll
    for (int q = 0; q < 3; q++) {
        const int k = tid + q * TU_THREADS;
        if (k < P2) out[k] = acc[q];
    }
}

// Leaf level of the upward pass on the FP64 tensor cores (orders <= 23): qhat[k1][k2] = sum_j (lx_k1(xi_j) Gamma_j) lz_k2(zeta_j)
// is a (P1 x n) x (n x P1) product per cell.  A warp takes 4 vortices per step: the lanes with lane & 3 = q hold vortex q's
// basis values at k = (lane >> 2) + 8 t, t < 3, in exactly the A- (rows k1) and B- (columns k2) fragment layouts, the
// normalisation sums run over those 8 lanes by shuffles, and 9 MMAs add the step to the 3 x 3 tiles of the result.  The
// four warps of the CTA split the cell's vortices and are summed in warp order.  (k_tree_up: 5 % of the DFMA rate, the
// tile loop is bound by shared-memory loads.)
__global__ void __launch_bounds__(128) k_tree_up_leaf_mma(const __grid_constant__ TreeGeom G, const int *startS, const double *xs,
                                                          const double *zs, const double *gs, double *qhat)
{
    const int c = blockIdx.x, b = startS[c], e = startS[c + 1];
    if (e - b <= G.pth) return;
    const int P1 = G.P1, l = G.L;
    const double h = ldexp(G.side, -(l + 1)), inv_h = 1.0 / h;
    const double cx = G.x0 + (2.0 * compact16((unsigned)c) + 1.0) * h, cz = G.z0 + (2.0 * compact16((unsigned)c >> 1) + 1.0) * h;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, fr = lane >> 2, fk = lane & 3;
    double acc[3][3][2];
#pragma unroll
    for (int m = 0; m < 3; m++)
#pragma unroll
        for (int n = 0; n < 3; n++) acc[m][n][0] = acc[m][n][1] = 0.0;
    for (int j0 = b + 4 * warp; j0 < e; j0 += 16) {
        const int j = j0 + fk;
        const bool valid = j < e;
        const int jj = valid ? j : e - 1;
        const double xi = (xs[jj] - cx) * inv_h, ze = (zs[jj] - cz) * inv_h, g = valid ? gs[jj] : 0.0;
        double ax[3], bz[3], sx = 0.0, sz = 0.0;
        int hx = -1, hz = -1;
#pragma unroll
        for (int t = 0; t < 3; t++) {
            const int k = fr + 8 * t;
            ax[t] = bz[t] = 0.0;
            if (k < P1) {
                double dx = xi - G.s[k], dz = ze - G.s[k];
                if (dx == 0.0) { hx = k; dx = 1.0; }
                if (dz == 0.0) { hz = k; dz = 1.0; }
                ax[t] = G.bw[k] / dx;
                bz[t] = G.bw[k] / dz;
                sx += ax[t];
                sz += bz[t];
            }
        }
#pragma unroll
        for (int o = 4; o < 32; o <<= 1) {      // the 8 lanes of a vortex: lane & 3 fixed
            sx += __shfl_xor_sync(~0u, sx, o);
            sz += __shfl_xor_sync(~0u, sz, o);
            hx = max(hx, __shfl_xor_sync(~0u, hx, o));
            hz = max(hz, __shfl_xor_sync(~0u, hz, o));
        }
        const double ix = g / sx, iz = 1.0 / sz;
#pragma unroll
        for (int t = 0; t < 3; t++) {
            const int k = fr + 8 * t;
            ax[t] = hx >= 0 ? (k == hx ? g : 0.0) : ax[t] * ix;      // lx_k1 Gamma_j
            bz[t] = hz >= 0 ? (k == hz ? 1.0 : 0.0) : bz[t] * iz;
        }
#pragma unroll
        for (int m = 0; m < 3; m++)
#pragma unroll
            for (int n = 0; n < 3; n++) dmma_m8n8k4(acc[m][n][0], acc[m][n][1], ax[m], bz[n]);
    }
    // sum the four warps in warp order (fixed), then write the P1 x P1 corner
    __shared__ double red[4][3][3][2][32];
#pragma unroll
    for (int m = 0; m < 3; m++)
#pragma unroll
        for (int n = 0; n < 3; n++) {
            red[warp][m][n][0][lane] = acc[m][n][0];
            red[warp][m][n][1][lane] = acc[m][n][1];
        }
    __syncthreads();
    double *out = qhat + (level_offset(l) + c) * G.P2;
    for (int idx = threadIdx.x; idx < 3 * 3 * 2 * 32; idx += blockDim.x) {
        const int ln = idx & 31, ee = (idx >> 5) & 1, n = (idx >> 6) % 3, m = (idx >> 6) / 3;
        const int k1 = 8 * m + (ln >> 2), k2 = 8 * n + 2 * (ln & 3) + ee;
        if (k1 < P1 && k2 < P1)
            out[k1 * P1 + k2] = ((red[0][m][n][ee][ln] + red[1][m][n][ee][ln]) + red[2][m][n][ee][ln]) + red[3][m][n][ee][ln];
    }
}

// ---------------------------------------------------------------------------------------------------
// evaluation.  A cell with more than pth source vortices also carries a LOCAL field: the velocity induced by everything
// outside its neighbourhood, sampled at its own P2 Chebyshev points (M2L: the far list of the cell's level acting on the
// points, the same pair arithmetic; L2L: the parent's local field interpolated to the child's points).  A target then
// takes (a) the local field of its deepest ancestor that has one, interpolated at the target (L2P), (b) the far lists of
// the levels below that ancestor evaluated directly, and (c) the 3x3 neighbour leaves directly.  Which cells carry a local
// field depends on the SOURCES only, so a target's sum does not depend on which other targets a rank was given.
// One launch holds the M2L items of every level (they depend on the upward pass only) and the leaf items.
// ---------------------------------------------------------------------------------------------------
struct TreeEval {
    const int *startS, *startT, *permT, *keyT;
    const double *xs, *zs, *gs, *qhat;     // sorted sources, proxies
    const double *xt, *zt;                 // targets, original order
    double *u, *w;                         // original order
    double *uloc, *wloc;                   // local fields, laid out like qhat
    unsigned long long *pairs;             // pair evaluations (diagnostic)
    int np;
};

struct TreeSmem {
    int ent_a[TR_MAX_SLOTS + 32], ent_len[TR_MAX_SLOTS + 32], ent_lvl[TR_MAX_SLOTS + 32], pre[TR_MAX_SLOTS + 33];
    int nent;
    double2 sxz[2][TE_TILE];
    double sg[2][TE_TILE];
};

// targets of a leaf item: the leaf's points (sorted order t -> original index)
struct TgtLeafPts {
    const int *permT;
    const double *xt, *zt;
    double *u, *w;
    __device__ __forceinline__ void load(int t, double &x, double &z) const
    {
        const int oi = permT[t];
        x = xt[oi];
        z = zt[oi];
    }
    __device__ __forceinline__ void store(int t, double uu, double ww) const
    {
        const int oi = permT[t];
        u[oi] = uu;
        w[oi] = ww;
    }
};
// targets of an M2L item: the cell's own Chebyshev points
struct TgtNodePts {
    double cx, cz, h;
    const double *s;
    int P1;
    double *u, *w;
    __device__ __forceinline__ void load(int k, double &x, double &z) const
    {
        const int k1 = k / P1, k2 = k - k1 * P1;
        x = fma(h, s[k1], cx);
        z = fma(h, s[k2], cz);
    }
    __device__ __forceinline__ void store(int k, double uu, double ww) const
    {
        u[k] = uu;
        w[k] = ww;
    }
};

// source j of the CTA's flattened list -> (x, z, g / 2 pi)
__device__ __forceinline__ void tree_fetch(const TreeGeom &G, const TreeEval &A, const TreeSmem &sm, int j, int total,
                                           double &x, double &z, double &g)
{
    if (j >= total) { x = z = g = 0.0; return; }
    int lo = 0, hi = sm.nent;
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (sm.pre[mid] <= j) lo = mid;
        else hi = mid;
    }
    const int o = j - sm.pre[lo], l = sm.ent_lvl[lo], a = sm.ent_a[lo];
    if (l < 0) {
        x = A.xs[a + o];
        z = A.zs[a + o];
        g = A.gs[a + o];
    } else {
        const int k1 = o / G.P1, k2 = o - k1 * G.P1;
        const double h = ldexp(G.side, -(l + 1));
        x = fma(h, G.s[k1], G.x0 + (2.0 * compact16((unsigned)a) + 1.0) * h);
        z = fma(h, G.s[k2], G.z0 + (2.0 * compact16((unsigned)a >> 1) + 1.0) * h);
        g = A.qhat[(level_offset(l) + a) * G.P2 + o];
    }
}

// Interaction list of cell (cx, cz) of level lc into shared memory: the 3x3 neighbours (near; lc == L) and the far cells
// of levels lmin .. lmax <= lc (a coarser level's list is the ancestor's).  Every candidate has a fixed slot, so the list
// order (= the summation order) never depends on scheduling; empty slots are dropped afterwards, order kept.
__device__ __forceinline__ int tree_build_list(const TreeGeom &G, const TreeEval &A, int cx, int cz, int lc, bool near, int lmin,
                                               int lmax, TreeSmem &sm, bool skip_proxies = false)
{
    const int tid = threadIdx.x, lane = tid & 31, L = G.L, P2 = G.P2;
    const int nslots = 9 + 36 * (L - 1);
    for (int s = tid; s < nslots; s += TE_THREADS) {
        int a = 0, len = 0, lvl = -1;
        if (s < 9) {
            const int jx = cx + s % 3 - 1, jz = cz + s / 3 - 1;
            if (near && jx >= 0 && jz >= 0 && jx < (1 << L) && jz < (1 << L)) {
                const int cc = morton2(jx, jz);
                a = A.startS[cc];
                len = A.startS[cc + 1] - a;
            }
        } else {
            const int t = s - 9, l = 2 + t / 36, r = t % 36, pn = r >> 2, ch = r & 3;
            if (l >= lmin && l <= lmax) {
                const int cxl = cx >> (lc - l), czl = cz >> (lc - l);
                const int qx = (cxl >> 1) + pn % 3 - 1, qz = (czl >> 1) + pn / 3 - 1;
                if (qx >= 0 && qz >= 0 && qx < (1 << (l - 1)) && qz < (1 << (l - 1))) {
                    const int jx = 2 * qx + (ch & 1), jz = 2 * qz + (ch >> 1);
                    if (max(abs(jx - cxl), abs(jz - czl)) > 1) {
                        const int cc = morton2(jx, jz), sh = 2 * (L - l);
                        const int b = A.startS[(long)cc << sh], n = A.startS[((long)cc + 1) << sh] - b;
                        if (n > G.pth) { a = cc; len = skip_proxies ? 0 : P2; lvl = l; }
                        else { a = b; len = n; }
                    }
                }
            }
        }
        sm.ent_a[s] = a;
        sm.ent_len[s] = len;
        sm.ent_lvl[s] = lvl;
    }
    __syncthreads();
    if (tid < 32) {
        int base = 0;
        for (int s0 = 0; s0 < nslots; s0 += 32) {
            const int s = s0 + lane;
            const int a = s < nslots ? sm.ent_a[s] : 0, len = s < nslots ? sm.ent_len[s] : 0, lvl = s < nslots ? sm.ent_lvl[s] : 0;
            const unsigned m = __ballot_sync(~0u, len > 0);
            __syncwarp();
            if (len > 0) {
                const int pos = base + __popc(m & ((1u << lane) - 1u));
                sm.ent_a[pos] = a;
                sm.ent_len[pos] = len;
                sm.ent_lvl[pos] = lvl;
            }
            base += __popc(m);
            __syncwarp();
        }
        const int nent = base;
        int run = 0;
        for (int s0 = 0; s0 < nent; s0 += 32) {
            const int s = s0 + lane;
            const int v = s < nent ? sm.ent_len[s] : 0;
            int inc = v;
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(~0u, inc, o);
                if (lane >= o) inc += t;
            }
            if (s < nent) sm.pre[s] = run + inc - v;
            run += __shfl_sync(~0u, inc, 31);
        }
        if (lane == 0) {
            sm.pre[nent] = run;
            sm.nent = nent;
        }
    }
    __syncthreads();
    return sm.pre[sm.nent];
}

// one pass: targets [t0, t1) of T, t1 - t0 <= R * TE_THREADS, against the CTA's whole list
template <int R, class Tgt>
__device__ __forceinline__ void tree_eval_rows(const TreeGeom &G, const TreeEval &A, const Tgt &T, TreeSmem &sm, int t0, int t1,
                                               int total)
{
    const int tid = threadIdx.x;
    const double vc4 = G.vc4;
    double xp[R], zp[R], au[R], aw[R];
#pragma unroll
    for (int r = 0; r < R; r++) {
        T.load(min(t0 + tid + r * TE_THREADS, t1 - 1), xp[r], zp[r]);
        au[r] = aw[r] = 0.0;
    }
    const int ntiles = (total + TE_TILE - 1) / TE_TILE;
    double nx, nz, ng;
    tree_fetch(G, A, sm, tid, total, nx, nz, ng);
    __syncthreads();                       // the previous pass has finished reading both buffers
    sm.sxz[0][tid] = make_double2(nx, nz);
    sm.sg[0][tid] = ng;
    __syncthreads();
    for (int k = 0; k < ntiles; k++) {
        const int buf = k & 1;
        if (k + 1 < ntiles) tree_fetch(G, A, sm, (k + 1) * TE_TILE + tid, total, nx, nz, ng);   // in flight during the tile
        const int len = min(TE_TILE, total - k * TE_TILE);
#pragma unroll 4
        for (int j = 0; j < len; j++) {
            const double2 s = sm.sxz[buf][j];
            const double gj = sm.sg[buf][j];
#pragma unroll
            for (int r = 0; r < R; r++) pair_fast(xp[r], zp[r], s.x, s.y, gj, vc4, au[r], aw[r]);
        }
        if (k + 1 < ntiles) {
            sm.sxz[buf ^ 1][tid] = make_double2(nx, nz);
            sm.sg[buf ^ 1][tid] = ng;
        }
        __syncthreads();
    }
#pragma unroll
    for (int r = 0; r < R; r++)
        if (t0 + tid + r * TE_THREADS < t1) T.store(t0 + tid + r * TE_THREADS, au[r], aw[r]);
}

// The item's targets [tb, te) are cut into row units of TE_THREADS, and the units into passes of <= 4 (rows per thread) as
// evenly as possible; passes are spread over blockIdx.y so that an item is several CTAs (wave quantisation).
template <class Tgt>
__device__ __forceinline__ void tree_eval_item(const TreeGeom &G, const TreeEval &A, const Tgt &T, TreeSmem &sm, int tb, int te,
                                               int total)
{
    const int units = (te - tb + TE_THREADS - 1) / TE_THREADS, npass = (units + 3) >> 2;
    const int base = units / npass, extra = units - base * npass;
    for (int pass = blockIdx.y; pass < npass; pass += gridDim.y) {
        const int R = base + (pass < extra ? 1 : 0);
        const int t0 = tb + (pass * base + min(pass, extra)) * TE_THREADS, t1 = min(te, t0 + R * TE_THREADS);
        if (total == 0) {
            for (int t = t0 + threadIdx.x; t < t1; t += TE_THREADS) T.store(t, 0.0, 0.0);
        } else if (R == 1) tree_eval_rows<1>(G, A, T, sm, t0, t1, total);
        else if (R == 2) tree_eval_rows<2>(G, A, T, sm, t0, t1, total);
        else if (R == 3) tree_eval_rows<3>(G, A, T, sm, t0, t1, total);
        else tree_eval_rows<4>(G, A, T, sm, t0, t1, total);
    }
}

// Does cell c of level l carry a local field?  More than P2 sources -- or, for grid targets of known density, more than P2
// grid points.  Both are independent of which targets a rank was given, and both hold for the parent when they hold for a child.
__device__ __forceinline__ bool tree_has_local(const TreeGeom &G, const int *startS, int l, long c)
{
    const int sh = 2 * (G.L - l);
    if (startS[(c + 1) << sh] - startS[c << sh] > G.pth) return true;
    const double a = ldexp(G.side, -l);
    return G.tdens * a * a > (double)G.P2;
}
// deepest level whose ancestor of leaf c carries a local field, or 1
__device__ __forceinline__ int tree_local_level(const TreeGeom &G, const int *startS, int c)
{
    for (int l = G.L; l >= 2; l--)
        if (tree_has_local(G, startS, l, (long)(c >> (2 * (G.L - l))))) return l;
    return 1;
}

__global__ void __launch_bounds__(TE_THREADS, 4) k_tree_eval(const __grid_constant__ TreeGeom G, const __grid_constant__ TreeEval A)
{
    __shared__ __align__(16) TreeSmem sm;
    const int L = G.L, P2 = G.P2;
    const int nm2l = (int)level_offset(L + 1);
    if ((int)blockIdx.x < nm2l) {
        // M2L item: cell c of level l
        int l = 2;
        while (level_offset(l + 1) <= (long)blockIdx.x) l++;
        const int c = (int)(blockIdx.x - level_offset(l)), sh = 2 * (L - l);
        if (!tree_has_local(G, A.startS, l, c)) return;                                   // no local field here
        if (A.startT[((long)c + 1) << sh] == A.startT[(long)c << sh]) return;           // none of this rank's targets below
        if ((int)blockIdx.y >= (((P2 + TE_THREADS - 1) / TE_THREADS + 3) >> 2)) return;
        const int cx = (int)compact16((unsigned)c), cz = (int)compact16((unsigned)c >> 1);
        const int total = tree_build_list(G, A, cx, cz, l, false, l, l, sm, true);   // proxy cells: k_tree_m2l_dmma
        const double h = ldexp(G.side, -(l + 1));
        const long off = (level_offset(l) + c) * P2;
        TgtNodePts T{G.x0 + (2.0 * cx + 1.0) * h, G.z0 + (2.0 * cz + 1.0) * h, h, G.s, G.P1, A.uloc + off, A.wloc + off};
        if (threadIdx.x == 0 && blockIdx.y == 0 && A.pairs) atomicAdd(A.pairs, (unsigned long long)P2 * (unsigned long long)total);
        tree_eval_item(G, A, T, sm, 0, P2, total);
        return;
    }
    const int c = (int)blockIdx.x - nm2l;
    const int tb = A.startT[c], te = A.startT[c + 1];
    if (tb == te) return;
    if ((int)blockIdx.y >= (((te - tb + TE_THREADS - 1) / TE_THREADS + 3) >> 2)) return;
    const int lstar = tree_local_level(G, A.startS, c);
    const int total = tree_build_list(G, A, (int)compact16((unsigned)c), (int)compact16((unsigned)c >> 1), L, true, lstar + 1, L, sm);
    if (threadIdx.x == 0 && blockIdx.y == 0 && A.pairs) atomicAdd(A.pairs, (unsigned long long)(te - tb) * (unsigned long long)total);
    TgtLeafPts T{A.permT, A.xt, A.zt, A.u, A.w};
    tree_eval_item(G, A, T, sm, tb, te, total);
}

// ---------------------------------------------------------------------------------------------------
// M2L between proxy cells as matrix products.  The proxies of a cell sit at fixed points of the cell, so the velocity
// that the P2 proxies of cell B induce at the P2 points of cell A of the same level depends on the cells' offset
// (dx, dz) in [-3, 3]^2 only: U_A += Mu[l][off] q_B, W_A += Mw[l][off] q_B with two P2 x P2 matrices per level and offset
// (per level: the core radius does not scale with the cells).  An entry costs one FMA per component instead of the 13
// slots + MUFU of a pair evaluation, and a matrix is shared by every pair of cells with that offset.  k_tree_m2l_mats
// builds the matrices; k_tree_m2l_dmma applies them on the FP64 tensor cores, a CTA per (points) x (cells) tile of the
// local fields of one level, walking the 40 offsets and the P2 proxies.  List entries that are plain vortices (cells
// with <= pth of them) stay with k_tree_eval.  The order of the sums is fixed (offsets, then proxies, ascending),
// whatever tile a cell lands in.  Measurements: DESIGN.md 4b.
// ---------------------------------------------------------------------------------------------------
#define TM_NOFF 49

// matrices [level - 2][off][j][i], i fastest
__global__ void __launch_bounds__(128) k_tree_m2l_mats(const __grid_constant__ TreeGeom G, double *Mu, double *Mw)
{
    const int j = blockIdx.x, off = blockIdx.y, l = 2 + blockIdx.z, P1 = G.P1, P2 = G.P2;
    const int dx = off % 7 - 3, dz = off / 7 - 3;
    if (max(abs(dx), abs(dz)) <= 1) return;
    const double h = ldexp(G.side, -(l + 1));
    const int j1 = j / P1, j2 = j - j1 * P1;
    const double xs = fma(h, G.s[j1], 2.0 * h * dx), zs = fma(h, G.s[j2], 2.0 * h * dz);   // relative to A's centre
    const size_t base = (((size_t)(l - 2) * TM_NOFF + off) * P2 + j) * P2;
    for (int i = threadIdx.x; i < P2; i += blockDim.x) {
        const int i1 = i / P1, i2 = i - i1 * P1;
        double u = 0.0, w = 0.0;
        pair_fast(h * G.s[i1], h * G.s[i2], xs, zs, 1.0, G.vc4, u, w);
        Mu[base + i] = u;
        Mw[base + i] = w;
    }
}

// Cells of every level that carry a local field and have targets of this rank beneath them, one list per level and per
// parity (ax & 1, az & 1) of the cell in its parent: cells of one parity share the 27 valid offsets of the 49, so a tile
// of them does no wasted products.  Any order inside a list: a cell's result does not depend on its neighbours in it.
__global__ void __launch_bounds__(256) k_tree_alist(const __grid_constant__ TreeGeom G, const int *startS, const int *startT,
                                                    int *alist, int *acount)
{
    const long b = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= level_offset(G.L + 1)) return;
    int l = 2;
    while (level_offset(l + 1) <= b) l++;
    const long c = b - level_offset(l);
    const int sh = 2 * (G.L - l);
    if (!tree_has_local(G, startS, l, c)) return;
    if (startT[(c + 1) << sh] == startT[c << sh]) return;
    const int par = (int)(c & 3);                                     // Morton: bit 0 = ax & 1, bit 1 = az & 1
    alist[level_offset(l) + ((long)par << (2 * (l - 1))) + atomicAdd(acount + 4 * l + par, 1)] = (int)c;
}

// The M2L products on the FP64 tensor cores (mma.sync.m8n8k4.f64; Blackwell's tcgen05 has no FP64 kind, so this is the
// FP64 tensor path of sm_100a).  CTA tile 64 points x 64 cells, 8 warps as 4 (points) x 2 (cells), warp tile 16 x 32 =
// 2 x 4 MMA tiles per component: per k-step of 4 proxies a thread reads 8 doubles of fragments for 16 MMAs (4096 FMA per
// warp), 0.5 bytes of shared memory per FMA where a register-tiled CUDA-core loop needs 4 and is bound by shared-memory
// bandwidth.  Fragment layout (PTX ISA, m8n8k4
// .f64): A[row = lane >> 2][k = lane & 3], B[k = lane & 3][col = lane >> 2], C[row = lane >> 2][col = 2 (lane & 3) + {0, 1}].
// Row strides of 68 doubles make the fragment loads conflict-free (stride = 4 mod 16 bank pairs).
#define TD_TI 64
#define TD_TC 64
#define TD_JC 16
#define TD_LD 68

__global__ void __launch_bounds__(256, 2) k_tree_m2l_dmma(const __grid_constant__ TreeGeom G, const int *startS, const int *alist,
                                                          const int *acount, const double *Mu, const double *Mw,
                                                          const double *qhat, double *uloc, double *wloc)
{
    const int P2 = G.P2, tid = threadIdx.x;
    int l = 2, tile = blockIdx.y, ntp;
    for (;; l++) {
        ntp = (int)(((1L << (2 * (l - 1))) + TD_TC - 1) / TD_TC);
        if (tile < 4 * ntp) break;
        tile -= 4 * ntp;
    }
    const int par = tile / ntp;
    tile -= par * ntp;
    const int nA = acount[4 * l + par];
    if (tile * TD_TC >= nA) return;
    const long abase = level_offset(l) + ((long)par << (2 * (l - 1)));
    const int i0 = blockIdx.x * TD_TI;
    __shared__ int Acell[TD_TC], Bcell[TD_TC];
    __shared__ __align__(16) double sMu[TD_JC][TD_LD], sMw[TD_JC][TD_LD], sQ[TD_JC][TD_LD];
    const int warp = tid >> 5, lane = tid & 31;
    const int iw = (warp & 3) * 16, cw = (warp >> 2) * 32;      // warp tile origin
    const int fr = lane >> 2, fk = lane & 3;                    // fragment row / k index of this lane
    double cu[2][4][2], cv[2][4][2];
#pragma unroll
    for (int a = 0; a < 2; a++)
#pragma unroll
        for (int b = 0; b < 4; b++) cu[a][b][0] = cu[a][b][1] = cv[a][b][0] = cv[a][b][1] = 0.0;
    if (tid < TD_TC) Acell[tid] = tile * TD_TC + tid < nA ? alist[abase + tile * TD_TC + tid] : -1;
    const double *Ml_u = Mu + (size_t)(l - 2) * TM_NOFF * P2 * P2, *Ml_w = Mw + (size_t)(l - 2) * TM_NOFF * P2 * P2;
    const double *ql = qhat + level_offset(l) * P2;
    const int sh = 2 * (G.L - l), nc = 1 << l;
    for (int off = 0; off < TM_NOFF; off++) {
        const int dx = off % 7 - 3, dz = off / 7 - 3;
        if (max(abs(dx), abs(dz)) <= 1) continue;
        if (dx < -2 - (par & 1) || dx > 3 - (par & 1) || dz < -2 - (par >> 1) || dz > 3 - (par >> 1)) continue;
        __syncthreads();
        if (tid < TD_TC) {
            int bcell = -1;
            const int a = Acell[tid];
            if (a >= 0) {
                const int ax = (int)compact16((unsigned)a), az = (int)compact16((unsigned)a >> 1), bx = ax + dx, bz = az + dz;
                if (bx >= 0 && bz >= 0 && bx < nc && bz < nc) {
                    const long bc = morton2(bx, bz);
                    if (startS[(bc + 1) << sh] - startS[bc << sh] > G.pth) bcell = (int)bc;
                }
            }
            Bcell[tid] = bcell;
        }
        if (!__syncthreads_or(tid < TD_TC && Bcell[tid] >= 0)) continue;
        const double *Mo_u = Ml_u + (size_t)off * P2 * P2, *Mo_w = Ml_w + (size_t)off * P2 * P2;
        double pmu[4], pmw[4], pq[4];     // TD_JC x 64 elements of each tile / 256 threads
        auto fetch = [&](int j0) {
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const int e = tid + 256 * q, jj = e >> 6, ii = e & 63, j = j0 + jj, i = i0 + ii;
                const bool ok = j < P2 && i < P2;
                pmu[q] = ok ? Mo_u[(size_t)j * P2 + i] : 0.0;
                pmw[q] = ok ? Mo_w[(size_t)j * P2 + i] : 0.0;
                const int cc = e / TD_JC, kj = e - cc * TD_JC, bcell = Bcell[cc];
                pq[q] = (bcell >= 0 && j0 + kj < P2) ? ql[(size_t)bcell * P2 + j0 + kj] : 0.0;
            }
        };
        auto put = [&]() {
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const int e = tid + 256 * q, jj = e >> 6, ii = e & 63;
                sMu[jj][ii] = pmu[q];
                sMw[jj][ii] = pmw[q];
                const int cc = e / TD_JC, kj = e - cc * TD_JC;
                sQ[kj][cc] = pq[q];
            }
        };
        fetch(0);
        for (int j0 = 0; j0 < P2; j0 += TD_JC) {
            __syncthreads();
            put();
            __syncthreads();
            if (j0 + TD_JC < P2) fetch(j0 + TD_JC);
#pragma unroll
            for (int k0 = 0; k0 < TD_JC; k0 += 4) {
                double a_u[2], a_w[2], b[4];
#pragma unroll
                for (int mt = 0; mt < 2; mt++) {
                    a_u[mt] = sMu[k0 + fk][iw + mt * 8 + fr];
                    a_w[mt] = sMw[k0 + fk][iw + mt * 8 + fr];
                }
#pragma unroll
                for (int nt = 0; nt < 4; nt++) b[nt] = sQ[k0 + fk][cw + nt * 8 + fr];
#pragma unroll
                for (int mt = 0; mt < 2; mt++)
#pragma unroll
                    for (int nt = 0; nt < 4; nt++) {
                        dmma_m8n8k4(cu[mt][nt][0], cu[mt][nt][1], a_u[mt], b[nt]);
                        dmma_m8n8k4(cv[mt][nt][0], cv[mt][nt][1], a_w[mt], b[nt]);
                    }
            }
        }
    }
    __syncthreads();
#pragma unroll
    for (int nt = 0; nt < 4; nt++)
#pragma unroll
        for (int e = 0; e < 2; e++) {
            const int a = Acell[cw + nt * 8 + 2 * fk + e];
            if (a < 0) continue;
            const size_t o = (size_t)(level_offset(l) + a) * P2;
#pragma unroll
            for (int mt = 0; mt < 2; mt++) {
                const int i = i0 + iw + mt * 8 + fr;
                if (i < P2) {
                    uloc[o + i] += cu[mt][nt][e];
                    wloc[o + i] += cv[mt][nt][e];
                }
            }
        }
}

// L2L: the parent's local field interpolated to the points of child cell c of level l (l >= 3), added to the child's M2L sums
__global__ void __launch_bounds__(256) k_tree_l2l(const __grid_constant__ TreeGeom G, int l, const int *startS, const int *startT,
                                                  double *uloc, double *wloc)
{
    const int c = blockIdx.x, sh = 2 * (G.L - l), tid = threadIdx.x, P1 = G.P1, P2 = G.P2;
    if (!tree_has_local(G, startS, l, c)) return;
    if (startT[((long)c + 1) << sh] == startT[(long)c << sh]) return;
    __shared__ double Up[TR_MAX_P1 * TR_MAX_P1], Wp[TR_MAX_P1 * TR_MAX_P1], Tu[TR_MAX_P1 * TR_MAX_P1], Tw[TR_MAX_P1 * TR_MAX_P1];
    __shared__ double Bx[TR_MAX_P1][TR_MAX_P1], Bz[TR_MAX_P1][TR_MAX_P1];
    const long poff = (level_offset(l - 1) + (c >> 2)) * P2, coff = (level_offset(l) + c) * P2;
    const int ch = c & 3;
    for (int k = tid; k < P2; k += 256) {
        Up[k] = uloc[poff + k];
        Wp[k] = wloc[poff + k];
    }
    if (tid < 2 * P1) {
        const int k = tid >> 1, dim = tid & 1;
        const double xi = (G.s[k] + (double)(dim ? (ch >> 1) * 2 - 1 : (ch & 1) * 2 - 1)) * 0.5;
        tree_basis(G, xi, dim ? Bz[k] : Bx[k]);
    }
    __syncthreads();
    for (int idx = tid; idx < P2; idx += 256) {      // T[m1][k2] = sum_m2 Bz[k2][m2] U[m1][m2]
        const int m1 = idx / P1, k2 = idx - m1 * P1;
        double a = 0.0, b = 0.0;
        for (int m2 = 0; m2 < P1; m2++) {
            a = fma(Bz[k2][m2], Up[m1 * P1 + m2], a);
            b = fma(Bz[k2][m2], Wp[m1 * P1 + m2], b);
        }
        Tu[idx] = a;
        Tw[idx] = b;
    }
    __syncthreads();
    for (int idx = tid; idx < P2; idx += 256) {      // child[k1][k2] += sum_m1 Bx[k1][m1] T[m1][k2]
        const int k1 = idx / P1, k2 = idx - k1 * P1;
        double a = 0.0, b = 0.0;
        for (int m1 = 0; m1 < P1; m1++) {
            a = fma(Bx[k1][m1], Tu[m1 * P1 + k2], a);
            b = fma(Bx[k1][m1], Tw[m1 * P1 + k2], b);
        }
        uloc[coff + idx] += a;
        wloc[coff + idx] += b;
    }
}

// L2P: every target adds the local field of its deepest ancestor that carries one, interpolated at the target
__global__ void __launch_bounds__(128) k_tree_l2p(const __grid_constant__ TreeGeom G, const __grid_constant__ TreeEval A)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= A.np) return;
    const int oi = A.permT[t], c = A.keyT[oi];
    const int l = tree_local_level(G, A.startS, c);
    if (l < 2) return;
    const int a = c >> (2 * (G.L - l)), P1 = G.P1;
    const double h = ldexp(G.side, -(l + 1)), inv_h = 1.0 / h;
    const double cx = G.x0 + (2.0 * compact16((unsigned)a) + 1.0) * h, cz = G.z0 + (2.0 * compact16((unsigned)a >> 1) + 1.0) * h;
    double bx[TR_MAX_P1], bz[TR_MAX_P1];
    tree_basis(G, (A.xt[oi] - cx) * inv_h, bx);
    tree_basis(G, (A.zt[oi] - cz) * inv_h, bz);
    const double *U = A.uloc + (level_offset(l) + a) * G.P2, *W = A.wloc + (level_offset(l) + a) * G.P2;
    double su = 0.0, sw = 0.0;
    for (int k1 = 0; k1 < P1; k1++) {
        double tu = 0.0, tw = 0.0;
        for (int k2 = 0; k2 < P1; k2++) {
            tu = fma(bz[k2], U[k1 * P1 + k2], tu);
            tw = fma(bz[k2], W[k1 * P1 + k2], tw);
        }
        su = fma(bx[k1], tu, su);
        sw = fma(bx[k1], tw, sw);
    }
    A.u[oi] += su;
    A.w[oi] += sw;
}

// L2P on the FP64 tensor cores (orders <= 19).  The scalar kernel above reads the cell's 2 P2 field values once PER TARGET
// (two loads per multiply-add, ~5 ms for the 16.7M points of a 4096^2 grid); here a warp takes 8 targets of one leaf at a
// time and the field sits in its registers as MMA B-fragments, loaded once per leaf:
//     D[target][k1] = sum_k2 lz_k2(zeta_target) U[k1][k2]            (15 MMAs per component: k2 in 5 steps of 4, k1 in 3 tiles of 8)
//     u_target     = sum_k1 lx_k1(xi_target) D[target][k1]          (each lane its 6 columns, then a 4-lane shuffle sum)
// The barycentric bases are computed in the fragment layouts directly (the 4 lanes of a target share the normalisation).
#define L2P_KS 5
#define L2P_NT 3
__global__ void __launch_bounds__(128) k_tree_l2p_mma(const __grid_constant__ TreeGeom G, const __grid_constant__ TreeEval A)
{
    const int c = blockIdx.x;                                   // target leaf
    const int tb = A.startT[c], te = A.startT[c + 1];
    if (tb == te) return;
    const int l = tree_local_level(G, A.startS, c);
    if (l < 2) return;
    const int a = c >> (2 * (G.L - l)), P1 = G.P1;
    const double h = ldexp(G.side, -(l + 1)), inv_h = 1.0 / h;
    const double cx = G.x0 + (2.0 * compact16((unsigned)a) + 1.0) * h, cz = G.z0 + (2.0 * compact16((unsigned)a >> 1) + 1.0) * h;
    const double *U = A.uloc + (level_offset(l) + a) * G.P2, *W = A.wloc + (level_offset(l) + a) * G.P2;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, fr = lane >> 2, fk = lane & 3;
    // B fragments: B[k2][k1] = U[k1][k2], this lane holds row k2 = fk + 4 s, column k1 = fr + 8 nt
    double bu[L2P_KS][L2P_NT], bw[L2P_KS][L2P_NT];
#pragma unroll
    for (int s = 0; s < L2P_KS; s++)
#pragma unroll
        for (int nt = 0; nt < L2P_NT; nt++) {
            const int k2 = fk + 4 * s, k1 = fr + 8 * nt;
            const bool ok = k1 < P1 && k2 < P1;
            bu[s][nt] = ok ? U[k1 * P1 + k2] : 0.0;
            bw[s][nt] = ok ? W[k1 * P1 + k2] : 0.0;
        }
    for (int t0 = tb + 8 * warp; t0 < te; t0 += 8 * (blockDim.x >> 5)) {
        const int t = t0 + fr;
        const bool valid = t < te;
        const int oi = A.permT[valid ? t : te - 1];
        const double xi = (A.xt[oi] - cx) * inv_h, ze = (A.zt[oi] - cz) * inv_h;
        // bases in fragment layout: lz at k2 = fk + 4 s (A fragment), lx at k1 = 8 nt + 2 fk + e (D fragment columns)
        double az[L2P_KS], ax[L2P_NT][2];
        double sz = 0.0, sx = 0.0;
        int hz = -1, hx = -1;
#pragma unroll
        for (int s = 0; s < L2P_KS; s++) {
            const int k = fk + 4 * s;
            az[s] = 0.0;
            if (k < P1) {
                double d = ze - G.s[k];
                if (d == 0.0) { hz = k; d = 1.0; }
                az[s] = G.bw[k] / d;
                sz += az[s];
            }
        }
#pragma unroll
        for (int nt = 0; nt < L2P_NT; nt++)
#pragma unroll
            for (int e = 0; e < 2; e++) {
                const int k = 8 * nt + 2 * fk + e;
                ax[nt][e] = 0.0;
                if (k < P1) {
                    double d = xi - G.s[k];
                    if (d == 0.0) { hx = k; d = 1.0; }
                    ax[nt][e] = G.bw[k] / d;
                    sx += ax[nt][e];
                }
            }
        sz += __shfl_xor_sync(~0u, sz, 1); sz += __shfl_xor_sync(~0u, sz, 2);     // the 4 lanes of a target
        sx += __shfl_xor_sync(~0u, sx, 1); sx += __shfl_xor_sync(~0u, sx, 2);
        hz = max(hz, __shfl_xor_sync(~0u, hz, 1)); hz = max(hz, __shfl_xor_sync(~0u, hz, 2));
        hx = max(hx, __shfl_xor_sync(~0u, hx, 1)); hx = max(hx, __shfl_xor_sync(~0u, hx, 2));
        const double iz = 1.0 / sz, ix = 1.0 / sx;
#pragma unroll
        for (int s = 0; s < L2P_KS; s++) az[s] = hz >= 0 ? (fk + 4 * s == hz ? 1.0 : 0.0) : az[s] * iz;
#pragma unroll
        for (int nt = 0; nt < L2P_NT; nt++)
#pragma unroll
            for (int e = 0; e < 2; e++) ax[nt][e] = hx >= 0 ? (8 * nt + 2 * fk + e == hx ? 1.0 : 0.0) : ax[nt][e] * ix;
        double du[L2P_NT][2], dw[L2P_NT][2];
#pragma unroll
        for (int nt = 0; nt < L2P_NT; nt++) du[nt][0] = du[nt][1] = dw[nt][0] = dw[nt][1] = 0.0;
#pragma unroll
        for (int s = 0; s < L2P_KS; s++)
#pragma unroll
            for (int nt = 0; nt < L2P_NT; nt++) {
                dmma_m8n8k4(du[nt][0], du[nt][1], az[s], bu[s][nt]);
                dmma_m8n8k4(dw[nt][0], dw[nt][1], az[s], bw[s][nt]);
            }
        double su = 0.0, sw = 0.0;
#pragma unroll
        for (int nt = 0; nt < L2P_NT; nt++)
#pragma unroll
            for (int e = 0; e < 2; e++) {
                su = fma(ax[nt][e], du[nt][e], su);
                sw = fma(ax[nt][e], dw[nt][e], sw);
            }
        su += __shfl_xor_sync(~0u, su, 1); su += __shfl_xor_sync(~0u, su, 2);
        sw += __shfl_xor_sync(~0u, sw, 1); sw += __shfl_xor_sync(~0u, sw, 2);
        if (valid && fk == 0) {
            A.u[oi] += su;
            A.w[oi] += sw;
        }
    }
}

__global__ void __launch_bounds__(256) k_tree_euler(const double *x, const double *z, const double *u, const double *w, double dt,
                                                    int n, double *xo, double *zo)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    xo[i] = __dadd_rn(x[i], __dmul_rn(dt, u[i]));   // forward Euler, LUDVM.py:1108-1127
    zo[i] = __dadd_rn(z[i], __dmul_rn(dt, w[i]));
}

// ---------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------
struct TreeBufs {
    int *keyS, *slotS, *keyT, *slotT, *cntS, *cntT, *startS, *startT, *tmpS, *permS, *tmpT, *permT;
    double *xs, *zs, *gs, *qhat, *uloc, *wloc;
    double *Mu, *Mw;   // M2L matrices [L - 1][TM_NOFF][P2][P2]
    int *alist, *acount;
    unsigned long long *pairs;
    int *maxcnt;   // [2]: largest leaf population, sources / targets
};
static size_t tree_layout(Arena &a, TreeBufs &b, long nw, long np, int L, int P2)
{
    const size_t ncell = (size_t)1 << (2 * L);
    b.keyS = a.take<int>(nw); b.slotS = a.take<int>(nw); b.keyT = a.take<int>(np); b.slotT = a.take<int>(np);
    b.cntS = a.take<int>(ncell + 1); b.cntT = a.take<int>(ncell + 1);
    b.startS = a.take<int>(ncell + 1); b.startT = a.take<int>(ncell + 1);
    b.tmpS = a.take<int>(nw); b.permS = a.take<int>(nw); b.tmpT = a.take<int>(np); b.permT = a.take<int>(np);
    b.xs = a.take<double>(nw); b.zs = a.take<double>(nw); b.gs = a.take<double>(nw);
    b.qhat = a.take<double>((size_t)level_offset(L + 1) * P2);
    b.uloc = a.take<double>((size_t)level_offset(L + 1) * P2);
    b.wloc = a.take<double>((size_t)level_offset(L + 1) * P2);
    b.Mu = a.take<double>((size_t)(L - 1) * TM_NOFF * P2 * P2);
    b.Mw = a.take<double>((size_t)(L - 1) * TM_NOFF * P2 * P2);
    b.alist = a.take<int>((size_t)level_offset(L + 1));
    b.acount = a.take<int>(64);
    b.pairs = a.take<unsigned long long>(1);
    b.maxcnt = a.take<int>(2);
    return a.off;
}

int tree_velocity_device(ludvm_ctx *ctx, cudaStream_t st, const double *g, const double *xw, const double *zw, double vc4,
                         long nw, const double *xp, const double *zp, long np_, int order, int leaf, double *u, double *w,
                         double *stats, double tdens, const double *box_x, const double *box_z, int nbox)
{
    // (box_x, box_z)[nbox]: points that span the targets' bounding box, used for it in place of the targets themselves --
    // a slab of a grid passes the full grid's corners, so that every slab builds the tree of the full grid
    if (order <= 0) order = 18;
    if (order < 2 || order > TR_MAX_ORDER) return set_error(LUDVM_E_ARG, "tree order %d outside 2..%d", order, TR_MAX_ORDER);
    void *p;
    int rc;
    if ((rc = scratch_reserve(ctx, SLOT_TREE_COUNTERS, 256, &p))) return rc;
    unsigned long long *mm = (unsigned long long *)p;
    {
        unsigned long long init[8] = {~0ull, 0, ~0ull, 0, ~0ull, 0, ~0ull, 0};
        CUDA_TRY(cudaMemcpyAsync(mm, init, sizeof(init), cudaMemcpyHostToDevice, st));
        const int blocks = (int)std::min<long>((nw + np_ + 1023) / 1024, (long)ctx->sm_count * 8);
        if (nbox > 0) k_tree_bbox<<<blocks, 256, 0, st>>>(xw, zw, (int)nw, box_x, box_z, nbox, mm);
        else k_tree_bbox<<<blocks, 256, 0, st>>>(xw, zw, (int)nw, xp, zp, (int)np_, mm);
        ctx->launches++;
        unsigned long long out[8];
        CUDA_TRY(cudaMemcpyAsync(out, mm, sizeof(out), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        for (int k = 0; k < 8; k += 2)
            if (out[k] > out[k + 1]) return set_error(LUDVM_E_ARG, "tree: no finite coordinates");
        TreeGeom G = {};
        const double xlo = dkey_inv(out[0]), xhi = dkey_inv(out[1]), zlo = dkey_inv(out[2]), zhi = dkey_inv(out[3]);
        const double sxl = dkey_inv(out[4]), sxh = dkey_inv(out[5]), szl = dkey_inv(out[6]), szh = dkey_inv(out[7]);
        double side = std::max(xhi - xlo, zhi - zlo);
        side = side * (1.0 + 1e-12) + 1e-300;
        if (!(side < 1e300)) return set_error(LUDVM_E_ARG, "tree: coordinates not finite");
        // leaf level from the wanted mean leaf population over the sources' own bounding box.  Per target a leaf costs
        // 9 x population pair evaluations and (27 x P2^2 / population) tensor-core FMA: the default population is P2
        // (the depth is an integer, so the actual population lands between P2 / 2 and 2 P2).
        const int P1 = order + 1, P2 = P1 * P1;
        // (dense grid targets: the near field is what is left per target, so small leaves; M2L does not grow with them)
        const double pop = leaf > 0 ? (double)leaf : (tdens > 0.0 ? 64.0 : 1.0 * P2);
        const double area = std::max((sxh - sxl) * (szh - szl), side * side * 1e-12);
        const double a0 = std::sqrt(pop * area / (double)std::max(1L, nw));
        int L = (int)std::lround(std::log2(std::max(side / a0, 1.0)));
        int lcap = 2;                                    // no more than ~16 leaf cells per source vortex
        while (lcap < TR_MAX_LEVEL && (1L << (2 * (lcap - 1))) < nw) lcap++;
        L = std::max(2, std::min(std::min(TR_MAX_LEVEL, lcap), L));
        if (const char *le = getenv("LUDVM_TREE_LEVEL")) L = std::max(2, std::min(TR_MAX_LEVEL, atoi(le)));
        G.x0 = xlo; G.z0 = zlo; G.side = side; G.inv_leaf = (double)(1 << L) / side; G.vc4 = vc4; G.tdens = tdens;
        // proxies (and a local field) from a quarter of P2 vortices on: with M2L on the tensor cores a proxy-to-proxy
        // interaction is ~10x cheaper than a pair evaluation, so a cell is worth representing by more proxies than it
        // has vortices (order 14, 2^20 vortices: 7.7 -> 5.7 ms with leaves of 160; profiles/r03q_tree_probe_pth.txt)
        G.pth = std::max(1, P2 / 4);
        G.L = L; G.P1 = P1; G.P2 = P2;
        for (int k = 0; k < P1; k++) {
            G.s[k] = std::sin(M_PI * (double)(order - 2 * k) / (double)(2 * order));
            G.bw[k] = ((k & 1) ? -1.0 : 1.0) * ((k == 0 || k == order) ? 0.5 : 1.0);
        }
        if ((order & 1) == 0) G.s[order / 2] = 0.0;
        for (int k = 0; k < P1 / 2; k++) G.s[order - k] = -G.s[k];

        Arena sizer;
        TreeBufs B;
        const size_t bytes = tree_layout(sizer, B, nw, np_, L, P2);
        if ((rc = scratch_reserve(ctx, SLOT_TREE_ARENA, bytes, &p))) return rc;
        Arena ar{(char *)p};
        tree_layout(ar, B, nw, np_, L, P2);
        const int ncell = 1 << (2 * L);
        CUDA_TRY(cudaMemsetAsync(B.cntS, 0, (size_t)(ncell + 1) * sizeof(int), st));
        CUDA_TRY(cudaMemsetAsync(B.cntT, 0, (size_t)(ncell + 1) * sizeof(int), st));
        CUDA_TRY(cudaMemsetAsync(B.pairs, 0, sizeof(unsigned long long), st));
        const int sort_blocks = std::min(ceil_div(ncell, 8), ctx->sm_count * 16);
        const int big_blocks = std::min(ncell, ctx->sm_count * 32);
        cudaEvent_t ev0 = nullptr;
        if (stats) {
            CUDA_TRY(cudaEventCreate(&ev0));
            CUDA_TRY(cudaEventRecord(ev0, st));
        }
        // targets == sources (the self-convection step of the whole cloud): one sort serves both
        const bool same = xp == xw && zp == zw && np_ == nw;
        if (same) { B.keyT = B.keyS; B.startT = B.startS; B.permT = B.permS; }
        CUDA_TRY(cudaMemsetAsync(B.maxcnt, 0, 2 * sizeof(int), st));
        k_tree_keys<<<ceil_div(nw, 256), 256, 0, st>>>(G, xw, zw, (int)nw, B.keyS, B.slotS, B.cntS);
        k_tree_scan<<<1, 1024, 0, st>>>(B.cntS, B.startS, ncell, B.maxcnt);
        ctx->launches += 2;
        if (!same) {
            k_tree_keys<<<ceil_div(np_, 256), 256, 0, st>>>(G, xp, zp, (int)np_, B.keyT, B.slotT, B.cntT);
            k_tree_scan<<<1, 1024, 0, st>>>(B.cntT, B.startT, ncell, B.maxcnt + 1);
            ctx->launches += 2;
        }
        // The sources of a cell are ordered by counting (O(population^2) per cell): a leaf of the deepest allowed tree that
        // still holds this many vortices means the cloud is far too clustered for a uniform-depth tree, and the
        // all-pairs kernels are the right tool.
        int maxcnt[2] = {0, 0};
        CUDA_TRY(cudaMemcpyAsync(maxcnt, B.maxcnt, sizeof(maxcnt), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        if (same) maxcnt[1] = maxcnt[0];
        if (maxcnt[0] > TR_MAX_LEAF_POP)
            return set_error(LUDVM_E_UNSUPPORTED, "tree: a leaf cell of level %d holds %d vortices (limit %d): the cloud is too "
                             "clustered for the uniform-depth tree, use the all-pairs modes", L, maxcnt[0], TR_MAX_LEAF_POP);
        k_tree_place<<<ceil_div(nw, 256), 256, 0, st>>>(B.keyS, B.slotS, B.startS, (int)nw, B.tmpS);
        k_tree_cellsort<<<sort_blocks, 256, 0, st>>>(B.tmpS, B.startS, ncell, B.permS);
        if (maxcnt[0] > TR_SORT_WARP_MAX) k_tree_cellsort_big<<<big_blocks, 256, 0, st>>>(B.tmpS, B.startS, ncell, B.permS);
        k_tree_gather<<<ceil_div(nw, 256), 256, 0, st>>>(B.permS, xw, zw, g, (int)nw, B.xs, B.zs, B.gs);
        ctx->launches += 3 + (maxcnt[0] > TR_SORT_WARP_MAX ? 1 : 0);
        if (!same) {   // targets: any order inside a cell will do (a target's sum does not involve the other targets)
            k_tree_place<<<ceil_div(np_, 256), 256, 0, st>>>(B.keyT, B.slotT, B.startT, (int)np_, B.permT);
            ctx->launches++;
        }
        for (int l = L; l >= 2; l--) {
            if (l == L && P1 <= 24) k_tree_up_leaf_mma<<<ncell, 128, 0, st>>>(G, B.startS, B.xs, B.zs, B.gs, B.qhat);
            else k_tree_up<<<1 << (2 * l), TU_THREADS, 0, st>>>(G, l, B.startS, B.xs, B.zs, B.gs, B.qhat);
            ctx->launches++;
        }
        TreeEval A = {B.startS, B.startT, B.permT, B.keyT, B.xs, B.zs, B.gs, B.qhat, xp, zp, u, w, B.uloc, B.wloc, B.pairs,
                      (int)np_};
        cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
        if (stats) {
            for (int k = 1; k < 3; k++) CUDA_TRY(cudaEventCreate(&ev[k]));
            CUDA_TRY(cudaEventRecord(ev[1], st));
        }
        // passes of <= 512 targets of one leaf are spread over blockIdx.y: enough of it for the most crowded leaf
        const long items = (long)ncell + level_offset(L + 1);
        int ysplit = std::max(4, (maxcnt[1] + 4 * TE_THREADS - 1) / (4 * TE_THREADS));
        ysplit = (int)std::max(1L, std::min<long>(ysplit, (1L << 24) / items));
        k_tree_eval<<<dim3((unsigned)items, ysplit), TE_THREADS, 0, st>>>(G, A);
        ctx->launches++;
        CUDA_TRY(cudaMemsetAsync(B.acount, 0, 64 * sizeof(int), st));
        k_tree_m2l_mats<<<dim3(P2, TM_NOFF, L - 1), 128, 0, st>>>(G, B.Mu, B.Mw);
        k_tree_alist<<<ceil_div(level_offset(L + 1), 256), 256, 0, st>>>(G, B.startS, B.startT, B.alist, B.acount);
        long tiles = 0;
        for (int l = 2; l <= L; l++) tiles += 4 * (((1L << (2 * (l - 1))) + TD_TC - 1) / TD_TC);
        k_tree_m2l_dmma<<<dim3((P2 + TD_TI - 1) / TD_TI, (unsigned)tiles), 256, 0, st>>>(G, B.startS, B.alist, B.acount, B.Mu, B.Mw,
                                                                                       B.qhat, B.uloc, B.wloc);
        ctx->launches += 3;
        for (int l = 3; l <= L; l++) {
            k_tree_l2l<<<1 << (2 * l), 256, 0, st>>>(G, l, B.startS, B.startT, B.uloc, B.wloc);
            ctx->launches++;
        }
        if (P1 <= 4 * L2P_KS) k_tree_l2p_mma<<<ncell, 128, 0, st>>>(G, A);
        else k_tree_l2p<<<ceil_div(np_, 128), 128, 0, st>>>(G, A);
        ctx->launches++;
        if (stats) CUDA_TRY(cudaEventRecord(ev[2], st));
        CUDA_TRY(cudaGetLastError());
        ctx->plan[0] = LUDVM_K_TREE; ctx->plan[1] = 4; ctx->plan[2] = L; ctx->plan[3] = 0; ctx->plan[4] = 1;
        ctx->plan[5] = order; ctx->plan[6] = TE_THREADS / 32; ctx->plan[7] = 1;
        if (stats) {
            unsigned long long pairs = 0;
            CUDA_TRY(cudaMemcpyAsync(&pairs, B.pairs, sizeof(pairs), cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaStreamSynchronize(st));
            stats[0] = L; stats[1] = side / (double)(1 << L); stats[2] = (double)pairs; stats[3] = (double)np_ * (double)nw;
            stats[4] = P2; stats[5] = (double)bytes;
            float ms_build = 0.f, ms_eval = 0.f;
            cudaEventElapsedTime(&ms_build, ev0, ev[1]);
            cudaEventElapsedTime(&ms_eval, ev[1], ev[2]);
            stats[6] = ms_build; stats[7] = ms_eval;
            cudaEventDestroy(ev0);
            for (auto &e : ev) if (e) cudaEventDestroy(e);
        }
    }
    return LUDVM_OK;
}

}  // namespace ludvm

using namespace ludvm;

LUDVM_API int ludvm_induced_velocity_tree(ludvm_ctx *ctx, const double *gamma, const double *xw, const double *zw, double vc4,
                                          long nw, const double *xp, const double *zp, long np_, int order, int leaf,
                                          double *u, double *w, int ptr_kind, double *stats)
{
    ARG_CHECK(ctx != nullptr);
    ARG_CHECK(nw >= 0 && np_ >= 0 && nw < (1L << 30) && np_ < (1L << 30));
    ARG_CHECK(ptr_kind == LUDVM_PTR_HOST || ptr_kind == LUDVM_PTR_DEVICE);
    ARG_CHECK(vc4 >= 0.0);
    if (np_ == 0) return LUDVM_OK;
    ARG_CHECK(u && w && xp && zp);
    ARG_CHECK(nw == 0 || (gamma && xw && zw));
    DeviceGuard g(ctx->device);
    int rc;
    const bool host = ptr_kind == LUDVM_PTR_HOST;
    const double *dg = gamma, *dxw = xw, *dzw = zw, *dxp = xp, *dzp = zp;
    double *du = u, *dw = w;
    if (host && ((rc = stage_in(ctx, {{gamma, nw, &dg}, {xw, nw, &dxw}, {zw, nw, &dzw}, {xp, np_, &dxp}, {zp, np_, &dzp}})) ||
                 (rc = stage_out(ctx, {{u, np_, &du}, {w, np_, &dw}}))))
        return rc;
    if (nw == 0) {
        CUDA_TRY(cudaMemsetAsync(du, 0, (size_t)np_ * sizeof(double), ctx->stream));
        CUDA_TRY(cudaMemsetAsync(dw, 0, (size_t)np_ * sizeof(double), ctx->stream));
        if (stats) memset(stats, 0, 8 * sizeof(double));
    } else if ((rc = tree_velocity_device(ctx, ctx->stream, dg, dxw, dzw, vc4, nw, dxp, dzp, np_, order, leaf, du, dw, stats))) {
        return rc;
    }
    return host ? copy_back(ctx, {{u, np_, &du}, {w, np_, &dw}}) : LUDVM_OK;
}

LUDVM_API int ludvm_selfconv_step_tree(ludvm_ctx *ctx, const double *gamma, const double *x, const double *z, double vc4, long n,
                                       long row0, long nrows, double dt, int order, int leaf, double *x_out, double *z_out,
                                       double *u_out, double *w_out, double *stats)
{
    ARG_CHECK(ctx != nullptr);
    ARG_CHECK(n > 0 && n < (1L << 30) && row0 >= 0 && nrows >= 0 && row0 + nrows <= n);
    ARG_CHECK(gamma && x && z && x_out && z_out && vc4 >= 0.0);
    if (nrows == 0) return LUDVM_OK;
    DeviceGuard g(ctx->device);
    int rc;
    double *du = u_out, *dw = w_out;
    if (!du || !dw) {
        void *o;
        if ((rc = scratch_reserve(ctx, SLOT_OUT, 2 * (size_t)nrows * sizeof(double), &o))) return rc;
        du = (double *)o;
        dw = du + nrows;
    }
    if ((rc = tree_velocity_device(ctx, ctx->stream, gamma, x, z, vc4, n, x + row0, z + row0, nrows, order, leaf, du, dw, stats))) return rc;
    k_tree_euler<<<ceil_div(nrows, 256), 256, 0, ctx->stream>>>(x + row0, z + row0, du, dw, dt, (int)nrows, x_out + row0,
                                                                z_out + row0);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return LUDVM_OK;
}

namespace ludvm {
// the 'ij' mesh rows [row0, row0 + nrows) of x1 x z1 as explicit target arrays
__global__ void __launch_bounds__(256) k_tree_grid_points(const double *x1, int nx, const double *z1, int nz, int row0, long npts,
                                                          double *xp, double *zp, double *box)
{
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) {   // corners of the FULL grid: box[0..1] = x, box[2..3] = z
        box[0] = x1[0]; box[1] = x1[nx - 1]; box[2] = z1[0]; box[3] = z1[nz - 1];
    }
    if (i >= npts) return;
    const int r = (int)(i / nz), j = (int)(i - (long)r * nz);
    xp[i] = x1[row0 + r];
    zp[i] = z1[j];
}
}  // namespace ludvm

LUDVM_API int ludvm_flowfield_velocity_tree(ludvm_ctx *ctx, const double *ga, const double *xa, const double *za, long na, double vc4,
                                            const double *x1, long nx, const double *z1, long nz, long row0, long nrows,
                                            double tgt_density, int order, int leaf, double *u, double *w, int ptr_kind,
                                            double *stats)
{
    ARG_CHECK(ctx != nullptr);
    ARG_CHECK(na > 0 && nx > 0 && nz > 0 && row0 >= 0 && nrows >= 0 && row0 + nrows <= nx);
    ARG_CHECK(na < (1L << 30) && nrows * nz < (1L << 30) && vc4 >= 0.0 && tgt_density >= 0.0);
    ARG_CHECK(ga && xa && za && x1 && z1 && u && w);
    ARG_CHECK(ptr_kind == LUDVM_PTR_HOST || ptr_kind == LUDVM_PTR_DEVICE);
    if (nrows == 0) return LUDVM_OK;
    DeviceGuard g(ctx->device);
    const long npts = nrows * nz;
    int rc;
    const bool host = ptr_kind == LUDVM_PTR_HOST;
    const double *dga = ga, *dxa = xa, *dza = za, *dx1 = x1, *dz1 = z1;
    double *du = u, *dw = w;
    if (host && ((rc = stage_in(ctx, {{ga, na, &dga}, {xa, na, &dxa}, {za, na, &dza}, {x1, nx, &dx1}, {z1, nz, &dz1}})) ||
                 (rc = stage_out(ctx, {{u, npts, &du}, {w, npts, &dw}}))))
        return rc;
    void *tp;
    if ((rc = scratch_reserve(ctx, SLOT_TREE_GRID, (2 * (size_t)npts + 4) * sizeof(double), &tp))) return rc;
    double *xp = (double *)tp, *zp = xp + npts, *box = zp + npts;
    k_tree_grid_points<<<ceil_div(npts, 256), 256, 0, ctx->stream>>>(dx1, (int)nx, dz1, (int)nz, (int)row0, npts, xp, zp, box);
    ctx->launches++;
    if ((rc = tree_velocity_device(ctx, ctx->stream, dga, dxa, dza, vc4, na, xp, zp, npts, order, leaf, du, dw, stats, tgt_density, box, box + 2, 2)))
        return rc;
    return host ? copy_back(ctx, {{u, npts, &du}, {w, npts, &dw}}) : LUDVM_OK;
}
