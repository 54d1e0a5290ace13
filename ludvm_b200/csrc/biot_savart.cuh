// biot_savart.cuh -- device templates of the all-pairs Vatistas-core Biot-Savart sum (LUDVM.py:549-570).
//
// Three evaluation strategies, all writing PARTIAL row sums [chunk][row] that a combine step folds in a fixed
// order (so results never depend on grid size, GPU count or scheduling):
//
//   exact  lane-group   8 lanes own one target row and reproduce numpy's pairwise-summation tree: lane k owns
//                       accumulator r[k] of the 8-way unrolled leaf loop, the leaf is closed with an xor-butterfly
//                       ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)) and the up-to-7 tail terms are added in order; leaves
//                       are folded with an explicit stack exactly as the recursion does.  A "chunk" is a node of
//                       the tree at depth d, so 2^d warps can share one row and the combine is the top of the tree.
//   fast   lane-group   same decomposition with FMA arithmetic and equal-length chunks (few targets, many sources:
//                       the 80 chord stations of airfoil_downwash, LUDVM.py:572-595).
//   fast   tiled        one thread owns R target rows in registers, sources are staged through shared memory in
//                       tiles and broadcast to the warp (the O(N^2) convection, LUDVM.py:1095-1127, flow-field
//                       grids, LUDVM.py:1193-1220).  13 FP64-pipe slots + 1 MUFU per pair.
#pragma once
#include "common.cuh"

namespace ludvm {

// Logical concatenation of up to three physical segments of one SoA (TEV ++ LEV ++ FREE, LUDVM.py:743-745).
struct SrcView {
    const double *x, *z, *g, *vc4;  // vc4 == nullptr: scalar core
    double vc4s;
    int n;         // logical length
    int n0, n01;   // logical [0,n0) -> phys [0,n0); [n0,n01) -> phys o1+..; [n01,n) -> phys o2+..
    int o1, o2;
    int gstride;   // 0: broadcast g[0]
    __device__ __forceinline__ int phys(int j) const
    {
        return j < n0 ? j : (j < n01 ? j - n0 + o1 : j - n01 + o2);
    }
};

__host__ __device__ inline SrcView make_src(const double *g, int gstride, const double *x, const double *z,
                                            const double *vc4, double vc4s, int n)
{
    SrcView s;
    s.x = x; s.z = z; s.g = g; s.vc4 = vc4; s.vc4s = vc4s;
    s.n = n; s.n0 = n; s.n01 = n; s.o1 = 0; s.o2 = 0; s.gstride = gstride;
    return s;
}

struct TgtArray {
    const double *x, *z;
    __device__ __forceinline__ void get(int r, double &xp, double &zp) const { xp = x[r]; zp = z[r]; }
};

// 'ij' mesh of x1 x z1 (LUDVM.py:1193-1195): row r -> (x1[row0 + r / nz], z1[r % nz]).
struct TgtGrid {
    const double *x1, *z1;
    int nz, row0;
    __device__ __forceinline__ void get(int r, double &xp, double &zp) const
    {
        int i = r / nz;
        xp = x1[row0 + i];
        zp = z1[r - i * nz];
    }
};

// ---------------------------------------------------------------------------------------------------
// exact lane-group
// ---------------------------------------------------------------------------------------------------
struct ExactSrc { double x, z, g, vc4; };
__device__ __forceinline__ ExactSrc exact_load(const SrcView &S, int j)
{
    int p = S.phys(j);
    ExactSrc s;
    s.vc4 = S.vc4 ? S.vc4[p] : S.vc4s;
    s.x = S.x[p]; s.z = S.z[p]; s.g = S.g[p * S.gstride];
    return s;
}
__device__ __forceinline__ void exact_term(const SrcView &S, double xp, double zp, int j, double &tu, double &tw)
{
    ExactSrc s = exact_load(S, j);
    pair_exact(xp, zp, s.x, s.z, s.g, s.vc4, tu, tw);
}

// K consecutive terms (sources j0, j0+8, ...) of one lane's accumulators for its R target rows: branch-free fast
// paths so the R*K div/sqrt chains interleave, library routines only if a range flag came back set; the adds keep
// numpy's order.  A source is loaded once for the lane's R rows.
template <int R, int K, bool FLAGS = true>
__device__ __forceinline__ void exact_batch(const SrcView &S, const double (&xp)[R], const double (&zp)[R], int j0,
                                            double (&au)[R], double (&aw)[R])
{
    double xw[R * K], zw[R * K], g[R * K], vc4[R * K], xps[R * K], zps[R * K], tu[R * K], tw[R * K];
#pragma unroll
    for (int k = 0; k < K; k++) {
        ExactSrc s = exact_load(S, j0 + 8 * k);
#pragma unroll
        for (int r = 0; r < R; r++) {
            xw[k * R + r] = s.x; zw[k * R + r] = s.z; g[k * R + r] = s.g; vc4[k * R + r] = s.vc4;
            xps[k * R + r] = xp[r]; zps[k * R + r] = zp[r];
        }
    }
    if (!pair_exact_try_batch<R * K, FLAGS>(xps, zps, xw, zw, g, vc4, tu, tw)) {
#pragma unroll
        for (int c = 0; c < R * K; c++) pair_exact_ref(xps[c], zps[c], xw[c], zw[c], g[c], vc4[c], tu[c], tw[c]);
    }
#pragma unroll
    for (int k = 0; k < K; k++)
#pragma unroll
        for (int r = 0; r < R; r++) {
            au[r] = __dadd_rn(au[r], tu[k * R + r]);
            aw[r] = __dadd_rn(aw[r], tw[k * R + r]);
        }
}

// One leaf (n <= 128) of numpy's pairwise sum for the R rows of each 8-lane group.  Result on every lane.
template <int R, bool FLAGS = true>
__device__ __forceinline__ void exact_leaf_group(const SrcView &S, const double (&xp)[R], const double (&zp)[R],
                                                 int off, int m, int lane8, double (&au)[R], double (&aw)[R])
{
    constexpr int K = 4 / R;   // four chains in flight per thread
    const unsigned full = 0xffffffffu;
    int body = (m >= 8) ? (m & ~7) : 0;
#pragma unroll
    for (int r = 0; r < R; r++) au[r] = aw[r] = -0.0;   // -0.0 + t == t bit for bit: no special case for the first term
    if (body) {
        const int nb = body >> 3;  // terms per lane, uniform across the warp
        int b = 0;
        for (; b + K <= nb; b += K) exact_batch<R, K, FLAGS>(S, xp, zp, off + 8 * b + lane8, au, aw);
        if (K == 4) {
            switch (nb - b) {
            case 3: exact_batch<R, 3, FLAGS>(S, xp, zp, off + 8 * b + lane8, au, aw); break;
            case 2: exact_batch<R, 2, FLAGS>(S, xp, zp, off + 8 * b + lane8, au, aw); break;
            case 1: exact_batch<R, 1, FLAGS>(S, xp, zp, off + 8 * b + lane8, au, aw); break;
            default: break;
            }
        } else if (nb - b) {
            exact_batch<R, 1, FLAGS>(S, xp, zp, off + 8 * b + lane8, au, aw);
        }
#pragma unroll
        for (int r = 0; r < R; r++)
#pragma unroll
            for (int s = 1; s < 8; s <<= 1) {
                au[r] = __dadd_rn(au[r], __shfl_xor_sync(full, au[r], s));
                aw[r] = __dadd_rn(aw[r], __shfl_xor_sync(full, aw[r], s));
            }
    }
    int rem = m - body;  // 0..7, uniform across the warp
    if (rem) {
        double tu[R], tw[R];
#pragma unroll
        for (int r = 0; r < R; r++) {
            tu[r] = tw[r] = 0.0;
            if (lane8 < rem) exact_term(S, xp[r], zp[r], off + body + lane8, tu[r], tw[r]);
        }
        for (int t = 0; t < rem; t++)
#pragma unroll
            for (int r = 0; r < R; r++) {
                au[r] = __dadd_rn(au[r], __shfl_sync(full, tu[r], t, 8));
                aw[r] = __dadd_rn(aw[r], __shfl_sync(full, tw[r], t, 8));
            }
    }
}

// Pairwise sum over the logical source range [off, off+n) -- a node of the tree -- for the group's R targets.
// Must be called by all 32 lanes with identical (off, n).
template <int R, bool FLAGS = true>
__device__ inline void exact_node_group(const SrcView &S, const double (&xp)[R], const double (&zp)[R], int off, int n,
                                        int lane8, double (&su)[R], double (&sw)[R])
{
    int r_off[PW_MAX_STACK], r_len[PW_MAX_STACK];
    double l_u[PW_MAX_STACK][R], l_w[PW_MAX_STACK][R];
    unsigned has_l = 0;
    int sp = 0;
    for (;;) {
        while (n > PW_BLOCK) {
            int n2 = pw_left(n);
            r_off[sp] = off + n2;
            r_len[sp] = n - n2;
            has_l &= ~(1u << sp);
            sp++;
            n = n2;
        }
        double ru[R], rw[R];
        exact_leaf_group<R, FLAGS>(S, xp, zp, off, n, lane8, ru, rw);
        for (;;) {
            if (sp == 0) {
#pragma unroll
                for (int r = 0; r < R; r++) { su[r] = ru[r]; sw[r] = rw[r]; }
                return;
            }
            if (!((has_l >> (sp - 1)) & 1u)) {
#pragma unroll
                for (int r = 0; r < R; r++) { l_u[sp - 1][r] = ru[r]; l_w[sp - 1][r] = rw[r]; }
                has_l |= 1u << (sp - 1);
                off = r_off[sp - 1];
                n = r_len[sp - 1];
                break;
            }
#pragma unroll
            for (int r = 0; r < R; r++) {
                ru[r] = __dadd_rn(l_u[sp - 1][r], ru[r]);
                rw[r] = __dadd_rn(l_w[sp - 1][r], rw[r]);
            }
            sp--;
        }
    }
}

// Warp task t -> (tree node b, row group q of 4*R rows: 8-lane group k owns rows q*4R + k*R .. +R).
// Partials: pu[b * nrows + row].
template <int R = 1, bool FLAGS = true, class Tgt>
__device__ __forceinline__ void exact_rows_warp_task(const SrcView &S, const Tgt &T, int nrows, int d, long t,
                                                     int lane, double *__restrict__ pu, double *__restrict__ pw_)
{
    int ngroups = (nrows + 4 * R - 1) / (4 * R);
    int b = (int)(t / ngroups);
    int q = (int)(t - (long)b * ngroups);
    int row0 = (q * 4 + (lane >> 3)) * R;
    double xp[R], zp[R];
#pragma unroll
    for (int r = 0; r < R; r++) T.get(min(row0 + r, nrows - 1), xp[r], zp[r]);
    int off, len;
    pw_node(S.n, d, b, off, len);
    double su[R], sw[R];
    exact_node_group<R, FLAGS>(S, xp, zp, off, len, lane & 7, su, sw);
    if ((lane & 7) == 0) {
#pragma unroll
        for (int r = 0; r < R; r++)
            if (row0 + r < nrows) {
                pu[(size_t)b * nrows + row0 + r] = su[r];
                pw_[(size_t)b * nrows + row0 + r] = sw[r];
            }
    }
}

// ---------------------------------------------------------------------------------------------------
// exact tiled: many target rows.  ONE THREAD owns one target row and all eight accumulators r0..r7 of numpy's
// unrolled leaf loop in registers; the sources of the block's tree node are staged through shared memory in tiles
// and broadcast to the warp (two LDS.128 per source serve 32 pairs), so the per-pair instruction overhead of the
// lane-group form -- per-lane global loads, index mapping, shuffles -- disappears and the kernel is bound by the
// FP64 pipe rather than by instruction issue.  Four consecutive sources go to four different accumulators: four
// independent div/sqrt chains per thread without reordering a single addition.  The traversal of the tree is
// uniform across the block (it depends on the node only).  Same partial layout as the lane-group kernel.
// ---------------------------------------------------------------------------------------------------
#define ET_THREADS 128
#define ET_TILE 1024   // sources per staged tile (a leaf is <= 128): 32 KB of shared memory

// Staged sources of the exact tiled kernels: (x, z) pairs plus either (Gamma, vc^4) pairs or Gamma alone with a
// scalar core (the one-CTA driver, where shared memory is scarce).
struct SmemSrc4 {
    const double2 *xz, *gv;
    __device__ __forceinline__ SmemSrc4 at(int j) const { return SmemSrc4{xz + j, gv + j}; }
    __device__ __forceinline__ void get(int k, double &x, double &z, double &g, double &v) const
    {
        const double2 a = xz[k], b = gv[k];
        x = a.x; z = a.y; g = b.x; v = b.y;
    }
    __device__ __forceinline__ void get_again(int k, double &x, double &z, double &g, double &v) const
    {
        const volatile double *a = (const volatile double *)(xz + k), *b = (const volatile double *)(gv + k);
        x = a[0]; z = a[1]; g = b[0]; v = b[1];
    }
};
struct SmemSrc3 {
    const double2 *xz;
    const double *gam;
    double vc4;
    __device__ __forceinline__ SmemSrc3 at(int j) const { return SmemSrc3{xz + j, gam + j, vc4}; }
    __device__ __forceinline__ void get(int k, double &x, double &z, double &g, double &v) const
    {
        const double2 a = xz[k];
        x = a.x; z = a.y; g = gam[k]; v = vc4;
    }
    __device__ __forceinline__ void get_again(int k, double &x, double &z, double &g, double &v) const
    {
        const volatile double *a = (const volatile double *)(xz + k), *b = (const volatile double *)(gam + k);
        x = a[0]; z = a[1]; g = b[0]; v = vc4;
    }
};

// au[k] += term(source k), k = 0..3, for one target.
template <bool FLAGS = true, class Src>
__device__ __forceinline__ void exact_quad_smem(const Src src, double xp, double zp, double &u0, double &u1, double &u2,
                                                double &u3, double &w0, double &w1, double &w2, double &w3)
{
    double xw[4], zw[4], g[4], vc4[4], xps[4], zps[4], tu[4], tw[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        src.get(k, xw[k], zw[k], g[k], vc4[k]);
        xps[k] = xp; zps[k] = zp;
    }
    if (!pair_exact_try_batch<4, FLAGS>(xps, zps, xw, zw, g, vc4, tu, tw)) {
#pragma unroll
        for (int k = 0; k < 4; k++) {   // rare: re-read the sources rather than keep them alive across the batch
            double x, z, gg, v;
            src.get_again(k, x, z, gg, v);
            pair_exact_ref(xp, zp, x, z, gg, v, tu[k], tw[k]);
        }
    }
    u0 = __dadd_rn(u0, tu[0]); u1 = __dadd_rn(u1, tu[1]); u2 = __dadd_rn(u2, tu[2]); u3 = __dadd_rn(u3, tu[3]);
    w0 = __dadd_rn(w0, tw[0]); w1 = __dadd_rn(w1, tw[1]); w2 = __dadd_rn(w2, tw[2]); w3 = __dadd_rn(w3, tw[3]);
}

// One leaf (m <= 128 staged sources) of numpy's pairwise sum for the thread's target.
template <bool FLAGS = true, class Src>
__device__ __forceinline__ void exact_leaf_thread(const Src src, int m, double xp, double zp, double &ru, double &rw)
{
    const int body = (m >= 8) ? (m & ~7) : 0;
    double su = -0.0, sw = -0.0;
    if (body) {
        double u[8], w[8];
#pragma unroll
        for (int k = 0; k < 8; k++) u[k] = w[k] = -0.0;   // -0.0 + t == t bit for bit
        for (int i = 0; i < body; i += 8) {
            exact_quad_smem<FLAGS>(src.at(i), xp, zp, u[0], u[1], u[2], u[3], w[0], w[1], w[2], w[3]);
            exact_quad_smem<FLAGS>(src.at(i + 4), xp, zp, u[4], u[5], u[6], u[7], w[4], w[5], w[6], w[7]);
        }
        su = __dadd_rn(__dadd_rn(__dadd_rn(u[0], u[1]), __dadd_rn(u[2], u[3])),
                       __dadd_rn(__dadd_rn(u[4], u[5]), __dadd_rn(u[6], u[7])));
        sw = __dadd_rn(__dadd_rn(__dadd_rn(w[0], w[1]), __dadd_rn(w[2], w[3])),
                       __dadd_rn(__dadd_rn(w[4], w[5]), __dadd_rn(w[6], w[7])));
    }
    for (int i = body; i < m; i++) {   // <= 7 tail terms, in order
        double x, z, g, v, tu, tw;
        src.get(i, x, z, g, v);
        pair_exact(xp, zp, x, z, g, v, tu, tw);
        su = __dadd_rn(su, tu);
        sw = __dadd_rn(sw, tw);
    }
    ru = su;
    rw = sw;
}

// The whole pairwise tree over n sources resident in shared memory, for the thread's target (no barriers inside:
// threads may call it a different number of times).
template <bool FLAGS = true, class Src>
__device__ __forceinline__ void exact_tree_thread(const Src src, int n, double xp, double zp, double &su, double &sw)
{
    int r_off[PW_MAX_STACK], r_len[PW_MAX_STACK];
    double l_u[PW_MAX_STACK], l_w[PW_MAX_STACK];
    unsigned has_l = 0;
    int sp = 0, off = 0;
    for (;;) {
        while (n > PW_BLOCK) {
            int n2 = pw_left(n);
            r_off[sp] = off + n2;
            r_len[sp] = n - n2;
            has_l &= ~(1u << sp);
            sp++;
            n = n2;
        }
        double ru, rw;
        exact_leaf_thread<FLAGS>(src.at(off), n, xp, zp, ru, rw);
        for (;;) {
            if (sp == 0) {
                su = ru;
                sw = rw;
                return;
            }
            if (!((has_l >> (sp - 1)) & 1u)) {
                l_u[sp - 1] = ru;
                l_w[sp - 1] = rw;
                has_l |= 1u << (sp - 1);
                off = r_off[sp - 1];
                n = r_len[sp - 1];
                break;
            }
            ru = __dadd_rn(l_u[sp - 1], ru);
            rw = __dadd_rn(l_w[sp - 1], rw);
            sp--;
        }
    }
}

template <bool FLAGS = true, class Tgt>
__device__ __forceinline__ void exact_tiled_block(const SrcView &S, const Tgt &T, int nrows, int row_block, int d, int b,
                                                  double *__restrict__ pu, double *__restrict__ pw_, double2 *sxz,
                                                  double2 *sgv)
{
    const int row = row_block * ET_THREADS + threadIdx.x;
    double xp, zp;
    T.get(min(row, nrows - 1), xp, zp);
    int off, n;
    pw_node(S.n, d, b, off, n);
    const int node_end = off + n;
    int tile0 = off, tile1 = off;   // staged logical source range
    int r_off[PW_MAX_STACK], r_len[PW_MAX_STACK];
    double l_u[PW_MAX_STACK], l_w[PW_MAX_STACK];
    unsigned has_l = 0;
    int sp = 0;
    double ru, rw;
    for (;;) {
        while (n > PW_BLOCK) {
            int n2 = pw_left(n);
            r_off[sp] = off + n2;
            r_len[sp] = n - n2;
            has_l &= ~(1u << sp);
            sp++;
            n = n2;
        }
        if (off + n > tile1) {   // uniform across the block: leaves come in increasing source order
            __syncthreads();
            tile0 = off;
            tile1 = min(off + ET_TILE, node_end);
            for (int j = threadIdx.x; j < tile1 - tile0; j += ET_THREADS) {
                int p = S.phys(tile0 + j);
                sxz[j] = make_double2(S.x[p], S.z[p]);
                sgv[j] = make_double2(S.g[p * S.gstride], S.vc4 ? S.vc4[p] : S.vc4s);
            }
            __syncthreads();
        }
        exact_leaf_thread<FLAGS>(SmemSrc4{sxz + (off - tile0), sgv + (off - tile0)}, n, xp, zp, ru, rw);
        bool done = false;
        for (;;) {
            if (sp == 0) {
                done = true;
                break;
            }
            if (!((has_l >> (sp - 1)) & 1u)) {
                l_u[sp - 1] = ru;
                l_w[sp - 1] = rw;
                has_l |= 1u << (sp - 1);
                off = r_off[sp - 1];
                n = r_len[sp - 1];
                break;
            }
            ru = __dadd_rn(l_u[sp - 1], ru);
            rw = __dadd_rn(l_w[sp - 1], rw);
            sp--;
        }
        if (done) break;
    }
    if (row < nrows) {
        pu[(size_t)b * nrows + row] = ru;
        pw_[(size_t)b * nrows + row] = rw;
    }
}

// Fold the 2^d node partials of one row: the top d levels of the tree are a perfect binary tree in index order;
// finish with numpy's additive identity (np.sum = 0.0 + pairwise).
__device__ __forceinline__ double exact_combine_row(const double *part, int nrows, int row, int d)
{
    double st[PW_MAX_STACK];
    int sp = 0;
    int nn = 1 << d;
    for (int i = 0; i < nn; i++) {
        double v = part[(size_t)i * nrows + row];
        for (int k = i; k & 1; k >>= 1) v = __dadd_rn(st[--sp], v);
        st[sp++] = v;
    }
    return __dadd_rn(0.0, st[0]);
}

// ---------------------------------------------------------------------------------------------------
// fast lane-group (few targets)
// ---------------------------------------------------------------------------------------------------
template <class Tgt>
__device__ __forceinline__ void fast_rows_warp_task(const SrcView &S, const Tgt &T, int nrows, int nchunks, long t,
                                                    int lane, double *__restrict__ pu, double *__restrict__ pw_)
{
    const unsigned full = 0xffffffffu;
    int nquads = (nrows + 3) >> 2;
    int c = (int)(t / nquads);
    int q = (int)(t - (long)c * nquads);
    int row = q * 4 + (lane >> 3);
    bool valid = row < nrows;
    double xp, zp;
    T.get(valid ? row : nrows - 1, xp, zp);
    int clen = (S.n + nchunks - 1) / nchunks;
    clen = (clen + 7) & ~7;
    int j0 = c * clen, j1 = min(S.n, j0 + clen);
    double au = 0.0, aw = 0.0, bu = 0.0, bw = 0.0;
    int j = j0 + (lane & 7);
    for (; j + 8 < j1; j += 16) {  // two independent chains
        int p = S.phys(j), p2 = S.phys(j + 8);
        pair_fast(xp, zp, S.x[p], S.z[p], S.g[p * S.gstride] * LUDVM_INV_TWO_PI, S.vc4 ? S.vc4[p] : S.vc4s, au, aw);
        pair_fast(xp, zp, S.x[p2], S.z[p2], S.g[p2 * S.gstride] * LUDVM_INV_TWO_PI, S.vc4 ? S.vc4[p2] : S.vc4s, bu, bw);
    }
    if (j < j1) {
        int p = S.phys(j);
        pair_fast(xp, zp, S.x[p], S.z[p], S.g[p * S.gstride] * LUDVM_INV_TWO_PI, S.vc4 ? S.vc4[p] : S.vc4s, au, aw);
    }
    au += bu;
    aw += bw;
#pragma unroll
    for (int s = 1; s < 8; s <<= 1) {
        au += __shfl_xor_sync(full, au, s);
        aw += __shfl_xor_sync(full, aw, s);
    }
    if (valid && (lane & 7) == 0) {
        pu[(size_t)c * nrows + row] = au;
        pw_[(size_t)c * nrows + row] = aw;
    }
}

__device__ __forceinline__ double fast_combine_row(const double *part, int nrows, int row, int nchunks)
{
    double s = 0.0;
    for (int c = 0; c < nchunks; c++) s += part[(size_t)c * nrows + row];
    return s;
}

// ---------------------------------------------------------------------------------------------------
// fast tiled (many targets).  Block = 256 threads, R rows per thread (row = base + r*256 + tid: coalesced),
// sources [c0, c1) of the block's chunk in tiles of FT_TILE.
// ---------------------------------------------------------------------------------------------------
#define FT_THREADS 256
#define FT_TILE 512
#ifndef FT_UNROLL
#define FT_UNROLL 4       // source-loop unroll of the thread-staged tiled block
#endif
#ifndef FT_UNROLL32
#define FT_UNROLL32 4     // source-loop unroll of the packed fp32x2 block
#endif
#ifndef FT_UNROLL_TMA
#define FT_UNROLL_TMA 2   // source-loop unroll of the TMA-staged kernel.  Measured at N = 2^20 (ms per step): 1: 905.5, 2: 872.6,
                          // 3: 874.2, 4: 903.2, 6: 890.8, 8: 875.1, 16: 871.8 -- not monotonic (instruction scheduling), 2 is the
                          // smallest code among the fast ones
#endif

template <int R, class Tgt>
__device__ __forceinline__ void fast_tiled_block(const SrcView &S, const Tgt &T, int nrows, int row_block, int c0,
                                                 int c1, double *__restrict__ pu, double *__restrict__ pw_,
                                                 double *sx, double *sz, double *sg, double *sv)
{
    constexpr int UNROLL = R <= 2 ? 8 : FT_UNROLL;   // few rows per thread: a deeper unroll supplies the independent chains
    double tx[R], tz[R], au[R], aw[R];
    int base = row_block * (FT_THREADS * R) + threadIdx.x;
#pragma unroll
    for (int r = 0; r < R; r++) {
        int row = min(base + r * FT_THREADS, nrows - 1);
        T.get(row, tx[r], tz[r]);
        au[r] = 0.0;
        aw[r] = 0.0;
    }
    for (int t0 = c0; t0 < c1; t0 += FT_TILE) {
        __syncthreads();
        for (int j = threadIdx.x; j < FT_TILE; j += FT_THREADS) {
            int s = t0 + j;
            bool ok = s < c1;
            int p = ok ? S.phys(s) : 0;
            sx[j] = ok ? S.x[p] : 0.0;
            sz[j] = ok ? S.z[p] : 0.0;
            sg[j] = ok ? S.g[p * S.gstride] * LUDVM_INV_TWO_PI : 0.0;
            sv[j] = ok ? (S.vc4 ? S.vc4[p] : S.vc4s) : 1.0;
        }
        __syncthreads();
        const int cnt = min(FT_TILE, c1 - t0);   // a ragged last tile costs only its own sources
#pragma unroll UNROLL
        for (int j = 0; j < cnt; j++) {
            double x = sx[j], z = sz[j], g = sg[j], v = sv[j];
#pragma unroll
            for (int r = 0; r < R; r++) pair_fast(tx[r], tz[r], x, z, g, v, au[r], aw[r]);
        }
    }
#pragma unroll
    for (int r = 0; r < R; r++) {
        int row = base + r * FT_THREADS;
        if (row < nrows) {
            pu[row] = au[r];
            pw_[row] = aw[r];
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// fast tiled, TMA-staged: for one contiguous source segment with a scalar core the x / z / Gamma tiles are brought
// into shared memory by the copy engine (cp.async.bulk + mbarrier complete_tx, SASS UBLKCP), double-buffered so the
// load of tile k+1 overlaps the FP64 work on tile k and only one __syncthreads per tile remains.  1/(2 pi) is folded
// into the row result.  Requires 16-byte aligned source pointers; a ragged last tile is loaded by the threads.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    uint32_t ok;
    do {
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
                     : "=r"(ok)
                     : "r"(smem_u32(bar)), "r"(parity)
                     : "memory");
    } while (!ok);
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

struct TmaTiles {  // [stage][x | z | g][FT_TILE]
    double buf[2][3][FT_TILE];
    uint64_t full[2];
};

template <int R, class Tgt>
__device__ __forceinline__ void fast_tiled_block_tma(const SrcView &S, const Tgt &T, int nrows, int row_block, int c0,
                                                     int c1, double *__restrict__ pu, double *__restrict__ pw_,
                                                     TmaTiles &sm)
{
    constexpr int UNROLL_TMA = FT_UNROLL_TMA;
    double tx[R], tz[R], au[R], aw[R];
    int base = row_block * (FT_THREADS * R) + threadIdx.x;
#pragma unroll
    for (int r = 0; r < R; r++) {
        int row = min(base + r * FT_THREADS, nrows - 1);
        T.get(row, tx[r], tz[r]);
        au[r] = 0.0;
        aw[r] = 0.0;
    }
    const double vc4 = S.vc4s;
    const int ntiles = (c1 - c0 + FT_TILE - 1) / FT_TILE;
    if (threadIdx.x == 0) {
        mbar_init(&sm.full[0], 1);
        mbar_init(&sm.full[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    // producer: thread 0 hands whole tiles to the copy engine; a ragged tile is filled by all threads instead
    auto issue = [&](int k) {
        int t0 = c0 + k * FT_TILE, cnt = min(FT_TILE, c1 - t0), st = k & 1;
        if (cnt == FT_TILE) {
            if (threadIdx.x == 0) {
                mbar_expect_tx(&sm.full[st], 3 * FT_TILE * sizeof(double));
                bulk_g2s(sm.buf[st][0], S.x + t0, FT_TILE * sizeof(double), &sm.full[st]);
                bulk_g2s(sm.buf[st][1], S.z + t0, FT_TILE * sizeof(double), &sm.full[st]);
                bulk_g2s(sm.buf[st][2], S.g + t0, FT_TILE * sizeof(double), &sm.full[st]);
            }
        } else {
            for (int j = threadIdx.x; j < cnt; j += FT_THREADS) {
                sm.buf[st][0][j] = S.x[t0 + j];
                sm.buf[st][1][j] = S.z[t0 + j];
                sm.buf[st][2][j] = S.g[t0 + j];
            }
            __threadfence_block();
            if (threadIdx.x == 0) mbar_arrive(&sm.full[st]);
        }
    };
    if (ntiles > 0) issue(0);
    for (int k = 0; k < ntiles; k++) {
        if (k + 1 < ntiles) issue(k + 1);  // stage (k+1)&1 was released by the __syncthreads of iteration k-1
        const int st = k & 1, cnt = min(FT_TILE, c1 - (c0 + k * FT_TILE));
        if (cnt != FT_TILE) __syncthreads();  // thread-filled tile: make every thread's stores visible
        mbar_wait(&sm.full[st], (k >> 1) & 1);
        const double *sx = sm.buf[st][0], *sz = sm.buf[st][1], *sg = sm.buf[st][2];
#pragma unroll UNROLL_TMA
        for (int j = 0; j < cnt; j++) {
            double x = sx[j], z = sz[j], g = sg[j];
#pragma unroll
            for (int r = 0; r < R; r++) pair_fast(tx[r], tz[r], x, z, g, vc4, au[r], aw[r]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int r = 0; r < R; r++) {
        int row = base + r * FT_THREADS;
        if (row < nrows) {
            pu[row] = au[r] * LUDVM_INV_TWO_PI;
            pw_[row] = aw[r] * LUDVM_INV_TWO_PI;
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// fast fused ("warp-split"): the whole row sum inside one thread-block cluster -- no partial sums in global memory
// and no combine kernel.  A CTA owns 32*R target rows; each of its FW_WARPS warps holds ALL of those rows (R per lane) and
// walks ONE source chunk with its own private, double-buffered bulk-copy pipeline (cp.async.bulk + mbarrier, SASS
// UBLKCP/SYNCS), so the main loop has no block-wide barrier at all.  A cluster of CL CTAs (1 or 2: clusters of two
// pack the 148 SMs perfectly) covers FW_WARPS*CL source chunks: 8 chunks = one 8-warp CTA, 16 chunks = a cluster of two
// 8-warp CTAs.  The chunk partials meet in shared memory and are folded IN
// CHUNK ORDER through distributed shared memory -- the same canonical order as fast_combine_row, so the result is
// bitwise equal to the partial-sum path and independent of grid size and GPU count.  The epilogue applies the forward
// Euler update (LUDVM.py:1108-1127) and the peer stores of the fused all-gather.
// ---------------------------------------------------------------------------------------------------
#ifndef FW_SUB
#define FW_SUB 128       // sources per warp-private stage: three 1 KB bulk copies
#endif
#define FW_STAGES 2
#define FW_WARPS 8       // warps per CTA, one source chunk each

// source-loop unroll of the fused kernel: few rows per lane need a deeper unroll for independent chains
__host__ __device__ constexpr int fw_unroll(int R) { return R == 1 ? 8 : 4; }

struct FwWarpStage {
    double x[FW_SUB], z[FW_SUB], g[FW_SUB];
};
struct FwSmem {
    FwWarpStage st[FW_WARPS][FW_STAGES];   // 6 KB per warp; the front of each warp's region is reused for its partials
    uint64_t full[FW_WARPS][FW_STAGES];
};

// Where the finished row sums go, for the fused kernel and k_combine alike.
struct RowOut {
    double *u, *w;           // velocities (nullable)
    const double *x, *z;     // Euler inputs, already offset to the first row (nullable: no update)
    double *xo, *zo;         // Euler outputs (nullable)
    double dt;
    int npeers;
    double *xo_peer[LUDVM_MAX_PEERS], *zo_peer[LUDVM_MAX_PEERS];
};

// Store one finished row sum s of component comp (0: u and x, 1: w and z): the velocity, the forward Euler update
// (LUDVM.py:1108-1127) and its copies in the peers' buffers (the all-gather, fused: st.global on mapped peer pointers).
__device__ __forceinline__ void store_row(const RowOut &O, int comp, int row, double s)
{
    double *vout = comp ? O.w : O.u;
    if (vout) vout[row] = s;
    const double *pin = comp ? O.z : O.x;
    if (pin) {
        const double pn = __dadd_rn(pin[row], __dmul_rn(O.dt, s));
        double *pout = comp ? O.zo : O.xo;
        if (pout) pout[row] = pn;
        for (int p = 0; p < O.npeers; p++) (comp ? O.zo_peer[p] : O.xo_peer[p])[row] = pn;
    }
}

__device__ __forceinline__ void cluster_sync_all()
{
    asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}
// generic address of `p` (a shared-memory address of this CTA) in CTA `rank` of the cluster
__device__ __forceinline__ const double *cluster_map(const double *p, unsigned rank)
{
    uint64_t out;
    asm volatile("mapa.u64 %0, %1, %2;" : "=l"(out) : "l"((uint64_t)p), "r"(rank));
    return (const double *)out;
}

template <int R, int CL, int V, class Tgt>
__device__ __forceinline__ void fast_fused_block(const SrcView &S, const Tgt &T, int nrows, int chunk_len, int nchunks,
                                                 const RowOut &O, FwSmem &sm)
{
    constexpr int UNROLL = fw_unroll(R);
    constexpr int ROWS = 32 * R;
    // the warp index through a shuffle: ptxas then knows it is warp-uniform and keeps the stage addresses and the loop
    // counter on the uniform datapath (ULEA / UIADD3 + LDS [UR + imm]) instead of vector integer instructions
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const unsigned crank = CL > 1 ? blockIdx.y : 0;
    const int base = blockIdx.x * ROWS + lane;
    double tx[R], tz[R], au[R], aw[R];
#pragma unroll
    for (int r = 0; r < R; r++) {
        T.get(min(base + 32 * r, nrows - 1), tx[r], tz[r]);
        au[r] = 0.0;
        aw[r] = 0.0;
    }
    double vc4;   // opaque copy: otherwise ptxas re-reads the kernel parameter (LDCU.64) in every trip of the source loop
    asm volatile("mov.f64 %0, %1;" : "=d"(vc4) : "d"(S.vc4s));
    const int c = (int)crank * FW_WARPS + warp;                      // this warp's source chunk
    const int c0 = min(S.n, c * chunk_len), c1 = c < nchunks ? min(S.n, c0 + chunk_len) : c0;
    const int nsub = (c1 - c0 + FW_SUB - 1) / FW_SUB;
    FwWarpStage *st = sm.st[warp];
    uint64_t *full = sm.full[warp];
    if (lane == 0) {
        mbar_init(&full[0], 1);
        mbar_init(&full[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    // producer = lane 0 of each warp: whole stages go through the copy engine, a ragged last stage is filled by the lanes
    auto issue = [&](int k) {
        const int t0 = c0 + k * FW_SUB, cnt = min(FW_SUB, c1 - t0);
        FwWarpStage &b = st[k & 1];
        if (cnt == FW_SUB) {
            if (lane == 0) {
                mbar_expect_tx(&full[k & 1], 3 * FW_SUB * sizeof(double));
                bulk_g2s(b.x, S.x + t0, FW_SUB * sizeof(double), &full[k & 1]);
                bulk_g2s(b.z, S.z + t0, FW_SUB * sizeof(double), &full[k & 1]);
                bulk_g2s(b.g, S.g + t0, FW_SUB * sizeof(double), &full[k & 1]);
            }
        } else {
            for (int j = lane; j < cnt; j += 32) {
                b.x[j] = S.x[t0 + j];
                b.z[j] = S.z[t0 + j];
                b.g[j] = S.g[t0 + j];
            }
        }
    };
    if (nsub > 0) issue(0);
    for (int k = 0; k < nsub; k++) {
        __syncwarp();                                   // every lane is done with stage (k+1)&1 (sub-tile k-1)
        if (k + 1 < nsub) issue(k + 1);
        const int cnt = min(FW_SUB, c1 - (c0 + k * FW_SUB));
        if (cnt == FW_SUB) mbar_wait(&full[k & 1], (k >> 1) & 1);
        else __syncwarp();                              // lane-filled (always the last sub-tile)
        const FwWarpStage &b = st[k & 1];
#pragma unroll UNROLL
        for (int j = 0; j < cnt; j++) {
            const double x = b.x[j], z = b.z[j], g = b.g[j];
#pragma unroll
            for (int r = 0; r < R; r++) pair_fast_v<V>(tx[r], tz[r], x, z, g, vc4, au[r], aw[r]);
        }
    }
    // chunk partials [warp][component][row] over the front of the warp's own stage memory (all its copies have landed)
    __syncwarp();
    double *part = (double *)st;
#pragma unroll
    for (int r = 0; r < R; r++) {
        part[32 * r + lane] = au[r] * LUDVM_INV_TWO_PI;
        part[ROWS + 32 * r + lane] = aw[r] * LUDVM_INV_TWO_PI;
    }
    if (CL > 1) cluster_sync_all();
    else __syncthreads();
    // fold in chunk order; CTA `crank` of the cluster finishes rows [crank*ROWS/CL, (crank+1)*ROWS/CL), one thread
    // per (component, row)
    constexpr int RPC = ROWS / CL;
    if ((int)threadIdx.x < 2 * RPC) {
        const int comp = (int)threadIdx.x / RPC, lrow = (int)crank * RPC + (int)threadIdx.x % RPC;
        const int row = blockIdx.x * ROWS + lrow;
        double s = 0.0;
#pragma unroll
        for (int q = 0; q < CL; q++) {
            const double *p0 = (const double *)sm.st[0] + comp * ROWS + lrow;
            const double *p = (CL > 1) ? cluster_map(p0, (unsigned)q) : p0;
#pragma unroll
            for (int wq = 0; wq < FW_WARPS; wq++)
                if (q * FW_WARPS + wq < nchunks) s += p[wq * (sizeof(FwWarpStage) * FW_STAGES / sizeof(double))];
        }
        if (row < nrows) store_row(O, comp, row, s);
    }
    if (CL > 1) cluster_sync_all();                     // nobody leaves while a peer still reads its shared memory
}

// ---------------------------------------------------------------------------------------------------
// fast symmetric ("k_fast_sym"): the whole-cloud self-convection sum with every unordered pair evaluated ONCE.
// Terms (i, j) and (j, i) share r^2, q and y = rsqrt_fast(q) (10 of pair_fast's 13 FP64 slots); only gg = G y and the
// two accumulating FMAs belong to each direction, so a term costs 8 slots instead of 13.  Because RN(-a) = -RN(a),
// the transposed term fma(G_i y, -dz_ij, u_j), fma(G_i y, dx_ij, w_j) is bit for bit what pair_fast computes for
// target j (a signed zero only matters on a -0 accumulator, and one that starts at +0 never becomes -0).
//
// Summation order is kept: every (target, source chunk) chain -- the chunks of fast_chunking -- is fed its terms in
// source order from +0, then scaled by 1/(2 pi) into the [chunk][target] partials that k_combine folds.  The rows are
// cut into 128-row blocks.  A work item ("strip") is one row block p of chunk a against the columns of chunk c >= a:
//   row role     the chains (i in p, chunk c) advance over the strip's columns, held in registers;
//   column role  each column's chain (j, chunk a) comes in from strip p - 1 (through the partials array), advances
//                over the 128 rows of p in order and goes out to strip p + 1.
// For c == a the strip starts at the diagonal block (p, p): the chains of p's rows arrive in column form, take their
// own block's 128 ordered terms unshared (pair_fast, self term included, as k_fast_fused) and continue in row role
// over the columns after the block.
//
// Inside a strip one warp holds the 128 rows (lane k: rows 4k..4k+3) and runs a skewed (systolic) schedule: at step
// s lane k evaluates column s - k against its four rows in order, then hands that column's (u, w) to lane k + 1 with
// a shuffle.  Lane 0 takes incoming column states from shared memory, lane 31 stores outgoing ones.  Row chains see
// columns in increasing order, column chains see rows in increasing order.  Source data comes from a warp-private
// ring of bulk-copy stages.
//
// Scheduling: a persistent grid; warps take strips from one atomic ticket in an order where the producer of every
// strip (p - 1, same chunk pair) holds a smaller ticket, so a waiting warp only ever waits on a running one.  Column
// states are published per (row block, chunk) as a progress counter (release / acquire at GPU scope).  A wait that
// exceeds FS_SPIN_LIMIT sets an error flag and abandons the launch instead of hanging the GPU.
// ---------------------------------------------------------------------------------------------------
#define FS_ROWS 128          // rows of a row block (one warp, four rows per lane)
#define FS_STAGE 64          // columns per bulk-copy stage = steps per block of the step loop
#define FS_RING 4            // stages in a warp's ring: the 31-step skew reads two, one is in flight
#define FS_WARPS 8
#define FS_SPIN_LIMIT (1u << 24)   // polls of 64+ ns: a lost producer becomes an error, not a hung GPU

struct FsWarpSmem {
    double x[FS_RING * FS_STAGE], z[FS_RING * FS_STAGE], g[FS_RING * FS_STAGE];   // column c of the strip at c % ring
    double2 cin[2][FS_STAGE];   // incoming column states (u, w) of this block of steps and the next
    uint64_t full[FS_RING];
};
struct FsSmem {
    FsWarpSmem w[FS_WARPS];
};

struct SymArgs {
    const double *x, *z, *g;
    double vc4;
    int n, chunk_len, nchunks;
    int bpc, blast;          // row blocks of a full chunk / of the last chunk
    int npairs;              // chunk pairs a <= c
    long nitems;             // strips
    double *pu, *pw;         // [chunk][n] chain states, then partial sums
    unsigned *progress;      // [row block][chunk]: absolute end of the column states stored by that strip
    unsigned *ticket;
    int *abort;              // device: a warp gave up, the others stop waiting
    int *timeout;            // host-mapped copy of the same verdict, read by the host without a synchronisation
};

__device__ __forceinline__ unsigned ld_acquire_gpu(const unsigned *p)
{
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_gpu(unsigned *p, unsigned v)
{
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// Wait (all lanes) until *p >= need.  false: the limit was hit or another warp already gave up.
__device__ __forceinline__ bool fs_wait(const SymArgs &A, const unsigned *p, unsigned need)
{
    unsigned spins = 0;
    while (ld_acquire_gpu(p) < need) {
        if (*(volatile int *)A.abort) return false;
        if (++spins > FS_SPIN_LIMIT) {
            *(volatile int *)A.abort = 1;
            *(volatile int *)A.timeout = 1;
            return false;
        }
        __nanosleep(64);
    }
    return true;
}

// One step for the lane's four rows against column (xj, zj, gj): row chains au, aw and the column chain cu, cw.
// MASK: the lane's column lies outside the strip (skew prologue / epilogue), its row chains must not move.
template <bool MASK>
__device__ __forceinline__ void fs_step(const double (&xr)[4], const double (&zr)[4], const double (&gr)[4],
                                        double (&au)[4], double (&aw)[4], double xj, double zj, double gj, double vc4,
                                        double &cu, double &cw, bool valid)
{
#pragma unroll
    for (int r = 0; r < 4; r++) {
        const double dx = xr[r] - xj;
        const double dz = zr[r] - zj;
        const double r2 = fma(dz, dz, dx * dx);
        const double q = fma(r2, r2, vc4);
        const double y = rsqrt_fast(q);
        const double ggr = gj * y, ggc = gr[r] * y;
        const double nu = fma(ggr, dz, au[r]), nw = fma(-ggr, dx, aw[r]);
        au[r] = (!MASK || valid) ? nu : au[r];
        aw[r] = (!MASK || valid) ? nw : aw[r];
        cu = fma(ggc, -dz, cu);
        cw = fma(ggc, dx, cw);
    }
}

__device__ __forceinline__ void fast_sym_warp(const SymArgs &A, FsWarpSmem &sm)
{
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    double vc4;   // opaque copy: keeps ptxas from re-reading the kernel parameter inside the step loop
    asm volatile("mov.f64 %0, %1;" : "=d"(vc4) : "d"(A.vc4));
    const int last = A.nchunks - 1;
    const size_t n = (size_t)A.n;
    for (;;) {
        unsigned tk = 0;
        if (lane == 0) tk = atomicAdd(A.ticket, 1u);
        const long t = (long)__shfl_sync(full, tk, 0);
        if (t >= A.nitems || *(volatile int *)A.abort) return;
        // ticket -> (round r, chunk pair): round-major, the pair (last, last) -- fewer row blocks -- listed last
        int r, pr;
        const long head = (long)A.blast * A.npairs;
        if (t < head) { r = (int)(t / A.npairs); pr = (int)(t % A.npairs); }
        else { r = A.blast + (int)((t - head) / (A.npairs - 1)); pr = (int)((t - head) % (A.npairs - 1)); }
        int a = last, c = last;
        if (pr < A.npairs - 1) {
            a = 0;
            while (pr >= last - a + 1) { pr -= last - a + 1; a++; }
            c = a + pr;
        }
        const int p = a * A.bpc + r;
        const int c0 = c * A.chunk_len, c1 = min(A.n, c0 + A.chunk_len);
        const int cstart = min(c1, a == c ? (p + 1) * FS_ROWS : c0);   // first column of the skewed stream
        const int L = c1 - cstart;
        const bool has_prev = r > 0;
        const unsigned *prog_in = A.progress + (size_t)max(p - 1, 0) * A.nchunks + c;   // read only if has_prev
        unsigned *prog_out = A.progress + (size_t)p * A.nchunks + c;
        double *cu_g = A.pu + (size_t)a * n, *cw_g = A.pw + (size_t)a * n;   // column chains (j, a)

        const int row0 = p * FS_ROWS + 4 * lane;
        double xr[4], zr[4], gr[4], au[4], aw[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int i = min(row0 + k, A.n - 1);
            xr[k] = A.x[i]; zr[k] = A.z[i]; gr[k] = A.g[i];
            au[k] = 0.0; aw[k] = 0.0;
        }
        if (a == c) {   // diagonal block: the rows' chains arrive as column states
            const int dend = min(c1, (p + 1) * FS_ROWS);
            if (has_prev) {
                if (!fs_wait(A, prog_in, (unsigned)dend)) return;
#pragma unroll
                for (int k = 0; k < 4; k++)
                    if (row0 + k < A.n) { au[k] = __ldcg(cu_g + row0 + k); aw[k] = __ldcg(cw_g + row0 + k); }
            }
            for (int j = p * FS_ROWS; j < dend; j++) {
                const double xj = A.x[j], zj = A.z[j], gj = A.g[j];
#pragma unroll
                for (int k = 0; k < 4; k++) pair_fast(xr[k], zr[k], xj, zj, gj, vc4, au[k], aw[k]);
            }
        }

        if (L > 0) {
            const int nst = (L + FS_STAGE - 1) / FS_STAGE;
            const int nblk = (L + 31 + FS_STAGE - 1) / FS_STAGE;
            if (lane == 0) {
#pragma unroll
                for (int k = 0; k < FS_RING; k++) mbar_init(&sm.full[k], 1);
                asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // lane-filled stages of the last strip
            }
            __syncwarp();
            // stage m = columns [64 m, 64 m + 64) of the stream: the copy engine for a whole stage, the lanes for a ragged
            // last one
            auto issue = [&](int m) {
                const int t0 = cstart + m * FS_STAGE, cnt = min(FS_STAGE, c1 - t0), o = (m % FS_RING) * FS_STAGE;
                if (cnt == FS_STAGE) {
                    if (lane == 0) {
                        uint64_t *bar = &sm.full[m % FS_RING];
                        mbar_expect_tx(bar, 3 * FS_STAGE * sizeof(double));
                        bulk_g2s(sm.x + o, A.x + t0, FS_STAGE * sizeof(double), bar);
                        bulk_g2s(sm.z + o, A.z + t0, FS_STAGE * sizeof(double), bar);
                        bulk_g2s(sm.g + o, A.g + t0, FS_STAGE * sizeof(double), bar);
                    }
                } else {
                    for (int j = lane; j < cnt; j += 32) {
                        sm.x[o + j] = A.x[t0 + j];
                        sm.z[o + j] = A.z[t0 + j];
                        sm.g[o + j] = A.g[t0 + j];
                    }
                }
            };
            // incoming column states of stream columns [64 b, 64 b + 64): two per lane
            double2 pre[2] = {make_double2(0.0, 0.0), make_double2(0.0, 0.0)};
            auto fetch = [&](int b) -> bool {
                const int e = min(L, (b + 1) * FS_STAGE);
                if (!fs_wait(A, prog_in, (unsigned)(cstart + e))) return false;
#pragma unroll
                for (int h = 0; h < 2; h++) {
                    const int jr = b * FS_STAGE + 32 * h + lane;
                    if (jr < e) pre[h] = make_double2(__ldcg(cu_g + cstart + jr), __ldcg(cw_g + cstart + jr));
                }
                return true;
            };
            if (has_prev) {
                if (!fetch(0)) return;
                sm.cin[0][lane] = pre[0];
                sm.cin[0][lane + 32] = pre[1];
            } else {   // the first row block of chunk a starts every column chain at +0
                sm.cin[0][lane] = sm.cin[0][lane + 32] = sm.cin[1][lane] = sm.cin[1][lane + 32] = make_double2(0.0, 0.0);
            }
            issue(0);
            double cu = 0.0, cw = 0.0;
            for (int b = 0; b < nblk; b++) {
                __syncwarp();   // stage b - 2 and cin[(b + 1) & 1] are no longer read; lane-filled data is visible
                if (b + 1 < nst) issue(b + 1);
                const bool more = has_prev && (b + 1) * FS_STAGE < L;
                if (more && !fetch(b + 1)) return;
                if (b < nst && min(FS_STAGE, c1 - (cstart + b * FS_STAGE)) == FS_STAGE)
                    mbar_wait(&sm.full[b % FS_RING], (b / FS_RING) & 1);
                const double2 *cin = sm.cin[b & 1];
                const int s0 = b * FS_STAGE;
                if (s0 >= 31 && s0 + FS_STAGE <= L) {
#pragma unroll 2
                    for (int tt = 0; tt < FS_STAGE; tt++) {
                        const int idx = (s0 + tt - lane) & (FS_RING * FS_STAGE - 1);
                        const double xj = sm.x[idx], zj = sm.z[idx], gj = sm.g[idx];
                        cu = __shfl_up_sync(full, cu, 1);
                        cw = __shfl_up_sync(full, cw, 1);
                        if (lane == 0) { const double2 v = cin[tt]; cu = v.x; cw = v.y; }
                        fs_step<false>(xr, zr, gr, au, aw, xj, zj, gj, vc4, cu, cw, true);
                        if (lane == 31) { __stcg(cu_g + cstart + s0 + tt - 31, cu); __stcg(cw_g + cstart + s0 + tt - 31, cw); }
                    }
                } else {
                    for (int tt = 0; tt < FS_STAGE; tt++) {
                        const int jr = s0 + tt - lane;
                        const bool valid = jr >= 0 && jr < L;
                        const int idx = jr & (FS_RING * FS_STAGE - 1);
                        const double xj = sm.x[idx], zj = sm.z[idx], gj = sm.g[idx];
                        cu = __shfl_up_sync(full, cu, 1);
                        cw = __shfl_up_sync(full, cw, 1);
                        if (lane == 0) { const double2 v = cin[tt]; cu = v.x; cw = v.y; }
                        fs_step<true>(xr, zr, gr, au, aw, xj, zj, gj, vc4, cu, cw, valid);
                        if (lane == 31 && valid) { __stcg(cu_g + cstart + jr, cu); __stcg(cw_g + cstart + jr, cw); }
                    }
                }
                if (more) {
                    sm.cin[(b + 1) & 1][lane] = pre[0];
                    sm.cin[(b + 1) & 1][lane + 32] = pre[1];
                }
                // lane 31 has stored stream columns [0, 64 b + 33)
                if (lane == 31) st_release_gpu(prog_out, (unsigned)(cstart + min(L, s0 + FS_STAGE - 31)));
            }
            if (a < c && r == A.bpc - 1) {   // the last row block of chunk a: its column chains are finished, scale them
                __syncwarp();
                for (int j = cstart + lane; j < c1; j += 32) {
                    cu_g[j] = __ldcg(cu_g + j) * LUDVM_INV_TWO_PI;
                    cw_g[j] = __ldcg(cw_g + j) * LUDVM_INV_TWO_PI;
                }
            }
        }
        // the rows' chains (i, c) are finished
#pragma unroll
        for (int k = 0; k < 4; k++)
            if (row0 + k < A.n) {
                A.pu[(size_t)c * n + row0 + k] = au[k] * LUDVM_INV_TWO_PI;
                A.pw[(size_t)c * n + row0 + k] = aw[k] * LUDVM_INV_TWO_PI;
            }
        __syncwarp();   // the next strip re-initialises the ring's barriers
    }
}

// fp32 pair arithmetic; R rows per thread.
template <int R, class Tgt>
__device__ __forceinline__ void fast32_tiled_block(const SrcView &S, const Tgt &T, int nrows, int row_block, int c0,
                                                   int c1, double *__restrict__ pu, double *__restrict__ pw_,
                                                   float4 *ssrc)
{
    float tx[R], tz[R];
    double au[R], aw[R];  // per-tile fp32 sums are flushed into fp64 row accumulators
    int base = row_block * (FT_THREADS * R) + threadIdx.x;
#pragma unroll
    for (int r = 0; r < R; r++) {
        int row = min(base + r * FT_THREADS, nrows - 1);
        double xd, zd;
        T.get(row, xd, zd);
        tx[r] = (float)xd;
        tz[r] = (float)zd;
        au[r] = 0.0;
        aw[r] = 0.0;
    }
    for (int t0 = c0; t0 < c1; t0 += FT_TILE) {
        __syncthreads();
        for (int j = threadIdx.x; j < FT_TILE; j += FT_THREADS) {
            int s = t0 + j;
            bool ok = s < c1;
            int p = ok ? S.phys(s) : 0;
            float4 v;
            v.x = ok ? (float)S.x[p] : 0.f;
            v.y = ok ? (float)S.z[p] : 0.f;
            v.z = ok ? (float)(S.g[p * S.gstride] * LUDVM_INV_TWO_PI) : 0.f;
            v.w = ok ? (float)(S.vc4 ? S.vc4[p] : S.vc4s) : 1.f;
            ssrc[j] = v;
        }
        __syncthreads();
        float fu[R], fw[R];
#pragma unroll
        for (int r = 0; r < R; r++) {
            fu[r] = 0.f;
            fw[r] = 0.f;
        }
#pragma unroll 8
        for (int j = 0; j < FT_TILE; j++) {
            float4 v = ssrc[j];
#pragma unroll
            for (int r = 0; r < R; r++) pair_fast32(tx[r], tz[r], v.x, v.y, v.z, v.w, fu[r], fw[r]);
        }
#pragma unroll
        for (int r = 0; r < R; r++) {
            au[r] += (double)fu[r];
            aw[r] += (double)fw[r];
        }
    }
#pragma unroll
    for (int r = 0; r < R; r++) {
        int row = base + r * FT_THREADS;
        if (row < nrows) {
            pu[row] = au[r];
            pw_[row] = aw[r];
        }
    }
}

// fp32 pair arithmetic with Blackwell's packed fp32x2 instructions (FADD2 / FMUL2 / FFMA2, sm_100+): one thread owns
// 2*RP target rows as RP float2 pairs, a source is broadcast from shared memory already duplicated into both halves
// ({-x,-x}, {-z,-z}, {g,g}: one LDS.64 each, no register shuffling), so a pair of interactions costs 8 packed FP32
// instructions + 2 MUFU.RSQ instead of 16 + 2 issue slots.  The scalar kernel is issue-bound (10 slots per pair at 4
// issues/clk/SM); packed, the bound becomes the FP32 pipe / MUFU rate (16 pairs/clk/SM).
// The w accumulator holds +sum(g K dx) and is negated once at the end.
struct Src32x2 {
    float2 nx, nz, g;
};

template <int RP, class Tgt>
__device__ __forceinline__ void fast32x2_tiled_block(const SrcView &S, const Tgt &T, int nrows, int row_block, int c0,
                                                     int c1, double *__restrict__ pu, double *__restrict__ pw_,
                                                     Src32x2 *ssrc)
{
    constexpr int UNROLL32 = FT_UNROLL32;
    constexpr int R = 2 * RP;
    float2 tx[RP], tz[RP];
    double au[R], aw[R];
    const int base = row_block * (FT_THREADS * R) + threadIdx.x;
#pragma unroll
    for (int r = 0; r < RP; r++) {
        double xa, za, xb, zb;
        T.get(min(base + (2 * r) * FT_THREADS, nrows - 1), xa, za);
        T.get(min(base + (2 * r + 1) * FT_THREADS, nrows - 1), xb, zb);
        tx[r] = make_float2((float)xa, (float)xb);
        tz[r] = make_float2((float)za, (float)zb);
        au[2 * r] = au[2 * r + 1] = aw[2 * r] = aw[2 * r + 1] = 0.0;
    }
    const float vcs = (float)S.vc4s;
    const float2 vc4 = make_float2(vcs, vcs);
    for (int t0 = c0; t0 < c1; t0 += FT_TILE) {
        __syncthreads();
        for (int j = threadIdx.x; j < FT_TILE; j += FT_THREADS) {
            int s = t0 + j;
            bool ok = s < c1;
            int p = ok ? S.phys(s) : 0;
            float x = ok ? -(float)S.x[p] : 0.f, z = ok ? -(float)S.z[p] : 0.f;
            float g = ok ? (float)(S.g[p * S.gstride] * LUDVM_INV_TWO_PI) : 0.f;
            Src32x2 v;
            v.nx = make_float2(x, x);
            v.nz = make_float2(z, z);
            v.g = make_float2(g, g);
            ssrc[j] = v;
        }
        __syncthreads();
        float2 fu[RP], fw[RP];
#pragma unroll
        for (int r = 0; r < RP; r++) fu[r] = fw[r] = make_float2(0.f, 0.f);
#pragma unroll UNROLL32
        for (int j = 0; j < FT_TILE; j++) {
            const Src32x2 v = ssrc[j];
#pragma unroll
            for (int r = 0; r < RP; r++) {
                float2 dx = __fadd2_rn(tx[r], v.nx), dz = __fadd2_rn(tz[r], v.nz);
                float2 r2 = __ffma2_rn(dz, dz, __fmul2_rn(dx, dx));
                float2 q = __ffma2_rn(r2, r2, vc4);
                float2 y;
                asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y.x) : "f"(q.x));
                asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y.y) : "f"(q.y));
                float2 gg = __fmul2_rn(v.g, y);
                fu[r] = __ffma2_rn(gg, dz, fu[r]);
                fw[r] = __ffma2_rn(gg, dx, fw[r]);
            }
        }
#pragma unroll
        for (int r = 0; r < RP; r++) {
            au[2 * r] += (double)fu[r].x;
            au[2 * r + 1] += (double)fu[r].y;
            aw[2 * r] -= (double)fw[r].x;
            aw[2 * r + 1] -= (double)fw[r].y;
        }
    }
#pragma unroll
    for (int r = 0; r < R; r++) {
        int row = base + r * FT_THREADS;
        if (row < nrows) {
            pu[row] = au[r];
            pw_[row] = aw[r];
        }
    }
}

}  // namespace ludvm
