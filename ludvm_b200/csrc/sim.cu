// sim.cu -- the on-device time step of LUDVM.time_loop (LUDVM.py:597-1171).
//
// This translation unit is compiled with -fmad=false: the scalar phases of the step are written as plain C
// expressions in the reference's operation order and must not be contracted into FMAs (SURVEY.md 4.3, A.5).
// The fast pair arithmetic uses explicit fma() and is unaffected.
//
// The vortex state (x, z, Gamma of TEV | LEV | FREE) stays in HBM in one SoA with three fixed segments, addressed
// through the logical->physical map of SrcView so that the reference's np.append(TEV[:..], LEV[:..], FREE)
// ordering -- which fixes the shape of numpy's summation tree -- is reproduced without moving data.
//
// One time step i is four phases (device functions below):
//   phase_wake_on_foil   partial sums of the existing wake at the P gamma points          (LUDVM.py:743-746)
//   phase_solve          one CTA: TEV placement, T1/T2/T3, Kelvin + LESP solve (Faure closed form / 2x2, or the
//                        Ramesh Newton iterations), Fourier coefficients, bound vortices  (LUDVM.py:672-1010)
//   phase_conv_partials  partial sums of the updated wake at the gamma points (loads) and at every wake vortex
//                        (convection), plus the bound vortices on the wake               (LUDVM.py:1049-1054, 1095-1124)
//   phase_finish_*       loads Fn, Fs, L, D, T, M; fold partials, forward-Euler update in place, history snapshot
//                                                                                         (LUDVM.py:1069-1090, 1108-1127)
// and these drivers run them:
//   * coop path   -- k_sim_persist: one thread-block cluster (smallest wakes) or one persistent cooperative grid (one CTA per SM) runs all steps while the wake is
//                    small (latency-bound), grid barriers between the phases, the solve CTA's tables resident in
//                    shared memory.
//   * graph path  -- four kernels per step, grid-wide warp pools, K steps captured once in a CUDA graph and replayed
//                    (step index and vortex counts are read from device memory; graphs cached per power-of-two
//                    bracket of the wake size).  In fast mode with wakes >= SIM_TILED_MIN_WAKE the step is the
//                    overlapped one: the old wake's self-convection (shared-memory tiled kernel) on a second graph
//                    branch beside phase 1 + solve.
//   * far-field steps -- opt-in (ludvm_sim_enable_far_field), wakes >= SIM_FAR_FIELD_MIN_WAKE: the overlapped step with the
//                    old wake's self-convection through the treecode (tree.cu), enqueued step by step from the host.
//   * CTA path    -- k_sim_cta: one persistent CTA runs ALL steps of one case with __syncthreads() between phases;
//                    cases are pulled from an atomic counter.  Used for batched parameter sweeps (config 4: 4096
//                    independent cases, no collective).
// Both methods take the coop and graph paths.  method='Ramesh' differs only in the solve (its Newton loops run on the
// solve CTA, grid_downwash) and, in exact mode, in phase 1, which evaluates the step's Newton wake instead of the old one.
// The once-per-step scalar reductions live in block_reduce.cuh.  -DLUDVM_TRACE adds clock64 phase traces (scripts/
// solve_trace.py); it is off in the shipped library.
#include <algorithm>
#include <chrono>
#include <map>

#include "biot_savart.cuh"
#include "block_reduce.cuh"

namespace ludvm {

#define SIM_DMAX 11          // at most 2^11 tree nodes per row are evaluated by separate warps
#define SOLVE_THREADS 256
#define CTA_THREADS 256
#define PI_D 3.141592653589793
#define SIM_TILED_MIN_WAKE 2048   // fast mode: wakes at least this large use the tiled convection kernel (measured: 8192 -> 5.48 s,
                                  // 4096 -> 5.31 s, 2048 -> 5.30 s, 1024 -> 5.29 s for the 20 000-step dt = 2e-3 run)
#define SIM_TILED_CHUNKS_MAX 64   // partial-sum slots per row of the tiled convection
#define SIM_EXACT_TILED_MIN_WAKE 8192   // exact mode, graph path: wakes at least this large use k_conv_partials_exact_tiled
#define SIM_COOP_MAX_WAKE 8192    // wakes up to this size are stepped by the persistent cooperative kernel
#define SIM_CLUSTER_CTAS 16       // the single-cluster persistent kernel: CTAs (16 = the non-portable maximum) x 256 threads
#define SIM_CLUSTER_MAX_WAKE 512  // wakes up to this size are stepped by the single-cluster kernel.  README
                                  // case, us per step over the 400 steps, exact / fast: cluster up to 128: 32.2 / 26.1, 256: 31.1 / 25.3,
                                  // 384: 30.2 / 24.8, 512: 29.6 / 24.4, all 604: 31.0 / 25.0; cooperative grid alone 33.4 / 26.9
                                  // (profiles/r02l_coop_probe.txt): past ~500 vortices the O(N^2) phases want more than 16 SMs
#define SIM_FAR_FIELD_MIN_WAKE 65536   // far_field_order set: steps whose wake bound is at least this take the far-field step.
                                       // Fast-mode ms per step, all pairs / far field at order 18, gust of nfree vortices
                                       // (profiles/far_field_time_loop_probe.txt; B200, 1000 W): 2^14 0.35 / 1.53,
                                       // 2^15 1.01 / 1.94, 2^16 3.67 / 2.14, 2^17 14.4 / 2.74
static_assert(SIM_FAR_FIELD_MIN_WAKE >= SIM_TILED_MIN_WAKE, "the far-field step replaces branch B of the overlapped step");
#define FINISH_STAGE 4096         // doubles of staging in the loads block of k_finish
#define SOLVE_SMEM_LIMIT (200 * 1024)   // dynamic shared memory of the solve kernel (bytes)
#define LUDVM_MAX_PANELS 1024     // Npoints - 1 <= this: 18 doubles per panel of the solve kernel's fixed shared memory


struct SimDev {
    int nt, P, Nc, nfree, nv, method, mode, store_history;   // store_history = k >= 1: TEV/LEV rows of steps i % k == 0 are kept
    int target_warps;   // parallelism target used to pick split depths (same value in every phase of a case)
    int sum_nodes;      // doubles of shared-memory staging (block_np_sum tree nodes, block_fold / block_trapz batches)
    int sinn_smem;      // 1: the sin(n theta) table [Nc,P] is copied to shared memory at the head of the solve phase
    int wof_single;     // 1: phase 1 leaves ONE finished sum per gamma point in pa_u / pa_w (one-CTA driver, fast mode)
    int range_bad_init; // host verdict on the tables and vc^4 (1: outside the range-proof window, or LUDVM_EXACT_FLAGS set)
    int af_stride;      // row stride of the [nv,P] bound-vortex arrays (P, or 0 in compact sweep mode)
    int fourier_rows;   // nt, or 2 in compact sweep mode (row i lives at i % fourier_rows)
    double dt, Uinf, chord, rho, piv, vc4, ic, sum_free, maxerror, epsilon, lespcrit0, a0_init, a1_init;
    int maxiter;
    // tables
    const double *cos_a, *sin_a, *alpha_dot, *h_dot, *gp, *le, *te;
    const double *detadx_p, *eta_p, *x_p, *theta_p, *dtheta, *cos_tp, *sin_tp, *cosn, *sinn, *free_g, *free_xz;
    // resident vortex state: [TEV nv | LEV nv | FREE nfree]
    double *wx, *wz, *wg;
    // results
    double *g_bound, *g_airfoil, *gamma_airfoil, *Gamma_airfoil, *fourier, *lesp, *lesp_prev, *lev_shed;
    double *Fn, *Fs, *L, *D, *T, *M;
    double *path_tev, *path_lev, *path_free;  // nullable
    double *dp;           // nullable: chordwise pressure jump [nt,P] (ludvm_sim_enable_pressure)
    // step bookkeeping
    long long *counters;  // [0] steps done, [1] itev of the last step, [2] ilev of the last step, [3] error flags
    int *ilev_arr;        // [nt+1]: ilev at the start of step i
    double *lespcrit_cur; // sign-carrying LESPcrit (LUDVM.py:802-805)
    // scratch
    double *pa_u, *pa_w;  // wake-on-foil partials        [2^d1][P]
    double *pb_u, *pb_w;  // loads+convection partials    [2^d2][P + Nw2]
    double *foil_u, *foil_w;  // bound vortices on the wake [Nw2]
    double *gp_u, *gp_w;      // overlapped step: wake velocity at the gamma points [P]
    double *pre_sums;         // graph path: np.sum(Gamma_TEV[:itev]), np.sum(Gamma_LEV[:ilev]) of the current step
    // exact mode: sticky verdict of the range proof behind the flag-free pair arithmetic (common.cuh,
    // coord_in_safe_window).  0 = every coordinate the all-pairs kernels have seen so far -- host tables, free vortices,
    // every vortex placed or moved by a step -- lies in the window, so the per-pair range words are skipped; set to 1
    // (by the host for the tables / vc^4, by k_case_init, the solve and the Euler update on the device) it sends every
    // later evaluation through the flagged instantiation.
    int *range_bad;
};

__device__ __forceinline__ bool range_safe(const SimDev &S) { return *(volatile const int *)S.range_bad == 0; }
__device__ __forceinline__ void range_note(const SimDev &S, double x, double z)
{
    if (!(coord_in_safe_window(x) && coord_in_safe_window(z))) *(volatile int *)S.range_bad = 1;
}

__host__ __device__ __forceinline__ int ilog2_ceil_i(int v)
{
    int l = 0;
    while ((1 << l) < v) l++;
    return l;
}

// Split depth for `nrows` target rows against n sources (identical on host and device, in every phase).
__host__ __device__ __forceinline__ int sim_depth(int n, int nrows, int target_warps)
{
    int quads = (nrows + 3) >> 2;
    int want = ilog2_ceil_i(max(1, target_warps / max(1, quads)));
    int d = min(pw_max_depth(n), want);
    return min(d, SIM_DMAX);
}
__host__ __device__ __forceinline__ int sim_chunks(int n, int nrows, int target_warps)
{
    int quads = (nrows + 3) >> 2;
    int c = max(1, target_warps / max(1, quads));
    c = min(c, (n + 63) / 64);
    return min(max(c, 1), 1 << SIM_DMAX);
}

// Phase 1 has only P target rows: its partials per row are capped (2^6 tree nodes / 64 chunks) so that the fold at
// the head of the solve kernel -- the step's critical path -- stays short; 64 x P/4 warp tasks still cover every SM.
#define SIM_WOF_MAX_DEPTH 6
__host__ __device__ __forceinline__ int wof_fold(int mode, int n, int P, int target_warps, int single = 0)
{
    if (single && mode != LUDVM_EXACT_F64) return 1;
    return mode == LUDVM_EXACT_F64 ? min(sim_depth(n, P, target_warps), SIM_WOF_MAX_DEPTH)
                                   : min(sim_chunks(n, P, target_warps), 1 << SIM_WOF_MAX_DEPTH);
}

// Node of numpy's pairwise tree over n elements, cut at depth d (pw_node's numbering), that holds logical element e.
__device__ __forceinline__ int pw_node_of(int n, int d, int e)
{
    int b = 0;
    for (int l = d - 1; l >= 0; l--) {
        const int n2 = pw_left(n);
        if (e >= n2) {
            b |= 1 << l;
            e -= n2;
            n -= n2;
        } else {
            n = n2;
        }
    }
    return b;
}

struct Step {
    int i, itev, ilev;
};

struct Pool {  // the warps / threads that cooperate on a phase
    int wid, nwarps, lane, tid, nth;
};

__device__ __forceinline__ Pool grid_pool()
{
    Pool p;
    p.lane = threadIdx.x & 31;
    p.wid = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    p.nwarps = gridDim.x * (blockDim.x >> 5);
    p.tid = blockIdx.x * blockDim.x + threadIdx.x;
    p.nth = gridDim.x * blockDim.x;
    return p;
}
__device__ __forceinline__ Pool block_pool()
{
    Pool p;
    p.lane = threadIdx.x & 31;
    p.wid = threadIdx.x >> 5;
    p.nwarps = blockDim.x >> 5;
    p.tid = threadIdx.x;
    p.nth = blockDim.x;
    return p;
}

__device__ __forceinline__ bool step_begin(const SimDev &S, int s, Step &st)
{
    long long i = S.counters[0] + s + 1;
    if (i >= S.nt) return false;
    st.i = (int)i;
    st.itev = st.i - 1;
    st.ilev = S.ilev_arr[st.i];
    return true;
}

// wake = TEV[:nT] ++ LEV[:nL] ++ FREE
__device__ __forceinline__ SrcView wake_view(const SimDev &S, int nT, int nL)
{
    SrcView v;
    v.x = S.wx; v.z = S.wz; v.g = S.wg; v.vc4 = nullptr; v.vc4s = S.vc4;
    v.n0 = nT; v.n01 = nT + nL; v.n = nT + nL + S.nfree;
    v.o1 = S.nv; v.o2 = 2 * S.nv; v.gstride = 1;
    return v;
}

struct TgtGamma {  // the P gamma points of step i
    const double *x, *z;
    __device__ __forceinline__ void get(int r, double &xp, double &zp) const { xp = x[r]; zp = z[r]; }
};

struct TgtGammaWake {  // rows [0,P): gamma points; rows [P, P+Nw): wake vortices in logical order
    const double *gx, *gz;
    int P;
    SrcView W;
    __device__ __forceinline__ void get(int r, double &xp, double &zp) const
    {
        if (r < P) {
            xp = gx[r];
            zp = gz[r];
        } else {
            int p = W.phys(r - P);
            xp = W.x[p];
            zp = W.z[p];
        }
    }
};

struct TgtWake {
    SrcView W;
    __device__ __forceinline__ void get(int r, double &xp, double &zp) const
    {
        int p = W.phys(r);
        xp = W.x[p];
        zp = W.z[p];
    }
};

// Positions of the two vortices a step may add, from data known before the solve (LUDVM.py:672-681, :784-800).
__device__ __forceinline__ void place_tev(const SimDev &S, int i, int itev, double &xt, double &zt)
{
    if (itev == 0) {
        xt = S.te[0] + 0.5 * S.Uinf * S.dt;
        zt = S.te[1] + 0.0;
    } else {
        double tex = S.te[(size_t)i * 2], tez = S.te[(size_t)i * 2 + 1];
        xt = tex + 1.0 / 3 * (S.wx[itev - 1] - tex);
        zt = tez + 1.0 / 3 * (S.wz[itev - 1] - tez);
    }
}
__device__ __forceinline__ void place_lev(const SimDev &S, int i, int ilev, double &xl, double &zl)
{
    double lex = S.le[(size_t)i * 2], lez = S.le[(size_t)i * 2 + 1];
    xl = lex;
    zl = lez;
    if (ilev > 0 && S.lev_shed[i - 1] != -1.0) {
        xl = lex + 1.0 / 3 * (S.wx[S.nv + ilev - 1] - lex);
        zl = lez + 1.0 / 3 * (S.wz[S.nv + ilev - 1] - lez);
    }
}

struct TgtWakePlus {  // rows [0, n): the old wake; n: the new TEV; n + 1: the LEV if one is shed; n + 2: the idle LEV slot (origin)
    SrcView W;
    double xt, zt, xl, zl;
    __device__ __forceinline__ void get(int r, double &xp, double &zp) const
    {
        if (r < W.n) {
            int p = W.phys(r);
            xp = W.x[p];
            zp = W.z[p];
        } else if (r == W.n) {
            xp = xt; zp = zt;
        } else if (r == W.n + 1) {
            xp = xl; zp = zl;
        } else {
            xp = 0.0; zp = 0.0;
        }
    }
};

// ---------------------------------------------------------------------------------------------------
// phase 1: wake TEV[:nT] ++ LEV[:nL] ++ FREE on the gamma points (LUDVM.py:584 via :692, :746)
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void phase_wake_on_foil(const SimDev &S, const Step &st, int nT, int nL, const Pool &pl)
{
    SrcView W = wake_view(S, nT, nL);
    TgtGamma T{S.gp + ((size_t)st.i * 2 + 0) * S.P, S.gp + ((size_t)st.i * 2 + 1) * S.P};
    long nquads = (S.P + 3) >> 2;
    const int fold = wof_fold(S.mode, W.n, S.P, S.target_warps, 0);
    if (S.mode == LUDVM_EXACT_F64) {
        if (range_safe(S))
            for (long t = pl.wid; t < (nquads << fold); t += pl.nwarps)
                exact_rows_warp_task<1, false>(W, T, S.P, fold, t, pl.lane, S.pa_u, S.pa_w);
        else
            for (long t = pl.wid; t < (nquads << fold); t += pl.nwarps)
                exact_rows_warp_task<1, true>(W, T, S.P, fold, t, pl.lane, S.pa_u, S.pa_w);
    } else {
        for (long t = pl.wid; t < nquads * fold; t += pl.nwarps)
            fast_rows_warp_task(W, T, S.P, fold, t, pl.lane, S.pa_u, S.pa_w);
    }
}

// ---------------------------------------------------------------------------------------------------
// phase 2 helpers
// ---------------------------------------------------------------------------------------------------

// unit-strength influence of a vortex at (xv, zv) on panel j (LUDVM.py:749-754): T = detadx*ut - un
__device__ __noinline__ double unit_T(const SimDev &S, double xa, double za, double xv, double zv, double ca,
                                         double sa, double detadx)
{
    double tu, tw;
    pair_exact(xa, za, xv, zv, 1.0, S.vc4, tu, tw);
    double u = 0.0 + (-0.0 + tu), w = 0.0 + (-0.0 + tw);  // np.sum over one element
    double ut = u * ca - w * sa;
    double un = u * sa + w * ca;
    return detadx * ut - un;
}

// LAPACK dgesv on a 2x2 system (SURVEY.md A.3)
__device__ __forceinline__ void solve2x2(double a00, double a01, double a10, double a11, double b0, double b1,
                                         double &x0, double &x1)
{
    if (fabs(a10) > fabs(a00)) {
        double t;
        t = a00; a00 = a10; a10 = t;
        t = a01; a01 = a11; a11 = t;
        t = b0; b0 = b1; b1 = t;
    }
    double l = a10 * (1.0 / a00);
    double u11 = a11 - l * a01;
    double y1 = fma(-l, b0, b1);
    x1 = y1 / u11;
    x0 = fma(-a01, x1, b0) / a00;
}

// Constant per-case tables of the scalar phases, resident in shared memory: panel tables [P] always, the
// cos(n theta) / sin(n theta) tables [Nc,P] when they fit (S.sinn_smem), else read from global memory.  Staged once
// per kernel launch (k_solve), once per case (one-CTA driver) or once per launch of the persistent grid.
struct StepTables {
    double *dth, *cm1, *ones, *detadx, *eta, *xp, *costp, *sintp, *dtheta, *dxp;  // cm1, ones adjacent (block_trapz operands)
    const double *cosn, *sinn;
    __device__ __forceinline__ StepTables(double *sm, const SimDev &S)
    {
        const int P = S.P;
        dth = sm; cm1 = dth + P; ones = cm1 + P; detadx = ones + P; eta = detadx + P; xp = eta + P; costp = xp + P;
        sintp = costp + P; dtheta = sintp + P; dxp = dtheta + P;
        cosn = S.sinn_smem ? dxp + P : S.cosn;
        sinn = S.sinn_smem ? dxp + P + (size_t)S.Nc * P : S.sinn;
    }
};
#define SINN_SMEM_MAX 4096   // largest cos/sin(n theta) table (doubles each) kept in shared memory
#define TABLE_SMEM_DOUBLES(P, Nc, big) (10 * (P) + ((big) ? 2 * (Nc) * (P) : 0))

// Fill the tables (all threads of the block).  The two large tables travel asynchronously (cp.async); call
// tables_wait() and a block barrier before reading them.
__device__ __forceinline__ void stage_tables(const SimDev &S, const StepTables &t)
{
    const int P = S.P, tid = threadIdx.x, nth = blockDim.x;
    if (S.sinn_smem) {
        const int n = S.Nc * P;
        double *dc = const_cast<double *>(t.cosn), *ds = const_cast<double *>(t.sinn);
        for (int idx = tid; idx < n; idx += nth) {
            asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(dc + idx)), "l"(S.cosn + idx));
            asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(ds + idx)), "l"(S.sinn + idx));
        }
        asm volatile("cp.async.commit_group;");
    }
    for (int j = tid; j < P; j += nth) {
        t.dth[j] = (j + 1 < P) ? S.theta_p[j + 1] - S.theta_p[j] : 0.0;   // np.trapz's d = x[1:] - x[:-1]
        t.cm1[j] = S.cos_tp[j] - 1;
        t.ones[j] = 1.0;
        t.detadx[j] = S.detadx_p[j];
        t.eta[j] = S.eta_p[j];
        t.xp[j] = S.x_p[j];
        t.costp[j] = S.cos_tp[j];
        t.sintp[j] = S.sin_tp[j];
        t.dtheta[j] = S.dtheta[j];
        t.dxp[j] = (j + 1 < P) ? S.x_p[j + 1] - S.x_p[j] : 0.0;
    }
}
__device__ __forceinline__ void tables_wait() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

struct Kin {  // per-step kinematics
    double ca, sa, ad, hd;
    const double *xa, *za;
};

// airfoil_downwash epilogue (LUDVM.py:587-593): global (u1,w1) at gamma point j -> normal downwash W_j
__device__ __noinline__ double downwash_at(const SimDev &S, const StepTables &t, const Kin &k, const double *u1,
                                           const double *w1, int j)
{
    double s1 = S.Uinf * k.ca + k.hd * k.sa, us = S.Uinf * k.sa, hc = k.hd * k.ca;
    double u = u1[j] * k.ca - w1[j] * k.sa;
    double w = u1[j] * k.sa + w1[j] * k.ca;
    return t.detadx[j] * (s1 + u - k.ad * t.eta[j]) - us - k.ad * (t.xp[j] - S.piv) + hc - w;
}

struct SolveSmem {  // carve-up of the solve phase's scratch shared memory (after the tables)
    double *u1, *w1, *T1, *T2, *T3, *W, *dG, *Wu, *A, *sc, *nodes;
    __device__ __forceinline__ SolveSmem(double *sm, int P, int Nc)
    {
        u1 = sm; w1 = u1 + P; T1 = w1 + P; T2 = T1 + P; T3 = T2 + P; W = T3 + P; dG = W + P; Wu = dG + P;
        A = Wu + P; sc = A + Nc; nodes = sc + 32;
    }
};
#define SOLVE_SCRATCH_DOUBLES(P, Nc, sum_nodes) (8 * (P) + (Nc) + 32 + (sum_nodes))
#define SOLVE_SMEM_DOUBLES(P, Nc, sum_nodes, big) (TABLE_SMEM_DOUBLES(P, Nc, big) + SOLVE_SCRATCH_DOUBLES(P, Nc, sum_nodes))

// Fold the phase-1 partials into u1, w1 (block-wide; ends with a barrier).
__device__ __forceinline__ void fold_wake_on_foil(const SimDev &S, int n1, const SolveSmem &m)
{
    block_fold(S.pa_u, S.pa_w, S.P, S.P, wof_fold(S.mode, n1, S.P, S.target_warps, S.wof_single), S.mode == LUDVM_EXACT_F64,
               m.nodes, S.sum_nodes, m.u1, m.w1);
}

// Fourier coefficients n0 .. n0+nq-1 of the downwash into A[]: A0 = -1/pi*trapz(W/Uinf), An = 2/pi*trapz(W/Uinf*
// cos(n theta)) (LUDVM.py:694-695, :769-771).  Wu[j] = W[j] / Uinf (tabulated: the same division); row 0 of the
// cos(n theta) table is cos(0) = 1.0 exactly, so A0's integrand W/Uinf * 1.0 needs no special case.  Block-wide.
__device__ __forceinline__ void block_fourier(const SimDev &S, const StepTables &t, const SolveSmem &m, int n0, int nq,
                                              double *A)
{
    block_trapz(m.Wu, 0, 0, t.cosn + (size_t)n0 * S.P, 0, S.P, t.dth, S.P, nq, m.nodes, S.sum_nodes, A + n0);
    for (int n = n0 + threadIdx.x; n < n0 + nq; n += blockDim.x) A[n] = (n == 0 ? (-1 / PI_D) : (2 / PI_D)) * A[n];
    __syncthreads();
}

// Whole-block airfoil_downwash of the wake TEV[:nT] ++ LEV[:nL] ++ FREE (used by the Ramesh iterations):
// fills W and Wu = W / Uinf.
__device__ __noinline__ void cta_downwash(const SimDev &S, const StepTables &t, const Step &st, const Kin &k, int nT, int nL,
                                          const SolveSmem &m)
{
    __syncthreads();  // circulation guesses written by thread 0 are visible
    phase_wake_on_foil(S, st, nT, nL, block_pool());
    fold_wake_on_foil(S, nT + nL + S.nfree, m);
    for (int j = threadIdx.x; j < S.P; j += blockDim.x) {
        double w = downwash_at(S, t, k, m.u1, m.w1, j);
        m.W[j] = w;
        m.Wu[j] = w / S.Uinf;
    }
    __syncthreads();
}

// The same downwash on the grid drivers, whose phase 1 ran grid-wide before the solve; the wake is not summed again.
// Between the Newton evaluations of a step only two elements of the wake change: logical itev (the TEV) and itev+1+ilev
// (the LEV slot), in circulation, plus the LEV position set once before the 2-D loop.
//   exact: phase 1 left the tree-node partials of the Newton wake TEV[:itev+1] ++ LEV[:ilev+1] ++ FREE (same cut and
//          [node][P] layout as here).  The <= 2 nodes holding those elements are evaluated again over their slots, then
//          folded.  A node's partial is a pure function of its range, so this is the full evaluation bit for bit.
//   fast:  m.T1 / m.T2 hold the folded sums of the old wake TEV[:itev] ++ LEV[:ilev] ++ FREE (Faure's phase 1); the two
//          new vortices' terms are added at each gamma point, in k_conv_new's order.
__device__ __noinline__ void grid_downwash(const SimDev &S, const StepTables &t, const Step &st, const Kin &k,
                                           const SolveSmem &m)
{
    __syncthreads();  // circulation guesses written by thread 0 are visible
    const int P = S.P, itev = st.itev, lev = S.nv + st.ilev;
    if (S.mode == LUDVM_EXACT_F64) {
        const SrcView W = wake_view(S, itev + 1, st.ilev + 1);
        const TgtGamma T{k.xa, k.za};
        const int d = wof_fold(S.mode, W.n, P, S.target_warps);
        const int b0 = pw_node_of(W.n, d, itev), b1 = pw_node_of(W.n, d, itev + 1 + st.ilev);
        const int ng = (P + 3) >> 2, ntask = (b0 == b1 ? 1 : 2) * ng;
        const Pool pl = block_pool();
        const bool safe = range_safe(S);
        for (int q = pl.wid; q < ntask; q += pl.nwarps) {
            const long task = q < ng ? (long)b0 * ng + q : (long)b1 * ng + (q - ng);
            if (safe) exact_rows_warp_task<1, false>(W, T, P, d, task, pl.lane, S.pa_u, S.pa_w);
            else exact_rows_warp_task<1, true>(W, T, P, d, task, pl.lane, S.pa_u, S.pa_w);
        }
        fold_wake_on_foil(S, W.n, m);
    } else {
        const double xt = S.wx[itev], zt = S.wz[itev], gt = S.wg[itev] * LUDVM_INV_TWO_PI;
        const double xl = S.wx[lev], zl = S.wz[lev], gl = S.wg[lev] * LUDVM_INV_TWO_PI;
        for (int j = threadIdx.x; j < P; j += blockDim.x) {
            double u = m.T1[j], w = m.T2[j];
            pair_fast(k.xa[j], k.za[j], xt, zt, gt, S.vc4, u, w);
            pair_fast(k.xa[j], k.za[j], xl, zl, gl, S.vc4, u, w);
            m.u1[j] = u;
            m.w1[j] = w;
        }
    }
    for (int j = threadIdx.x; j < P; j += blockDim.x) {
        double w = downwash_at(S, t, k, m.u1, m.w1, j);
        m.W[j] = w;
        m.Wu[j] = w / S.Uinf;
    }
    __syncthreads();
}

// Downwash of the Newton wake TEV[:itev+1] ++ LEV[:ilev+1] ++ FREE into W, Wu.
template <bool GRID>
__device__ __forceinline__ void newton_downwash(const SimDev &S, const StepTables &t, const Step &st, const Kin &k,
                                                const SolveSmem &m)
{
    if (GRID) grid_downwash(S, t, st, k, m);
    else cta_downwash(S, t, st, k, st.itev + 1, st.ilev + 1, m);
}

// Kelvin residual of the Newton loops (LUDVM.py:697-699, :825-827).  Leaves A0 in sc[20], A1 in sc[21], the bound
// circulation in sc[24]; returns the residual on every thread.  One copy per GRID (phase_solve): the sweep driver's copy
// sees its descriptor in shared memory only, and keeps the code it had before the grid drivers called it.
template <bool GRID>
__device__ __noinline__ double cta_kelvin_f(const SimDev &S, const StepTables &t, const Step &st, const SolveSmem &m)
{
    block_fourier(S, t, m, 0, 2, m.sc + 20);
    double sT = block_np_sum(S.wg, st.itev + 1, m.nodes, S.sum_nodes);
    double sL = block_np_sum(S.wg + S.nv, st.ilev + 1, m.nodes, S.sum_nodes);
    double cb = S.Uinf * S.chord * PI_D * (m.sc[20] + m.sc[21] / 2);
    double f = cb + sT + sL + S.sum_free - S.ic;
    if (threadIdx.x == 0) m.sc[24] = cb;
    __syncthreads();
    return f;
}

// ---------------------------------------------------------------------------------------------------
// phase 2: the scalar phases (one CTA).  Faure expects the phase-1 partials of TEV[:itev] ++ LEV[:ilev] ++ FREE.
// Every reduction over the panels (np.trapz, np.sum) is evaluated by an 8-lane group in numpy's own order, so the
// 30 Fourier coefficients, the I/J integrals and the row folds all run side by side; scalars that every thread
// needs are recomputed by every thread from shared operands (identical arithmetic) instead of being broadcast
// through another barrier.
// ---------------------------------------------------------------------------------------------------
// `tab` = shared memory of the StepTables (staged here when stage_now, else already resident), `sm` = scratch.
// GRID (Ramesh): phase 1 ran grid-wide before this solve, so the Newton evaluations use grid_downwash; the one-CTA sweep
// driver keeps cta_downwash.
template <int METHOD, bool GRID = false>
__device__ void phase_solve(const SimDev &S, const Step &st, double *tab, double *sm, const double *pre_sums,
                            bool stage_now)
{
    const int P = S.P, Nc = S.Nc, tid = threadIdx.x, nth = blockDim.x;
    const int i = st.i, itev = st.itev, ilev = st.ilev, nv = S.nv;
    const StepTables t(tab, S);
    const SolveSmem m(sm, P, Nc);
    double *const T1 = m.T1, *const T2 = m.T2, *const T3 = m.T3, *const W = m.W, *const Wu = m.Wu, *const dG = m.dG;
    double *const A = m.A, *const sc = m.sc;
    // sc[]: 0 xt, 1 zt, 4 I1, 5 I2, 6 trapz(T1), 7 trapz(T2), 8 I3, 9 trapz(T3), 10 gtev, 11 glev, 13 xl, 14 zl,
    //       15 lespcrit, 16 bound, 20.. Newton scratch
    Kin k{S.cos_a[i], S.sin_a[i], S.alpha_dot[i], S.h_dot[i], S.gp + ((size_t)i * 2 + 0) * P,
          S.gp + ((size_t)i * 2 + 1) * P};
    const double ca = k.ca, sa = k.sa;
    const double Uinf = S.Uinf, chord = S.chord, dt = S.dt;
    constexpr bool ramesh = METHOD == LUDVM_METHOD_RAMESH;
    double *F = S.fourier + (size_t)(i % S.fourier_rows) * 2 * Nc;
    const double *Fprev = S.fourier + (size_t)((i - 1) % S.fourier_rows) * 2 * Nc;

    TRACE(0);
    // operands of the TEV placement: loads issued first, consumed after the table set-up below
    double tex = 0.0, tez = 0.0, pxw = 0.0, pzw = 0.0, lc0 = 0.0;
    if (tid == 0) {
        const size_t it = itev == 0 ? 0 : (size_t)i;
        tex = S.te[it * 2];
        tez = S.te[it * 2 + 1];
        if (itev > 0) {
            pxw = S.wx[itev - 1];
            pzw = S.wz[itev - 1];
        }
        lc0 = *S.lespcrit_cur;
    }
    if (stage_now) stage_tables(S, t);
    // TEV placement (LUDVM.py:672-681)
    if (tid == 0) {
        double xt, zt;
        if (itev == 0) {
            xt = tex + 0.5 * Uinf * dt;
            zt = tez + 0.0;
        } else {
            xt = tex + 1.0 / 3 * (pxw - tex);
            zt = tez + 1.0 / 3 * (pzw - tez);
        }
        sc[0] = xt;
        sc[1] = zt;
        S.wx[itev] = xt;
        S.wz[itev] = zt;
        range_note(S, xt, zt);
        sc[15] = lc0;
        sc[11] = 0.0;
        if (ramesh && ilev < nv) {  // row i of path['LEV'] starts with a zero slot (SURVEY.md B.3)
            S.wx[nv + ilev] = 0.0;
            S.wz[nv + ilev] = 0.0;
        }
    }
    double sT = 0.0, sL = 0.0;  // np.sum(circulation['TEV'][:itev]), np.sum(circulation['LEV'][:ilev])
    if (!ramesh) {
        // Faure closed form (LUDVM.py:741-773)
        TRACE(1);
        fold_wake_on_foil(S, itev + ilev + S.nfree, m);
        TRACE(2);
        if (pre_sums) {   // evaluated beside phase 1 (graph path): identical arithmetic, off the critical path
            sT = pre_sums[0];
            sL = pre_sums[1];
        } else {
            sT = block_np_sum(S.wg, itev, m.nodes, S.sum_nodes);       // LUDVM.py:758-759
            TRACE(3);
            sL = block_np_sum(S.wg + nv, ilev, m.nodes, S.sum_nodes);
        }
        TRACE(4);
        for (int idx = tid; idx < 2 * P; idx += nth) {
            if (idx < P) T1[idx] = downwash_at(S, t, k, m.u1, m.w1, idx);
            else T2[idx - P] = unit_T(S, k.xa[idx - P], k.za[idx - P], sc[0], sc[1], ca, sa, t.detadx[idx - P]);
        }
        TRACE(5);
        // I1, I2 (LUDVM.py:756-757) -> sc[4], sc[5] and -- needed only if a LEV is shed, but free here -- the raw
        // integrals of J1, J2 (LUDVM.py:940-941) -> sc[6], sc[7]   (T2 = T1 + P, ones = cm1 + P in the layout)
        if (stage_now) tables_wait();   // the barrier inside block_trapz publishes the async copies
        block_trapz(T1, 1, P, t.cm1, 1, P, t.dth, P, 4, m.nodes, S.sum_nodes, sc + 4);
        TRACE(6);
        const double I1 = sc[4], I2 = sc[5];
        const double gtev = -(I1 + sT + sL + S.sum_free - S.ic) / (1 + I2);  // LUDVM.py:758-760
        if (tid == 0) {
            sc[10] = gtev;
            sc[16] = I1 + gtev * I2;                                          // circulation['bound'], LUDVM.py:762
        }
        for (int j = tid; j < P; j += nth) {                                  // LUDVM.py:767
            double w = T1[j] + gtev * T2[j];
            W[j] = w;
            Wu[j] = w / Uinf;
        }
        TRACE(7);
        block_fourier(S, t, m, 0, Nc, A);                                        // LUDVM.py:769-773
        for (int n = tid; n < Nc; n += nth) F[Nc + n] = (A[n] - Fprev[n]) / dt;
        TRACE(8);
    } else {
        // Ramesh 1-D Newton on the TEV strength (LUDVM.py:683-739)
        if (tid == 0) {
            sc[26] = 1.0;   // f
            sc[27] = -1.0;  // shed_vortex_gamma
        }
        if (stage_now) tables_wait();
        __syncthreads();
        if (GRID && S.mode != LUDVM_EXACT_F64) {   // the old wake's sums at the gamma points, fixed for the step
            fold_wake_on_foil(S, itev + ilev + S.nfree, m);
            for (int j = tid; j < P; j += nth) {
                T1[j] = m.u1[j];
                T2[j] = m.w1[j];
            }
        }
        int niter = 1;
        while (fabs(sc[26]) > S.maxerror && niter < S.maxiter) {
            double shed = sc[27];
            if (tid == 0) S.wg[itev] = shed;
            newton_downwash<GRID>(S, t, st, k, m);
            double f = cta_kelvin_f<GRID>(S, t, st, m);
            if (tid == 0) S.wg[itev] = shed + S.epsilon;
            newton_downwash<GRID>(S, t, st, k, m);
            double fdelta = cta_kelvin_f<GRID>(S, t, st, m);
            if (tid == 0) {
                double fprime = (fdelta - f) / S.epsilon;
                sc[27] = shed - f / fprime;
                sc[26] = f;
                S.wg[itev] = sc[27];
            }
            __syncthreads();
            niter++;
        }
        newton_downwash<GRID>(S, t, st, k, m);
        block_fourier(S, t, m, 0, Nc, A);
        for (int n = tid; n < Nc; n += nth) F[Nc + n] = (A[n] - Fprev[n]) / dt;
        if (tid == 0) {
            sc[10] = S.wg[itev];
            sc[16] = Uinf * chord * PI_D * (A[0] + A[1] / 2);  // LUDVM.py:734
        }
        __syncthreads();
    }
    // LESP test (LUDVM.py:775-781); |.| makes the comparison blind to the sign flip thread 0 applies below
    if (tid == 0) S.lesp_prev[itev] = A[0];
    const bool shed = fabs(A[0]) >= fabs(sc[15]);
    if (shed) {
        // LEV placement (LUDVM.py:784-805), evaluated by every thread
        double lex = S.le[(size_t)i * 2], lez = S.le[(size_t)i * 2 + 1], xl = lex, zl = lez;
        if (ilev > 0 && S.lev_shed[i - 1] != -1.0) {
            xl = lex + 1.0 / 3 * (S.wx[nv + ilev - 1] - lex);
            zl = lez + 1.0 / 3 * (S.wz[nv + ilev - 1] - lez);
        }
        if (!ramesh) {
            // Faure 2x2 linear system (LUDVM.py:916-961); T1, T2, I1, I2 are unchanged recomputations there
            for (int j = tid; j < P; j += nth) T3[j] = unit_T(S, k.xa[j], k.za[j], xl, zl, ca, sa, t.detadx[j]);
            __syncthreads();   // every thread has evaluated `shed` and read lev_shed[i-1]
            if (tid == 0) {
                sc[13] = xl;
                sc[14] = zl;
                sc[15] = (A[0] < 0) ? -fabs(sc[15]) : fabs(sc[15]);
                S.lev_shed[i] = (double)ilev;
            }
            block_trapz(T3, 0, 0, t.cm1, 0, P, t.dth, P, 2, m.nodes, S.sum_nodes, sc + 8);  // I3, raw J3 -> sc[8], sc[9]
            // LUDVM.py:945-959, on every thread
            const double I1 = sc[4], I2 = sc[5], I3 = sc[8];
            const double J1 = (-1 / PI_D) * sc[6], J2 = (-1 / PI_D) * sc[7], J3 = (-1 / PI_D) * sc[9];
            const double b1 = -(I1 + sT + sL + S.sum_free - S.ic), b2 = sc[15] - J1;
            double x0, x1;
            solve2x2(1 + I2, 1 + I3, J2, J3, b1, b2, x0, x1);
            for (int j = tid; j < P; j += nth) {
                double w = T1[j] + x0 * T2[j] + x1 * T3[j];
                W[j] = w;
                Wu[j] = w / Uinf;
            }
            __syncthreads();
            if (tid == 0) {
                sc[10] = x0;
                sc[11] = x1;
                sc[16] = I1 + x0 * I2 + x1 * I3;
                A[0] = J1 + x0 * J2 + x1 * J3;
            }
            block_fourier(S, t, m, 1, Nc - 1, A);  // LUDVM.py:960-961
        } else {
            __syncthreads();   // every thread has evaluated `shed` and read lev_shed[i-1]
            if (tid == 0) {
                sc[13] = xl;
                sc[14] = zl;
                sc[15] = (A[0] < 0) ? -fabs(sc[15]) : fabs(sc[15]);
                S.lev_shed[i] = (double)ilev;
                S.wx[nv + ilev] = xl;
                S.wz[nv + ilev] = zl;
                range_note(S, xl, zl);
                // Ramesh 2-D Newton on (LEV, TEV) strengths (LUDVM.py:807-909)
                sc[26] = 0.1;          // f1
                sc[27] = 0.1;          // f2
                sc[28] = S.wg[itev];   // TEV_shed_gamma
                sc[29] = S.wg[itev];   // LEV_shed_gamma
            }
            __syncthreads();
            int niter = 1;
            while ((fabs(sc[26]) > S.maxerror || fabs(sc[27]) > S.maxerror) && niter < S.maxiter) {
                double tg = sc[28], lg = sc[29];
                if (tid == 0) { S.wg[itev] = tg; S.wg[nv + ilev] = lg; }
                newton_downwash<GRID>(S, t, st, k, m);
                double f1 = cta_kelvin_f<GRID>(S, t, st, m);
                double cbound = sc[24], f2 = sc[15] - sc[20];
                __syncthreads();
                if (tid == 0) { S.wg[itev] = tg + S.epsilon; S.wg[nv + ilev] = lg; }
                newton_downwash<GRID>(S, t, st, k, m);
                double f1dT = cta_kelvin_f<GRID>(S, t, st, m), f2dT = sc[15] - sc[20];
                __syncthreads();
                if (tid == 0) { S.wg[itev] = tg; S.wg[nv + ilev] = lg + S.epsilon; }
                newton_downwash<GRID>(S, t, st, k, m);
                double f1dL = cta_kelvin_f<GRID>(S, t, st, m), f2dL = sc[15] - sc[20];
                __syncthreads();
                if (tid == 0) {
                    double eps = S.epsilon, x0, x1;
                    solve2x2((f1dL - f1) / eps, (f1dT - f1) / eps, (f2dL - f2) / eps, (f2dT - f2) / eps, f1, f2, x0, x1);
                    sc[29] = lg + (-x0);
                    sc[28] = tg + (-x1);
                    sc[26] = f1;
                    sc[27] = f2;
                    S.wg[itev] = sc[28];
                    S.wg[nv + ilev] = sc[29];
                    sc[16] = cbound;
                }
                __syncthreads();
                niter++;
            }
            newton_downwash<GRID>(S, t, st, k, m);
            block_fourier(S, t, m, 0, Nc, A);  // LUDVM.py:902-909
            if (tid == 0) {
                sc[10] = S.wg[itev];
                sc[11] = S.wg[nv + ilev];
                sc[16] = Uinf * chord * PI_D * (A[0] + A[1] / 2);
            }
            __syncthreads();
        }
    }
    // commit the step's circulations and bookkeeping
    TRACE(9);
    if (tid == 0) {
        S.wg[itev] = sc[10];
        if (shed) {
            S.wg[nv + ilev] = sc[11];
            S.wx[nv + ilev] = sc[13];
            S.wz[nv + ilev] = sc[14];
            range_note(S, sc[13], sc[14]);
        } else if (ilev < nv) {  // untouched slot of row i: zero circulation at the origin (SURVEY.md B.3)
            S.wx[nv + ilev] = 0.0;
            S.wz[nv + ilev] = 0.0;
        }
        S.g_bound[itev] = sc[16];
        S.lesp[itev] = A[0];  // LUDVM.py:971
        S.ilev_arr[i + 1] = ilev + (shed ? 1 : 0);
        *S.lespcrit_cur = sc[15];
    }
    for (int n = tid; n < Nc; n += nth) F[n] = A[n];
    // bound-vortex distribution (LUDVM.py:986-1010)
    const size_t arow = (size_t)itev * S.af_stride;
    const double *sinn = t.sinn;
    for (int j = tid; j < P; j += nth) {
        double term2 = 0;
#pragma unroll 4
        for (int n = 1; n < Nc; n++) term2 = A[n] * sinn[(size_t)n * P + j] + term2;
        double term1 = A[0] * (1 + t.costp[j]) / t.sintp[j];
        double gamma = 2 * Uinf * (term1 + term2);
        double dg = gamma * chord / 2 * t.sintp[j] * t.dtheta[j];
        dG[j] = dg;
        S.g_airfoil[arow + j] = dg;
        S.gamma_airfoil[arow + j] = gamma;
    }
    TRACE(10);
}

// Gamma_j = np.sum(dGamma[:j+1]) (LUDVM.py:1008-1010) of one row of dGamma
__device__ __forceinline__ double gamma_cum_at(const double *dG, int j)
{
    auto f = [&](int kk) { return dG[kk]; };
    return 0.0 + pw_seq(f, 0, j + 1);
}

// Nothing in the step consumes Gamma, so it runs beside the loads.
__device__ __forceinline__ void phase_gamma_cumsum(const SimDev &S, const Step &st, int t0, int nthreads)
{
    const double *dG = S.g_airfoil + (size_t)st.itev * S.af_stride;
    double *out = S.Gamma_airfoil + (size_t)st.itev * S.af_stride;
    for (int j = t0; j < S.P; j += nthreads) out[j] = gamma_cum_at(dG, j);
}

// Pressure jump of step i, the array the reference allocates but never fills (LUDVM.py:1059-1064):
//   dp[i,j] = rho ((Uinf cos a + hdot sin a + u_j) gamma[itev,j] + (Gamma[itev,j] - Gamma[itev-1,j]) / dt)
// u_j = the loads' tangential wake velocity at gamma point j, which phase_finish_loads left in dp[i,j] (same thread, same
// j).  Gamma row itev is summed by another CTA while the loads run (or after them, in the one-CTA driver), so it is formed
// again here with the same expression; row itev - 1 is complete.  Called after the loads, where little else is live
// (inside the loads' loop, or out of line, it cost the kernels around it spills); on the graph path it is a kernel of its
// own after k_finish / k_finish_ov (k_pressure), which keep their register allocation.  In the one-CTA driver
// (the DP sweep instantiations) it runs before that CTA's own phase_gamma_cumsum, so a
// compact sweep case, whose one Gamma row every step overwrites (af_stride = 0), still holds row itev - 1 in it here:
// each thread reads Gprev[j] before the same thread (same j mapping) writes that element in phase_gamma_cumsum.
__device__ __forceinline__ void pressure_row(const SimDev &S, const Step &st)
{
    const int i = st.i, itev = st.itev;
    const double vrel = S.Uinf * S.cos_a[i] + S.h_dot[i] * S.sin_a[i];
    const double *gam = S.gamma_airfoil + (size_t)itev * S.af_stride, *dG = S.g_airfoil + (size_t)itev * S.af_stride;
    const double *Gprev = S.Gamma_airfoil + (size_t)(itev - 1) * S.af_stride;
    double *row = S.dp + (size_t)i * S.P;
    for (int j = threadIdx.x; j < S.P; j += blockDim.x) {
        const double u = row[j], G = gamma_cum_at(dG, j), Gp = itev >= 1 ? Gprev[j] : 0.0;
        row[j] = S.rho * ((vrel + u) * gam[j] + (G - Gp) / S.dt);
    }
}

// ---------------------------------------------------------------------------------------------------
// phase 3: updated wake on (gamma points ++ wake) and bound vortices on the wake
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void phase_conv_partials(const SimDev &S, const Step &st, const Pool &pl)
{
    const int P = S.P;
    SrcView W = wake_view(S, st.itev + 1, st.ilev + 1);
    const double *gx = S.gp + ((size_t)st.i * 2 + 0) * P, *gz = S.gp + ((size_t)st.i * 2 + 1) * P;
    TgtGammaWake TA{gx, gz, P, W};
    TgtWake TW{W};
    SrcView Fo = make_src(S.g_airfoil + (size_t)st.itev * S.af_stride, 1, gx, gz, nullptr, S.vc4, P);
    const int nrows = P + W.n;
    long nquadsA = (nrows + 3) >> 2, nquadsW = (W.n + 3) >> 2;
    if (S.mode == LUDVM_EXACT_F64) {
        int d = sim_depth(W.n, nrows, S.target_warps);
        long nA = nquadsA << d;
        if (range_safe(S)) {
            for (long t = pl.wid; t < nA + nquadsW; t += pl.nwarps) {
                if (t < nA) exact_rows_warp_task<1, false>(W, TA, nrows, d, t, pl.lane, S.pb_u, S.pb_w);
                else exact_rows_warp_task<1, false>(Fo, TW, W.n, 0, t - nA, pl.lane, S.foil_u, S.foil_w);
            }
        } else {
            for (long t = pl.wid; t < nA + nquadsW; t += pl.nwarps) {
                if (t < nA) exact_rows_warp_task<1, true>(W, TA, nrows, d, t, pl.lane, S.pb_u, S.pb_w);
                else exact_rows_warp_task<1, true>(Fo, TW, W.n, 0, t - nA, pl.lane, S.foil_u, S.foil_w);
            }
        }
    } else {
        int c = sim_chunks(W.n, nrows, S.target_warps);
        long nA = nquadsA * c;
        for (long t = pl.wid; t < nA + nquadsW; t += pl.nwarps) {
            if (t < nA) fast_rows_warp_task(W, TA, nrows, c, t, pl.lane, S.pb_u, S.pb_w);
            else fast_rows_warp_task(Fo, TW, W.n, 1, t - nA, pl.lane, S.foil_u, S.foil_w);
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// phase 4: loads (one CTA) and convection update + history (thread pool)
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ int conv_fold(const SimDev &S, const Step &st, int tiled_chunks)
{
    if (tiled_chunks > 0) return tiled_chunks;
    int nw = st.itev + 1 + st.ilev + 1 + S.nfree;
    return S.mode == LUDVM_EXACT_F64 ? sim_depth(nw, S.P + nw, S.target_warps) : sim_chunks(nw, S.P + nw, S.target_warps);
}

// `tab` = shared memory of resident StepTables, or nullptr: then the three tables needed here are built in `sm`.
// `ov`: the wake velocity at the gamma points was already assembled in S.gp_u / S.gp_w (overlapped step).
// DP: the driver can carry the pressure jump (S.dp non-null): u is left in the dp row for pressure_row.  The sweep
// instantiations of k_sim_cta without it compile without the store.
template <bool DP>
__device__ void phase_finish_loads(const SimDev &S, const Step &st, double *tab, double *sm, int tiled_chunks, int cap,
                                   bool ov = false)  // LUDVM.py:1035-1090
{
    const int P = S.P, i = st.i, itev = st.itev, tid = threadIdx.x, nth = blockDim.x;
    const int nrows = P + st.itev + 1 + st.ilev + 1 + S.nfree;
    const bool exact = S.mode == LUDVM_EXACT_F64;
    const int fold = conv_fold(S, st, tiled_chunks);
    double *ug = sm, *ugx = ug + P, *sc = ugx + P, *stage = sc + 8;
    const double *dxp, *ones, *xp;
    const double ca = S.cos_a[i], sa = S.sin_a[i], hd = S.h_dot[i];
    const double *gam = S.gamma_airfoil + (size_t)itev * S.af_stride;
    if (tab) {
        const StepTables t(tab, S);
        dxp = t.dxp; ones = t.ones; xp = t.xp;
    } else {
        double *d = stage + cap, *o = d + P, *x = o + P;
        for (int j = tid; j < P; j += nth) {
            d[j] = (j + 1 < P) ? S.x_p[j + 1] - S.x_p[j] : 0.0;
            o[j] = 1.0;
            x[j] = S.x_p[j];
        }
        dxp = d; ones = o; xp = x;
    }
    if (ov) {
        for (int j = tid; j < P; j += nth) {
            ug[j] = S.gp_u[j];
            ugx[j] = S.gp_w[j];
        }
        __syncthreads();
    } else {
        block_fold(S.pb_u, S.pb_w, nrows, P, fold, exact, stage, cap, ug, ugx);  // wake velocity at the gamma points
    }
    for (int j = tid; j < P; j += nth) {
        double u1 = ug[j], w1 = ugx[j];
        double u = u1 * ca - w1 * sa;
        if (DP && S.dp) S.dp[(size_t)i * P + j] = u;   // pressure_row's input
        ug[j] = u * gam[j];
        ugx[j] = u * gam[j] * xp[j];
    }
    block_trapz(ug, 1, P, ones, 0, 0, dxp, P, 2, stage, cap, sc);   // trapz(ug, x_p), trapz(ugx, x_p)
    if (tid == 0) {
        const double *F = S.fourier + (size_t)(i % S.fourier_rows) * 2 * S.Nc, *Fd = F + S.Nc;
        const double rho = S.rho, chord = S.chord, Uinf = S.Uinf;
        double A0 = F[0], A1 = F[1], A2 = F[2], A0d = Fd[0], A1d = Fd[1], A2d = Fd[2], A3d = Fd[3];
        double vrel = Uinf * ca + hd * sa;
        double Fn = rho * PI_D * chord * Uinf *
                        (vrel * (A0 + 0.5 * A1) + chord * (3.0 / 4 * A0d + 1.0 / 4 * A1d + 1.0 / 8 * A2d)) +
                    rho * sc[0];
        double Fs = rho * PI_D * chord * (Uinf * Uinf) * (A0 * A0);
        double Lf = Fn * ca + Fs * sa;
        double Df = Fn * sa - Fs * ca;
        double Mo = S.piv * Fn -
                    rho * PI_D * (chord * chord) * Uinf *
                        (vrel * (1.0 / 4 * A0 + 1.0 / 4 * A1 - 1.0 / 8 * A2) +
                         chord * (7.0 / 16 * A0d + 3.0 / 16 * A1d + 1.0 / 16 * A2d - 1.0 / 64 * A3d)) -
                    rho * sc[1];
        S.Fn[i] = Fn; S.Fs[i] = Fs; S.L[i] = Lf; S.D[i] = Df; S.T[i] = -Df; S.M[i] = Mo;
        S.counters[1] = itev;
        S.counters[2] = st.ilev;
    }
}

// convection, LUDVM.py:1095-1127: x += dt*(u_wake + u_foil) for TEV[:nT], LEV[:nL], FREE, in place
__device__ __forceinline__ void phase_finish_update(const SimDev &S, const Step &st, long t0, long nthreads,
                                                    int tiled_chunks)
{
    const int P = S.P, i = st.i, nv = S.nv;
    const int nT = st.itev + 1, nL = st.ilev + 1;
    SrcView W = wake_view(S, nT, nL);
    const int nrows = P + W.n;
    const bool exact = S.mode == LUDVM_EXACT_F64;
    const int fold = conv_fold(S, st, tiled_chunks);
    const double dt = S.dt;
    for (long r = t0; r < W.n; r += nthreads) {
        int row = P + (int)r;
        double uw, ww, uf, wf;
        if (exact) {
            uw = exact_combine_row(S.pb_u, nrows, row, fold);
            ww = exact_combine_row(S.pb_w, nrows, row, fold);
            uf = 0.0 + S.foil_u[r];
            wf = 0.0 + S.foil_w[r];
        } else {
            uw = fast_combine_row(S.pb_u, nrows, row, fold);
            ww = fast_combine_row(S.pb_w, nrows, row, fold);
            uf = S.foil_u[r];
            wf = S.foil_w[r];
        }
        int p = W.phys((int)r);
        double xn = S.wx[p] + dt * (uw + uf);
        double zn = S.wz[p] + dt * (ww + wf);
        S.wx[p] = xn;
        S.wz[p] = zn;
        if (exact) range_note(S, xn, zn);
        if (S.store_history) {   // snapshot row i / k of the strided TEV / LEV history; the FREE history is kept in full
            double *hx, *hz;
            const bool snap = (i % S.store_history) == 0;
            const size_t hrow = (size_t)(i / S.store_history);
            if (r < nT) {
                if (!snap) continue;
                hx = S.path_tev + (hrow * 2) * nv + r;
                hz = hx + nv;
            } else if (r < nT + nL) {
                if (!snap) continue;
                hx = S.path_lev + (hrow * 2) * nv + (r - nT);
                hz = hx + nv;
            } else {
                hx = S.path_free + ((size_t)i * 2) * S.nfree + (r - nT - nL);
                hz = hx + S.nfree;
            }
            *hx = xn;
            *hz = zn;
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// graph path: four kernels per step
// ---------------------------------------------------------------------------------------------------
// Ramesh in exact mode: the partials of the step's Newton wake TEV[:itev+1] ++ LEV[:ilev+1] ++ FREE, whatever the two new
// slots hold now (grid_downwash evaluates their nodes again); fast mode and Faure: the old wake TEV[:itev] ++ LEV[:ilev] ++ FREE.
template <int METHOD>
__device__ __forceinline__ int wof_extra(const SimDev &S)
{
    return (METHOD == LUDVM_METHOD_RAMESH && S.mode == LUDVM_EXACT_F64) ? 1 : 0;
}

template <int METHOD>
__global__ void __launch_bounds__(256) k_wake_on_foil(SimDev S, int s)
{
    Step st;
    if (!step_begin(S, s, st)) return;
    if (blockIdx.x == gridDim.x - 1) {  // the last block evaluates the two circulation sums of LUDVM.py:758-759
        __shared__ double s_nodes[1024];
        double sT = block_np_sum(S.wg, st.itev, s_nodes, 1024);
        double sL = block_np_sum(S.wg + S.nv, st.ilev, s_nodes, 1024);
        if (threadIdx.x == 0) {
            S.pre_sums[0] = sT;
            S.pre_sums[1] = sL;
        }
        return;
    }
    Pool pl = grid_pool();
    pl.nwarps -= blockDim.x >> 5;
    pl.nth -= blockDim.x;
    phase_wake_on_foil(S, st, st.itev + wof_extra<METHOD>(S), st.ilev + wof_extra<METHOD>(S), pl);
}
template __global__ void k_wake_on_foil<LUDVM_METHOD_FAURE>(SimDev, int);   // emission order: see method_kernels

template <int METHOD>
__global__ void __launch_bounds__(SOLVE_THREADS) k_solve(SimDev S, int s)
{
    extern __shared__ double sm[];
    Step st;
    TRACE(20);
    if (!step_begin(S, s, st)) return;
    TRACE(21);
    phase_solve<METHOD, METHOD == LUDVM_METHOD_RAMESH>(S, st, sm, sm + TABLE_SMEM_DOUBLES(S.P, S.Nc, S.sinn_smem),
                                                       S.pre_sums, true);
    __syncthreads();
    TRACE(22);
}
template __global__ void k_solve<LUDVM_METHOD_FAURE>(SimDev, int);

__global__ void __launch_bounds__(256) k_conv_partials(SimDev S, int s)
{
    Step st;
    if (!step_begin(S, s, st)) return;
    phase_conv_partials(S, st, grid_pool());
}

// Large wakes in exact mode: one thread per target row, the eight accumulators of numpy's leaf loop in registers,
// sources broadcast from shared memory (exact_tiled_block, biot_savart.cuh) -- the FP64 pipe instead of instruction
// issue bounds it.  grid = (row blocks, 2^dcap + 1): y < 2^d evaluates tree node y of the wake on (gamma points ++
// wake), the last y the P bound vortices on the wake.  Same partial layout as k_conv_partials, so k_finish is shared.
__global__ void __launch_bounds__(ET_THREADS, 3) k_conv_partials_exact_tiled(SimDev S, int s)
{
    __shared__ __align__(16) double2 sxz[ET_TILE], sgv[ET_TILE];
    Step st;
    if (!step_begin(S, s, st)) return;
    const int P = S.P;
    SrcView W = wake_view(S, st.itev + 1, st.ilev + 1);
    const double *gx = S.gp + ((size_t)st.i * 2 + 0) * P, *gz = S.gp + ((size_t)st.i * 2 + 1) * P;
    const int nrows = P + W.n;
    if (blockIdx.y + 1 < gridDim.y) {
        const int d = sim_depth(W.n, nrows, S.target_warps);
        if ((long)blockIdx.x * ET_THREADS >= nrows) return;
        TgtGammaWake TA{gx, gz, P, W};
        if (range_safe(S))
            for (int b = blockIdx.y; b < (1 << d); b += gridDim.y - 1)   // normally one node per CTA
                exact_tiled_block<false>(W, TA, nrows, blockIdx.x, d, b, S.pb_u, S.pb_w, sxz, sgv);
        else
            for (int b = blockIdx.y; b < (1 << d); b += gridDim.y - 1)
                exact_tiled_block<true>(W, TA, nrows, blockIdx.x, d, b, S.pb_u, S.pb_w, sxz, sgv);
    } else {
        if ((long)blockIdx.x * ET_THREADS >= W.n) return;
        SrcView Fo = make_src(S.g_airfoil + (size_t)st.itev * S.af_stride, 1, gx, gz, nullptr, S.vc4, P);
        TgtWake TW{W};
        if (range_safe(S)) exact_tiled_block<false>(Fo, TW, W.n, blockIdx.x, 0, 0, S.foil_u, S.foil_w, sxz, sgv);
        else exact_tiled_block<true>(Fo, TW, W.n, blockIdx.x, 0, 0, S.foil_u, S.foil_w, sxz, sgv);
    }
}

// Large wakes in fast mode: the O(N^2) part goes through the shared-memory tiled kernel (13 FP64 slots/pair at
// ~94% of the DFMA rate) instead of the lane-group tasks.  grid = (row blocks, chunks + 1): y < chunks evaluates the
// wake on (gamma points ++ wake) for one source chunk; y == chunks evaluates the P bound vortices on the wake.
template <int R>
__global__ void __launch_bounds__(FT_THREADS, 2) k_conv_partials_tiled(SimDev S, int s, int chunks)
{
    __shared__ double sx[FT_TILE], sz[FT_TILE], sg[FT_TILE], sv[FT_TILE];
    Step st;
    if (!step_begin(S, s, st)) return;
    const int P = S.P;
    SrcView W = wake_view(S, st.itev + 1, st.ilev + 1);
    const double *gx = S.gp + ((size_t)st.i * 2 + 0) * P, *gz = S.gp + ((size_t)st.i * 2 + 1) * P;
    const int nrows = P + W.n;
    if ((int)blockIdx.y < chunks) {
        if ((long)blockIdx.x * (FT_THREADS * R) >= nrows) return;
        TgtGammaWake TA{gx, gz, P, W};
        int chunk_len = ((W.n + chunks - 1) / chunks + FT_TILE - 1) / FT_TILE * FT_TILE;
        int c0 = blockIdx.y * chunk_len, c1 = min(W.n, c0 + chunk_len);
        size_t po = (size_t)blockIdx.y * nrows;
        fast_tiled_block<R>(W, TA, nrows, blockIdx.x, c0, c1, S.pb_u + po, S.pb_w + po, sx, sz, sg, sv);
    } else {
        if ((long)blockIdx.x * (FT_THREADS * R) >= W.n) return;
        SrcView Fo = make_src(S.g_airfoil + (size_t)st.itev * S.af_stride, 1, gx, gz, nullptr, S.vc4, P);
        TgtWake TW{W};
        fast_tiled_block<R>(Fo, TW, W.n, blockIdx.x, 0, P, S.foil_u, S.foil_w, sx, sz, sg, sv);
    }
}

// ---------------------------------------------------------------------------------------------------
// overlapped step (fast mode, tiled wakes).  The O(N^2) part of the convection -- the OLD wake TEV[:itev] ++ LEV[:ilev]
// ++ FREE acting on itself and on the positions the step's two new vortices will take -- does not depend on the
// circulations solved in this step, so it runs on a second graph branch beside phase 1 + the solve (which keep one
// CTA busy for tens of microseconds while 147 SMs would idle):
//   branch A: k_wake_on_foil -> k_solve_small                   branch B: k_conv_old_tiled
//   join:     k_conv_new  (the two new vortices + the P bound vortices on every wake row; wake velocity at the gamma
//                          points = phase-1 sums + the two new vortices)  ->  k_finish_ov (loads, Euler update)
// For the solve CTA to start while the convection grid occupies every SM it must fit into the hole ONE retiring
// convection CTA leaves (256 threads x <= 70 registers): k_solve_small is the solve compiled for 64 registers (a
// 128-register solve CTA was measured to start only when the convection kernel drained, DESIGN.md 5).
// Summation order differs from the serial step (fast mode carries no order guarantee); exact mode keeps the serial step.
// ---------------------------------------------------------------------------------------------------
// Source chunking of the old-wake convection, chosen from the ACTUAL wake size (a graph serves a 2:1 range of sizes):
// about eight waves of CTAs over the resident slots, chunk length a multiple of 64 sources, at most
// SIM_TILED_CHUNKS_MAX chunks.  With chunks fixed per graph the grid was 2.4 waves at 22k vortices (79 % occupancy of
// the last wave's worth of time).  Identical in the producer and in k_finish_ov.
struct TiledGeom {
    int chunk_len, chunks;
    // `slots` = resident CTA slots of the convection kernel.
    __host__ __device__ __forceinline__ TiledGeom(int nrows, int nsrc, int R, int slots)
    {
        const int rb = (nrows + FT_THREADS * R - 1) / (FT_THREADS * R);
        int want = (8 * slots + rb - 1) / rb;
        want = want < 1 ? 1 : (want > SIM_TILED_CHUNKS_MAX ? SIM_TILED_CHUNKS_MAX : want);
        chunk_len = (((nsrc + want - 1) / want + 63) / 64) * 64;
        chunks = (nsrc + chunk_len - 1) / chunk_len;
    }
};

template <int METHOD>
__global__ void __launch_bounds__(SOLVE_THREADS, 4) k_solve_small(SimDev S, int s)
{
    extern __shared__ double sm[];
    Step st;
    if (!step_begin(S, s, st)) return;
    phase_solve<METHOD, METHOD == LUDVM_METHOD_RAMESH>(S, st, sm, sm + TABLE_SMEM_DOUBLES(S.P, S.Nc, S.sinn_smem),
                                                       S.pre_sums, true);
}
template __global__ void k_solve_small<LUDVM_METHOD_FAURE>(SimDev, int);

template <int R>
__global__ void __launch_bounds__(FT_THREADS, 2) k_conv_old_tiled(SimDev S, int s, int slots)
{
    __shared__ __align__(16) double sx[4 * FT_TILE];
    Step st;
    if (!step_begin(S, s, st)) return;
    SrcView W = wake_view(S, st.itev, st.ilev);
    const int nrows = W.n + 3;   // + the new TEV, the LEV if shed, the idle LEV slot: their rows need no solve either
    const TiledGeom G(nrows, W.n, R, slots);
    if ((long)blockIdx.x * (FT_THREADS * R) >= nrows || (int)blockIdx.y >= G.chunks) return;
    TgtWakePlus TW;
    TW.W = W;
    place_tev(S, st.i, st.itev, TW.xt, TW.zt);
    place_lev(S, st.i, st.ilev, TW.xl, TW.zl);
    int c0 = blockIdx.y * G.chunk_len, c1 = min(W.n, c0 + G.chunk_len);
    size_t po = (size_t)blockIdx.y * nrows;
    fast_tiled_block<R>(W, TW, nrows, blockIdx.x, c0, c1, S.pb_u + po, S.pb_w + po, sx, sx + FT_TILE, sx + 2 * FT_TILE,
                        sx + 3 * FT_TILE);
}

// Row of the updated wake TEV[:itev+1] ++ LEV[:ilev+1] ++ FREE -> row of k_conv_old_tiled's partials (nold = rows of
// the old wake; the step's two additions map to the extra rows, see TgtWakePlus).
__device__ __forceinline__ int old_row(int r, int itev, int ilev, int nold, bool shed)
{
    if (r < itev) return r;
    if (r == itev) return nold;
    if (r < itev + 1 + ilev) return r - 1;
    if (r == itev + 1 + ilev) return shed ? nold + 1 : nold + 2;
    return r - 2;
}

__global__ void __launch_bounds__(256) k_conv_new(SimDev S, int s)
{
    __shared__ double sx[260], sz[260], sg[260];   // P bound vortices + the two new wake vortices (P <= 256)
    Step st;
    if (!step_begin(S, s, st)) return;
    const int P = S.P, tid = threadIdx.x, itev = st.itev, ilev = st.ilev, nv = S.nv;
    SrcView W = wake_view(S, itev + 1, ilev + 1);
    const double *gx = S.gp + ((size_t)st.i * 2 + 0) * P, *gz = S.gp + ((size_t)st.i * 2 + 1) * P;
    const double *ga = S.g_airfoil + (size_t)itev * S.af_stride;
    if (blockIdx.x == 0) {   // gamma points: old wake (phase-1 partials) + the two new vortices  (LUDVM.py:1049-1054)
        const int fold = wof_fold(S.mode, itev + ilev + S.nfree, P, S.target_warps);
        const double xt = S.wx[itev], zt = S.wz[itev], gt = S.wg[itev] * LUDVM_INV_TWO_PI;
        const double xl = S.wx[nv + ilev], zl = S.wz[nv + ilev], gl = S.wg[nv + ilev] * LUDVM_INV_TWO_PI;
        for (int j = tid; j < P; j += blockDim.x) {
            double u = fast_combine_row(S.pa_u, P, j, fold), w = fast_combine_row(S.pa_w, P, j, fold);
            pair_fast(gx[j], gz[j], xt, zt, gt, S.vc4, u, w);
            pair_fast(gx[j], gz[j], xl, zl, gl, S.vc4, u, w);
            S.gp_u[j] = u;
            S.gp_w[j] = w;
        }
        return;
    }
    // every wake row (the two new ones included): the P bound vortices and the two new wake vortices
    for (int j = tid; j < P + 2; j += blockDim.x) {
        if (j < P) { sx[j] = gx[j]; sz[j] = gz[j]; sg[j] = ga[j] * LUDVM_INV_TWO_PI; }
        else {
            int q = j == P ? itev : nv + ilev;
            sx[j] = S.wx[q]; sz[j] = S.wz[q]; sg[j] = S.wg[q] * LUDVM_INV_TWO_PI;
        }
    }
    __syncthreads();
    for (long r = (long)(blockIdx.x - 1) * blockDim.x + tid; r < W.n; r += (long)(gridDim.x - 1) * blockDim.x) {
        const int p = W.phys((int)r);
        const double xp = S.wx[p], zp = S.wz[p];
        double u0 = 0.0, w0 = 0.0, u1 = 0.0, w1 = 0.0;
        int j = 0;
        for (; j + 1 < P + 2; j += 2) {
            pair_fast(xp, zp, sx[j], sz[j], sg[j], S.vc4, u0, w0);
            pair_fast(xp, zp, sx[j + 1], sz[j + 1], sg[j + 1], S.vc4, u1, w1);
        }
        if (j < P + 2) pair_fast(xp, zp, sx[j], sz[j], sg[j], S.vc4, u0, w0);
        S.foil_u[r] = u0 + u1;
        S.foil_w[r] = w0 + w1;
    }
}

// `chunks` = partial sums per row of pb_u / pb_w: 0 = k_conv_old_tiled's (TiledGeom of the actual wake), 1 = the
// far-field step's single finished row.
__global__ void __launch_bounds__(256) k_finish_ov(SimDev S, int s, int R, int slots, int chunks)
{
    extern __shared__ double sm[];
    Step st;
    if (!step_begin(S, s, st)) return;
    if (blockIdx.x == 0) {
        phase_finish_loads<true>(S, st, nullptr, sm, 1, FINISH_STAGE, true);
        return;
    }
    if (blockIdx.x == 1) {
        phase_gamma_cumsum(S, st, threadIdx.x, blockDim.x);
        return;
    }
    // convection (LUDVM.py:1095-1127): old-wake partials + k_conv_new's terms
    const int i = st.i, nv = S.nv, nT = st.itev + 1, nL = st.ilev + 1;
    SrcView W = wake_view(S, nT, nL);
    const int nold = W.n - 2, npart = nold + 3;
    if (chunks == 0) chunks = TiledGeom(npart, nold, R, slots).chunks;
    const bool shed = S.lev_shed[i] != -1.0;
    const double dt = S.dt;
    for (long r = (long)(blockIdx.x - 2) * blockDim.x + threadIdx.x; r < W.n; r += (long)(gridDim.x - 2) * blockDim.x) {
        const int ro = old_row((int)r, st.itev, st.ilev, nold, shed);
        const double u = S.foil_u[r] + fast_combine_row(S.pb_u, npart, ro, chunks);
        const double w = S.foil_w[r] + fast_combine_row(S.pb_w, npart, ro, chunks);
        const int p = W.phys((int)r);
        const double xn = S.wx[p] + dt * u, zn = S.wz[p] + dt * w;
        S.wx[p] = xn;
        S.wz[p] = zn;
        if (S.store_history) {
            double *hx, *hz;
            const bool snap = (i % S.store_history) == 0;
            const size_t hrow = (size_t)(i / S.store_history);
            if (r < nT) {
                if (!snap) continue;
                hx = S.path_tev + (hrow * 2) * nv + r;
                hz = hx + nv;
            } else if (r < nT + nL) {
                if (!snap) continue;
                hx = S.path_lev + (hrow * 2) * nv + (r - nT);
                hz = hx + nv;
            } else {
                hx = S.path_free + ((size_t)i * 2) * S.nfree + (r - nT - nL);
                hz = hx + S.nfree;
            }
            *hx = xn;
            *hz = zn;
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// far-field step (LUDVM(..., far_field_order=p), fast mode, wakes >= SIM_FAR_FIELD_MIN_WAKE): branch B of the
// overlapped step with the old wake's self-convection evaluated by the treecode (tree.cu) instead of k_conv_old_tiled.
//   k_ff_gather       the old wake TEV[:itev] ++ LEV[:ilev] ++ FREE, contiguous, in logical order (the tree's sources
//                     and targets: one sort serves both)
//   tree              rows 0 .. nold-1 of pb_u / pb_w, one finished sum per row
//   k_ff_extra_rows   rows nold .. nold+2 (TgtWakePlus: the new TEV, the LEV, the idle LEV slot at the origin) against
//                     the old wake by all pairs; kept out of the tree, whose bounding box the origin would stretch
// The join (k_conv_new -> k_finish_ov with one partial per row) is the overlapped step's.  Every sum has a fixed order, so
// the step is bitwise reproducible run to run.
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_ff_gather(SimDev S, double *x, double *z, double *g)
{
    Step st;
    if (!step_begin(S, 0, st)) return;
    const SrcView W = wake_view(S, st.itev, st.ilev);
    for (long r = (long)blockIdx.x * blockDim.x + threadIdx.x; r < W.n; r += (long)gridDim.x * blockDim.x) {
        const int p = W.phys((int)r);
        x[r] = S.wx[p];
        z[r] = S.wz[p];
        g[r] = S.wg[p];
    }
}

#define FF_EXTRA_THREADS 1024
__global__ void __launch_bounds__(FF_EXTRA_THREADS) k_ff_extra_rows(SimDev S, const double *x, const double *z,
                                                                    const double *g, int n)
{
    __shared__ double su[FF_EXTRA_THREADS], sw[FF_EXTRA_THREADS];
    Step st;
    if (!step_begin(S, 0, st)) return;
    const int row = blockIdx.x, tid = threadIdx.x;   // 0: the new TEV, 1: the LEV, 2: the idle LEV slot
    double xp = 0.0, zp = 0.0;
    if (row == 0) place_tev(S, st.i, st.itev, xp, zp);
    else if (row == 1) place_lev(S, st.i, st.ilev, xp, zp);
    double u = 0.0, w = 0.0;
    for (int j = tid; j < n; j += FF_EXTRA_THREADS) pair_fast(xp, zp, x[j], z[j], g[j] * LUDVM_INV_TWO_PI, S.vc4, u, w);
    su[tid] = u;
    sw[tid] = w;
    for (int h = FF_EXTRA_THREADS / 2; h > 0; h >>= 1) {   // fixed-shape tree: the same sum on every run
        __syncthreads();
        if (tid < h) {
            su[tid] += su[tid + h];
            sw[tid] += sw[tid + h];
        }
    }
    if (tid == 0) {
        S.pb_u[n + row] = su[0];
        S.pb_w[n + row] = sw[0];
    }
}

__global__ void __launch_bounds__(256) k_finish(SimDev S, int s, int tiled_chunks)
{
    extern __shared__ double sm[];
    Step st;
    if (!step_begin(S, s, st)) return;
    if (blockIdx.x == 0) {
        phase_finish_loads<true>(S, st, nullptr, sm, tiled_chunks, FINISH_STAGE);
        return;
    }
    if (blockIdx.x == 1) {
        phase_gamma_cumsum(S, st, threadIdx.x, blockDim.x);
        return;
    }
    phase_finish_update(S, st, (long)(blockIdx.x - 2) * blockDim.x + threadIdx.x, (long)(gridDim.x - 2) * blockDim.x,
                        tiled_chunks);
}

// Graph path with the pressure jump enabled: row i of dp after k_finish / k_finish_ov (one CTA).
__global__ void __launch_bounds__(256) k_pressure(SimDev S, int s)
{
    Step st;
    if (!step_begin(S, s, st)) return;
    pressure_row(S, st);
}

__global__ void k_advance(SimDev S, int k)
{
    long long v = S.counters[0] + k;
    S.counters[0] = v > S.nt - 1 ? S.nt - 1 : v;
}

// ---------------------------------------------------------------------------------------------------
// cooperative path: one persistent grid (one CTA per SM) runs many steps of ONE simulation with grid-wide barriers
// between the phases.  For small wakes a step is latency-bound: four dependent launches per step cost more than the
// arithmetic, and every launch starts with cold instruction and data caches.  Here the phases are the same device
// functions over the same warp pools, the solve CTA stays on its SM (warm caches), and a phase boundary is one
// arrive + spin on a counter in L2.  Launched with cudaLaunchCooperativeKernel (co-residency guaranteed).
// ---------------------------------------------------------------------------------------------------
#define COOP_SPIN_LIMIT (1u << 27)   // ~1 s of polling: a lost CTA turns into an error flag, not a hung GPU

// Two-level grid barrier on monotonically increasing counters (all zeroed by the host before the launch): CTAs arrive
// on the counter of their group of COOP_GROUP CTAs (distinct L2 lines, so the groups' atomics proceed in parallel);
// the last arriver of a group arrives on the root counter; the last arriver there publishes the barrier index in a
// flag word that every CTA polls with plain volatile loads.  A single counter would serialise 148 atomics on one
// address (~27 cycles each, measured ~2.5-5 us per barrier); this chain is 16 + 10 atomics deep.
// Memory protocol as in cooperative_groups::grid_group::sync(): block barrier, fence, arrive, poll, fence, block barrier.
#define COOP_GROUP 16
#define COOP_BAR_WORDS (16 * 20)   // root, flag and up to 16 group counters, one 128-byte line each
__device__ __forceinline__ void grid_barrier(unsigned long long *bar, unsigned long long &k, long long *counters)
{
    __syncthreads();
    if (threadIdx.x == 0) {
        k += 1;
        const unsigned nb = gridDim.x, g = blockIdx.x / COOP_GROUP, ng = (nb + COOP_GROUP - 1) / COOP_GROUP;
        const unsigned gsize = min((unsigned)COOP_GROUP, nb - g * COOP_GROUP);
        unsigned long long *root = bar, *flag = bar + 16, *grp = bar + 32 + 16 * g;
        __threadfence();
        if (atomicAdd(grp, 1ULL) + 1 == k * gsize) {
            __threadfence();
            if (atomicAdd(root, 1ULL) + 1 == k * ng) {
                __threadfence();
                *(volatile unsigned long long *)flag = k;
            }
        }
        unsigned spins = 0;
        while (*(volatile unsigned long long *)flag < k) {
            if (++spins > COOP_SPIN_LIMIT) {
                counters[3] = 1;  // error flag
                break;
            }
        }
        __threadfence();
    }
    __syncthreads();
}

// One persistent kernel, two ways of keeping its CTAs in step:
//   CLUSTER = false  a cooperative grid of one CTA per SM with the L2 grid barrier above (wakes up to a few thousand);
//   CLUSTER = true   ONE thread-block cluster (up to 16 CTAs, co-scheduled on one GPC) whose phase boundary is the hardware
//                    cluster barrier (barrier.cluster, release/acquire at cluster scope: ~0.2 us instead of ~1.7-3 us).
//                    A README-size step is four barriers and ~10 us of O(N^2) work spread thin over 148 SMs, so fewer
//                    CTAs with a cheap barrier win while the wake is small (SIM_CLUSTER_MAX_WAKE).
// The loads (LUDVM.py:1035-1090) and the cumulative bound circulation of step i feed nothing inside the loop, and the
// solve of step i + 1 keeps one CTA busy for ~11 us while every other CTA waits: CTA 1 evaluates the loads and CTA 2 the
// cumulative sums of step i during that window (both have the constant tables / scratch of their own).  What they read --
// the convection partials at the gamma points, gamma_airfoil / g_airfoil row itev, fourier row i -- is not rewritten
// before phase 3 of step i + 1, which the barrier after the solve holds back until they are done.
template <bool CLUSTER>
__device__ __forceinline__ void persist_barrier(unsigned long long *bar, unsigned long long &k, long long *counters)
{
    if (CLUSTER) cluster_sync_all();
    else grid_barrier(bar, k, counters);
}

// 256 threads per CTA on both paths: 512 threads halve the O(N^2) phases' rounds but cap the kernel at 128 registers and
// slow the solve by ~3 us: README case 30.4 / 25.7 us per step (exact / fast) against 28.7 / 24.0 with 256
// (profiles/r02s_coop_probe_1.txt).
template <bool CLUSTER, int METHOD>
__global__ void __launch_bounds__(256, 1) k_sim_persist(SimDev S, int nsteps, unsigned long long *bar)
{
    extern __shared__ double sm[];
    unsigned long long epoch = 0;
    const int first = (int)S.counters[0] + 1;
    const int last = min(S.nt - 1, first + nsteps - 1);
    const int nb = gridDim.x;
    double *const tab = sm, *const scr = sm + TABLE_SMEM_DOUBLES(S.P, S.Nc, S.sinn_smem);
    if (blockIdx.x <= 1) {   // the solve CTA and the loads CTA keep the constant tables in shared memory for the whole launch
        stage_tables(S, StepTables(tab, S));
        tables_wait();
    }
    __syncthreads();
#ifdef LUDVM_TRACE
#define COOP_T(k) do { if (blockIdx.x == 0 && threadIdx.x == 0) { long long t__ = clock64(); acc[k] += t__ - tlast; tlast = t__; } } while (0)
    long long acc[8] = {0, 0, 0, 0, 0, 0, 0, 0}, tlast = clock64();
#else
#define COOP_T(k) do { } while (0)
#endif
    auto deferred_tail = [&](int ip) {
        Step sp{ip, ip - 1, ((volatile int *)S.ilev_arr)[ip]};
        if (blockIdx.x == 1) {
            phase_finish_loads<true>(S, sp, tab, scr, 0, S.sum_nodes);
            if (S.dp) pressure_row(S, sp);
        } else if (blockIdx.x == 2) phase_gamma_cumsum(S, sp, threadIdx.x, blockDim.x);
    };
    for (int i = first; i <= last; i++) {
        Step st{i, i - 1, ((volatile int *)S.ilev_arr)[i]};
        // phase 1: the wake on the gamma points; the last CTA evaluates the two circulation sums instead
        if (blockIdx.x == nb - 1) {
            double sT = block_np_sum(S.wg, st.itev, scr, S.sum_nodes);
            double sL = block_np_sum(S.wg + S.nv, st.ilev, scr, S.sum_nodes);
            if (threadIdx.x == 0) {
                S.pre_sums[0] = sT;
                S.pre_sums[1] = sL;
            }
        } else {
            Pool pl = grid_pool();
            pl.nwarps -= blockDim.x >> 5;
            pl.nth -= blockDim.x;
            phase_wake_on_foil(S, st, st.itev + wof_extra<METHOD>(S), st.ilev + wof_extra<METHOD>(S), pl);
        }
        COOP_T(0);
        persist_barrier<CLUSTER>(bar, epoch, S.counters);
        COOP_T(1);
        if (blockIdx.x == 0) phase_solve<METHOD, METHOD == LUDVM_METHOD_RAMESH>(S, st, tab, scr, S.pre_sums, false);
        else if (i > first) deferred_tail(i - 1);
        COOP_T(2);
        persist_barrier<CLUSTER>(bar, epoch, S.counters);
        COOP_T(3);
        phase_conv_partials(S, st, grid_pool());
        COOP_T(4);
        persist_barrier<CLUSTER>(bar, epoch, S.counters);
        COOP_T(5);
        phase_finish_update(S, st, (long)blockIdx.x * blockDim.x + threadIdx.x, (long)nb * blockDim.x, 0);
        COOP_T(6);
        persist_barrier<CLUSTER>(bar, epoch, S.counters);
        COOP_T(7);
    }
    if (last >= first) deferred_tail(last);
#ifdef LUDVM_TRACE
    if (blockIdx.x == 0 && threadIdx.x == 0)
        for (int q = 0; q < 8; q++) g_trace[40 + q] = acc[q];
#endif
    if (blockIdx.x == 0 && threadIdx.x == 0) S.counters[0] = last;
}

// ---------------------------------------------------------------------------------------------------
// CTA path: one persistent CTA per case, all steps
// ---------------------------------------------------------------------------------------------------
// Out-of-line copies of the O(N^2) phases for the one-CTA driver: their hot loops get a register allocation of their own
// instead of sharing one with the scalar phases inlined around them.
__device__ __noinline__ void cta_wake_on_foil(const SimDev &S, const Step &st)
{
    phase_wake_on_foil(S, st, st.itev, st.ilev, block_pool());
}
__device__ __noinline__ void cta_conv_partials(const SimDev &S, const Step &st)
{
    phase_conv_partials(S, st, block_pool());
}

// Fast-mode phase 1 of the one-CTA driver (the wake TEV[:itev] ++ LEV[:ilev] ++ FREE on the P gamma points): the lane-group
// tasks spend three global loads per pair on 8 warps (19 us per step alone on an SM, a fifth of the driver's step,
// profiles/r02u_sweep_trace.txt).  Here the wake is staged once in shared memory, the block is cut into blockDim / P
// slices of the sources, every thread of a slice owns one gamma point, and the slices' partial sums are added in slice
// order: one finished sum per gamma point (SimDev::wof_single).  Needs P <= blockDim and 3 n + 2 P (blockDim / P) doubles.
__device__ __noinline__ void cta_wof_tiled_fast(const SimDev &S, const Step &st, double *smt)
{
    const int P = S.P, tid = threadIdx.x, nth = blockDim.x;
    SrcView W = wake_view(S, st.itev, st.ilev);
    const int n = W.n, nslice = nth / P;
    const double *gx = S.gp + ((size_t)st.i * 2 + 0) * P, *gz = S.gp + ((size_t)st.i * 2 + 1) * P;
    double *sx = smt, *sz = sx + n, *sg = sz + n, *pu = sg + n, *pw = pu + nslice * P;
    __syncthreads();
    for (int j = tid; j < n; j += nth) {
        const int p = W.phys(j);
        sx[j] = S.wx[p]; sz[j] = S.wz[p]; sg[j] = S.wg[p] * LUDVM_INV_TWO_PI;
    }
    __syncthreads();
    const int slice = tid / P, row = tid - slice * P;
    if (slice < nslice) {
        const int len = (n + nslice - 1) / nslice, j0 = slice * len, j1 = min(n, j0 + len);
        const double xp = gx[row], zp = gz[row];
        double u0 = 0.0, w0 = 0.0, u1 = 0.0, w1 = 0.0;
        int j = j0;
#pragma unroll 2
        for (; j + 1 < j1; j += 2) {
            pair_fast(xp, zp, sx[j], sz[j], sg[j], S.vc4, u0, w0);
            pair_fast(xp, zp, sx[j + 1], sz[j + 1], sg[j + 1], S.vc4, u1, w1);
        }
        if (j < j1) pair_fast(xp, zp, sx[j], sz[j], sg[j], S.vc4, u0, w0);
        pu[slice * P + row] = u0 + u1;
        pw[slice * P + row] = w0 + w1;
    }
    __syncthreads();
    if (tid < P) {
        double u = 0.0, w = 0.0;
        for (int q = 0; q < nslice; q++) { u += pu[q * P + tid]; w += pw[q * P + tid]; }
        S.pa_u[tid] = u;
        S.pa_w[tid] = w;
    }
}

// Fast-mode convection of the one-CTA driver when the whole wake fits in shared memory (parameter sweeps: <= ~800
// vortices): the lane-group tasks spend 3 loads per pair and are LSU-bound (48 % of the DFMA rate measured); here the
// wake (x, z, Gamma/2pi) is staged once, every thread keeps R target rows in registers and the sources are broadcast
// from shared memory -- 3 LDS per R pairs.  Writes complete row sums: pb_u/w[row] (one partial, what conv_fold
// expects of this driver) for the gamma points ++ wake, foil_u/w[r] for the bound vortices on the wake.
template <int R>
__device__ __forceinline__ void cta_tiled_rows(const double *sx, const double *sz, const double *sg, int nsrc, double vc4,
                                               const double *tx_, const double *tz_, int nrows, double *ou, double *ow)
{
    for (int base = 0; base < nrows; base += R * (int)blockDim.x) {
        double tx[R], tz[R], au[R], aw[R];
#pragma unroll
        for (int r = 0; r < R; r++) {
            int row = min(base + r * (int)blockDim.x + (int)threadIdx.x, nrows - 1);
            tx[r] = tx_[row]; tz[r] = tz_[row];
            au[r] = 0.0; aw[r] = 0.0;
        }
#pragma unroll 4
        for (int j = 0; j < nsrc; j++) {
            const double x = sx[j], z = sz[j], g = sg[j];
#pragma unroll
            for (int r = 0; r < R; r++) pair_fast(tx[r], tz[r], x, z, g, vc4, au[r], aw[r]);
        }
#pragma unroll
        for (int r = 0; r < R; r++) {
            int row = base + r * (int)blockDim.x + (int)threadIdx.x;
            if (row < nrows) { ou[row] = au[r]; ow[row] = aw[r]; }
        }
    }
}

__device__ __noinline__ void cta_conv_tiled_fast(const SimDev &S, const Step &st, double *smt)
{
    const int P = S.P, tid = threadIdx.x, nth = blockDim.x;
    SrcView W = wake_view(S, st.itev + 1, st.ilev + 1);
    const int n = W.n, nrows = P + n;
    const double *gx = S.gp + ((size_t)st.i * 2 + 0) * P, *gz = S.gp + ((size_t)st.i * 2 + 1) * P;
    const double *ga = S.g_airfoil + (size_t)st.itev * S.af_stride;
    // shared layout: targets [P + n] (gamma points ++ wake), then the wake strengths [n] and the bound strengths [P];
    // the wake's own coordinates are the tail of the target arrays
    double *tx = smt, *tz = tx + nrows, *sgw = tz + nrows, *sgf = sgw + n;
    __syncthreads();
    for (int r = tid; r < nrows; r += nth) {
        if (r < P) { tx[r] = gx[r]; tz[r] = gz[r]; sgf[r] = ga[r] * LUDVM_INV_TWO_PI; }
        else {
            int p = W.phys(r - P);
            tx[r] = S.wx[p]; tz[r] = S.wz[p]; sgw[r - P] = S.wg[p] * LUDVM_INV_TWO_PI;
        }
    }
    __syncthreads();
    // rows per thread = ceil(rows / threads): with 256 threads and <= 684 rows a fixed R = 4 left a third of the row
    // slots empty (684 / 1024); R = 3 fills 684 / 768
    if (nrows > 3 * nth) {
        cta_tiled_rows<4>(tx + P, tz + P, sgw, n, S.vc4, tx, tz, nrows, S.pb_u, S.pb_w);
        cta_tiled_rows<4>(tx, tz, sgf, P, S.vc4, tx + P, tz + P, n, S.foil_u, S.foil_w);
    } else if (nrows > 2 * nth) {
        cta_tiled_rows<3>(tx + P, tz + P, sgw, n, S.vc4, tx, tz, nrows, S.pb_u, S.pb_w);
        cta_tiled_rows<3>(tx, tz, sgf, P, S.vc4, tx + P, tz + P, n, S.foil_u, S.foil_w);
    } else if (nrows > nth) {
        cta_tiled_rows<2>(tx + P, tz + P, sgw, n, S.vc4, tx, tz, nrows, S.pb_u, S.pb_w);
        cta_tiled_rows<2>(tx, tz, sgf, P, S.vc4, tx + P, tz + P, n, S.foil_u, S.foil_w);
    } else {
        cta_tiled_rows<1>(tx + P, tz + P, sgw, n, S.vc4, tx, tz, nrows, S.pb_u, S.pb_w);
        cta_tiled_rows<1>(tx, tz, sgf, P, S.vc4, tx + P, tz + P, n, S.foil_u, S.foil_w);
    }
}
// Exact-mode twin: the wake ((x, z) pairs and Gamma) is staged once, every thread owns whole target rows and walks
// numpy's summation tree with the eight leaf accumulators in registers and four div/sqrt chains in flight
// (exact_tree_thread).  3 (P + n) doubles of scratch (+ 1 for 16-byte alignment).  One partial per row, as above.
__device__ __noinline__ void cta_conv_tiled_exact(const SimDev &S, const Step &st, double *smt)
{
    const int P = S.P, tid = threadIdx.x, nth = blockDim.x;
    SrcView W = wake_view(S, st.itev + 1, st.ilev + 1);
    const int n = W.n, nrows = P + n;
    const double *gx = S.gp + ((size_t)st.i * 2 + 0) * P, *gz = S.gp + ((size_t)st.i * 2 + 1) * P;
    const double *ga = S.g_airfoil + (size_t)st.itev * S.af_stride;
    // shared layout: (x, z) of the gamma points [P] ++ wake [n], then Gamma of the bound vortices [P] ++ wake [n]
    double2 *txz = reinterpret_cast<double2 *>(smt + ((reinterpret_cast<size_t>(smt) >> 3) & 1));
    double *tg = reinterpret_cast<double *>(txz + nrows);
    __syncthreads();
    for (int r = tid; r < nrows; r += nth) {
        if (r < P) { txz[r] = make_double2(gx[r], gz[r]); tg[r] = ga[r]; }
        else {
            int p = W.phys(r - P);
            txz[r] = make_double2(S.wx[p], S.wz[p]); tg[r] = S.wg[p];
        }
    }
    __syncthreads();
    const SmemSrc3 wake{txz + P, tg + P, S.vc4}, foil{txz, tg, S.vc4};
    const bool safe = range_safe(S);
    for (int row = tid; row < nrows; row += nth) {
        const double2 t = txz[row];
        double u, w;
        if (safe) exact_tree_thread<false>(wake, n, t.x, t.y, u, w);
        else exact_tree_thread<true>(wake, n, t.x, t.y, u, w);
        S.pb_u[row] = u; S.pb_w[row] = w;
    }
    for (int row = tid; row < n; row += nth) {
        const double2 t = txz[P + row];
        double u, w;
        if (safe) exact_tree_thread<false>(foil, P, t.x, t.y, u, w);
        else exact_tree_thread<true>(foil, P, t.x, t.y, u, w);
        S.foil_u[row] = u; S.foil_w[row] = w;
    }
}
__device__ __noinline__ void cta_finish_update(const SimDev &S, const Step &st)
{
    phase_finish_update(S, st, threadIdx.x, blockDim.x, 0);
}

#ifndef SWEEP_CTAS_PER_SM
#define SWEEP_CTAS_PER_SM 3   // resident one-CTA-per-case drivers per SM.  The driver is a chain of short phases separated by
                              // block barriers, i.e. latency-bound, so a third resident case pays even though it caps the kernel
                              // at 80 registers (more spills): 4096-case sweep 0.582 -> 0.564 s fast, 1.008 -> 0.896 s exact
                              // (profiles/r02o_sweep_occupancy.txt); 4 would need 280 KB of shared memory per SM
#endif
// DP: the cases may carry the pressure jump (S.dp non-null); without it the store of u and pressure_row are compiled out.
template <int THREADS, int METHOD, bool DP>
__global__ void __launch_bounds__(THREADS, THREADS <= 128 ? 6 : (THREADS <= 256 ? SWEEP_CTAS_PER_SM : 1)) k_sim_cta(const SimDev *cases, int ncases, int *next_case, int nsteps)
{
    extern __shared__ double sm[];
    __shared__ int s_case;
    __shared__ SimDev s_sim;  // the case descriptor lives in shared memory (a by-value copy would sit in local memory)
    for (;;) {
        __syncthreads();
        if (threadIdx.x == 0) s_case = atomicAdd(next_case, 1);
        __syncthreads();
        const int c = s_case;
        if (c >= ncases) return;
        {
            const int *src = reinterpret_cast<const int *>(cases + c);
            int *dst = reinterpret_cast<int *>(&s_sim);
            for (int w = threadIdx.x; w < (int)(sizeof(SimDev) / sizeof(int)); w += blockDim.x) dst[w] = src[w];
        }
        __syncthreads();
        const SimDev &S = s_sim;
        double *const tab = sm, *const scr = sm + TABLE_SMEM_DOUBLES(S.P, S.Nc, S.sinn_smem);
        stage_tables(S, StepTables(tab, S));   // once per case
        tables_wait();
        __syncthreads();
        const int first = (int)S.counters[0] + 1;
        const int last = min(S.nt - 1, first + nsteps - 1);
#ifdef LUDVM_TRACE
#define CTA_T(k) do { __syncthreads(); if (threadIdx.x == 0) { long long t__ = clock64(); acc[k] += t__ - tlast; tlast = t__; } } while (0)
        long long acc[6] = {0, 0, 0, 0, 0, 0}, tlast = clock64();
#else
#define CTA_T(k) do { } while (0)
#endif
        for (int i = first; i <= last; i++) {
            __syncthreads();
            Step st{i, i - 1, S.ilev_arr[i]};
            CTA_T(5);
            if (METHOD == LUDVM_METHOD_FAURE) {
                if (S.wof_single) cta_wof_tiled_fast(S, st, scr);
                else cta_wake_on_foil(S, st);
                __syncthreads();
            }
            CTA_T(0);
            phase_solve<METHOD>(S, st, tab, scr, nullptr, false);
            __syncthreads();
            CTA_T(1);
            // fast mode with the wake in shared memory: 3 (P + n) + P doubles of the scratch area
            // (exact mode: the same footprint; only the 256-thread driver has the registers for it)
            const bool fits = 3 * (S.P + st.itev + st.ilev + 2 + S.nfree) + S.P <= SOLVE_SCRATCH_DOUBLES(S.P, S.Nc, S.sum_nodes);
            if (S.mode != LUDVM_EXACT_F64 && fits)
                cta_conv_tiled_fast(S, st, scr);
            else if (THREADS <= 256 && fits && st.itev + st.ilev + 2 + S.nfree >= 8)
                cta_conv_tiled_exact(S, st, scr);
            else
                cta_conv_partials(S, st);
            __syncthreads();
            CTA_T(2);
            phase_finish_loads<DP>(S, st, tab, scr, 0, S.sum_nodes);
            if (DP && S.dp) pressure_row(S, st);
            CTA_T(3);
            cta_finish_update(S, st);
            phase_gamma_cumsum(S, st, threadIdx.x, blockDim.x);
            CTA_T(4);
        }
#ifdef LUDVM_TRACE
        if (threadIdx.x == 0)
            for (int q = 0; q < 6; q++) atomicAdd((unsigned long long *)&g_trace[40 + q], (unsigned long long)acc[q]);
#endif
        __syncthreads();
        if (threadIdx.x == 0) S.counters[0] = last;
    }
}

// Per-case initial state (LUDVM.py:618, :645-654): free vortices, fourier[0,0,:2], LEV_shed = -1, LESPcrit.
__global__ void __launch_bounds__(256) k_case_init(const SimDev *cases, int ncases)
{
    int c = blockIdx.x;
    if (c >= ncases) return;
    const SimDev S = cases[c];
    for (int j = threadIdx.x; j < S.nt; j += blockDim.x) S.lev_shed[j] = -1.0;
    if (threadIdx.x == 0 && S.range_bad_init) *S.range_bad = 1;
    for (int j = threadIdx.x; j < S.nfree; j += blockDim.x) {
        S.wg[2 * S.nv + j] = S.free_g[j];
        S.wx[2 * S.nv + j] = S.free_xz[j];
        S.wz[2 * S.nv + j] = S.free_xz[S.nfree + j];
        range_note(S, S.free_xz[j], S.free_xz[S.nfree + j]);
        if (S.store_history) {
            S.path_free[j] = S.free_xz[j];
            S.path_free[S.nfree + j] = S.free_xz[S.nfree + j];
        }
    }
    if (threadIdx.x == 0) {
        S.fourier[0] = S.a0_init;
        S.fourier[1] = S.a1_init;
        *S.lespcrit_cur = S.lespcrit0;
    }
}

// Sweep results: out[c][f][nt] with f in LUDVM_SW_* order (the three circulation rows hold nt-1 values + a 0).
__global__ void __launch_bounds__(256) k_sweep_gather(const SimDev *cases, int ncases, double *out)
{
    int c = blockIdx.x;
    if (c >= ncases) return;
    const SimDev S = cases[c];
    const double *src[LUDVM_SWEEP_FIELDS] = {S.Fn, S.Fs, S.L, S.D, S.T, S.M, S.lesp, S.lesp_prev, S.lev_shed,
                                             S.wg, S.wg + S.nv, S.g_bound};
    double *o = out + (size_t)c * LUDVM_SWEEP_FIELDS * S.nt;
    for (int f = 0; f < LUDVM_SWEEP_FIELDS; f++) {
        int n = f < 9 ? S.nt : S.nt - 1;
        for (int j = threadIdx.x; j < S.nt; j += blockDim.x) o[(size_t)f * S.nt + j] = j < n ? src[f][j] : 0.0;
    }
}

struct DevTables {  // device copies of one ludvm_sim_tables
    const double *cos_a, *sin_a, *alpha_dot, *h_dot, *gp, *le, *te;
    const double *detadx_p, *eta_p, *x_p, *theta_p, *dtheta, *cos_tp, *sin_tp, *cosn, *sinn, *free_g, *free_xz;
    bool coords_in_window;   // every gamma-point / LE / TE coordinate passes coord_in_safe_window (host scan)
};

static bool host_coords_in_window(const double *a, size_t n)
{
    for (size_t i = 0; i < n; i++) {
        uint64_t b;
        memcpy(&b, &a[i], 8);
        const unsigned h = (unsigned)(b >> 32) & 0x7fffffffu;
        if (!((h >= LUDVM_SAFE_LO && h < LUDVM_SAFE_HI) || (h == 0u && (unsigned)b == 0u))) return false;
    }
    return true;
}

static int check_params(const ludvm_sim_params *p, const ludvm_sim_tables *t)
{
    ARG_CHECK(p->nt >= 2 && p->nt < (1 << 24) && p->P >= 2 && p->Nc >= 4 && p->Nc <= 512);
    if (p->P > LUDVM_MAX_PANELS)
        return set_error(LUDVM_E_UNSUPPORTED, "Npoints - 1 = %ld panels; the solve kernel keeps 18 doubles per panel in "
                         "shared memory and supports at most %d", (long)p->P, LUDVM_MAX_PANELS);
    ARG_CHECK(p->nfree >= 1 && p->nfree < (1 << 28));
    ARG_CHECK(p->mode == LUDVM_EXACT_F64 || p->mode == LUDVM_FAST_F64);
    ARG_CHECK(p->method == LUDVM_METHOD_FAURE || p->method == LUDVM_METHOD_RAMESH);
    ARG_CHECK(t->cos_a && t->sin_a && t->alpha_dot && t->h_dot && t->gp && t->le && t->te && t->detadx_p && t->eta_p &&
              t->x_p && t->theta_p && t->dtheta && t->cos_tp && t->sin_tp && t->cosn && t->sinn && t->free_g &&
              t->free_xz);
    return LUDVM_OK;
}

// Fill the scalar fields and carve the per-case state out of the arena.  `compact` keeps only what a parameter
// sweep reads back (no [nv,P] bound-vortex histories, two Fourier rows, no vortex path history).
static void layout_case(SimDev &D, const ludvm_sim_params &p, const DevTables &t, Arena &a, int target_warps,
                        int sum_nodes, bool compact, int cta_threads = CTA_THREADS)
{
    const size_t nt = p.nt, P = p.P, Nc = p.Nc, nf = p.nfree, nv = nt - 1, nstate = 2 * nv + nf;
    D.nt = (int)nt; D.P = (int)P; D.Nc = (int)Nc; D.nfree = (int)nf; D.nv = (int)nv;
    D.method = p.method; D.mode = p.mode; D.store_history = compact ? 0 : std::max(0, p.store_history);
    D.target_warps = target_warps; D.sum_nodes = sum_nodes;
    // (the 128-thread sweep driver reads cos/sin(n theta) from global memory: six resident cases per SM need <= 37 KB each)
    D.sinn_smem = (Nc * P <= SINN_SMEM_MAX && !(compact && cta_threads <= 128)) ? 1 : 0;
    D.af_stride = compact ? 0 : (int)P;
    D.fourier_rows = compact ? 2 : (int)nt;
    D.dt = p.dt; D.Uinf = p.Uinf; D.chord = p.chord; D.rho = p.rho; D.piv = p.piv; D.vc4 = p.vc4; D.ic = p.ic;
    D.sum_free = p.sum_free; D.maxerror = p.maxerror; D.epsilon = p.epsilon; D.maxiter = (int)p.maxiter;
    D.lespcrit0 = p.lespcrit; D.a0_init = p.a0_init; D.a1_init = p.a1_init;
    D.cos_a = t.cos_a; D.sin_a = t.sin_a; D.alpha_dot = t.alpha_dot; D.h_dot = t.h_dot; D.gp = t.gp; D.le = t.le;
    D.te = t.te; D.detadx_p = t.detadx_p; D.eta_p = t.eta_p; D.x_p = t.x_p; D.theta_p = t.theta_p;
    D.dtheta = t.dtheta; D.cos_tp = t.cos_tp; D.sin_tp = t.sin_tp; D.cosn = t.cosn; D.sinn = t.sinn;
    D.free_g = t.free_g; D.free_xz = t.free_xz;
    {   // one-CTA driver, fast mode: phase 1 from a shared-memory copy of the wake (cta_wof_tiled_fast)
        const long nth = cta_threads, nsl = P ? nth / (long)P : 0, nmax = (long)nstate + 2;
        D.wof_single = (compact && p.mode != LUDVM_EXACT_F64 && p.method == LUDVM_METHOD_FAURE && nsl >= 1 &&
                        3 * nmax + 2 * (long)P * nsl <= (long)SOLVE_SCRATCH_DOUBLES(P, Nc, sum_nodes)) ? 1 : 0;
    }
    D.range_bad_init = (t.coords_in_window && vc4_in_safe_window(p.vc4) && !getenv("LUDVM_EXACT_FLAGS")) ? 0 : 1;
    D.range_bad = a.take<int>(1);
    D.wx = a.take<double>(nstate); D.wz = a.take<double>(nstate); D.wg = a.take<double>(nstate);
    D.g_bound = a.take<double>(nv);
    const size_t afrows = compact ? 1 : nv;
    D.g_airfoil = a.take<double>(afrows * P);
    D.gamma_airfoil = a.take<double>(afrows * P);
    D.Gamma_airfoil = a.take<double>(afrows * P);
    D.fourier = a.take<double>((size_t)D.fourier_rows * 2 * Nc);
    D.lesp = a.take<double>(nt); D.lesp_prev = a.take<double>(nt); D.lev_shed = a.take<double>(nt);
    D.Fn = a.take<double>(nt); D.Fs = a.take<double>(nt); D.L = a.take<double>(nt); D.D = a.take<double>(nt);
    D.T = a.take<double>(nt); D.M = a.take<double>(nt);
    if (D.store_history) {
        const size_t hrows = (nt - 1) / D.store_history + 1;
        D.path_tev = a.take<double>(hrows * 2 * nv);
        D.path_lev = a.take<double>(hrows * 2 * nv);
        D.path_free = a.take<double>(nt * 2 * nf);
    } else {
        D.path_tev = D.path_lev = D.path_free = nullptr;
    }
    D.dp = nullptr;   // ludvm_sim_enable_pressure
    D.counters = a.take<long long>(4);
    D.ilev_arr = a.take<int>(nt + 2);
    D.lespcrit_cur = a.take<double>(1);
    const size_t quadsP = (P + 3) / 4;
    const size_t pa = std::min<size_t>((size_t)1 << SIM_DMAX, std::max<size_t>(1, 2 * (size_t)target_warps / quadsP)) * P + P;
    D.pa_u = a.take<double>(pa); D.pa_w = a.take<double>(pa);
    const size_t rows_max = P + nstate + 2;
    size_t pb = std::max(rows_max, (size_t)16 * target_warps + rows_max);
    if (!compact && p.mode != LUDVM_EXACT_F64) pb = std::max(pb, (size_t)SIM_TILED_CHUNKS_MAX * rows_max);
    D.pb_u = a.take<double>(pb); D.pb_w = a.take<double>(pb);
    D.foil_u = a.take<double>(nstate + 8); D.foil_w = a.take<double>(nstate + 8);
    D.pre_sums = a.take<double>(2);
    D.gp_u = a.take<double>(P); D.gp_w = a.take<double>(P);
}

// Shared-memory staging area of the block-wide folds / integrals (block_reduce.cuh batches whatever does not fit):
// `want` doubles if the solve kernel's total stays inside SOLVE_SMEM_LIMIT, else what is left -- never less than one
// np.trapz row (P) or one row of 64 + 1 partials.  The fixed part is 18 P + Nc + 32 doubles (+ the cos/sin(n theta)
// tables when they are small enough to be resident), so P <= LUDVM_MAX_PANELS always fits.
static int clamp_sum_nodes(long P, long Nc, long want)
{
    const bool big = Nc * P <= SINN_SMEM_MAX;
    const long fixed = SOLVE_SMEM_DOUBLES(P, Nc, 0, big);
    const long room = SOLVE_SMEM_LIMIT / (long)sizeof(double) - fixed;
    return (int)std::max<long>(std::max<long>(P, 130), std::min(want, room));
}

static size_t solve_smem_bytes(const SimDev &D) { return (size_t)SOLVE_SMEM_DOUBLES(D.P, D.Nc, D.sum_nodes, D.sinn_smem) * sizeof(double); }

}  // namespace ludvm

using namespace ludvm;

struct ludvm_sim {
    ludvm_ctx *ctx = nullptr;
    ludvm_sim_params p{};
    SimDev d{};
    std::vector<void *> allocs;
    SimDev *d_case = nullptr;  // device copy of `d` (k_case_init)
    long steps_enqueued = 0;
    int K = 50;
    std::map<int, cudaGraphExec_t> graphs;  // (bracket, length) -> instantiated graph
    size_t solve_smem = 0, finish_smem = 0;
    unsigned long long *d_bar = nullptr;  // grid-barrier counter of the cooperative path
    int coop_grid = 0;                    // CTAs of the cooperative kernel (0: path not available on this device)
    int cluster_ctas = 0;                 // CTAs of the single-cluster kernel (0: not available)
    cudaStream_t cap_stream2 = nullptr;   // second capture stream: the overlapped step's old-wake convection branch
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    cudaStream_t cap_stream = nullptr;  // private stream used only to record graphs (the context's stream may be
                                        // the legacy default stream, which cannot be captured)
    // far field (ludvm_sim_enable_far_field): order (0 = off), the old wake compacted for the tree [3][2 nv + nfree],
    // and far_field_info's counters
    int ff_order = 0;
    double *ff_xzg = nullptr;
    long long ff_steps = 0, ff_fallback = 0, ff_leaf_level = 0;
};

namespace ludvm {

// Device memory comes from the stream-ordered allocator (the context raises the pool's release threshold, so the
// arenas of successive simulations / sweeps are recycled without driver calls: cudaMalloc + cudaFree of a 4096-case
// sweep's arenas was measured at 0.2-3 s per call on the pool's boxes, more than the kernel).
static int dev_malloc(ludvm_ctx *ctx, std::vector<void *> &allocs, size_t bytes, void **out)
{
    void *p = nullptr;
    cudaError_t e = cudaMallocAsync(&p, std::max<size_t>(bytes, 256), ctx->stream);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return set_error(LUDVM_E_NOMEM, "cudaMallocAsync(%zu) failed: %s", bytes, cudaGetErrorString(e));
    }
    allocs.push_back(p);
    *out = p;
    return LUDVM_OK;
}

// Upload one host table set into its own arena; returns device pointers.
static int upload_tables(ludvm_ctx *ctx, std::vector<void *> &allocs, const ludvm_sim_params &p,
                         const ludvm_sim_tables &t, DevTables *out)
{
    const size_t nt = p.nt, P = p.P, Nc = p.Nc, nf = p.nfree;
    struct Item { const double *h; size_t n; const double **d; };
    Item items[] = {{t.cos_a, nt, &out->cos_a}, {t.sin_a, nt, &out->sin_a}, {t.alpha_dot, nt, &out->alpha_dot},
                    {t.h_dot, nt, &out->h_dot}, {t.gp, nt * 2 * P, &out->gp}, {t.le, nt * 2, &out->le},
                    {t.te, nt * 2, &out->te}, {t.detadx_p, P, &out->detadx_p}, {t.eta_p, P, &out->eta_p},
                    {t.x_p, P, &out->x_p}, {t.theta_p, P, &out->theta_p}, {t.dtheta, P, &out->dtheta},
                    {t.cos_tp, P, &out->cos_tp}, {t.sin_tp, P, &out->sin_tp}, {t.cosn, Nc * P, &out->cosn},
                    {t.sinn, Nc * P, &out->sinn}, {t.free_g, nf, &out->free_g}, {t.free_xz, 2 * nf, &out->free_xz}};
    Arena a;
    for (auto &it : items) a.take<double>(it.n);
    void *base;
    int rc = dev_malloc(ctx, allocs, a.off + 256, &base);
    if (rc) return rc;
    Arena b;
    b.base = (char *)base;
    for (auto &it : items) {
        double *d = b.take<double>(it.n);
        CUDA_TRY(cudaMemcpyAsync(d, it.h, it.n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        *it.d = d;
    }
    out->coords_in_window = host_coords_in_window(t.gp, nt * 2 * P) && host_coords_in_window(t.le, nt * 2) &&
                            host_coords_in_window(t.te, nt * 2);
    return LUDVM_OK;
}

// Upper bound of the wake size reached within steps [first, first+K)
static long wake_upper(const ludvm_sim *s, long first_step)
{
    long i = std::min<long>(first_step + s->K, s->p.nt - 1);
    return 2 * i + 2 + s->p.nfree;
}

static int bracket_of(long n)
{
    int b = 6;
    while ((1L << b) < n) b++;
    return b;
}

// Launch geometry of one step for every wake size up to 2^bracket.
struct StepPlan {
    int g1, g3, g4, g5, R, tchunks, slots;
    bool tiled, ov, tiled_exact;
    dim3 gto;
    dim3 gt;
    dim3 gte;
};

// The kernels of one method's step (the rest of the step does not depend on the method).
struct MethodKernels {
    void (*wake_on_foil)(SimDev, int);
    void (*solve)(SimDev, int);
    void (*solve_small)(SimDev, int);
    const void *persist_coop, *persist_cluster;   // k_sim_persist<false / true, METHOD>
};
static const MethodKernels &method_kernels(int method);

typedef void (*conv_old_fn)(SimDev, int, int);
static conv_old_fn conv_old_kernel(int R)
{
    return R == 4 ? k_conv_old_tiled<4> : (R == 2 ? k_conv_old_tiled<2> : k_conv_old_tiled<1>);
}

static StepPlan plan_step(const ludvm_sim *s, int bracket)
{
    const SimDev &D = s->d;
    const int nw = (int)std::min<long>(1L << bracket, 2L * D.nv + D.nfree + 2);  // wake-size upper bound
    const int sm = s->ctx->sm_count;
    StepPlan pl{};
    // worst-case warp-task counts over every wake size n <= nw (split depth is monotone in n, capped by the target)
    const int dcap = std::min(pw_max_depth(nw), SIM_DMAX);
    const long quadsP = (D.P + 3) / 4;
    long t1 = D.mode == LUDVM_EXACT_F64 ? quadsP << std::min(dcap, SIM_WOF_MAX_DEPTH)
                                        : quadsP * wof_fold(D.mode, nw, D.P, D.target_warps);
    pl.g1 = 1 + (int)std::max<long>(1, std::min<long>((t1 + 7) / 8, (long)sm * 8));  // + 1: the circulation-sum block
    const long quadsA = (D.P + nw + 3) / 4, quadsW = (nw + 3) / 4;
    long t3 = std::min<long>(quadsA << dcap, std::max<long>(quadsA, 2L * D.target_warps)) + quadsW;
    if (D.mode != LUDVM_EXACT_F64) t3 = std::max<long>(quadsA, (long)D.target_warps + quadsA) + quadsW;
    pl.g3 = (int)std::max<long>(1, std::min<long>((t3 + 7) / 8, (long)sm * 16));
    pl.g4 = 2 + (int)std::max<long>(1, std::min<long>((nw + 255) / 256, (long)sm * 8));
    pl.tiled = D.mode != LUDVM_EXACT_F64 && nw >= SIM_TILED_MIN_WAKE;
    pl.ov = false;
    pl.tiled_exact = D.mode == LUDVM_EXACT_F64 && nw >= SIM_EXACT_TILED_MIN_WAKE && !getenv("LUDVM_NO_EXACT_TILED");
    // grid.y covers the deepest split any wake served by this bracket's graph can ask for (the actual wake may be a
    // quarter of the bound when no LEV is shed); deeper splits, if any, are looped over inside the kernel
    const int dplan = std::min(dcap, ilog2_ceil_i(std::max(1, D.target_warps / std::max(1, (D.P + nw / 4 + 3) / 4))));
    pl.gte = dim3((unsigned)((D.P + nw + ET_THREADS - 1) / ET_THREADS), (1u << dplan) + 1u);
    pl.g5 = 1;
    pl.slots = 0;
    pl.R = 1;
    pl.tchunks = 0;
    pl.gt = dim3(1, 1);
    if (pl.tiled) {
        const long rows_up = D.P + nw;
        // rows per thread (measured on the dt = 2e-3 run: R = 1 only 5.48 s; R = 2 from 8192 rows 5.26 s; R = 4 from 16384-65536
        // rows no better than R = 2)
        pl.R = rows_up >= 131072 ? 4 : (rows_up >= 8192 ? 2 : 1);
        const long row_blocks = (rows_up + FT_THREADS * pl.R - 1) / (FT_THREADS * pl.R);
        pl.tchunks = (int)std::max<long>(1, std::min<long>(std::min<long>(16, nw / (2 * FT_TILE)),
                                                           ((long)sm * 2 * 6 + row_blocks - 1) / row_blocks));
        pl.gt = dim3((unsigned)row_blocks, (unsigned)pl.tchunks + 1);
        // overlapped step: old-wake convection on a second graph branch beside phase 1 + solve
        pl.ov = D.P <= 256;
        pl.gto = dim3((unsigned)((nw + 3 + FT_THREADS * pl.R - 1) / (FT_THREADS * pl.R)), (unsigned)SIM_TILED_CHUNKS_MAX);
        pl.slots = sm * (pl.R == 1 ? 3 : 2);   // resident CTAs of k_conv_old_tiled<R>: 70 registers -> 3 per SM, 112-120 -> 2
        {   // resident CTAs of the chosen instantiation, from the occupancy calculator
            int per_sm = 0;
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, conv_old_kernel(pl.R), FT_THREADS, 0) == cudaSuccess &&
                per_sm > 0)
                pl.slots = sm * per_sm;
            else
                cudaGetLastError();
        }
        pl.g5 = 1 + (int)std::max<long>(1, std::min<long>((nw + 255) / 256, (long)sm * 8));
    }
    return pl;
}

// Enqueue kernel `which` of step offset k: 0 wake-on-foil, 1 solve, 2 convection partials, 3 finish; for the overlapped
// step 2 = old-wake convection (independent of 0 and 1), 4 = the new-vortex / bound-vortex terms, 3 = finish.  With the
// pressure jump enabled, 3 is followed by k_pressure.
static void enqueue_step_kernel(const ludvm_sim *s, const StepPlan &pl, int which, int k, cudaStream_t cs)
{
    const SimDev &D = s->d;
    const MethodKernels &mk = method_kernels(D.method);
    switch (which) {
    case 0: mk.wake_on_foil<<<pl.g1, 256, 0, cs>>>(D, k); break;
    case 1: (pl.ov ? mk.solve_small : mk.solve)<<<1, SOLVE_THREADS, s->solve_smem, cs>>>(D, k); break;
    case 2:
        if (pl.tiled_exact) k_conv_partials_exact_tiled<<<pl.gte, ET_THREADS, 0, cs>>>(D, k);
        else if (!pl.tiled) k_conv_partials<<<pl.g3, 256, 0, cs>>>(D, k);
        else if (pl.ov) conv_old_kernel(pl.R)<<<pl.gto, FT_THREADS, 0, cs>>>(D, k, pl.slots);
        else if (pl.R == 4) k_conv_partials_tiled<4><<<pl.gt, FT_THREADS, 0, cs>>>(D, k, pl.tchunks);
        else if (pl.R == 2) k_conv_partials_tiled<2><<<pl.gt, FT_THREADS, 0, cs>>>(D, k, pl.tchunks);
        else k_conv_partials_tiled<1><<<pl.gt, FT_THREADS, 0, cs>>>(D, k, pl.tchunks);
        break;
    case 4: k_conv_new<<<pl.g5, 256, 0, cs>>>(D, k); break;
    default:
        if (pl.ov) k_finish_ov<<<pl.g4, 256, s->finish_smem, cs>>>(D, k, pl.R, pl.slots, 0);
        else k_finish<<<pl.g4, 256, s->finish_smem, cs>>>(D, k, pl.tchunks);
        if (D.dp) k_pressure<<<1, 256, 0, cs>>>(D, k);
        break;
    }
}

static int create_streams(ludvm_sim *s)
{
    if (s->cap_stream) return LUDVM_OK;
    int lo = 0, hi = 0;
    cudaDeviceGetStreamPriorityRange(&lo, &hi);   // lo = least, hi = greatest priority
    CUDA_TRY(cudaStreamCreateWithPriority(&s->cap_stream, cudaStreamNonBlocking, hi));   // latency-critical branch
    CUDA_TRY(cudaStreamCreateWithPriority(&s->cap_stream2, cudaStreamNonBlocking, lo));  // bulk old-wake convection
    CUDA_TRY(cudaEventCreateWithFlags(&s->ev_fork, cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&s->ev_join, cudaEventDisableTiming));
    return LUDVM_OK;
}

static int build_graph(ludvm_sim *s, int bracket, int ksteps, cudaGraphExec_t *out)
{
    const SimDev &D = s->d;
    const StepPlan pl = plan_step(s, bracket);
    cudaGraph_t graph;
    int rc = create_streams(s);
    if (rc) return rc;
    cudaStream_t cs = s->cap_stream, cs2 = s->cap_stream2;
    CUDA_TRY(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
    for (int k = 0; k < ksteps; k++) {
        if (pl.ov) {
            CUDA_TRY(cudaEventRecord(s->ev_fork, cs));
            CUDA_TRY(cudaStreamWaitEvent(cs2, s->ev_fork, 0));
            enqueue_step_kernel(s, pl, 0, k, cs);
            enqueue_step_kernel(s, pl, 2, k, cs2);
            enqueue_step_kernel(s, pl, 1, k, cs);
            // The new-vortex / bound-vortex terms need the solve, not the old-wake sums; enqueueing them beside the bulk
            // kernel instead of after the join measured no better (5.88 vs 5.84 s).
            CUDA_TRY(cudaEventRecord(s->ev_join, cs2));
            CUDA_TRY(cudaStreamWaitEvent(cs, s->ev_join, 0));
            enqueue_step_kernel(s, pl, 4, k, cs);
            enqueue_step_kernel(s, pl, 3, k, cs);
        } else {
            for (int which = 0; which < 4; which++) enqueue_step_kernel(s, pl, which, k, cs);
        }
    }
    k_advance<<<1, 1, 0, cs>>>(D, ksteps);
    cudaError_t e = cudaStreamEndCapture(cs, &graph);
    if (e != cudaSuccess) return set_error(LUDVM_E_CUDA, "graph capture failed: %s", cudaGetErrorString(e));
    e = cudaGraphInstantiate(out, graph, 0);
    cudaGraphDestroy(graph);
    if (e != cudaSuccess) return set_error(LUDVM_E_CUDA, "graph instantiate failed: %s", cudaGetErrorString(e));
    return LUDVM_OK;
}

// First step (0-based, as ludvm_sim::steps_enqueued) that the far field takes: the wake bound of step k alone,
// 2 min(k + 1, nt - 1) + 2 + nfree (wake_upper over one step), reaches SIM_FAR_FIELD_MIN_WAKE.  It does not depend on
// steps_per_graph or on how ludvm_sim_run is called, so neither changes which steps take which path.
static long far_field_first_step(const ludvm_sim *s)
{
    long k = 0;
    while (k < s->p.nt - 1 && 2 * std::min<long>(k + 1, s->p.nt - 1) + 2 + s->p.nfree < SIM_FAR_FIELD_MIN_WAKE) k++;
    return k;
}

// One far-field step, enqueued from the host (the tree's depth comes from its bounding box, read back to the host, so
// the step cannot be captured in a graph).  Forks from the context's stream onto the sim's two private streams and joins
// back, so the work stays ordered with whatever else the context's stream carries.  `pl` is the plan the graph path
// would use for this step: branch A, the join and, if the tree refuses the cloud, branch B are its kernels.
static int far_field_step(ludvm_sim *s, const StepPlan &pl)
{
    ludvm_ctx *ctx = s->ctx;
    const SimDev &D = s->d;
    int rc = create_streams(s);
    if (rc) return rc;
    // nold = itev + ilev + nfree of step i = steps_enqueued + 1 (ilev_arr[i] is written by step i - 1's solve)
    const long i = s->steps_enqueued + 1;
    int ilev = 0;
    CUDA_TRY(cudaMemcpyAsync(&ilev, D.ilev_arr + i, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    const long nold = (i - 1) + ilev + D.nfree;
    cudaStream_t cs = s->cap_stream, cs2 = s->cap_stream2;
    CUDA_TRY(cudaEventRecord(s->ev_fork, ctx->stream));
    CUDA_TRY(cudaStreamWaitEvent(cs, s->ev_fork, 0));
    CUDA_TRY(cudaStreamWaitEvent(cs2, s->ev_fork, 0));
    // branch A first, so that it runs while the host waits for the tree's read-backs
    enqueue_step_kernel(s, pl, 0, 0, cs);
    enqueue_step_kernel(s, pl, 1, 0, cs);
    double *xg = s->ff_xzg, *zg = xg + (2 * (size_t)D.nv + D.nfree), *gg = zg + (2 * (size_t)D.nv + D.nfree);
    k_ff_gather<<<(int)std::min<long>((nold + 255) / 256, (long)ctx->sm_count * 8), 256, 0, cs2>>>(D, xg, zg, gg);
    ctx->launches += 3;
    // The tree's scratch (ctx slots SLOT_TREE_*) may be reallocated inside this call: scratch_reserve synchronises the
    // context's stream before it frees, the tree has synchronised cs2 just before, and branch A on cs never touches
    // those slots, so no stream can still be using the memory freed.
    rc = tree_velocity_device(ctx, cs2, gg, xg, zg, D.vc4, nold, xg, zg, nold, s->ff_order, 0, D.pb_u, D.pb_w, nullptr);
    int chunks = 1;
    if (rc == LUDVM_E_UNSUPPORTED) {   // a leaf of the deepest tree would hold > 65 536 vortices: all pairs, as the graph
        enqueue_step_kernel(s, pl, 2, 0, cs2);
        ctx->launches++;
        chunks = 0;
        s->ff_fallback++;
    } else if (rc) {
        return rc;
    } else {
        k_ff_extra_rows<<<3, FF_EXTRA_THREADS, 0, cs2>>>(D, xg, zg, gg, (int)nold);
        ctx->launches++;
        s->ff_steps++;
        s->ff_leaf_level = ctx->plan[2];
    }
    CUDA_TRY(cudaEventRecord(s->ev_join, cs));
    CUDA_TRY(cudaStreamWaitEvent(ctx->stream, s->ev_join, 0));
    CUDA_TRY(cudaEventRecord(s->ev_join, cs2));
    CUDA_TRY(cudaStreamWaitEvent(ctx->stream, s->ev_join, 0));
    enqueue_step_kernel(s, pl, 4, 0, ctx->stream);
    k_finish_ov<<<pl.g4, 256, s->finish_smem, ctx->stream>>>(D, 0, pl.R, pl.slots, chunks);
    if (D.dp) k_pressure<<<1, 256, 0, ctx->stream>>>(D, 0);
    k_advance<<<1, 1, 0, ctx->stream>>>(D, 1);
    ctx->launches += 3 + (D.dp ? 1 : 0);
    CUDA_TRY(cudaGetLastError());
    s->steps_enqueued++;
    return LUDVM_OK;
}

static int set_smem_limits(size_t solve_smem, size_t finish_smem)
{
    if (solve_smem > SOLVE_SMEM_LIMIT + 4096) return set_error(LUDVM_E_UNSUPPORTED, "Npoints too large for the solve kernel");
    if (solve_smem > 48 * 1024) {
        for (int method : {LUDVM_METHOD_FAURE, LUDVM_METHOD_RAMESH}) {
            CUDA_TRY(cudaFuncSetAttribute(method_kernels(method).solve, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)solve_smem));
            CUDA_TRY(cudaFuncSetAttribute(method_kernels(method).solve_small, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)solve_smem));
        }
        CUDA_TRY(cudaFuncSetAttribute(k_sim_cta<CTA_THREADS, LUDVM_METHOD_FAURE, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)solve_smem));
        CUDA_TRY(cudaFuncSetAttribute(k_sim_cta<128, LUDVM_METHOD_FAURE, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)solve_smem));
        CUDA_TRY(cudaFuncSetAttribute(k_sim_cta<CTA_THREADS, LUDVM_METHOD_RAMESH, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)solve_smem));
        CUDA_TRY(cudaFuncSetAttribute(k_sim_cta<CTA_THREADS, LUDVM_METHOD_FAURE, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)solve_smem));
        CUDA_TRY(cudaFuncSetAttribute(k_sim_cta<128, LUDVM_METHOD_FAURE, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)solve_smem));
        CUDA_TRY(cudaFuncSetAttribute(k_sim_cta<CTA_THREADS, LUDVM_METHOD_RAMESH, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)solve_smem));
    }
    if (finish_smem > 48 * 1024)
        CUDA_TRY(cudaFuncSetAttribute(k_finish, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)finish_smem));
    return LUDVM_OK;
}

}  // namespace ludvm

LUDVM_API int ludvm_sim_create(ludvm_ctx *ctx, const ludvm_sim_params *p, const ludvm_sim_tables *t, ludvm_sim **out)
{
    ARG_CHECK(ctx && p && t && out);
    *out = nullptr;
    int rc = check_params(p, t);
    if (rc) return rc;
    DeviceGuard g(ctx->device);
    ludvm_sim *s = new ludvm_sim();
    s->ctx = ctx;
    s->p = *p;
    s->K = p->steps_per_graph > 0 ? p->steps_per_graph : 50;
#define TRY(x) do { if ((rc = (x)) != LUDVM_OK) { ludvm_sim_destroy(s); return rc; } } while (0)
#define CU(x) do { cudaError_t e__ = (x); if (e__ != cudaSuccess) { ludvm_sim_destroy(s); return set_error(LUDVM_E_CUDA, "%s failed: %s", #x, cudaGetErrorString(e__)); } } while (0)
    DevTables dt{};
    TRY(upload_tables(ctx, s->allocs, *p, *t, &dt));
    // exact mode splits the summation tree deeper: its large-wake convection kernel runs one 128-thread CTA per
    // (128 rows, tree node) and wants several waves of 4 CTAs/SM (the split depth never changes a result).  Measured on
    // the 20 000-step dt = 2e-3 run in exact mode: 96 x SMs 16.9 s, 192 x 15.1 s, 384 x 14.4 s.
    const int target = ctx->sm_count * (p->mode == LUDVM_EXACT_F64 ? 384 : 48);
    // shared-memory staging area of the block-wide folds / integrals: all Nc Fourier integrands, or 64 partials of
    // every (row, component), in one batch
    const int sum_nodes = clamp_sum_nodes(p->P, p->Nc, std::max<long>(4096, std::max<long>(p->Nc * p->P, 2 * p->P * 65)));
    Arena measure;
    layout_case(s->d, *p, dt, measure, target, sum_nodes, false);
    void *base;
    TRY(dev_malloc(ctx, s->allocs, measure.off + 256, &base));
    CU(cudaMemsetAsync(base, 0, measure.off + 256, ctx->stream));
    Arena real;
    real.base = (char *)base;
    layout_case(s->d, *p, dt, real, target, sum_nodes, false);
    void *dc;
    TRY(dev_malloc(ctx, s->allocs, sizeof(SimDev), &dc));
    s->d_case = (SimDev *)dc;
    {
        void *db;
        TRY(dev_malloc(ctx, s->allocs, COOP_BAR_WORDS * sizeof(unsigned long long), &db));
        s->d_bar = (unsigned long long *)db;
    }
    CU(cudaMemcpyAsync(s->d_case, &s->d, sizeof(SimDev), cudaMemcpyHostToDevice, ctx->stream));
    k_case_init<<<1, 256, 0, ctx->stream>>>(s->d_case, 1);
    ctx->launches++;
    s->solve_smem = solve_smem_bytes(s->d);
    s->finish_smem = (5 * (size_t)p->P + 8 + (size_t)std::max<long>(FINISH_STAGE, 2 * p->P)) * sizeof(double);
    TRY(set_smem_limits(s->solve_smem, s->finish_smem));
    {   // cooperative path: needs cooperative-launch support and one resident CTA per SM
        int coop = 0, per_sm = 0;
        cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, ctx->device);
        const void *kcoop = method_kernels(p->method).persist_coop;
        if (coop && cudaFuncSetAttribute(kcoop, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s->solve_smem) == cudaSuccess &&
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kcoop, 256, s->solve_smem) == cudaSuccess && per_sm >= 1)
            s->coop_grid = ctx->sm_count;
        cudaGetLastError();
        // cluster path: one thread-block cluster of SIM_CLUSTER_CTAS CTAs (16 needs the non-portable opt-in), if the
        // device can co-schedule it with this much shared memory per CTA
        if (!getenv("LUDVM_NO_CLUSTER")) {
            const void *kern = method_kernels(p->method).persist_cluster;
            if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s->solve_smem) == cudaSuccess &&
                cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess) {
                cudaLaunchConfig_t cfg = {};
                cfg.gridDim = dim3(SIM_CLUSTER_CTAS);
                cfg.blockDim = dim3(256);
                cfg.dynamicSmemBytes = s->solve_smem;
                cudaLaunchAttribute at[1];
                at[0].id = cudaLaunchAttributeClusterDimension;
                at[0].val.clusterDim.x = SIM_CLUSTER_CTAS; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
                cfg.attrs = at; cfg.numAttrs = 1;
                int nclusters = 0;
                if (cudaOccupancyMaxActiveClusters(&nclusters, kern, &cfg) == cudaSuccess && nclusters >= 1) s->cluster_ctas = SIM_CLUSTER_CTAS;
            }
            cudaGetLastError();
        }
    }
    CU(cudaStreamSynchronize(ctx->stream));  // the host tables may be freed by the caller after return
#undef TRY
#undef CU
    *out = s;
    return LUDVM_OK;
}

LUDVM_API int ludvm_sim_enable_pressure(ludvm_sim *s)
{
    ARG_CHECK(s != nullptr);
    if (s->steps_enqueued > 0) return set_error(LUDVM_E_STATE, "ludvm_sim_enable_pressure must precede the first step");
    if (s->d.dp) return LUDVM_OK;
    DeviceGuard g(s->ctx->device);
    const size_t bytes = (size_t)s->d.nt * s->d.P * sizeof(double);
    void *p;
    int rc = dev_malloc(s->ctx, s->allocs, bytes, &p);
    if (rc) return rc;
    CUDA_TRY(cudaMemsetAsync(p, 0, bytes, s->ctx->stream));   // row 0 and rows of steps not run stay zero
    s->d.dp = (double *)p;   // every driver takes `d` by value at launch
    CUDA_TRY(cudaStreamSynchronize(s->ctx->stream));
    return LUDVM_OK;
}

LUDVM_API int ludvm_sim_enable_far_field(ludvm_sim *s, int order)
{
    ARG_CHECK(s != nullptr);
    if (s->steps_enqueued > 0) return set_error(LUDVM_E_STATE, "ludvm_sim_enable_far_field must precede the first step");
    if (s->p.mode == LUDVM_EXACT_F64)
        return set_error(LUDVM_E_UNSUPPORTED, "the far field is an approximation; exact mode keeps numpy's sums bit for bit");
    if (s->p.method == LUDVM_METHOD_RAMESH)
        return set_error(LUDVM_E_UNSUPPORTED, "the far-field step is built for method Faure; method='Ramesh' convects by all pairs");
    if (s->p.P > 256)
        return set_error(LUDVM_E_UNSUPPORTED, "P = %ld: the far-field step builds on the overlapped step, which needs P <= 256",
                         (long)s->p.P);
    if (order < 2 || order > TR_MAX_ORDER)
        return set_error(LUDVM_E_ARG, "far-field order %d outside 2..%d", order, TR_MAX_ORDER);
    DeviceGuard g(s->ctx->device);
    if (!s->ff_xzg) {
        void *p;
        int rc = dev_malloc(s->ctx, s->allocs, 3 * (2 * (size_t)s->d.nv + s->d.nfree) * sizeof(double), &p);
        if (rc) return rc;
        s->ff_xzg = (double *)p;
    }
    s->ff_order = order;
    return LUDVM_OK;
}

LUDVM_API int ludvm_sim_far_field_info(ludvm_sim *s, int64_t out[4])
{
    ARG_CHECK(s != nullptr && out != nullptr);
    out[0] = s->ff_steps;
    out[1] = s->ff_fallback;
    out[2] = s->ff_order;
    out[3] = s->ff_leaf_level;
    return LUDVM_OK;
}

LUDVM_API int ludvm_sim_run(ludvm_sim *s, long nsteps)
{
    ARG_CHECK(s != nullptr && nsteps >= 0);
    DeviceGuard g(s->ctx->device);
    long total = s->p.nt - 1;
    long todo = std::min(nsteps, total - s->steps_enqueued);
    if (todo <= 0) return LUDVM_OK;
    // smallest wakes: ONE thread-block cluster with the hardware cluster barrier between the phases
    if (s->cluster_ctas >= 4) {
        const long last_small = (SIM_CLUSTER_MAX_WAKE - 2 - (long)s->p.nfree) / 2;
        long k = std::min(todo, last_small - s->steps_enqueued);
        if (k > 0) {
            SimDev dc = s->d;
            dc.target_warps = s->cluster_ctas * 8;
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3(s->cluster_ctas);
            cfg.blockDim = dim3(256);
            cfg.dynamicSmemBytes = s->solve_smem;
            cfg.stream = s->ctx->stream;
            cudaLaunchAttribute at[1];
            at[0].id = cudaLaunchAttributeClusterDimension;
            at[0].val.clusterDim.x = s->cluster_ctas; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
            cfg.attrs = at; cfg.numAttrs = 1;
            unsigned long long *nobar = nullptr;
            int ki = (int)k;
            void *args[] = {&dc, &ki, &nobar};
            CUDA_TRY(cudaLaunchKernelExC(&cfg, method_kernels(s->p.method).persist_cluster, args));
            s->ctx->launches++;
            s->steps_enqueued += k;
            todo -= k;
        }
    }
    // small wakes: the persistent cooperative kernel, all of those steps in one launch
    if (s->coop_grid >= 4 && !getenv("LUDVM_NO_COOP")) {
        // fast mode hands over to the graph path (tiled, overlapped step) earlier than exact mode does
        const long coop_max = s->p.mode == LUDVM_EXACT_F64 ? SIM_COOP_MAX_WAKE : SIM_TILED_MIN_WAKE;
        const long last_small = (coop_max - 2 - (long)s->p.nfree) / 2;   // wake after step i <= 2 i + 2 + nfree
        long k = std::min(todo, last_small - s->steps_enqueued);
        if (k > 0) {
            SimDev dc = s->d;
            dc.target_warps = s->coop_grid * 8;   // one wave of warp tasks over the resident grid
            int ki = (int)k;
            unsigned long long *bar = s->d_bar;
            void *args[] = {&dc, &ki, &bar};
            CUDA_TRY(cudaMemsetAsync(s->d_bar, 0, COOP_BAR_WORDS * sizeof(unsigned long long), s->ctx->stream));
            CUDA_TRY(cudaLaunchCooperativeKernel(method_kernels(s->p.method).persist_coop, dim3(s->coop_grid), dim3(256), args, s->solve_smem, s->ctx->stream));
            s->ctx->launches++;
            s->steps_enqueued += k;
            todo -= k;
        }
    }
    // graphs of K unrolled steps (a shorter one for a tail), cached per (wake-size bracket, length).  With the far field
    // enabled, the steps from far_field_first_step on are far-field steps, each with the plan of the graph it stands in for.
    const long ff_first = s->ff_order ? far_field_first_step(s) : total;
    while (todo > 0) {
        int k = (int)std::min<long>(s->K, todo);
        int b = bracket_of(wake_upper(s, s->steps_enqueued));
        if (s->steps_enqueued >= ff_first) {
            const StepPlan pl = plan_step(s, b);
            for (int j = 0; j < k; j++) {
                int rc = far_field_step(s, pl);
                if (rc) return rc;
            }
            todo -= k;
            continue;
        }
        k = (int)std::min<long>(k, ff_first - s->steps_enqueued);
        int key = b * 100000 + k;
        auto it = s->graphs.find(key);
        if (it == s->graphs.end()) {
            cudaGraphExec_t ge;
            int rc = build_graph(s, b, k, &ge);
            if (rc) return rc;
            it = s->graphs.emplace(key, ge).first;
        }
        CUDA_TRY(cudaGraphLaunch(it->second, s->ctx->stream));
        s->ctx->launches += (plan_step(s, b).ov ? 5L : 4L) * k + (s->d.dp ? k : 0) + 1;
        s->steps_enqueued += k;
        todo -= k;
    }
    return LUDVM_OK;
}

// Diagnostic twin of ludvm_sim_run for the graph path: the same kernels with the same launch geometry, launched one
// by one with CUDA events around each, so that the share of each phase in a step can be reported (profiles/).
LUDVM_API int ludvm_sim_profile_steps(ludvm_sim *s, long nsteps, double *ms_out)
{
    ARG_CHECK(s != nullptr && nsteps >= 0 && ms_out != nullptr);
    if (s->ff_order)
        return set_error(LUDVM_E_UNSUPPORTED, "the far-field step is not one of the graph path's phases; time ludvm_sim_run");
    DeviceGuard g(s->ctx->device);
    for (int q = 0; q < 5; q++) ms_out[q] = 0.0;
    long total = s->p.nt - 1;
    long todo = std::min(nsteps, total - s->steps_enqueued);
    if (todo <= 0) return LUDVM_OK;
    cudaStream_t st = s->ctx->stream;
    cudaEvent_t ev[5];
    for (auto &e : ev) CUDA_TRY(cudaEventCreate(&e));
    for (long k = 0; k < todo; k++) {
        const StepPlan pl = plan_step(s, bracket_of(wake_upper(s, s->steps_enqueued)));
        for (int which = 0; which < 4; which++) {
            CUDA_TRY(cudaEventRecord(ev[which], st));
            enqueue_step_kernel(s, pl, which, 0, st);
            if (which == 2 && pl.ov) enqueue_step_kernel(s, pl, 4, 0, st);
        }
        CUDA_TRY(cudaEventRecord(ev[4], st));
        k_advance<<<1, 1, 0, st>>>(s->d, 1);
        CUDA_TRY(cudaEventSynchronize(ev[4]));
        for (int which = 0; which < 4; which++) {
            float ms = 0.f;
            CUDA_TRY(cudaEventElapsedTime(&ms, ev[which], ev[which + 1]));
            ms_out[which] += ms;
            ms_out[4] += ms;
        }
        s->ctx->launches += s->d.dp ? 6 : 5;
        s->steps_enqueued += 1;
    }
    CUDA_TRY(cudaStreamSynchronize(st));
    for (auto &e : ev) cudaEventDestroy(e);
    CUDA_TRY(cudaGetLastError());
    return LUDVM_OK;
}

#ifdef LUDVM_TRACE
extern "C" __attribute__((visibility("default"))) int ludvm_debug_trace(long long *out)
{
    return cudaMemcpyFromSymbol(out, ludvm::g_trace, sizeof(long long) * 64) == cudaSuccess ? 0 : -1;
}
#endif

LUDVM_API int ludvm_sim_steps_done(ludvm_sim *s, long *out)
{
    ARG_CHECK(s && out);
    DeviceGuard g(s->ctx->device);
    long long v = 0;
    CUDA_TRY(cudaMemcpyAsync(&v, s->d.counters, sizeof(v), cudaMemcpyDeviceToHost, s->ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(s->ctx->stream));
    *out = (long)v;
    return LUDVM_OK;
}

static int field_info(ludvm_sim *s, int field, const void **ptr, size_t *bytes)
{
    const SimDev &D = s->d;
    const size_t nt = D.nt, nv = D.nv, P = D.P, Nc = D.Nc, nf = D.nfree, d8 = sizeof(double);
    switch (field) {
    case LUDVM_F_PATH_TEV: *ptr = D.path_tev; *bytes = ((nt - 1) / std::max(1, D.store_history) + 1) * 2 * nv * d8; break;
    case LUDVM_F_PATH_LEV: *ptr = D.path_lev; *bytes = ((nt - 1) / std::max(1, D.store_history) + 1) * 2 * nv * d8; break;
    case LUDVM_F_PATH_FREE: *ptr = D.path_free; *bytes = nt * 2 * nf * d8; break;
    case LUDVM_F_G_TEV: *ptr = D.wg; *bytes = nv * d8; break;
    case LUDVM_F_G_LEV: *ptr = D.wg + nv; *bytes = nv * d8; break;
    case LUDVM_F_G_BOUND: *ptr = D.g_bound; *bytes = nv * d8; break;
    case LUDVM_F_G_AIRFOIL: *ptr = D.g_airfoil; *bytes = nv * P * d8; break;
    case LUDVM_F_GAMMA_AIRFOIL: *ptr = D.gamma_airfoil; *bytes = nv * P * d8; break;
    case LUDVM_F_GAMMA_INT_AIRFOIL: *ptr = D.Gamma_airfoil; *bytes = nv * P * d8; break;
    case LUDVM_F_FOURIER: *ptr = D.fourier; *bytes = nt * 2 * Nc * d8; break;
    case LUDVM_F_LESP: *ptr = D.lesp; *bytes = nt * d8; break;
    case LUDVM_F_LESP_PREV: *ptr = D.lesp_prev; *bytes = nt * d8; break;
    case LUDVM_F_LEV_SHED: *ptr = D.lev_shed; *bytes = nt * d8; break;
    case LUDVM_F_FN: *ptr = D.Fn; *bytes = nt * d8; break;
    case LUDVM_F_FS: *ptr = D.Fs; *bytes = nt * d8; break;
    case LUDVM_F_L: *ptr = D.L; *bytes = nt * d8; break;
    case LUDVM_F_D: *ptr = D.D; *bytes = nt * d8; break;
    case LUDVM_F_T: *ptr = D.T; *bytes = nt * d8; break;
    case LUDVM_F_M: *ptr = D.M; *bytes = nt * d8; break;
    case LUDVM_F_COUNTERS: *ptr = D.counters; *bytes = 4 * sizeof(long long); break;
    case LUDVM_F_RANGE_BAD: *ptr = D.range_bad; *bytes = sizeof(int); break;
    case LUDVM_F_DP: *ptr = D.dp; *bytes = nt * P * d8; break;
    case LUDVM_F_CUR_TEV: case LUDVM_F_CUR_LEV: case LUDVM_F_CUR_FREE:
        *ptr = nullptr; *bytes = 2 * (field == LUDVM_F_CUR_FREE ? nf : nv) * d8; break;
    default: return set_error(LUDVM_E_ARG, "unknown field %d", field);
    }
    return LUDVM_OK;
}

LUDVM_API int ludvm_sim_field_bytes(ludvm_sim *s, int field, size_t *out)
{
    ARG_CHECK(s && out);
    const void *p;
    return field_info(s, field, &p, out);
}

// Several result fields in one call: every copy is enqueued, then ONE synchronisation (a run's results are ~25 fields;
// fetching them one by one costs a stream synchronisation each).
LUDVM_API int ludvm_sim_fetch_many(ludvm_sim *s, int nfields, const int *fields, void *const *dsts, const size_t *bytes)
{
    ARG_CHECK(s && nfields >= 0 && (nfields == 0 || (fields && dsts && bytes)));
    DeviceGuard g(s->ctx->device);
    cudaStream_t st = s->ctx->stream;
    for (int k = 0; k < nfields; k++) {
        ARG_CHECK(dsts[k] != nullptr);
        const void *p;
        size_t want;
        int rc = field_info(s, fields[k], &p, &want);
        if (rc) return rc;
        if (bytes[k] != want)
            return set_error(LUDVM_E_ARG, "field %d holds %zu bytes, caller passed %zu", fields[k], want, bytes[k]);
        if (fields[k] == LUDVM_F_CUR_TEV || fields[k] == LUDVM_F_CUR_LEV || fields[k] == LUDVM_F_CUR_FREE) {
            const SimDev &D = s->d;
            size_t off = fields[k] == LUDVM_F_CUR_TEV ? 0 : (fields[k] == LUDVM_F_CUR_LEV ? D.nv : 2 * (size_t)D.nv);
            size_t n = fields[k] == LUDVM_F_CUR_FREE ? D.nfree : D.nv;
            CUDA_TRY(cudaMemcpyAsync(dsts[k], D.wx + off, n * sizeof(double), cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaMemcpyAsync((double *)dsts[k] + n, D.wz + off, n * sizeof(double), cudaMemcpyDeviceToHost, st));
        } else {
            if (!p && fields[k] == LUDVM_F_DP) return set_error(LUDVM_E_STATE, "the pressure jump was not enabled (ludvm_sim_enable_pressure)");
            if (!p) return set_error(LUDVM_E_STATE, "field %d was not kept (store_history = 0)", fields[k]);
            CUDA_TRY(cudaMemcpyAsync(dsts[k], p, want, cudaMemcpyDeviceToHost, st));
        }
    }
    CUDA_TRY(cudaStreamSynchronize(st));
    return LUDVM_OK;
}

LUDVM_API int ludvm_sim_fetch(ludvm_sim *s, int field, void *dst, size_t bytes)
{
    return ludvm_sim_fetch_many(s, 1, &field, &dst, &bytes);
}

LUDVM_API int ludvm_sim_destroy(ludvm_sim *s)
{
    if (!s) return LUDVM_OK;
    DeviceGuard g(s->ctx->device);
    cudaStreamSynchronize(s->ctx->stream);
    for (auto &kv : s->graphs) cudaGraphExecDestroy(kv.second);
    if (s->cap_stream) cudaStreamDestroy(s->cap_stream);
    if (s->cap_stream2) cudaStreamDestroy(s->cap_stream2);
    if (s->ev_fork) cudaEventDestroy(s->ev_fork);
    if (s->ev_join) cudaEventDestroy(s->ev_join);
    for (void *p : s->allocs) cudaFreeAsync(p, s->ctx->stream);
    delete s;
    return LUDVM_OK;
}

// ---------------------------------------------------------------------------------------------------
// batched parameter sweep (BASELINE.json configs[3]): ncases independent simulations, one CTA per case
// ---------------------------------------------------------------------------------------------------
namespace ludvm {

using SweepKernel = void (*)(const SimDev *, int, int *, int);

template <int THREADS, int METHOD>
static SweepKernel sweep_kernel(bool dp)
{
    return dp ? k_sim_cta<THREADS, METHOD, true> : k_sim_cta<THREADS, METHOD, false>;
}

// ludvm_sweep_run (dp null) and ludvm_sweep_run_pressure: dp, if set, is a host buffer [ncases][nt][P].
static int sweep_run(ludvm_ctx *ctx, long ncases, const ludvm_sim_params *params, const ludvm_sim_tables *tables,
                     double *out, size_t out_doubles_per_case, double *dp, size_t dp_doubles_per_case)
{
    ARG_CHECK(ctx && params && tables && out && ncases > 0 && ncases < (1 << 24));
    int rc;
    const ludvm_sim_params &p0 = params[0];
    for (long c = 0; c < ncases; c++) {
        if ((rc = check_params(&params[c], &tables[c]))) return rc;
        ARG_CHECK(params[c].nt == p0.nt && params[c].P == p0.P && params[c].Nc == p0.Nc && params[c].nfree == p0.nfree &&
                  params[c].method == p0.method);
    }
    const size_t nt = p0.nt;
    ARG_CHECK(out_doubles_per_case == (size_t)LUDVM_SWEEP_FIELDS * nt);
    if (dp) ARG_CHECK(dp_doubles_per_case == nt * (size_t)p0.P);
    DeviceGuard g(ctx->device);
    std::vector<void *> allocs;
    auto cleanup = [&]() { for (void *p : allocs) cudaFreeAsync(p, ctx->stream); };
    const bool tm = getenv("LUDVM_SWEEP_TIMING") != nullptr;   // stderr breakdown of the call (diagnostic)
    auto now = [&]() { if (tm) cudaStreamSynchronize(ctx->stream); return std::chrono::steady_clock::now(); };
    auto t0 = now();
#define TRY(x) do { if ((rc = (x)) != LUDVM_OK) { cleanup(); return rc; } } while (0)
#define CU(x) do { cudaError_t e__ = (x); if (e__ != cudaSuccess) { cleanup(); return set_error(LUDVM_E_CUDA, "%s failed: %s", #x, cudaGetErrorString(e__)); } } while (0)
    // table sets shared by several cases (same host pointers) are uploaded once
    std::map<const double *, DevTables> uploaded;
    std::vector<SimDev> host_cases((size_t)ncases);
    std::vector<DevTables> dts((size_t)ncases);
    const bool ramesh = p0.method == LUDVM_METHOD_RAMESH;
    // threads per case: 256 (three resident cases per SM) in fast mode; in exact mode 128 threads with the cos/sin(n theta)
    // tables read from global memory put six cases on an SM and win (4096-case sweep, 256 / 128 threads: fast 0.511 / 0.537 s,
    // exact 0.899 / 0.832 s; profiles/r02v_sweep_threads.txt).
    const int cta_threads = (!ramesh && p0.mode == LUDVM_EXACT_F64) ? 128 : CTA_THREADS;
    const int target = 2 * (cta_threads / 32), sum_nodes = clamp_sum_nodes(p0.P, p0.Nc, std::max<long>(256, p0.Nc * p0.P));
    Arena measure;
    for (long c = 0; c < ncases; c++) {
        auto it = uploaded.find(tables[c].gp);
        if (it == uploaded.end()) {
            DevTables dt{};
            TRY(upload_tables(ctx, allocs, params[c], tables[c], &dt));
            it = uploaded.emplace(tables[c].gp, dt).first;
        }
        dts[c] = it->second;
        layout_case(host_cases[c], params[c], dts[c], measure, target, sum_nodes, true, cta_threads);
    }
    void *base;
    TRY(dev_malloc(ctx, allocs, measure.off + 256, &base));
    CU(cudaMemsetAsync(base, 0, measure.off + 256, ctx->stream));
    Arena real;
    real.base = (char *)base;
    for (long c = 0; c < ncases; c++) layout_case(host_cases[c], params[c], dts[c], real, target, sum_nodes, true, cta_threads);
    // the pressure jump lives outside the arena (a sweep without it keeps the arena's layout); row 0 of each case stays 0
    void *ddp = nullptr;
    const size_t dp_bytes = dp ? sizeof(double) * (size_t)ncases * dp_doubles_per_case : 0;
    if (dp) {
        TRY(dev_malloc(ctx, allocs, dp_bytes, &ddp));
        CU(cudaMemsetAsync(ddp, 0, dp_bytes, ctx->stream));
        for (long c = 0; c < ncases; c++) host_cases[c].dp = (double *)ddp + (size_t)c * dp_doubles_per_case;
    }
    void *dcases, *dnext;
    TRY(dev_malloc(ctx, allocs, sizeof(SimDev) * (size_t)ncases + 256, &dcases));
    TRY(dev_malloc(ctx, allocs, 256, &dnext));
    CU(cudaMemcpyAsync(dcases, host_cases.data(), sizeof(SimDev) * (size_t)ncases, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemsetAsync(dnext, 0, sizeof(int), ctx->stream));
    k_case_init<<<(unsigned)ncases, 256, 0, ctx->stream>>>((const SimDev *)dcases, (int)ncases);
    auto t1 = now();
    size_t smem = solve_smem_bytes(host_cases[0]);
    TRY(set_smem_limits(smem, 0));
    const SweepKernel kern = cta_threads == 128 ? sweep_kernel<128, LUDVM_METHOD_FAURE>(dp)
                             : ramesh          ? sweep_kernel<CTA_THREADS, LUDVM_METHOD_RAMESH>(dp)
                                               : sweep_kernel<CTA_THREADS, LUDVM_METHOD_FAURE>(dp);
    int per_sm = 1;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, cta_threads, smem));
    int grid = (int)std::min<long>(ncases, (long)ctx->sm_count * std::max(per_sm, 1));
    kern<<<grid, cta_threads, smem, ctx->stream>>>((const SimDev *)dcases, (int)ncases, (int *)dnext, (int)nt);
    ctx->launches += 2;
    CU(cudaGetLastError());
    auto t2 = now();
    void *dout;
    const size_t out_bytes = sizeof(double) * (size_t)ncases * out_doubles_per_case;
    TRY(dev_malloc(ctx, allocs, out_bytes, &dout));
    k_sweep_gather<<<(unsigned)ncases, 256, 0, ctx->stream>>>((const SimDev *)dcases, (int)ncases, (double *)dout);
    ctx->launches++;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(out, dout, out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    if (dp) CU(cudaMemcpyAsync(dp, ddp, dp_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    auto t3 = now();
#undef CU
#undef TRY
    cleanup();
    if (tm) {
        auto t4 = std::chrono::steady_clock::now();
        auto ms = [](auto a, auto b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
        fprintf(stderr, "ludvm_sweep_run: upload+alloc+init %.1f ms, kernel %.1f ms, gather+D2H %.1f ms, free %.1f ms (arena %.0f MB, "
                "dp %.0f MB, %d cases resident per SM)\n",
                ms(t0, t1), ms(t1, t2), ms(t2, t3), ms(t3, t4), measure.off / 1048576.0, dp_bytes / 1048576.0, per_sm);
    }
    return LUDVM_OK;
}

}  // namespace ludvm

LUDVM_API int ludvm_sweep_run(ludvm_ctx *ctx, long ncases, const ludvm_sim_params *params,
                              const ludvm_sim_tables *tables, double *out, size_t out_doubles_per_case)
{
    return sweep_run(ctx, ncases, params, tables, out, out_doubles_per_case, nullptr, 0);
}

LUDVM_API int ludvm_sweep_run_pressure(ludvm_ctx *ctx, long ncases, const ludvm_sim_params *params,
                                       const ludvm_sim_tables *tables, double *out, size_t out_doubles_per_case,
                                       double *dp, size_t dp_doubles_per_case)
{
    ARG_CHECK(dp != nullptr);
    return sweep_run(ctx, ncases, params, tables, out, out_doubles_per_case, dp, dp_doubles_per_case);
}

namespace ludvm {

// Defined last: the translation unit's device code is emitted in the order its kernels are first referenced, and that
// order feeds the device compiler's optimisation order.  With every Ramesh instantiation referenced here, after all Faure
// kernels (k_wake_on_foil / k_solve / k_solve_small<Faure> are instantiated explicitly at their definitions), the Faure
// kernels compile to the same SASS as before Ramesh had single-simulation drivers.
static const MethodKernels &method_kernels(int method)
{
    static const MethodKernels faure{k_wake_on_foil<LUDVM_METHOD_FAURE>, k_solve<LUDVM_METHOD_FAURE>,
                                     k_solve_small<LUDVM_METHOD_FAURE>, (const void *)k_sim_persist<false, LUDVM_METHOD_FAURE>,
                                     (const void *)k_sim_persist<true, LUDVM_METHOD_FAURE>};
    static const MethodKernels ramesh{k_wake_on_foil<LUDVM_METHOD_RAMESH>, k_solve<LUDVM_METHOD_RAMESH>,
                                      k_solve_small<LUDVM_METHOD_RAMESH>, (const void *)k_sim_persist<false, LUDVM_METHOD_RAMESH>,
                                      (const void *)k_sim_persist<true, LUDVM_METHOD_RAMESH>};
    return method == LUDVM_METHOD_RAMESH ? ramesh : faure;
}

}  // namespace ludvm
