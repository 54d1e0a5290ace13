/*
 * ludvm_b200.h -- C ABI of libludvm_b200.so: the B200 (sm_100a) implementation of the per-timestep
 * vortex-velocity hot path of jcatalang/LUDVM.
 *
 * The reference has no FFI layer of its own (it is a single numpy file); its boundary is the Python class
 * `LUDVM` (LUDVM.py:132).  Each entry point below replaces the arithmetic of one reference method and is
 * bound with ctypes by the drop-in class `ludvm_b200.LUDVM` (see INTEGRATION.md for the stub a reference
 * maintainer would add).  Citations are to /root/reference/LUDVM.py.
 *
 * Conventions
 *   - every function returns 0 on success, a negative LUDVM_E_* code otherwise; the message of the last
 *     failure on the calling thread is `ludvm_last_error()`;
 *   - no exceptions and no ownership cross the ABI: the caller owns every buffer, the library owns only the
 *     opaque handles it returns;
 *   - all arrays are contiguous IEEE float64 unless stated; `ptr_kind` says whether the array arguments of a
 *     call are host pointers (copied through the context's staging buffers on its stream, the call returns
 *     after the results are in the host buffers) or device pointers (the call only enqueues work on the
 *     context's stream);
 *   - a context owns one CUDA stream; a context is not thread-safe, distinct contexts are;
 *   - there is NO CPU fallback: without a CUDA device every call fails with LUDVM_E_CUDA.
 *
 * Arithmetic modes
 *   LUDVM_EXACT_F64  bit-reproduces the reference's numpy arithmetic: unfused IEEE + - * / sqrt in the
 *                    reference's operation order and numpy's pairwise-summation tree (np.sum / np.trapz),
 *                    LAPACK's 2x2 solve.  Needed because the time loop is chaotic (SURVEY.md 4.3).
 *   LUDVM_FAST_F64   FMA + MUFU.RSQ64H-seeded reciprocal square root (13 FP64-pipe slots per pair); per-call
 *                    results within 1e-12 of the reference relative to sum |terms|.
 *   LUDVM_FAST_F32   single-precision pair arithmetic (inputs/outputs still float64); reported separately.
 *   LUDVM_FAST12_F64 opt-in (all-pairs entry points only): 12 FP64-pipe slots per pair -- one second-order refinement of a
 *                    centred MUFU seed; |error| <= 4.3e-13 per pair (inside the 1e-12 statement, 2.3x margin) instead
 *                    of 2.7e-16, ~7 % faster.  Used by the fused single-launch kernel; launches that are not eligible
 *                    for it fall back to LUDVM_FAST_F64.  Reported separately.
 */
#ifndef LUDVM_B200_H
#define LUDVM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LUDVM_B200_ABI_VERSION 1

enum { LUDVM_EXACT_F64 = 0, LUDVM_FAST_F64 = 1, LUDVM_FAST_F32 = 2, LUDVM_FAST12_F64 = 3 };
enum { LUDVM_PTR_HOST = 0, LUDVM_PTR_DEVICE = 1 };
enum { LUDVM_METHOD_FAURE = 0, LUDVM_METHOD_RAMESH = 1 };

enum {
    LUDVM_OK = 0,
    LUDVM_E_ARG = -1,      /* bad argument (null pointer, negative size, unknown mode ...) */
    LUDVM_E_CUDA = -2,     /* CUDA runtime error (message in ludvm_last_error) */
    LUDVM_E_NOMEM = -3,    /* device or host allocation failed */
    LUDVM_E_STATE = -4,    /* call not valid in the handle's current state */
    LUDVM_E_UNSUPPORTED = -5
};

typedef struct ludvm_ctx ludvm_ctx;
typedef struct ludvm_sim ludvm_sim;

int ludvm_abi_version(void);
const char *ludvm_last_error(void);

/* Context = device + stream + scratch.  `cuda_stream` is a cudaStream_t to enqueue on (e.g. PyTorch's current
 * stream), or NULL to let the context create its own non-blocking stream. */
int ludvm_ctx_create(int device, void *cuda_stream, ludvm_ctx **out);
int ludvm_ctx_destroy(ludvm_ctx *ctx);
int ludvm_ctx_synchronize(ludvm_ctx *ctx);
/* Number of kernels this context has launched since creation (bench.py's `gpu_launches`). */
int ludvm_ctx_launch_count(ludvm_ctx *ctx, long long *out);
/* Which all-pairs kernel the last induced_velocity / selfconv_step / flowfield_velocity call on this context chose
 * (diagnostic; the parity tests assert that the instantiation a benchmark times is the one they checked):
 * out[0] = LUDVM_K_* kernel id, out[1] = target rows per thread (or per lane), out[2] = source chunks folded per row
 * (fast kernels) or depth of the summation-tree cut (exact kernels), out[3] = 1 if sources are staged with bulk
 * copies (TMA engine), out[4] = thread-block cluster size, out[5] = kernel variant (source-loop unroll of the fused
 * kernel; exact kernels: 1 = a range scan of the coordinates preceded the launch and selects, on the device, the
 * instantiation without per-pair range words), out[6] = warps per CTA of the fused kernel, out[7] = exact kernels
 * with out[5] = 1: the scan's verdict (0 = every coordinate inside the window, the flag-free instantiation ran;
 * 1 = the flagged instantiation ran; reading it synchronises the context's stream), fused kernel: 1 = 12-slot pair arithmetic. */
enum { LUDVM_K_NONE = 0, LUDVM_K_EXACT_ROWS = 1, LUDVM_K_EXACT_TILED = 2, LUDVM_K_FAST_ROWS = 3, LUDVM_K_FAST_TILED = 4,
       LUDVM_K_FAST_TILED_TMA = 5, LUDVM_K_FAST32_TILED = 6, LUDVM_K_FAST32X2_TILED = 7, LUDVM_K_FAST_FUSED = 8,
       LUDVM_K_TREE = 9 /* out[2] = leaf level of the quadtree, out[5] = interpolation order */,
       LUDVM_K_FAST_SYM = 10 /* ludvm_selfconv_step_all: out[1] = rows per lane, out[5] = columns per staged block */ };
int ludvm_ctx_last_plan(ludvm_ctx *ctx, int32_t out[8]);

/*
 * induced_velocity -- replaces LUDVM.induced_velocity (LUDVM.py:549-570).
 *   u_i =  sum_j G_j (z_i - z_j) / (2 pi sqrt(r_ij^4 + vc^4)),  w_i = -sum_j G_j (x_i - x_j) / (...)
 * gamma has ngamma == nw entries, or ngamma == 1 (broadcast, as the unit-strength calls LUDVM.py:751 do).
 * vc4 is the value of `v_core**4` evaluated by the caller (0.0 for viscous=False); vc4_per_source, when not
 * NULL, overrides it with one core radius^4 per source vortex (a superset of the reference).
 */
int ludvm_induced_velocity(ludvm_ctx *ctx, int mode, const double *gamma, long ngamma, const double *xw,
                           const double *zw, const double *vc4_per_source, double vc4, long nw,
                           const double *xp, const double *zp, long np, double *u, double *w, int ptr_kind);

/*
 * Self-convection of a vortex cloud, target-row shard [row0, row0+nrows) of n vortices (BASELINE.json
 * config 3; the convection phase LUDVM.py:1095-1127 without the aerofoil): forward Euler
 *   x_out[i] = x[i] + dt * u_i,  z_out[i] = z[i] + dt * w_i   for the shard's rows, against all n sources.
 * Device pointers only; x_out/z_out are full-length arrays (only the shard's rows are written), so that an
 * all-gather over the row shards completes the step.  u_out/w_out (nullable) receive the shard's velocities.
 */
int ludvm_selfconv_step(ludvm_ctx *ctx, int mode, const double *gamma, const double *x, const double *z,
                        const double *vc4_per_source, double vc4, long n, long row0, long nrows, double dt,
                        double *x_out, double *z_out, double *u_out, double *w_out);

/*
 * The same step for the whole cloud (row0 = 0, nrows = n), with the same results bit for bit.  In fast mode with one
 * finite core vc4 > 0 (vc4_per_source NULL), 16-byte aligned arrays and n >= 2^17 it evaluates every unordered pair
 * once and applies the shared part of the term to both vortices (LUDVM_K_FAST_SYM: 8 FP64-pipe slots per term instead
 * of 13); otherwise it does exactly what ludvm_selfconv_step(..., row0 = 0, nrows = n, ...) does.  A LUDVM_K_FAST_SYM
 * launch that stops making progress gives up instead of hanging; the next ludvm_selfconv_step_all or
 * ludvm_ctx_synchronize on the context then returns LUDVM_E_CUDA.
 */
int ludvm_selfconv_step_all(ludvm_ctx *ctx, int mode, const double *gamma, const double *x, const double *z,
                            const double *vc4_per_source, double vc4, long n, double dt, double *x_out, double *z_out,
                            double *u_out, double *w_out);

/*
 * Same step with the all-gather fused into the kernel epilogue: instead of writing the shard's rows locally for a
 * later NCCL all-gather, the Euler-update kernel stores them straight into the next-position buffers of all
 * `npeers` ranks (peer-mapped device pointers, e.g. from torch.distributed._symmetric_memory; include this rank's
 * own buffer) over NVLink/NVSwitch.  The caller separates consecutive steps with a cross-rank barrier.
 */
#define LUDVM_MAX_PEERS 16
int ludvm_selfconv_step_p2p(ludvm_ctx *ctx, int mode, const double *gamma, const double *x, const double *z,
                            const double *vc4_per_source, double vc4, long n, long row0, long nrows, double dt,
                            int npeers, double *const *x_out_peers, double *const *z_out_peers);

/*
 * O(N log N) far field for clouds with N >> 2^20 (SURVEY.md section 8(f)-4).  The reference has no counterpart: its
 * induced_velocity (LUDVM.py:549-570) is all-pairs, and these calls approximate exactly that sum.  A kernel-independent
 * treecode: quadtree in Morton order over the bounding square, the far field of a cell carried by (order + 1)^2 proxy
 * vortices at its tensor Chebyshev points (barycentric Lagrange anterpolation, nested over the levels), one-cell
 * separation lists; near field and proxies are evaluated with the LUDVM_FAST_F64 pair arithmetic.  `order` 2..24
 * (<= 0: 18) sets the accuracy -- measured against the all-pairs sum, relative to sum |terms|: order 12 ~ 2e-11,
 * 16 ~ 5e-14, 18 ~ 3e-15 -- and `leaf` the wanted mean number of vortices per leaf cell (<= 0: the proxies per cell,
 * (order + 1)^2).  Results are bitwise reproducible and do not depend on how target rows are split over GPUs.
 * stats (host pointer, nullable) receives 8 doubles: leaf level, leaf side, pair evaluations done, np * nw, proxies per
 * cell, device arena bytes, ms of tree build + upward pass, ms of the evaluation kernel; asking for it synchronises the
 * stream.
 */
int ludvm_induced_velocity_tree(ludvm_ctx *ctx, const double *gamma, const double *xw, const double *zw, double vc4,
                                long nw, const double *xp, const double *zp, long np, int order, int leaf, double *u,
                                double *w, int ptr_kind, double *stats);
/* ludvm_selfconv_step through the treecode (device pointers): rows [row0, row0 + nrows) of x_out / z_out are written. */
int ludvm_selfconv_step_tree(ludvm_ctx *ctx, const double *gamma, const double *x, const double *z, double vc4, long n,
                             long row0, long nrows, double dt, int order, int leaf, double *x_out, double *z_out,
                             double *u_out, double *w_out, double *stats);

/* ludvm_flowfield_velocity (one source set) through the same hierarchical far field: rows [row0, row0 + nrows) of the 'ij'
 * mesh x1 x z1.  tgt_density = grid points per unit area of the FULL grid, 1 / (dx dz) (not of the slab, so that slabs
 * reproduce the full-grid values bit for bit): cells holding more than (order+1)^2 grid points carry a local field even
 * where they hold few sources; 0 decides from the sources alone.  u, w: [nrows, nz] row-major. */
int ludvm_flowfield_velocity_tree(ludvm_ctx *ctx, const double *ga, const double *xa, const double *za, long na, double vc4,
                                  const double *x1, long nx, const double *z1, long nz, long row0, long nrows,
                                  double tgt_density, int order, int leaf, double *u, double *w, int ptr_kind, double *stats);

/*
 * Flow-field grid evaluation -- replaces the velocity part of LUDVM.flowfield (LUDVM.py:1193-1220) for one
 * snapshot: targets are the 'ij' mesh of x1[nx] x z1[nz] (np.arange values passed by the caller), rows
 * [row0, row0+nrows) of the x index.  Up to two source sets are summed the way the reference does
 * (u_wake + u_foil, LUDVM.py:1219); set B may be empty (nb = 0).  u, w: [nrows, nz] row-major.
 */
int ludvm_flowfield_velocity(ludvm_ctx *ctx, int mode, const double *ga, const double *xa, const double *za,
                             long na, const double *gb, const double *xb, const double *zb, long nb, double vc4,
                             const double *x1, long nx, const double *z1, long nz, long row0, long nrows,
                             double *u, double *w, int ptr_kind);
/* Velocity AND vorticity of one snapshot in one call (the body of LUDVM.flowfield's loop, LUDVM.py:1193-1292, for the
 * rows [row0, row0+nrows) of the grid, nrows >= 2): u, w, ome are [nrows, nz].  With host pointers the fields cross the
 * bus once.  The stencil is applied to the slab as given (one-sided at its first / last row). */
int ludvm_flowfield(ludvm_ctx *ctx, int mode, const double *ga, const double *xa, const double *za, long na,
                    const double *gb, const double *xb, const double *zb, long nb, double vc4, const double *x1, long nx,
                    const double *z1, long nz, long row0, long nrows, double *u, double *w, double *ome, int ptr_kind);
/* Vorticity stencil of LUDVM.py:1222-1292 (centred interior, one-sided edges/corners) on [ns, nx, nz] fields. */
int ludvm_flowfield_vorticity(ludvm_ctx *ctx, const double *x1, long nx, const double *z1, long nz,
                              const double *u, const double *w, long ns, double *ome, int ptr_kind);

/*
 * time_loop -- replaces LUDVM.time_loop (LUDVM.py:597-1171) with an on-device step replayed as a CUDA graph.
 * Every table is evaluated by the host exactly as the reference evaluates it with numpy (SURVEY.md A.4) and
 * uploaded once by ludvm_sim_create; vortex state stays resident in HBM across steps.
 */
typedef struct {
    int64_t nt;        /* len(self.t)                          LUDVM.py:254-255 */
    int64_t P;         /* Npoints - 1 panels / gamma points    LUDVM.py:345; at most 1024 (LUDVM_E_UNSUPPORTED above) */
    int64_t Nc;        /* Ncoeffs                              LUDVM.py:245     */
    int64_t nfree;     /* n_freevort >= 1                      LUDVM.py:268-277 */
    int32_t method;    /* LUDVM_METHOD_*                       LUDVM.py:252     */
    int32_t mode;      /* LUDVM_EXACT_F64 | LUDVM_FAST_F64 */
    int32_t store_history; /* 0: only the current positions exist; 1: keep path['TEV'/'LEV'/'FREE'] [nt,2,*] on the
                              device (LUDVM.py:615-617); k > 1: strided snapshots -- rows of steps i % k == 0 of
                              path['TEV'/'LEV'] ([(nt-1)/k + 1, 2, nt-1]; path['FREE'] stays [nt,2,nfree]) */
    int32_t steps_per_graph; /* K unrolled steps per captured graph; <= 0: library default */
    double dt, Uinf, chord, rho, piv, lespcrit;
    double vc4;        /* v_core**4                            LUDVM.py:260, :565 */
    double ic;         /* circulation['IC']                    LUDVM.py:649 */
    double sum_free;   /* np.sum(circulation['FREE'])          LUDVM.py:759 */
    double a0_init, a1_init; /* fourier[0,0,:2]                LUDVM.py:645-647 */
    double maxerror, epsilon; /* Newton constants              LUDVM.py:248-250 */
    int64_t maxiter;
} ludvm_sim_params;

typedef struct {
    const double *cos_a, *sin_a, *alpha_dot, *h_dot; /* [nt]: np.cos(alpha), np.sin(alpha), LUDVM.py:578-580 */
    const double *gp;          /* path['airfoil_gamma_points'] [nt,2,P]   LUDVM.py:447-448 */
    const double *le, *te;     /* path['airfoil'][:,:,0], [:,:,-1]  [nt,2] LUDVM.py:674-681, :790-800 */
    const double *detadx_p, *eta_p, *x_p, *theta_p; /* airfoil[...] panel tables [P] LUDVM.py:345-347 */
    const double *dtheta;      /* theta[1:] - theta[:-1]  [P]             LUDVM.py:995 */
    const double *cos_tp, *sin_tp; /* np.cos/np.sin(theta_panel) [P]      LUDVM.py:756, :1002 */
    const double *cosn, *sinn; /* np.cos(n*theta_panel), np.sin(n*theta_panel) [Nc,P] LUDVM.py:771, :1000;
                                  row 0 of cosn is cos(0) = 1.0 exactly and is used as the unit weight of A0 */
    const double *free_g;      /* circulation_freevort [nfree]            LUDVM.py:622 */
    const double *free_xz;     /* xy_freevort [2,nfree]                   LUDVM.py:618 */
} ludvm_sim_tables;            /* host pointers */

int ludvm_sim_create(ludvm_ctx *ctx, const ludvm_sim_params *p, const ludvm_sim_tables *t, ludvm_sim **out);
/* Advance `nsteps` time steps (clamped to the nt-1 total).  Asynchronous on the context's stream. */
int ludvm_sim_run(ludvm_sim *sim, long nsteps);
/* Steps completed so far (synchronises). */
int ludvm_sim_steps_done(ludvm_sim *sim, long *out);
/* Diagnostic twin of ludvm_sim_run (either method): advances `nsteps` steps launching the step's kernels one by one
 * with CUDA events around each.  ms_out[0..3] = summed milliseconds of wake-on-foil, solve, convection partials,
 * finish; ms_out[4] = their total.  Synchronises. */
int ludvm_sim_profile_steps(ludvm_sim *sim, long nsteps, double *ms_out);
/* Opt in to the chordwise pressure jump LUDVM_F_DP, which the reference allocates but never fills (LUDVM.py:1059-1064).
 * For step i >= 1 and gamma point j, with itev = i - 1:
 *   dp[i,j] = rho ((Uinf cos a_i + hdot_i sin a_i + u_j) gamma_airfoil[itev,j] + (Gamma_airfoil[itev,j] - Gamma_airfoil[itev-1,j]) / dt)
 * u_j = the tangential wake velocity at gamma point j that the loads integrate (LUDVM.py:1049-1057), Gamma_airfoil[-1] = 0;
 * row 0 and the rows of steps not yet run are zero.  Allocates and zeroes [nt,P] doubles.  Valid only before the first step
 * is run (LUDVM_E_STATE after); a second call does nothing. */
int ludvm_sim_enable_pressure(ludvm_sim *sim);
/* Opt in to the far-field convection (fast mode): every step whose wake bound 2 min(i, nt-1) + 2 + nfree (i = the step's
 * number, from 1) reaches the library's all-pairs / far-field crossover (SIM_FAR_FIELD_MIN_WAKE in sim.cu, DESIGN.md 4b)
 * convects the old wake TEV[:itev] ++ LEV[:ilev] ++ FREE through the treecode of ludvm_induced_velocity_tree at this
 * `order` (2..24; 18 matches the all-pairs fast kernel to ~1e-15 of sum|terms|) instead of all pairs.  Earlier steps are
 * unchanged.  The result is not bit-equal to the all-pairs run, but it is bitwise reproducible run to run and independent
 * of steps_per_graph and of how ludvm_sim_run is called.  A far-field step is not captured in a graph: ludvm_sim_run
 * enqueues it from the host and waits for the device within it (the step's vortex counts, then the tree's bounding box and
 * largest leaf), so ludvm_sim_run returns once the last far-field step's tree is enqueued.  A step whose cloud the tree
 * refuses (a leaf of the deepest tree would hold more than 65 536 vortices) runs the all-pairs kernels instead.
 * Valid only before the first step (LUDVM_E_STATE after); LUDVM_E_UNSUPPORTED in exact mode, for method Ramesh and for
 * P > 256; LUDVM_E_ARG for an order outside 2..24.  Allocates 3 (2 (nt-1) + nfree) doubles.
 * ludvm_sim_profile_steps returns LUDVM_E_UNSUPPORTED once it is enabled. */
int ludvm_sim_enable_far_field(ludvm_sim *sim, int order);
/* out[0] = steps convected through the far field so far, out[1] = qualifying steps that fell back to all pairs,
 * out[2] = the order (0: not enabled), out[3] = leaf level of the last tree (0: none yet).  Does not synchronise. */
int ludvm_sim_far_field_info(ludvm_sim *sim, int64_t out[4]);

enum {
    LUDVM_F_PATH_TEV = 0,  /* [(nt-1)/k+1,2,nt-1]  needs store_history = k >= 1  LUDVM.py:615 */
    LUDVM_F_PATH_LEV = 1,  /* [(nt-1)/k+1,2,nt-1]                                LUDVM.py:616 */
    LUDVM_F_PATH_FREE = 2, /* [nt,2,nfree]                      LUDVM.py:617 */
    LUDVM_F_G_TEV = 3,     /* [nt-1]                            LUDVM.py:620 */
    LUDVM_F_G_LEV = 4,     /* [nt-1]                            LUDVM.py:621 */
    LUDVM_F_G_BOUND = 5,   /* [nt-1]                            LUDVM.py:623 */
    LUDVM_F_G_AIRFOIL = 6, /* [nt-1,P]  dGamma                  LUDVM.py:624 */
    LUDVM_F_GAMMA_AIRFOIL = 7, /* [nt-1,P]                      LUDVM.py:626 */
    LUDVM_F_GAMMA_INT_AIRFOIL = 8, /* [nt-1,P] 'Gamma_airfoil'  LUDVM.py:627 */
    LUDVM_F_FOURIER = 9,   /* [nt,2,Nc]                         LUDVM.py:639 */
    LUDVM_F_LESP = 10,     /* [nt]                              LUDVM.py:640 */
    LUDVM_F_LESP_PREV = 11,/* [nt]                              LUDVM.py:641 */
    LUDVM_F_LEV_SHED = 12, /* [nt] float, -1 = none             LUDVM.py:654 */
    LUDVM_F_FN = 13, LUDVM_F_FS = 14, LUDVM_F_L = 15, LUDVM_F_D = 16, LUDVM_F_T = 17, LUDVM_F_M = 18, /* [nt] */
    LUDVM_F_CUR_TEV = 19,  /* current TEV positions [2,nt-1] (latest row of path['TEV']) */
    LUDVM_F_CUR_LEV = 20,  /* current LEV positions [2,nt-1] */
    LUDVM_F_CUR_FREE = 21, /* current FREE positions [2,nfree] */
    LUDVM_F_COUNTERS = 22, /* int64[4]: steps done, itev, ilev (next free slots), error flags */
    LUDVM_F_RANGE_BAD = 23, /* int32[1], exact mode: 0 = every coordinate seen so far lay inside the window in which the
                               pair arithmetic needs no per-pair range words (the flag-free instantiation ran), 1 = the
                               flagged instantiation took over (sticky) */
    LUDVM_F_DP = 24,       /* [nt,P] pressure jump; LUDVM_E_STATE unless ludvm_sim_enable_pressure was called */
    LUDVM_F__COUNT = 25
};
/* Copy a result field to a host buffer of `bytes` bytes (must equal the field's size).  Synchronises. */
int ludvm_sim_fetch(ludvm_sim *sim, int field, void *dst, size_t bytes);
/* The same for `nfields` fields at once: all copies are enqueued, then one synchronisation. */
int ludvm_sim_fetch_many(ludvm_sim *sim, int nfields, const int *fields, void *const *dsts, const size_t *bytes);
int ludvm_sim_field_bytes(ludvm_sim *sim, int field, size_t *out);
int ludvm_sim_destroy(ludvm_sim *sim);

/*
 * Batched parameter sweep (BASELINE.json configs[3]: e.g. 4096 cases LESPcrit x reduced frequency): `ncases`
 * independent time loops, one persistent CTA per case, all steps in one launch, no collective.  All cases must
 * share nt, P, Nc, nfree and method; table sets shared by several cases (identical host pointers) are uploaded once.
 * out is a host buffer [ncases][LUDVM_SWEEP_FIELDS][nt] (out_doubles_per_case = LUDVM_SWEEP_FIELDS * nt) with rows
 * Fn, Fs, L, D, T, M, LESP, LESP_prev, LEV_shed, circulation TEV, LEV, bound (the last three hold nt-1 values).
 * To split a sweep over GPUs call it once per device with that device's slice of the cases.
 */
#define LUDVM_SWEEP_FIELDS 12
enum { LUDVM_SW_FN = 0, LUDVM_SW_FS, LUDVM_SW_L, LUDVM_SW_D, LUDVM_SW_T, LUDVM_SW_M, LUDVM_SW_LESP,
       LUDVM_SW_LESP_PREV, LUDVM_SW_LEV_SHED, LUDVM_SW_G_TEV, LUDVM_SW_G_LEV, LUDVM_SW_G_BOUND };
int ludvm_sweep_run(ludvm_ctx *ctx, long ncases, const ludvm_sim_params *params, const ludvm_sim_tables *tables,
                    double *out, size_t out_doubles_per_case);
/* ludvm_sweep_run plus the pressure jump of ludvm_sim_enable_pressure for every case: dp is a host buffer
 * [ncases][nt][P] (dp_doubles_per_case = nt * P), row 0 of each case zero.  Same arguments and checks otherwise.
 * The call allocates ncases * nt * P doubles of device memory for it (LUDVM_E_NOMEM if that fails). */
int ludvm_sweep_run_pressure(ludvm_ctx *ctx, long ncases, const ludvm_sim_params *params, const ludvm_sim_tables *tables,
                             double *out, size_t out_doubles_per_case, double *dp, size_t dp_doubles_per_case);

/*
 * Roofline denominator: sustained FP64 FMA issue rate of this GPU, measured with a register-resident DFMA
 * chain kernel (MEASURED_PEAKS.json has no FP64 entry).  Returns DFMA/s (x2 = FLOP/s) over `ms_target` ms.
 */
int ludvm_measure_fp64_fma_rate(ludvm_ctx *ctx, double ms_target, double *dfma_per_s);
int ludvm_measure_fp32_fma_rate(ludvm_ctx *ctx, double ms_target, double *ffma_per_s);

#ifdef __cplusplus
}
#endif
#endif /* LUDVM_B200_H */
