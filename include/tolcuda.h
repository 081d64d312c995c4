/* libtolcuda -- B200 (sm_100a) evaluator for tol's SNOPT user function (F and sparse G).
 *
 * C ABI: plain pointers and sizes only.  Every entry point names the reference interface it
 * replaces (file:line into lingaqing/tol).  All functions return 0 on success, a positive
 * cudaError_t value on a CUDA failure, or a negative TOLCUDA_E* code; none throws across the ABI.
 * tolcuda_last_error() returns a human-readable message for the calling thread's last failure.
 *
 * There is NO CPU fallback: every evaluation runs the sm_100a kernels in fg_kernels.cu.
 *
 * Threading: a handle owns its streams and staging buffers and is NOT re-entrant -- one call at a time per
 * handle (the reference callback is single-threaded too: process-global `prob`, src/tol.cpp:3).  Different
 * handles, e.g. one per device, may be used from different threads concurrently (tolbatch does).  The
 * context-free queries (tolcuda_problem_*, tolcuda_compact_len, tolcuda_expand_compact_g, tolcuda_write_results_*,
 * tolcuda_read_params) are thread-safe. */
#ifndef TOLCUDA_H_
#define TOLCUDA_H_

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

/* formulations: reference src/tol.cpp:5-36 (mission_select) */
#define TOLCUDA_G7 7   /* guidance, reference src/problemG7.cpp */
#define TOLCUDA_S10 10 /* loiter,   reference src/problemS10.cpp */

/* wind models: reference src/problem.cpp:475-531 (modelWind cases 0 and 1; case 1 is what the
 * reference runs whenever its MongoDB wind server is unreachable, src/problem.cpp:63-78) */
#define TOLCUDA_WIND_NONE 0
#define TOLCUDA_WIND_LINEAR_LAYER 1
#define TOLCUDA_WIND_CUBE 3 /* modelWind case 3 (src/problem.cpp:544-695); set with tolcuda_set_wind_grid */

/* error codes (negative; positive values are cudaError_t) */
#define TOLCUDA_EINVAL (-1)      /* bad argument                                         */
#define TOLCUDA_EUNSUPPORTED (-2) /* formulation / wind model / ts outside what is built */
#define TOLCUDA_ENOCTX (-3)      /* DEFINEGusrfg_ called with no bound context            */
#define TOLCUDA_EIO (-4)         /* .param file missing or malformed                      */
#define TOLCUDA_ENOMEM (-5)

/* flags for tolcuda_eval_batch */
#define TOLCUDA_NEED_F 0x1
#define TOLCUDA_NEED_G 0x2
#define TOLCUDA_HOST_PTRS 0x10   /* x/F/G are host memory (staged through pinned buffers)  */
#define TOLCUDA_DEVICE_PTRS 0x20 /* x/F/G are device memory on the context's device        */
/* neither pointer flag: detected with cudaPointerGetAttributes on x */
#define TOLCUDA_NO_SYNC 0x40 /* device pointers only: return after enqueueing on the context's
                                stream instead of synchronising it                         */
#define TOLCUDA_COMPACT_G 0x80 /* G receives COMPACT rows (tolcuda_compact_len doubles each, see
                                  tolcuda_expand_compact_g) instead of rows in coordinate order */
#define TOLCUDA_FULL_G_COPY 0x100 /* host pointers only: copy full G rows across PCIe instead of
                                     compact rows expanded by host threads (see tolcuda_eval_batch) */

/* Device pointers + TOLCUDA_NO_SYNC only: this launch may START while the kernel enqueued immediately before it on
 * the stream is still finishing (programmatic dependent launch): its CTAs move into the SMs the previous grid's
 * tail has left.  The caller guarantees that x was not written by that preceding kernel (x is read early).
 *   TOLCUDA_OVERLAP           the kernel waits for the preceding kernel to complete before its first store, so
 *                             F/G/summary may alias whatever that kernel read or wrote (e.g. the same F/G again)
 *   TOLCUDA_OVERLAP_DISJOINT  no wait at all: the caller also guarantees that F/G/summary overlap nothing the
 *                             preceding kernel reads or writes (e.g. consecutive chunks of a batch, or two sets
 *                             of result buffers used alternately)
 * What the hardware orders: a dependent grid may begin once every CTA of its predecessor has STARTED; nothing more.
 * Launch i+2 can therefore only begin after every CTA of launch i+1 has started, i.e. after launch i+1 has worked
 * off all but its last wave -- with two buffer sets used alternately, launch i+2 meets launch i only if a single CTA
 * of launch i outlives (almost) all of launch i+1, which cannot happen once a launch is many CTA lifetimes long (a
 * CTA lives ~10-20 us; from a few thousand trajectories per launch on).  A caller that needs the ordering
 * unconditionally uses TOLCUDA_OVERLAP, or plain launches. */
#define TOLCUDA_OVERLAP 0x200
#define TOLCUDA_OVERLAP_DISJOINT 0x400
#define TOLCUDA_FLAGS_ALL 0x7f3 /* every bit defined above; others are rejected with TOLCUDA_EINVAL */

typedef struct tolcuda_ctx *tolcuda_handle;

/* What reference `problem::problem(arguments&)` gathers before the first callback
 * (src/problem.cpp:13-60, src/parameters.cpp:42-148):
 *   aircraft[15] = mm,b,SS,ee,AR,Cd0,CLmin,CLmax,phimax,Vamin,Vamax,gammamax,phidotmax,Tmin,Tmax
 *                  (file order, angles already in radians); the path uses mm,SS,ee,AR,Cd0
 *   gains[5]     = kT,kp,kv,ka,kdt
 *   goal[4]      = xg,yg,zg,rg in NED (xg = north_goal, yg = east_goal, zg = -up_goal;
 *                  src/problem.cpp:24-27)
 *   numbounds is implied by the formulation (12 for G7, 11 for S10; problems/<M>/snopt.param). */
typedef struct tolcuda_config {
    int formulation; /* TOLCUDA_G7 | TOLCUDA_S10 */
    int ts;          /* time segments ("N nodes"), >= 1 */
    int wind_model;  /* TOLCUDA_WIND_* */
    int device;      /* CUDA device ordinal */
    double aircraft[15];
    double gains[5];
    double goal[4];
    /* used only by the set-up queries below (not by F/G):
     *   limits[8]   = dtmin,dtmax,xmin,xmax,ymin,ymax,zmin,zmax (limits.param file order)
     *   solver_tol[2] = SNOPT major optimality / feasibility tolerance (snopt.param lines 6, 7) */
    double limits[8];
    double solver_tol[2];
} tolcuda_config;

/* Replaces the problemG7 / problemS10 construction in reference src/tol.cpp:5-36 for the
 * evaluation path: builds the sparsity pattern once (closed form of countG, src/problem.cpp:813-919),
 * builds the kernels' constants (handed to every launch as a __grid_constant__ parameter: constant bank, immediate
 * operands), creates the stream and pinned staging buffers. */
int tolcuda_create(const tolcuda_config *cfg, tolcuda_handle *out);

/* Same, reading the reference's own files: <root>aircraft/<aircraft>.param,
 * <root>problems/<mission>/{gains,snopt}.param (reference src/parameters.cpp:42-148; root must end
 * in '/').  east/north/up and the goal are the reference CLI's positional arguments
 * (src/arguments.cpp:32-46).  ts_override > 0 replaces the ts of snopt.param. */
int tolcuda_create_from_files(const char *root, const char *aircraft, const char *mission,
                              double east, double north, double up, double east_goal,
                              double north_goal, double up_goal, double radius_goal,
                              int ts_override, int device, tolcuda_handle *out);
/* The first half of tolcuda_create_from_files on its own (host only, no CUDA): the reference's files and command
 * line as a tolcuda_config -- what the reference's `aircraft`, `gain`, `limit`, `snopt` constructors and
 * problem::problem hold afterwards (src/parameters.cpp:42-148, src/problem.cpp:13-60: ENU -> NED goal, degrees ->
 * radians); wind model 1, the one the reference falls back to (src/problem.cpp:77). */
int tolcuda_config_from_files(const char *root, const char *aircraft, const char *mission,
                              double east, double north, double up, double east_goal,
                              double north_goal, double up_goal, double radius_goal,
                              int ts_override, int device, tolcuda_config *out);

/* Wind model 3 of the reference: the wind cube that reference cacheWind pulls from its MongoDB server
 * (src/problem.cpp:371-460: cache[i][j][k], i < ne, j < nn, k < nu) is handed over by the caller and kept in
 * device memory; the F/G kernels then interpolate it per node exactly as modelWind case 3 does
 * (src/problem.cpp:544-695: trilinear shape functions of the v component and of its gradient; u, w stay 0).
 *   gx[ne], gy[nn], gz[nu]  grid coordinates = cache[i][0][0].x, cache[0][j][0].y, cache[0][0][k].z (ENU, m)
 *   v[ne*nn*nu]             cache[i][j][k].v, i-major
 *   datum[3]                EastFromDatum, NorthFromDatum, UpFromDatum (src/problem.cpp:406-413)
 *   spacing[3]              xspacing, yspacing, zspacing (include/problem.h:87-89: 150 m each)
 * Switches the context to TOLCUDA_WIND_CUBE.  Nodes outside the cube use the nearest cell (the reference
 * indexes out of bounds there). */
int tolcuda_set_wind_grid(tolcuda_handle h, int ne, int nn, int nu, const double *gx, const double *gy,
                          const double *gz, const double *v, const double *datum, const double *spacing);

int tolcuda_destroy(tolcuda_handle h);

/* n, neF, neG as reference src/problem.cpp:151-152 and countG's final neG */
int tolcuda_dims(tolcuda_handle h, int *n, int *neF, int *neG);

/* iGfun/jGvar exactly as reference countG leaves them for snoptProblemA::setG
 * (src/problem.cpp:870-871, :1230): 0-based, sorted by row then column, neG entries each. */
int tolcuda_pattern(tolcuda_handle h, int *iGfun, int *jGvar);

/* The same two queries without a context (and without touching CUDA), for a driver that must size
 * and fill SNOPT's arrays before any device exists: closed form of reference countG
 * (src/problem.cpp:813-919) -- neG = 105*ts+48 (G7), 107*ts+37 (S10). */
int tolcuda_problem_dims(int formulation, int ts, int *n, int *neF, int *neG);
int tolcuda_problem_pattern(int formulation, int ts, int *iGfun, int *jGvar);

/* Set-up parity (host only, no CUDA): what the reference constructor leaves in SNOPT's arrays before
 * runSNOPT -- bit-identical to the reference's.
 *   initial guess  problemG7::InitialCond src/problemG7.cpp:19-217, problemS10::InitialCond
 *                  src/problemS10.cpp:19-219          -> x0[n]
 *   bounds         problem::setLimits src/problem.cpp:198-365 -> xlow,xupp[n], Flow,Fupp[neF]
 *                  (xstate, xmul, Fmul, Fstate are all zero there)
 *   solver options problem::runSNOPT src/problem.cpp:1223-1238: Derivative option 1, Iterations
 *                  limit 60000, tolerances from snopt.param, cold start, ObjRow 0, ObjAdd 0 */
int tolcuda_problem_initial_guess(const tolcuda_config *cfg, double *x0);
int tolcuda_problem_bounds(const tolcuda_config *cfg, double *xlow, double *xupp, double *Flow,
                           double *Fupp);
/* Result files of a finished solve (host only, no CUDA), byte for byte what the reference writes:
 *   JSON  problem::writeJSON src/problem.cpp:1247-1365 -- "snopt_results.json" (src/tol.cpp:30), the file the
 *         mission layer reads back (msl/mission.py:204-240): args, problem, FinalCost, dt, trajectory
 *         {time,x,y,z,Va,gam,chi,phi,CL,dphi,dCL,T}, aircraft, gains, limits, snopt; jsoncpp StyledWriter layout
 *   TXT   problem::writeTXT src/problem.cpp:1371-1418 (the reference ignores its file-name argument and always
 *         writes "snopt_output.txt"; here `path` is honoured)
 * aircraft/mission: the names given on the reference command line; east,north,up: its first three arguments;
 * x[n]: decision vector; final_cost: F[0].  cfg->limits and cfg->solver_tol must be filled (they are after
 * tolcuda_create_from_files + tolcuda_get_config). */
int tolcuda_write_results_json(const tolcuda_config *cfg, const char *aircraft, const char *mission, double east,
                               double north, double up, const double *x, double final_cost, const char *path);
int tolcuda_write_results_txt(const tolcuda_config *cfg, const double *x, double final_cost, const char *path);

/* The reference callback's per-call dump files (src/DefineFG.cpp:16-46, src/problem.cpp:740-756): on EVERY call the
 * reference rewrites, in its working directory, Xoutput.txt (x, before anything is evaluated), Woutput.txt (the 12
 * wind arrays per node, "%.6f "), Foutput.txt and Goutput.txt (one "%.14f" value per line) -- the live plotter
 * matlab/@plotSNOPT/plotSNOPT.m:108-125 polls Xoutput.txt to draw the iterates while SNOPT runs.  They are 88 % of
 * the reference's call time, so they are OFF by default here.  tolcuda_set_dump_dir(h, dir) (or TOLCUDA_DUMP_DIR in
 * the environment when the context is created) makes DEFINEGusrfg_ -- and only it, as in the reference -- write the
 * same files, byte for byte the reference's format, into `dir` ("." = where the reference puts them); NULL or ""
 * switches them off again.  Woutput.txt is written for wind models 0 and 1.  A file that cannot be written is
 * reported once on stderr and does not stop the solve.
 * tolcuda_write_dump / tolcuda_write_wind_dump are the two writers on their own (host only, no CUDA): `count` values
 * as "%.14f" lines; the wind arrays of modelWind case `wind_model` (0 or 1) along the trajectory x[1 + 11*(ts+1)]. */
int tolcuda_set_dump_dir(tolcuda_handle h, const char *dir);
int tolcuda_write_dump(const char *path, const double *values, long count);
int tolcuda_write_wind_dump(const char *path, int wind_model, int ts, const double *x);
/* the configuration a handle was created with (e.g. after tolcuda_create_from_files) */
int tolcuda_get_config(tolcuda_handle h, tolcuda_config *cfg);

/* One trajectory, host pointers: what reference DEFINEGusrfg_ computes (src/DefineFG.cpp:24-38)
 * without the debug dumps.  Writes F[0..neF) if needF > 0 and G[0..neG) if needG > 0. */
int tolcuda_eval(tolcuda_handle h, const double *x, int needF, double *F, int needG, double *G);

/* B independent trajectories in one launch, trajectory-major: trajectory b reads x + b*ldx
 * (n doubles) and writes F + b*ldF (neF doubles) and G + b*ldG (neG doubles, coordinate order of
 * tolcuda_pattern).  Leading dimensions are in doubles; padding them to a multiple of 16 keeps
 * every trajectory 128-byte aligned (tolcuda_padded_ld).  flags: TOLCUDA_NEED_* | pointer kind. */
/* Host pointers: chunks of trajectories are pipelined H2D(x) -> kernel -> D2H(F, G) over three streams.
 * 71 of the 104 G values of a collocation window are structural constants (the zeros and +-1 of reference
 * tabG, src/problem.cpp:1038,1084,1098,1112,1170,1182,1204) and two equal -dt, so by default only the
 * x-dependent values cross PCIe (compact rows) and a pool of host threads places them in the caller's G
 * and writes the constants as literals; the rows the caller sees are bit for bit those of the
 * device-pointer path.  TOLCUDA_FULL_G_COPY (or tolcuda_set_option(h, "compact_host", 0)) copies full rows instead. */
int tolcuda_eval_batch(tolcuda_handle h, int B, const double *x, long ldx, double *F, long ldF,
                       double *G, long ldG, int flags);

/* Compact G rows, for callers that move G themselves (e.g. gather it from several GPUs):
 *   [0, R0)                    objective-row block as in G (R0 = 3*ts+4 for S10, ts+6 for G7)
 *   [R0 + 31*k, R0 + 31*k+31)  the 31 x-dependent values of window k in coordinate order
 *   [R0 + 31*ts, + nbG)        boundary block as in G (nbG = 33 for S10, 42 for G7)
 *   [R0 + 31*ts + nbG]         -dt (value of the d/d(dphi) and d/d(dCL) entries of rows F7, F8)
 * tolcuda_compact_len returns the row length (or a negative TOLCUDA_E* code); tolcuda_eval_batch with
 * TOLCUDA_COMPACT_G writes such rows (ldG >= that length); tolcuda_expand_compact_g turns B of them into
 * rows in the coordinate order of tolcuda_pattern on `threads` host threads (0 = all cores available to
 * the process).  Host memory only, no CUDA call; no arithmetic on the values. */
long tolcuda_compact_len(int formulation, int ts);
int tolcuda_expand_compact_g(int formulation, int ts, long B, const double *Gc, long ldGc, double *G, long ldG,
                             int threads);
/* The same expansion on the device (expand_kernel.cu): B compact rows in device memory -> rows in coordinate
 * order in device memory, on the context's stream; bit-identical to what tolcuda_eval_batch writes without
 * TOLCUDA_COMPACT_G.  flags: 0 or TOLCUDA_NO_SYNC.  For results kept or gathered in compact form on the GPU. */
int tolcuda_expand_compact_g_device(tolcuda_handle h, long B, const double *Gc, long ldGc, double *G, long ldG,
                                    int flags);
/* Column-compressed (CSC) view of G for a device-side QP / factorisation (SURVEY.md 8f-4; nothing of the kind in
 * the reference, where SNOPT alone consumes G): colptr[n+1], rowidx[neG] (rows ascending within a column) and,
 * optionally, perm[neG] = coordinate-order position of CSC entry p.  Host only.
 * tolcuda_repack_csc_device gathers B rows of device memory from coordinate order into that order:
 * Gcsc[b*ldC + p] = G[b*ldG + perm[p]], on the context's stream (flags: 0 or TOLCUDA_NO_SYNC). */
int tolcuda_problem_pattern_csc(int formulation, int ts, int *colptr, int *rowidx, int *perm);
int tolcuda_repack_csc_device(tolcuda_handle h, long B, const double *G, long ldG, double *Gcsc, long ldC, int flags);
/* Matrix-free products with the Jacobian (a device-side consumer of G for an iterative QP / SQP step on the GPU;
 * SURVEY.md 8f-4, nothing of the kind in the reference): J(x_b) is the neF x n matrix whose coordinate entries
 * (tolcuda_pattern) are the G values tolcuda_eval_batch writes for x_b.  The kernels evaluate every window's
 * entries exactly as for G and consume them in registers -- G is never written, so a product moves
 * 8*(2n + neF) bytes per trajectory instead of 8*(n + neF + neG).
 *   tolcuda_jac_vec    y[b*ldy + i] = sum_j J_ij d[b*ldd + j]        d: n per row,   y: neF per row
 *   tolcuda_jac_tvec   z[b*ldz + j] = sum_i J_ij lambda[b*ldl + i]   lambda: neF,    z: n
 * Device pointers on the context's device; flags: 0 or TOLCUDA_NO_SYNC.  Sums run in ascending column (row)
 * order within a window, separately rounded products (no FMA contraction); they agree with products formed from
 * the G rows to rounding of the sums (tests/test_gpu_parity.py::test_matrix_free_jacobian_products). */
int tolcuda_jac_vec(tolcuda_handle h, int B, const double *x, long ldx, const double *d, long ldd, double *y, long ldy,
                    int flags);
int tolcuda_jac_tvec(tolcuda_handle h, int B, const double *x, long ldx, const double *lambda, long ldl, double *z,
                     long ldz, int flags);
/* Hessian of the Lagrangian times a vector (a truncated-Newton / trust-region CG step or an exact-Hessian SQP step on
 * the GPU), with J as above:
 *   w_b = D_x[ J(x_b)^T lambda_b ] d_b,   w[b*ldw + j] = sum_i lambda_i sum_l (dJ_ij / dx_l) d_l
 * x: n per row, lambda: neF (lambda[0] weights the objective row, IPOPT's sigma), d: n, w: n.  z, if not NULL,
 * receives J(x_b)^T lambda_b (n per row) bit for bit as tolcuda_jac_tvec writes it.  Where G is the gradient of F this
 * is the Hessian of lambda^T F times d.  G7's objective row is the gradient of 1/2 kT sum T^2 + kp ts dt / dist (kp
 * where F[0] uses kv, as in the reference), its boundary row 11 that of dist alone (the reference leaves out the
 * node-0 derivative of dmax); w differentiates those rows.  S10's boundary-row dt entries are the constant 0.  G holds
 * the wind and its gradient fixed while its entries depend on them, and w differentiates the entries with the wind
 * included: the operator is symmetric under wind model 0, not under models 1 and 3 (DESIGN.md 5).  The kernels evaluate every window's Jacobian entries in forward-mode dual arithmetic and
 * consume them in registers, moving 8*(3n + neF) bytes per trajectory (+ 8n with z).
 * Device pointers on the context's device; flags: 0 or TOLCUDA_NO_SYNC (TOLCUDA_HOST_PTRS: TOLCUDA_EUNSUPPORTED).  A
 * null x, lambda, d or w, or a leading dimension shorter than its row, is TOLCUDA_EINVAL; B = 0 launches nothing.
 * Evaluated with the context's goal (tolcuda_lag_hess_vec_goals: one per trajectory); the options "kernel", "per",
 * "lwarps" and "per_min_waves" apply as to tolcuda_jac_tvec, and every option gives the same bits except w[0] and z[0] (sums over the trajectory) under
 * kernel L. */
int tolcuda_lag_hess_vec(tolcuda_handle h, int B, const double *x, long ldx, const double *lambda, long ldl,
                         const double *d, long ldd, double *w, long ldw, double *z, long ldz, int flags);
/* host threads the host-pointer batch path of this context expands compact rows with (0 = default:
 * environment TOLCUDA_HOST_THREADS, else the cores available to the process / LOCAL_WORLD_SIZE) */
int tolcuda_set_host_threads(tolcuda_handle h, int threads);

/* Execution-strategy options of a context.  They choose between equivalent ways of running the same arithmetic:
 * every value of every option yields the same bits in F and G (tested), with one exception -- the tile-loop kernel
 * ("kernel" = 2, always used for ts > 256) adds the terms of the objective per lane over a warp's tiles first, so
 * F[0], and only F[0], can differ from the default kernel's in the last bits (and with "lwarps"):
 *   "kernel"         0 (default): one CTA per run of trajectories for ts <= 256, the tile-loop kernel beyond;
 *                    2: the tile-loop kernel for any ts
 *   "per"            trajectories per CTA, 1..4; 0 (default) = 2 for large batches, 1 below "per_min_waves" waves
 *   "per_min_waves"  waves of single-trajectory CTAs; -1 (default) = 24, 8 for TOLCUDA_OVERLAP_DISJOINT launches
 *   "tail_x4"        quarter-waves of single-trajectory CTAs a grid of runs ends on; -1 (default) = 2, and 0 for
 *                    TOLCUDA_OVERLAP_DISJOINT launches (the next grid fills the tail)
 *   "lwarps"         warps per CTA of the tile-loop kernel, 1..8; 0 (default) = the count that balances the tiles
 *   "zero_copy"      1 (default): the single-trajectory path lets the kernel read x / write F, G in mapped pinned
 *                    host memory; 0: staged cudaMemcpyAsync copies
 *   "compact_host"   1 (default): the host-pointer batch path moves compact G rows across PCIe and expands them on
 *                    host threads; 0: full rows cross PCIe (as with TOLCUDA_FULL_G_COPY)
 *   "full_rows_pct"  host-pointer batch path with compact_host = 1: this share of the chunks (0..100, default 0) crosses
 *                    PCIe as full rows straight into the caller's G while the others go as compact rows and are
 *                    expanded by the host threads -- the copy engines and the cores work side by side; the best share
 *                    depends on the host (bench.py and tolbatch --host-path auto calibrate it)
 *   "chunk_mb"       host-pointer batch path: upper limit of the device megabytes per pipeline lane (default 32;
 *                    a call is cut into ~160 chunks of at least 1 MB, so smaller batches use smaller chunks)
 * Returns TOLCUDA_EINVAL for an unknown name or a value out of range. */
int tolcuda_set_option(tolcuda_handle h, const char *name, long value);

/* Same evaluation plus a per-trajectory summary computed inside the kernel from values it already holds
 * (a device-side consumer of F; nothing of the kind exists in the reference, where SNOPT alone reads F):
 *   summary[b*lds + 0] = F[0]                      objective
 *   summary[b*lds + 1] = max |defect|              over the 8*ts dynamics rows
 *   summary[b*lds + 2] = max boundary violation    |row| for equality rows, max(row, 0) for G7's dist <= dmax
 *   summary[b*lds + 3] = sum of defect^2
 * Non-finite rows: the maxima are NaN when any of their rows is NaN (a NaN defect or boundary row is not hidden by
 * finite ones), +inf when a row is +-inf and none is NaN; the sum is NaN or +inf likewise.  Each entry is what
 * numpy's max / sum give on the F this call writes, so screening on summary[b*lds + 1] < tol rejects a trajectory
 * whose defects are NaN.
 * lds >= 4; same pointer kind as x/F/G.  With neither TOLCUDA_NEED_F nor TOLCUDA_NEED_G only the summary
 * is produced (F and G may then be NULL). */
int tolcuda_eval_batch_summary(tolcuda_handle h, int B, const double *x, long ldx, double *F, long ldF,
                               double *G, long ldG, double *summary, long lds, int flags);

/* Per-trajectory goals: one launch for trajectories of different missions (goal = the reference CLI's Eg Ng Ug Rg,
 * src/arguments.cpp:32-46, which F and G depend on: S10's cost and objective row through r_k - rg, G7's boundary rows
 * through chi_d = atan2(yg, xg) and dmax = |(xg, yg) - p_0|).  Aircraft, gains, ts and wind model stay the context's.
 *   tolcuda_set_goals         keeps a goal table on the context's device: row b is goal[b*ldg + 0..3] = xg, yg, zg, rg
 *                             in NED, as tolcuda_config.goal (ldg >= 4; host memory).  chi_d is derived per row on the
 *                             host exactly as tolcuda_create derives it.  Synchronises the context's stream before it
 *                             replaces the previous table, so TOLCUDA_NO_SYNC launches in flight (evaluations and
 *                             products) finish with the table they were enqueued with.  count = 0 frees the table.
 *   tolcuda_eval_batch_goals  as tolcuda_eval_batch_summary (summary may be NULL; every flag and option of it applies),
 *                             but trajectory b of this call uses goal row row0 + b of the table.
 *   tolcuda_jac_vec_goals, tolcuda_jac_tvec_goals, tolcuda_lag_hess_vec_goals
 *                             as tolcuda_jac_vec, tolcuda_jac_tvec and tolcuda_lag_hess_vec (same arguments after B, same
 *                             validation, flags and options; one launch per call), but trajectory b of this call uses
 *                             goal row row0 + b of the table: the matrix-free products of a batch of different missions.
 * Row b of F, G and summary (of y, z, w and the optional z) is bit for bit what a context created with row0 + b's goal
 * (and the same options) writes for the same x (and d, lambda); under kernel L the caveat of tolcuda_lag_hess_vec on
 * w[0] and z[0] applies unchanged.  No table, row0 < 0 or row0 + B > count (and a NULL handle, checked before any
 * CUDA call) return TOLCUDA_EINVAL and launch nothing.  The table lives in device memory: 64 bytes per row. */
int tolcuda_set_goals(tolcuda_handle h, long count, const double *goal, long ldg);
int tolcuda_eval_batch_goals(tolcuda_handle h, long row0, int B, const double *x, long ldx, double *F, long ldF,
                             double *G, long ldG, double *summary, long lds, int flags);
int tolcuda_jac_vec_goals(tolcuda_handle h, long row0, int B, const double *x, long ldx, const double *d, long ldd,
                          double *y, long ldy, int flags);
int tolcuda_jac_tvec_goals(tolcuda_handle h, long row0, int B, const double *x, long ldx, const double *lambda, long ldl,
                           double *z, long ldz, int flags);
int tolcuda_lag_hess_vec_goals(tolcuda_handle h, long row0, int B, const double *x, long ldx, const double *lambda,
                               long ldl, const double *d, long ldd, double *w, long ldw, double *z, long ldz, int flags);

/* page-locked host memory for x/F/G of the host-pointer batch path (full PCIe speed, asynchronous
 * copies); plain wrappers so that a C/C++ driver needs no CUDA headers */
int tolcuda_host_alloc(size_t bytes, void **ptr);
int tolcuda_host_free(void *ptr);
int tolcuda_device_count(int *count);

/* Result buffers that OTHER GPUs of the box write directly (SURVEY.md 8f-4: "optional NVLink gather of results
 * to one GPU"; nothing of the kind in the reference).  The F/G kernels store through ordinary global
 * addresses (F: coalesced stores, G: TMA bulk copies), so F/G of tolcuda_eval_batch may point into the memory of
 * a peer GPU: the shard then lands in the gathering GPU's rows over NVLink while it is being computed -- one
 * kernel, no staging copy and no collective afterwards.
 *   one process per GPU   the gathering process allocates with tolcuda_device_alloc, exports the allocation with
 *                         tolcuda_ipc_export (a CUDA IPC handle: TOLCUDA_IPC_HANDLE_BYTES opaque bytes to send over
 *                         any channel); every other process maps it with tolcuda_ipc_open on ITS device (peer access
 *                         is enabled by the mapping) and passes `mapped + offset of its rows` as F/G with
 *                         TOLCUDA_DEVICE_PTRS; after its call has returned (synchronised) its rows are visible
 *                         to the owner; tolcuda_ipc_close unmaps.
 *   one process, several devices (tolbatch)   tolcuda_enable_peer(device, peer) once per ordered pair, then any
 *                         cudaMalloc / tolcuda_device_alloc pointer of `peer` is valid in kernels of `device`.
 * x always stays on the evaluating GPU. */
#define TOLCUDA_IPC_HANDLE_BYTES 64
int tolcuda_device_alloc(int device, size_t bytes, void **ptr);
int tolcuda_device_free(int device, void *ptr);
int tolcuda_ipc_export(int device, const void *ptr, unsigned char handle[TOLCUDA_IPC_HANDLE_BYTES]);
int tolcuda_ipc_open(int device, const unsigned char handle[TOLCUDA_IPC_HANDLE_BYTES], void **ptr);
int tolcuda_ipc_close(int device, void *ptr);
int tolcuda_enable_peer(int device, int peer);
/* Stream-ordered 32-bit flags in device memory -- the context's own device or a peer's mapping -- so that a consumer
 * on one GPU can start on a chunk as soon as the producer's kernel for that chunk has finished on another, with no
 * host in between:
 *   tolcuda_stream_signal  enqueues "*flag = value" on the context's stream, after everything enqueued before it
 *                          (the preceding kernels' stores, peer stores included, are visible before the flag is)
 *   tolcuda_stream_wait    enqueues "wait until (int)(*flag - value) >= 0" on the context's stream
 * flag: 4-byte aligned.  (cuStreamWriteValue32 / cuStreamWaitValue32 of the CUDA driver.) */
int tolcuda_stream_signal(tolcuda_handle h, void *flag, unsigned int value);
int tolcuda_stream_wait(tolcuda_handle h, const void *flag, unsigned int value);

/* Fused evaluate + gather: all B rows of F and G of a batch whose shards are evaluated on `world` GPUs, in the memory
 * of ONE of them (rank `dst`), written there by the shards' own kernels over NVLink while they compute -- no send
 * buffer, no collective.  The protocol of the primitives above in one place (gather.cpp), for a C/C++ driver with
 * several devices (tolbatch --gather-gpu) and for one process per GPU alike.  Rank q owns the contiguous block of
 * trajectory indices [q*ceil(B/world), ...) (SURVEY.md 8e).
 *   tolcuda_gather_create   the gathering rank: allocates the buffer on its context's device (F rows | G rows |
 *                           staging for the peers' compact rows | chunk flags); ipc_handle (may be NULL) receives the
 *                           TOLCUDA_IPC_HANDLE_BYTES bytes other PROCESSES need
 *   tolcuda_gather_attach   every other rank, on its own context: `owner` = the creating rank's gather handle when it
 *                           lives in the same process (peer access is enabled), else NULL and `ipc_handle` = the bytes
 *                           the owner exported
 *   tolcuda_gather_send     a peer evaluates its shard (x: its rows on its device) in `chunks` launches; F goes to its
 *                           final place, G as compact rows into the staging region, each chunk followed by a
 *                           stream-ordered flag in the owner's memory.  Asynchronous (tolcuda_synchronize to wait).
 *   tolcuda_gather_collect  the owner evaluates its own shard in place and expands every peer chunk into rows in
 *                           coordinate order as soon as its flag arrives (no host in between); returns, after
 *                           synchronising, the device pointers and leading dimensions of the B rows.
 * All ranks call send / collect once per evaluation, with the same `chunks` (1..16).  A peer must not start the NEXT
 * send before the owner's collect of this one has returned (in one process: program order; across processes: a
 * barrier).  The rows are bit for bit those of a single GPU evaluating the whole batch. */
typedef struct tolcuda_gather *tolcuda_gather_handle;
int tolcuda_gather_create(tolcuda_handle h, long B, int world, int dst, tolcuda_gather_handle *out,
                          unsigned char *ipc_handle);
int tolcuda_gather_attach(tolcuda_handle h, long B, int world, int rank, int dst, tolcuda_gather_handle owner,
                          const unsigned char *ipc_handle, tolcuda_gather_handle *out);
int tolcuda_gather_send(tolcuda_gather_handle g, const double *x, long ldx, int chunks);
int tolcuda_gather_collect(tolcuda_gather_handle g, const double *x, long ldx, int chunks, double **F, long *ldF,
                           double **G, long *ldG);
int tolcuda_gather_buffer(tolcuda_gather_handle g, void **base, size_t *bytes); /* the owner's buffer as mapped here */
int tolcuda_gather_close(tolcuda_gather_handle g);
/* synchronous copies between host memory and memory of `device` (plain wrappers, like tolcuda_host_alloc) */
int tolcuda_copy_to_device(int device, void *dst, const void *src, size_t bytes);
int tolcuda_copy_to_host(int device, void *dst, const void *src, size_t bytes);

/* smallest multiple of 16 doubles (128 bytes) that holds `len` doubles */
long tolcuda_padded_ld(long len);

/* run the context's single-trajectory and device-pointer work on a caller-owned cudaStream_t (e.g.
 * torch's current stream) so that the caller's CUDA events bracket the kernels.  NULL is the legacy
 * default stream, as everywhere in CUDA; tolcuda_use_own_stream goes back to the context's own.
 * The context's own stream is created cudaStreamNonBlocking: it is NOT ordered against the legacy default stream or
 * any other stream.  With device pointers the caller orders its producers of x and its consumers (or earlier
 * writers, e.g. a memset) of F/G against the stream in use -- by handing over its own stream here, by
 * tolcuda_synchronize, or by events. */
int tolcuda_set_stream(tolcuda_handle h, void *cuda_stream);
int tolcuda_use_own_stream(tolcuda_handle h);
int tolcuda_synchronize(tolcuda_handle h);

/* number of kernel launches this context has issued (bench.py's gpu_launches) */
long tolcuda_launch_count(tolcuda_handle h);

/* Makes `h` the process-global context DEFINEGusrfg_ evaluates with, as reference `problem *prob`
 * (src/tol.cpp:3, include/global_objects.h:5) is for the reference callback.  NULL unbinds. */
int tolcuda_bind_global(tolcuda_handle h);

/* The snOptA user function, signature of snFunA (reference include/snopt/snopt.h:60-66), symbol and
 * argument meaning of reference include/DefineFG.h:5-17 / src/DefineFG.cpp:9-48, so
 * `setUserFun(DEFINEGusrfg_)` (src/problem.cpp:1234) binds it unchanged.  Success leaves *Status
 * untouched (the reference never writes it); a CUDA failure or a missing context sets *Status = -2
 * (SNOPT: terminate) and reports on stderr.  cu/iu/ru are ignored as in the reference. */
void DEFINEGusrfg_(int *Status, int *n, double x[], int *needF, int *neF, double F[], int *needG,
                   int *neG, double G[], char *cu, int *lencu, int iu[], int *leniu, double ru[],
                   int *lenru);

/* reference parameters::readparams (src/parameters.cpp:14-34): one leading number per line, text
 * from the first '/' on ignored, lines that do not start with a number skipped.  Stores up to
 * `cap` values and returns the number found in *count. */
int tolcuda_read_params(const char *path, double *values, int cap, int *count);

const char *tolcuda_last_error(void);
const char *tolcuda_version(void);

#ifdef __cplusplus
}
#endif
#endif /* TOLCUDA_H_ */
