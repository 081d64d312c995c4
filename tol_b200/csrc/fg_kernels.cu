// sm_100a kernels for tol's SNOPT user function: objective, defect + boundary constraints F and the
// sparse Jacobian values G in SNOPT coordinate order, for B independent trajectories per launch.
//
// Replaces (reference file:line, lingaqing/tol):
//   problem::modelWind            src/problem.cpp:475-531   (cases 0, 1)
//   problem::computeF             src/problem.cpp:765-774
//   problem::dynamicConstraints   src/problem.cpp:929-1021
//   problem::computeG             src/problem.cpp:782-806
//   problem::dynamicsGradients    src/problem.cpp:1035-1208
//   problemS10::{cost,boundaryConstraints,costGradient,boundaryGradients}  src/problemS10.cpp:227-415
//   problemG7::{cost,boundaryConstraints,costGradient,boundaryGradients}   src/problemG7.cpp:225-513
//
// Work decomposition.  One thread owns one collocation window k (node k and the 8 states of node
// k+1); one warp owns a tile of 32 consecutive windows of one trajectory and runs on its own.  The
// reference instead walks the neG coordinate entries and, for every single entry, re-evaluates the
// whole 12-column expression table of that entry's row (src/problem.cpp:785-802, 1074-1199); here
// every parenthesised sub-expression is evaluated once per node.
//
// Numerics.  Compiled with -fmad=false: every product and sum is rounded separately, in the C
// left-to-right association of the cited reference line, exactly like the reference's x86-64 -O2
// build (no FMA contraction).  Sub-expressions the reference multiplies by a wind-gradient
// component that is identically zero under the selected wind model are dropped: x + 0*y == x
// for finite y, so this changes no value (only, possibly, the sign of a zero).  Divisions by a
// denominator that occurs several times share one correctly rounded reciprocal and a Markstein
// correction (div_r; see there for what it guarantees and where it differs from `/`).  What is left to
// differ from the reference is the last-ulp behaviour of sin/cos (CUDA libdevice vs glibc).
//
// Memory.  The kernel is bound by its write stream (G is 91 % of the bytes), and on B200 that stream
// is limited by L2 write REQUESTS, not bytes: pieces smaller than whole 128-byte lines cost bandwidth
// (208-byte pieces measured 4.8 TB/s against 7.5 TB/s for a plain fill).  So G leaves as whole
// 832-byte window records, contiguous in SNOPT coordinate order:
//   * each warp stages the 33-node slice of x its windows need in shared memory (cp.async, 16-byte);
//   * a window's 104-value record is assembled in one of the warp's 8 record slots whose structural
//     constants (0, +-1) are written once per run of trajectories; per pass of 8 windows only the 33
//     x-dependent entries are stored, and the 8 finished records (6,656 contiguous bytes) go to the TMA unit
//     as one cp.async.bulk shared->global copy;
//   * F (8 defects per window) and the S10 objective-row entries go out through the dead x slice as
//     coalesced stores.  Cost sums use warp-shuffle reductions.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include <atomic>
#include <type_traits>
#include <utility>

#include "fg_const.h"
#include "fg_launch.h"

namespace {

constexpr int MAX_DEVICES = 64;  // power of two; device ordinals are folded into it
constexpr int PX = TOLCUDA_PX;
constexpr int PF = TOLCUDA_PF;
constexpr int REC = TOLCUDA_REC;
// Record buffer: one per warp, NPP = 8 dense record slots of REC doubles.  A drain pass hands 8 windows (lanes
// 8g .. 8g+7) to the TMA unit: each of those lanes places its 33 x-dependent values in its own slot (the slots'
// constants are written once per run of trajectories), then lane 0 issues the 8 records (6,656 bytes) as one bulk
// copy; a pass waits until the TMA unit has read the previous one, so a tile takes 4 passes.  Two buffers of 4
// records (8 passes, fill and read overlapped) need the same shared memory, twice the shared-store instructions,
// proxy fences and warp barriers of a tile, and measured 0.3 % slower; 16-record buffers leave room for only one
// CTA per SM and measured slower still (profiles/r1_history.md).
constexpr int NPP = 8;                 // windows per drain pass = record slots per warp
// + 16 doubles of slack: when the records of a trajectory start 8 mod 16 in global memory (odd ts, or an odd
// leading dimension) the slots are used shifted by one double, so that all but the first and the last double of
// a pass still form one 16-byte aligned bulk copy (see tile_drain); 16 keeps the tiles 128-byte aligned
constexpr int TILE_SLACK = 16;
constexpr int TILE_LEN = NPP * REC + TILE_SLACK;
constexpr int SX_LEN = 368;            // a warp's x slice: slot for x[11*k0] + 33 nodes = 364 doubles (tile stays 128-byte aligned)
constexpr int WARP_SMEM = SX_LEN + TILE_LEN;        // kernel A
constexpr int WARP_SMEM_B = 2 * SX_LEN + TILE_LEN;  // kernel L (and kernel A with runs): two x-slice buffers
constexpr int F_LD = 10;               // smem stride of a window's 8 defects (== 2 mod 4)
constexpr int NVAR = TOLCUDA_NVAR;     // x-dependent entries of a record (plus two -dt entries)
// kernel flavours: plain F/G; F/G + per-trajectory summary; F + COMPACT G (objective-row block, then the
// NVAR x-dependent entries of every window, then the boundary block) for the host-pointer path, where the
// structural constants are filled in on the host instead of crossing PCIe
constexpr int MODE_PLAIN = 0, MODE_SUMMARY = 1, MODE_COMPACT = 2;
// matrix-free consumers of the Jacobian (SURVEY.md 8f-4; G is never written): MODE_JVP  y = J(x) d  (the F pointer
// receives y, the G pointer holds d), MODE_VJP  z = J(x)^T lambda  (the F pointer holds lambda, the G pointer receives z)
constexpr int MODE_JVP = 3, MODE_VJP = 4;
// F alone (needG == 0 in a plain call: SNOPT's line-search evaluations, screening): the same window arithmetic up to the
// defects and nothing of the Jacobian's -- a third of the registers and no record slots, so three to four times the
// warps per SM for what is a latency-bound chain (x slice -> 3 sincos -> defects -> staged F)
constexpr int MODE_FONLY = 5;
// ... and the same with the per-trajectory summary (screening: x in, [objective, worst defect, worst boundary violation,
// sum of defect^2] out, F optional)
constexpr int MODE_FSUMM = 6;
// w = D_x[J(x)^T lambda] d, the Hessian of the Lagrangian times d (the F pointer holds lambda, the G pointer receives
// w; d and the optional z = J^T lambda travel as extra kernel arguments): MODE_VJP run in dual arithmetic (Dual)
constexpr int MODE_HVP = 7;
__host__ __device__ constexpr bool mode_is_fonly(int mode) { return mode == MODE_FONLY || mode == MODE_FSUMM; }
__host__ __device__ constexpr bool mode_has_summary(int mode) { return mode == 1 || mode == MODE_FSUMM; }
__host__ __device__ constexpr bool mode_is_op(int mode) { return mode == MODE_JVP || mode == MODE_VJP || mode == MODE_HVP; }
// the flavours that assemble whole records in the warp's record slots (the others use the tile as plain staging)
__host__ __device__ constexpr bool mode_has_records(int mode) { return mode == MODE_PLAIN || mode == MODE_SUMMARY; }
// doubles of a warp's tile in kernel A
__host__ __device__ constexpr int tile_len_of(int mode) { return mode_is_fonly(mode) ? 0 : TILE_LEN; }

// Programmatic dependent launch (FgLaunch::pdl).  Every CTA releases the NEXT launch on the stream as soon as it
// has started (griddepcontrol.launch_dependents), so the next grid's CTAs move into SMs the tail of this grid has
// left instead of waiting for its last CTA.  A grid launched as a dependent reads only x before its first global
// store; there it waits for the preceding grid to have completed (griddepcontrol.wait, FLOW_WAIT) -- unless the
// caller has declared the outputs of the two launches disjoint, in which case the two grids simply overlap.
// Both instructions are no-ops in a launch without the attribute.
constexpr int FLOW_WAIT = 1;
__device__ __forceinline__ void pdl_release() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// record position -> content: tolcuda_rec_kind (fg_const.h), the table compact.cpp and expand_kernel.cu use too
__host__ __device__ constexpr int rec_kind(int p) { return tolcuda_rec_kind(p); }
// the positions record_store / tile_init write by hand, checked against that table
constexpr bool record_slots_match_table() {
    constexpr int var_pos[TOLCUDA_NVAR] = {0,  4,  5,  6,  13, 17, 18, 19, 26, 30, 31, 39, 43, 44, 45, 47,
                                           50, 52, 56, 57, 58, 59, 60, 65, 69, 70, 71, 72, 73, 78, 91};
    for (int i = 0; i < TOLCUDA_NVAR; i++)
        if (rec_kind(var_pos[i]) != i) return false;
    int nvar = 0;
    for (int p = 0; p < TOLCUDA_REC; p++) {
        const int kd = rec_kind(p);
        nvar += kd >= 0;
        const bool minus1 = p == 1 || p == 15 || p == 29 || p == 85 || p == 99, plus1 = p % 13 == 12;
        if ((kd == -3) != minus1 || (kd == -2) != plus1 || (kd == -4) != (p == 87 || p == 101)) return false;
    }
    return nvar == TOLCUDA_NVAR;
}
static_assert(record_slots_match_table(), "record_store / tile_init disagree with tolcuda_rec_kind (fg_const.h)");
template <int P, class Num>
__device__ __forceinline__ Num rec_value(const Num *v, const Num mdt) {
    constexpr int kd = rec_kind(P);
    if constexpr (kd >= 0) return v[kd];
    else if constexpr (kd == -2) return 1.0;
    else if constexpr (kd == -3) return -1.0;
    else if constexpr (kd == -4) return mdt;
    else return 0.0;
}
// acc + R[P] * w, skipping structural zeros and multiplications by +-1 (Num = Dual: the constants' derivatives are 0)
template <int P, class Num>
__device__ __forceinline__ Num rec_madd(const Num acc, const Num *v, const Num mdt, const double w) {
    constexpr int kd = rec_kind(P);
    if constexpr (kd == -1) return acc;
    else if constexpr (kd == -2) return acc + w;
    else if constexpr (kd == -3) return acc - w;
    else return acc + rec_value<P>(v, mdt) * w;
}
// row S of a window's record times dv[0..12]; column J of it times lam[0..7]
template <int S, int... J>
__device__ __forceinline__ double rec_row_dot(const double *v, const double mdt, const double *dv, std::integer_sequence<int, J...>) {
    double a = 0.0;
    ((a = rec_madd<13 * S + J>(a, v, mdt, dv[J])), ...);
    return a;
}
template <int J, class Num, int... S>
__device__ __forceinline__ Num rec_col_dot(const Num *v, const Num mdt, const double *lam, std::integer_sequence<int, S...>) {
    Num a = 0.0;
    ((a = rec_madd<13 * S + J>(a, v, mdt, lam[S])), ...);
    return a;
}
template <int... S>
__device__ __forceinline__ void rec_times_vec(const double *v, const double mdt, const double *dv, double *y, std::integer_sequence<int, S...>) {
    ((y[S] = rec_row_dot<S>(v, mdt, dv, std::make_integer_sequence<int, 12>())), ...);  // column 12 (+1) by the caller
}
template <class Num, int... J>
__device__ __forceinline__ void rec_transposed_times_vec(const Num *v, const Num mdt, const double *lam, Num *z, std::integer_sequence<int, J...>) {
    ((z[J] = rec_col_dot<J>(v, mdt, lam, std::make_integer_sequence<int, TOLCUDA_PF>())), ...);
}

// per-lane partial results a tile hands back: cost sums and the feasibility summary of its defects
struct TileSums {
    double sumT, sump;  // sum of T^2, sum of (r-R)^2 (S10)
    double dmax, dssq;  // max |defect|, sum of defect^2 (SUMM instantiations only)
};

// the larger of a and b, NaN if either is NaN (fmax drops a NaN operand): a summary maximum over values one of which is
// NaN is NaN, as numpy's max of the same values, so a NaN defect or boundary row cannot hide behind finite ones
__device__ __forceinline__ double max_nan(double a, double b) { return (a > b || a != a) ? a : b; }

__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) v = max_nan(v, __shfl_xor_sync(0xffffffffu, v, m));
    return v;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
    return v;
}

// x / D given rD = RN(1/D): one product plus one Markstein correction.  For finite operands in the normal range this
// is the correctly rounded quotient in all but pathological cases (q = RN(x*rD) can be ~2 ulp off before the
// correction; 4e8 random operand pairs, all-ones mantissas included, gave 0 mismatches against `/`, DESIGN.md 3).
// For D == 0 or non-finite D the residual is NaN, so the result is NaN where the reference's `/` gives +-inf (or 0
// for an infinite D): non-finite either way, and SNOPT keeps Va and cos(gamma) away from 0 by bounds
// (tests/test_gpu_parity.py::test_degenerate_inputs_are_non_finite_where_the_reference_is compares finiteness there).
__device__ __forceinline__ double div_r(double x, double D, double rD) {
    const double q = x * rD;
    return fma(fma(-q, D, x), rD, q);
}

// ---- forward-mode dual numbers (MODE_HVP) ---------------------------------------------------------------
//
// A value and its derivative along the direction d.  The window arithmetic is written once, on a scalar type Num:
// double in every other mode, Dual in MODE_HVP.  The value part of every Dual operation is the double operation
// itself on the value parts (same operands, same order, -fmad=false), so the values of a Dual evaluation are bit for
// bit those of the double one; the derivative parts follow the product and quotient rules.
struct __align__(16) Dual {
    double v, d;
    Dual() = default;
    __device__ __forceinline__ Dual(double a, double b = 0.0) : v(a), d(b) {}
    __device__ __forceinline__ friend void sincos(const Dual a, Dual *s, Dual *c) {
        double sv, cv;
        sincos(a.v, &sv, &cv);
        *s = Dual(sv, cv * a.d);
        *c = Dual(cv, -(sv * a.d));
    }
    __device__ __forceinline__ friend Dual sqrt(const Dual a) {
        const double r = sqrt(a.v);
        return Dual(r, a.d / (2.0 * r));
    }
};
__device__ __forceinline__ Dual operator-(const Dual a) { return Dual(-a.v, -a.d); }
__device__ __forceinline__ Dual operator+(const Dual a, const Dual b) { return Dual(a.v + b.v, a.d + b.d); }
__device__ __forceinline__ Dual operator+(const Dual a, const double b) { return Dual(a.v + b, a.d); }
__device__ __forceinline__ Dual operator+(const double a, const Dual b) { return Dual(a + b.v, b.d); }
__device__ __forceinline__ Dual operator-(const Dual a, const Dual b) { return Dual(a.v - b.v, a.d - b.d); }
__device__ __forceinline__ Dual operator-(const Dual a, const double b) { return Dual(a.v - b, a.d); }
__device__ __forceinline__ Dual operator-(const double a, const Dual b) { return Dual(a - b.v, -b.d); }
__device__ __forceinline__ Dual operator*(const Dual a, const Dual b) { return Dual(a.v * b.v, a.v * b.d + a.d * b.v); }
__device__ __forceinline__ Dual operator*(const Dual a, const double b) { return Dual(a.v * b, a.d * b); }
__device__ __forceinline__ Dual operator*(const double a, const Dual b) { return Dual(a * b.v, a * b.d); }
__device__ __forceinline__ Dual operator/(const Dual a, const Dual b) {
    const double q = a.v / b.v;
    return Dual(q, (a.d - q * b.d) / b.v);
}
__device__ __forceinline__ Dual operator/(const Dual a, const double b) { return Dual(a.v / b, a.d / b); }
__device__ __forceinline__ Dual operator/(const double a, const Dual b) {
    const double q = a / b.v;
    return Dual(q, -(q * b.d) / b.v);
}
__device__ __forceinline__ Dual &operator+=(Dual &a, const Dual b) { return a = a + b; }
__device__ __forceinline__ Dual &operator+=(Dual &a, const double b) { return a = a + b; }
// value and derivative parts of either scalar type
__device__ __forceinline__ double val(const double a) { return a; }
__device__ __forceinline__ double val(const Dual a) { return a.v; }
__device__ __forceinline__ double der(const double) { return 0.0; }
__device__ __forceinline__ double der(const Dual a) { return a.d; }
// component j of a node: the staged x value, with (Dual) the matching component of d
template <class Num>
__device__ __forceinline__ Num node_in(const double *s, const double *ds, const int j) {
    if constexpr (std::is_same_v<Num, Dual>) return Num(s[j], __ldg(ds + j));
    else return s[j];
}
__device__ __forceinline__ double shfl(const double a, const int src) { return __shfl_sync(0xffffffffu, a, src); }
__device__ __forceinline__ Dual shfl(const Dual a, const int src) { return Dual(shfl(a.v, src), shfl(a.d, src)); }

// div_r (above) of dual operands: the value is div_r of the values, the derivative (x' - q D') / D
__device__ __forceinline__ Dual div_r(const Dual x, const Dual D, const Dual rD) {
    const double q = div_r(x.v, D.v, rD.v);
    return Dual(q, (x.d - q * D.d) * rD.v);
}
__device__ __forceinline__ Dual div_r(const Dual x, const double D, const double rD) {
    return Dual(div_r(x.v, D, rD), x.d * rD);
}

__device__ __forceinline__ void st2(double *p, double a, double b) {
    *reinterpret_cast<double2 *>(p) = make_double2(a, b);
}

// ---- asynchronous copies ---------------------------------------------------------------------------
//
// Shared-memory operands are 32-bit shared-window addresses computed ONCE per kernel (smem_addr): converting
// a generic pointer at every use costs an S2R of the CTA's cluster rank plus address arithmetic each time,
// and inside the kernels' loops ptxas re-materialises that instead of keeping it.
__device__ __forceinline__ uint32_t smem_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
// thread index read ONCE: as a plain threadIdx.x expression ptxas re-reads the special register (S2R, tens of
// cycles on the MIO path) at every use inside the kernels' loops when registers are tight; a volatile asm
// result cannot be re-materialised
__device__ __forceinline__ int thread_index() {
    int t;
    asm volatile("mov.u32 %0, %%tid.x;" : "=r"(t));
    return t;
}
__device__ __forceinline__ void cp_async16(uint32_t dst, const double *src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src));
}
__device__ __forceinline__ void cp_async8(uint32_t dst, const double *src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(src));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// enqueue the copy of `cnt` doubles xs[0..cnt) to shared address sx_s: 16-byte pieces when xs allows it
__device__ __forceinline__ void slice_prefetch(const uint32_t sx_s, const double *xs, const int cnt, const int lane) {
    if ((reinterpret_cast<uintptr_t>(xs) & 15) == 0) {
#pragma unroll
        for (int it = 0; it < (SX_LEN / 2 + 31) / 32; it++) {
            const int i = lane + 32 * it;
            if (2 * i + 1 < cnt) cp_async16(sx_s + 16 * i, xs + 2 * i);
            else if (2 * i < cnt) cp_async8(sx_s + 16 * i, xs + 2 * i);
        }
    } else {
        for (int i = lane; i < cnt; i += 32) cp_async8(sx_s + 8 * i, xs + i);
    }
}

// TMA bulk copy shared -> global of `bytes` (a multiple of 16; both sides 16-byte aligned)
__device__ __forceinline__ void bulk_issue(double *gdst, const uint32_t ssrc, const int bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(ssrc), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_store(double *gdst, const uint32_t ssrc, const int bytes) {
    bulk_issue(gdst, ssrc, bytes);
    bulk_commit();
}
// wait until all but the newest N bulk groups of the calling thread have finished READING shared memory
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}

// ---- per-trajectory goals (tolcuda_set_goals) ----------------------------------------------------------------------
//
// With a goal table, the values of a trajectory's row its formulation reads (S10: xg, yg, rg; G7: xg, yg, cos_chid,
// sin_chid) travel with the trajectory's first x slice, in the same cp.async group, into the last 4 doubles of the
// slice buffer: neither the slice (at most 1 + 11*33 doubles) nor the F / objective-row staging reaches them, so they
// stay readable through the trajectory's epilogue.  They are read from there at each use, not held in registers.
// Kernel L stages them for S10 only, whose tiles read them; G7 reads them once per trajectory, in the epilogue, from
// the table row itself (a pointer to the staged values, live across the tile loop, spills in the wind-cube instances).
constexpr int GOAL_SX = SX_LEN - 4;
static_assert(1 + PX * 33 <= GOAL_SX && 32 * F_LD <= GOAL_SX && 3 * 33 <= GOAL_SX, "goal values overlap the slice");
template <int FORM>
__device__ __forceinline__ void goal_prefetch(const uint32_t sx_s, const double *grow, const int lane) {
    if (lane < 4) cp_async8(sx_s + 8 * (GOAL_SX + lane), grow + (FORM != TOLCUDA_FORM_S10 && lane >= 2 ? lane + 1 : lane));
}
// the goal of the trajectory being evaluated: the context's immediates, or (GOALS) the values staged beside its slice
// (S10: xg, yg, rg; G7: xg, yg, cos_chid, sin_chid), or (GOALS, ROW) the trajectory's row of the table itself
template <int FORM, bool GOALS, bool ROW = false>
struct Goal {
    const double *s;  // slice buffer + GOAL_SX, or the table row
    __device__ __forceinline__ double get(const int i) const { return ROW ? __ldg(s + i) : s[i]; }
    __device__ __forceinline__ double xg(const FgConst &c) const { return GOALS ? get(0) : c.xg; }
    __device__ __forceinline__ double yg(const FgConst &c) const { return GOALS ? get(1) : c.yg; }
    __device__ __forceinline__ double rg(const FgConst &c) const {
        static_assert(FORM == TOLCUDA_FORM_S10, "only S10 stages rg");
        return GOALS ? get(2) : c.rg;
    }
    __device__ __forceinline__ double cos_chid(const FgConst &c) const {
        static_assert(FORM != TOLCUDA_FORM_S10, "only G7 stages cos_chid, sin_chid");
        return GOALS ? get(ROW ? 3 : 2) : c.cos_chid;
    }
    __device__ __forceinline__ double sin_chid(const FgConst &c) const {
        static_assert(FORM != TOLCUDA_FORM_S10, "only G7 stages cos_chid, sin_chid");
        return GOALS ? get(ROW ? 4 : 3) : c.sin_chid;
    }
};

// ---- record slots -------------------------------------------------------------------------------------
//
// Record layout (row s of the window at 13*s: [d/d dt, d/d c0..c10 @k, d/d c_s @k+1]).  Structural
// constants: tabG zero-initialisation and the +-1 entries (src/problem.cpp:1038, 1084, 1098, 1112, 1170,
// 1182, 1204); everything x-dependent is zeroed here and written per window by record_store.
// offset of record slot q (0 .. NPP-1) within the record buffer
__device__ __forceinline__ int slot_offset(const int q) { return q * REC; }
// lanes 0 .. NPP-1 each prepare one record slot: zeros, then the 13 structural +-1 entries.
// mis = 1: the slots sit one double further (records that start 8 mod 16 in global memory)
__device__ __forceinline__ void tile_init(double *tile, const int lane, const int mis) {
    if (lane >= NPP) return;
    double *rec = tile + slot_offset(lane) + mis;
    if (mis) {
        rec[0] = 0.0;
#pragma unroll
        for (int j = 1; j < REC - 1; j += 2) st2(rec + j, 0.0, 0.0);
        rec[REC - 1] = 0.0;
    } else {
#pragma unroll
        for (int j = 0; j < REC; j += 2) st2(rec + j, 0.0, 0.0);
    }
    rec[1] = -1.0;   // F1 d/dx
    rec[15] = -1.0;  // F2 d/dy
    rec[29] = -1.0;  // F3 d/dz
    rec[85] = -1.0;  // F7 d/dphi
    rec[99] = -1.0;  // F8 d/dCL
#pragma unroll
    for (int s = 0; s < PF; s++) rec[13 * s + 12] = 1.0;  // d/d(state s at node k+1)
}

// the x-dependent entries; adjacent (even, odd) positions leave as one 16-byte store
__device__ __forceinline__ void record_store(double *rec, const double *v, const double mdt) {
    rec[0] = v[0];  // F1: dt | Va, gam | chi          src/problem.cpp:1084-1088
    st2(rec + 4, v[1], v[2]);
    rec[6] = v[3];
    rec[13] = v[4];  // F2                              :1098-1102
    rec[17] = v[5];
    st2(rec + 18, v[6], v[7]);
    rec[26] = v[8];  // F3: dt | Va, gam                :1112-1115
    st2(rec + 30, v[9], v[10]);
    rec[39] = v[11];  // F4: dt | Va | gam, chi | CL | T :1125-1130
    rec[43] = v[12];
    st2(rec + 44, v[13], v[14]);
    rec[47] = v[15];
    rec[50] = v[16];
    rec[52] = v[17];  // F5: dt | Va, gam | chi, phi | CL :1140-1145
    st2(rec + 56, v[18], v[19]);
    st2(rec + 58, v[20], v[21]);
    rec[60] = v[22];
    rec[65] = v[23];  // F6                              :1155-1160
    rec[69] = v[24];
    st2(rec + 70, v[25], v[26]);
    st2(rec + 72, v[27], v[28]);
    rec[78] = v[29];  // F7: dt, d/ddphi = -dt           :1171-1172
    st2(rec + 86, 0.0, mdt);
    rec[91] = v[30];  // F8: dt, d/ddCL = -dt            :1183-1184
    st2(rec + 100, 0.0, mdt);
}

// the same entries into a slot that starts 8 mod 16: pairs are the (odd, even) neighbours
__device__ __forceinline__ void record_store_shifted(double *rec, const double *v, const double mdt) {
    rec[0] = v[0];
    rec[4] = v[1];
    st2(rec + 5, v[2], v[3]);
    rec[13] = v[4];
    st2(rec + 17, v[5], v[6]);
    rec[19] = v[7];
    rec[26] = v[8];
    rec[30] = v[9];
    rec[31] = v[10];
    rec[39] = v[11];
    st2(rec + 43, v[12], v[13]);
    rec[45] = v[14];
    rec[47] = v[15];
    rec[50] = v[16];
    rec[52] = v[17];
    rec[56] = v[18];
    st2(rec + 57, v[19], v[20]);
    st2(rec + 59, v[21], v[22]);
    rec[65] = v[23];
    st2(rec + 69, v[24], v[25]);
    st2(rec + 71, v[26], v[27]);
    rec[73] = v[28];
    rec[78] = v[29];
    rec[87] = mdt;
    rec[91] = v[30];
    rec[101] = mdt;
}

// ---- wind model 3: trilinear interpolation of the cached wind cube, src/problem.cpp:544-695 -------------
//
// Only the v component is interpolated by the reference (u, w and their gradients stay zero).  The cell
// search keeps the reference's comparisons (first index with coordinate - grid < spacing; sic: the x search
// is bounded by the cube's second dimension and the y search by its first); where the reference would then
// index past the cube (undefined behaviour) the last cell is used instead.
// Num = Dual: the cell search compares values only; the derivatives are those of the interpolant within the cell.
template <class Num>
__device__ __forceinline__ void wind_cube(const FgConst &c, const Num xn, const Num yn, const Num zn,
                                          Num &v, Num &dv_dx, Num &dv_dy, Num &dv_dz) {
    const Num xs = yn + c.datum[0];  // ENU <- NED, :551-553
    const Num ys = xn + c.datum[1];
    const Num zs = -zn + c.datum[2];
    const double dx = c.spacing[0], dy = c.spacing[1], dz = c.spacing[2];
    int xi, yi, zi;
    for (xi = 0; xi < c.grid_nn; xi++)
        if ((val(xs) - __ldg(c.grid_x + xi)) < dx) break;
    for (yi = 0; yi < c.grid_ne; yi++)
        if ((val(ys) - __ldg(c.grid_y + yi)) < dy) break;
    for (zi = 0; zi < c.grid_nu; zi++)
        if ((val(zs) - __ldg(c.grid_z + zi)) < dz) break;
    xi = min(xi, c.grid_ne - 2), yi = min(yi, c.grid_nn - 2), zi = min(zi, c.grid_nu - 2);
    const double *g0 = c.grid_v + ((size_t)xi * c.grid_nn + yi) * c.grid_nu + zi;
    const size_t sx = (size_t)c.grid_nn * c.grid_nu, sy = c.grid_nu;
    double vc[8];
    vc[0] = __ldg(g0), vc[1] = __ldg(g0 + sx), vc[2] = __ldg(g0 + sy), vc[3] = __ldg(g0 + sx + sy);
    vc[4] = __ldg(g0 + 1), vc[5] = __ldg(g0 + sx + 1), vc[6] = __ldg(g0 + sy + 1), vc[7] = __ldg(g0 + sx + sy + 1);
    const Num xrel = (xs - __ldg(c.grid_x + xi)), yrel = (ys - __ldg(c.grid_y + yi)), zrel = (zs - __ldg(c.grid_z + zi));
    const Num zeta = xrel / dx, eta = yrel / dy, mu = zrel / dz;
    const double dxdy = dx * dy, dxdz = dx * dz, dydz = dy * dz, dxdydz = dx * dy * dz;
    Num N[8], NX[8], NY[8], NZ[8];
    N[0] = (1 - zeta) * (1 - eta) * (1 - mu);  // :618-625
    N[1] = zeta * (1 - eta) * (1 - mu);
    N[2] = (1 - zeta) * eta * (1 - mu);
    N[3] = zeta * eta * (1 - mu);
    N[4] = (1 - zeta) * (1 - eta) * mu;
    N[5] = zeta * (1 - eta) * mu;
    N[6] = (1 - zeta) * eta * mu;
    N[7] = zeta * eta * mu;
    NX[0] = -((eta - 1.0) * (mu - 1.0)) / dx;  // :643-650 (yrel/dy == eta, zrel/dz == mu)
    NX[1] = ((eta - 1.0) * (mu - 1.0)) / dx;
    NX[2] = (yrel * (mu - 1.0)) / dxdy;
    NX[3] = -(yrel * (mu - 1.0)) / dxdy;
    NX[4] = (zrel * (eta - 1.0)) / dxdz;
    NX[5] = -(zrel * (eta - 1.0)) / dxdz;
    NX[6] = -(yrel * zrel) / dxdydz;
    NX[7] = (yrel * zrel) / dxdydz;
    NY[0] = -((zeta - 1.0) * (mu - 1.0)) / dy;  // :653-660
    NY[1] = (xrel * (mu - 1.0)) / dxdy;
    NY[2] = ((zeta - 1.0) * (mu - 1.0)) / dy;
    NY[3] = -(xrel * (mu - 1.0)) / dxdy;
    NY[4] = (zrel * (zeta - 1.0)) / dydz;
    NY[5] = -(xrel * zrel) / dxdydz;
    NY[6] = -(zrel * (zeta - 1.0)) / dydz;
    NY[7] = (xrel * zrel) / dxdydz;
    NZ[0] = -((zeta - 1.0) * (eta - 1.0)) / dz;  // :663-670
    NZ[1] = (xrel * (eta - 1.0)) / dxdz;
    NZ[2] = (yrel * (zeta - 1.0)) / dydz;
    NZ[3] = -(xrel * yrel) / dxdydz;
    NZ[4] = ((zeta - 1.0) * (eta - 1.0)) / dz;
    NZ[5] = -(xrel * (eta - 1.0)) / dxdz;
    NZ[6] = -(yrel * (zeta - 1.0)) / dydz;
    NZ[7] = (xrel * yrel) / dxdydz;
    v = 0.0, dv_dx = 0.0, dv_dy = 0.0, dv_dz = 0.0;
#pragma unroll
    for (int i = 0; i < 8; i++) {  // :631-635, :682-692
        v += N[i] * vc[i];
        dv_dx += NX[i] * vc[i];
        dv_dy += NY[i] * vc[i];
        dv_dz += NZ[i] * vc[i];
    }
}

// ---- drain: passes of NPP windows through the record buffer, whole records to global (tile_eval) ---------------
__device__ __forceinline__ void tile_drain(const FgConst &c, double *tile, const uint32_t tile_s, const int k0, const int nk,
                                           const int lane, double *__restrict__ Gb, int &tile_mis, const double *v,
                                           const double mdt) {
    // Pass g (windows k0+NPP*g ..) fills the buffer once the TMA unit has read the previous pass; lane 0 issues the
    // pass's records as one bulk copy.
    // Records that start 8 mod 16 in global memory (R0 is odd for odd ts; odd leading dimensions) are staged one
    // double further into the slots: all but the first and the last double of a pass then form one 16-byte
    // aligned bulk copy, and two lanes store those two doubles.
    double *Grec = Gb + c.R0 + (size_t)REC * k0;  // record of window k0
    const int mis = (int)(reinterpret_cast<uintptr_t>(Grec) >> 3) & 1;
    if (mis != tile_mis) {  // the slots' constants are in place for the other alignment
        __syncwarp();
        tile_init(tile, lane, mis);
        tile_mis = mis;
        __syncwarp();
    }
#pragma unroll 1
    for (int g = 0; g < 32 / NPP; g++) {
        if (g * NPP >= nk) break;
        if (g >= 1) {
            if (lane == 0) bulk_wait_read<0>();  // pass g-1 has been read: the buffer is free
            __syncwarp();
        }
        if ((lane / NPP) == g) {
            if (mis) record_store_shifted(tile + slot_offset(lane & (NPP - 1)) + 1, v, mdt);
            else record_store(tile + slot_offset(lane & (NPP - 1)), v, mdt);
            // the writers make their generic-proxy stores visible to the async proxy (the TMA unit) ...
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        }
        const int nrec = min(NPP, nk - g * NPP);
        double *dst = Grec + (size_t)REC * NPP * g;
        __syncwarp();  // ... and lane 0 issues the copy after all of them have done so
        if (mis) {
            // doubles [1, nrec*REC - 1) of the pass as one aligned copy; lanes 1 and 2 store the two ends
            if (lane == 0) bulk_store(dst + 1, tile_s + 16, (nrec * REC - 2) * 8);
            if (lane == 1) dst[0] = tile[1];
            if (lane == 2) dst[nrec * REC - 1] = tile[nrec * REC];
        } else if (lane == 0) {
            // nrec is 1 .. NPP here: the guard and the clamp are redundant, but without them ptxas compiles every
            // record-writing instance differently from the code the profiles were measured on
            if (0 < nrec) bulk_issue(dst, tile_s, min(NPP, nrec) * REC * 8);
            bulk_commit();
        }
    }
    if (lane == 0) bulk_wait_read<0>();  // the buffer is reused (or released) after this
    __syncwarp();
}

// ---- one warp, one tile of 32 windows ---------------------------------------------------------------
//
// sx: the warp's staged x slice (slot 0 = x[11*k0], node j of the slice at sx[1+11j]).  Once every lane
// has its window in registers the slice is dead and serves as staging area for F and the objective row.
// tile: the warp's NPP record slots, constants already in place (tile_init).
// dep_wait: this is the warp's first tile of a launch that may have started before the preceding launch on the
// stream had finished (pdl_wait before the first global store).
// MODE_HVP: Db is the trajectory's row of d, Zb its row of z (or null); the window arithmetic runs on Dual, and
// ts_out.sumT / ts_out.sump return the tile's shares of z[0] / w[0].
template <int FORM, int WIND, int MODE, bool GOALS>
__device__ __forceinline__ void tile_eval(const FgConst &c, double *sx, double *tile, const uint32_t tile_s, const double dt_in,
                                          const int k0, const int nk, const int lane,
                                          double *__restrict__ Fb, double *__restrict__ Gb,
                                          const int needF, const int needG, TileSums &ts_out,
                                          const bool dep_wait, int &tile_mis, const double *aux = nullptr,
                                          const double *__restrict__ Db = nullptr, double *__restrict__ Zb = nullptr) {
    double &sumT = ts_out.sumT, &sump = ts_out.sump;
    constexpr bool OP = mode_is_op(MODE);
    using Num = std::conditional_t<MODE == MODE_HVP, Dual, double>;
    if (MODE == MODE_JVP) {  // the window's slice of d (the G pointer) into the unused record buffer
        slice_prefetch(tile_s, Gb + (size_t)PX * k0, 1 + PX * (nk + 1), lane);
        cp_async_commit();
    }
    // MODE_VJP: the record buffer holds aux (22 doubles), then the tile's multipliers; MODE_HVP: aux (22 Duals), the
    // multipliers, then the staging area of z
    constexpr int LAM_OFF = MODE == MODE_HVP ? 48 : 32;
    constexpr int ZST_OFF = LAM_OFF + PF * 33;
    static_assert(ZST_OFF + SX_LEN <= TILE_LEN, "MODE_HVP staging exceeds the record buffer");
    if (MODE == MODE_VJP || MODE == MODE_HVP) {
        // lambda of window k0-1 (its +1 entries reach this tile's first node) and of the tile's own windows: 8 each
        if (k0 > 0) slice_prefetch(tile_s + 8 * LAM_OFF, Fb + 1 + (size_t)PF * (k0 - 1), PF * (nk + 1), lane);
        else slice_prefetch(tile_s + 8 * (LAM_OFF + PF), Fb + 1, PF * nk, lane);
        cp_async_commit();
    }
    constexpr bool X3 = (WIND == 3);             // wind cube: Wx with all three gradient components
    constexpr bool W = (WIND == 1) || X3;        // Wx and dWx/dz present
    constexpr bool S10 = (FORM == TOLCUDA_FORM_S10);
    const Goal<FORM, GOALS> gl{sx + GOAL_SX};
    const int ts = c.ts;
    const int k = k0 + lane;
    const bool active = lane < nk;
    const bool last_window = active && (k == ts - 1);  // also carries node ts
    const double *s0 = sx + 1 + PX * (active ? lane : 0);
    const double *s1 = s0 + PX;
    // MODE_HVP: the matching components of d (node k; node k+1 for the objective terms at node ts)
    const double *dk = MODE == MODE_HVP ? Db + 1 + PX * (size_t)(k0 + (active ? lane : 0)) : nullptr;
    const double *dk1 = MODE == MODE_HVP ? dk + PX : nullptr;
    const Num dt = node_in<Num>(&dt_in, Db, 0);
    const Num z = node_in<Num>(s0, dk, 2), Va = node_in<Num>(s0, dk, 3), gam = node_in<Num>(s0, dk, 4);
    const Num chi = node_in<Num>(s0, dk, 5), phi = node_in<Num>(s0, dk, 6), CL = node_in<Num>(s0, dk, 7);
    const Num dphi = node_in<Num>(s0, dk, 8), dCL = node_in<Num>(s0, dk, 9), T = node_in<Num>(s0, dk, 10);

    // ---- shared sub-expressions of the window ----
    Num sc, cc, sg, cg, sp, cp;
    sincos(chi, &sc, &cc);
    sincos(gam, &sg, &cg);
    sincos(phi, &sp, &cp);
    // wind, NED <- ENU (src/problem.cpp:970-981): Wx = v, dWx_dx = dv_dy, dWx_dy = dv_dx, dWx_dz = -dv_dz;
    // every other component is exactly zero under models 0, 1 and 3.
    //   model 1 (:522-524): v = -Vref*zs/href with zs = -z, dv_dz = -Vref/href
    //   model 3 (:544-695): v and its gradient interpolated from the wind cube (wind_cube)
    Num Wxz = c.wind_Wxz, Wxx = 0.0, Wxy = 0.0;
    Num Wx = 0.0;
    if (WIND == 1) {
        const Num zs = -z;
        Wx = -2.4 * zs / 10.0;
    }
    if (X3) {
        Num dv_dx, dv_dy, dv_dz;
        wind_cube(c, node_in<Num>(s0, dk, 0), node_in<Num>(s0, dk, 1), z, Wx, dv_dx, dv_dy, dv_dz);
        Wxx = dv_dy, Wxy = dv_dx, Wxz = -dv_dz;
    }
    // (Wx + Va*cos(chi)*cos(gam)), (Wy + Va*cos(gam)*sin(chi)), (Wz - Va*sin(gam))
    const Num Vacc = Va * cc, Vacg = Va * cg, Vasg = Va * sg;
    const Num vx = W ? Wx + Vacc * cg : Vacc * cg;
    const Num vy = Vacg * sc;
    const Num vz = -Vasg;
    // the z-column instances of the reference's repeated wind-gradient brackets
    Num az = 0, bz = 0, cz = 0, dz = 0, ez = 0, fz = 0;
    if (W) {
        const Num Wxzcc = Wxz * cc, Wxzsc = Wxz * sc;
        az = Wxzcc * cg;          // (dWx_dz*cc*cg - dWz_dz*sg + dWy_dz*cg*sc)
        bz = Wxzcc * sg;          // (dWz_dz*cg + dWx_dz*cc*sg + dWy_dz*sc*sg)
        cz = -Wxzsc;              // (dWy_dz*cc - dWx_dz*sc)
        dz = Wxzcc;               // (dWx_dz*cc + dWy_dz*sc)
        ez = -((Wxz * cg) * sc);  // (dWy_dz*cc*cg - dWx_dz*cg*sc)
        fz = -(Wxzsc * sg);       // (dWy_dz*cc*sg - dWx_dz*sc*sg)
    }
    // the x- and y-column instances of the same brackets (wind cube only)
    Num ax = 0, ay = 0, bx = 0, by = 0, cx = 0, cy = 0, dxw = 0, dyw = 0, ex = 0, ey = 0, fx = 0, fy = 0;
    if (X3) {
        const Num Wxxcc = Wxx * cc, Wxycc = Wxy * cc, Wxxsc = Wxx * sc, Wxysc = Wxy * sc;
        ax = Wxxcc * cg, ay = Wxycc * cg;
        bx = Wxxcc * sg, by = Wxycc * sg;
        cx = -Wxxsc, cy = -Wxysc;
        dxw = Wxxcc, dyw = Wxycc;
        ex = -((Wxx * cg) * sc), ey = -((Wxy * cg) * sc);
        fx = -(Wxxsc * sg), fy = -(Wxysc * sg);
    }
    const Num ccg = cc * cg, cgsc = cg * sc;                  // cos(chi)*cos(gam), cos(gam)*sin(chi)
    const Num Vaccsg = Vacc * sg, Vascsg = Va * sc * sg;       // Va*cos(chi)*sin(gam), Va*sin(chi)*sin(gam)
    const Num Vacccg = Vacc * cg;                              // Va*cos(chi)*cos(gam)
    const Num rVa = 1.0 / Va, rVacg = 1.0 / Vacg;
    const Num CdT = c.Cd0 + div_r(CL * CL, c.ARpiee, c.r_ARpiee);  // (Cd0 + CL*CL/(AR*pi*ee))
    const Num rSV = c.rhoSS * Va;                                  // rho*SS*Va
    const Num CLrS = CL * c.rho * c.SS;                            // CL*rho*SS
    const Num CLrSV = CLrS * Va;
    const Num Va2 = Va * Va;
    const Num Tmm = div_r(T, c.mm, c.r_mm);
    const Num gsg = c.g * sg, gcg = c.g * cg;
    // (vx*bx + vy*by + vz*bz - g*cos(gam))
    const Num n4 = X3 ? vx * bx + vy * by + vz * bz - gcg : (W ? vz * bz - gcg : -gcg);
    // (vx*ax + vy*ay + vz*az) and (vz*cz + cx*vx + vy*cy)
    const Num va3 = X3 ? vx * ax + vy * ay + vz * az : vz * az;
    const Num vc3 = X3 ? vz * cz + cx * vx + vy * cy : vz * cz;
    const Num Vadt = Va * dt, mdt = -dt;

    // ---- objective terms: src/problemS10.cpp:246-258, 340-372; src/problemG7.cpp:240-241, 370 ----
    sumT = 0.0, sump = 0.0;
    Num r0x = 0.0, r0y = 0.0, rex = 0.0, rey = 0.0;
    const Num Te = node_in<Num>(s1, dk1, 10);
    if (active) sumT = val(T * T);
    if (last_window) sumT += val(Te * Te);
    if constexpr (S10) {
        if (active) {
            const Num ddx = node_in<Num>(s0, dk, 0) - gl.xg(c), ddy = node_in<Num>(s0, dk, 1) - gl.yg(c);
            const Num r = sqrt(ddx * ddx + ddy * ddy);
            const Num rmR = r - gl.rg(c);
            const Num rr = 1.0 / r;
            sump = val(rmR * rmR);
            r0x = div_r(c.kp * rmR * ddx, r, rr);
            r0y = div_r(c.kp * rmR * ddy, r, rr);
        }
        if (last_window) {
            const Num ddx = node_in<Num>(s1, dk1, 0) - gl.xg(c), ddy = node_in<Num>(s1, dk1, 1) - gl.yg(c);
            const Num r = sqrt(ddx * ddx + ddy * ddy);
            const Num rmR = r - gl.rg(c);
            const Num rr = 1.0 / r;
            sump += val(rmR * rmR);
            rex = div_r(c.kp * rmR * ddx, r, rr);
            rey = div_r(c.kp * rmR * ddy, r, rr);
        }
    }

    // ---- defects, src/problem.cpp:1003-1019 ----
    double f[PF];
    {
        const Num drag3 = div_r(rSV * Va * CdT, c.twomm, c.r_twomm);
        const Num dx3 = X3 ? Tmm - vy * ay - vz * az - vx * ax - gsg - drag3
                           : (W ? Tmm - vz * az - gsg - drag3 : Tmm - gsg - drag3);
        const Num dx4 = div_r(n4 + div_r(CLrSV * Va * cp, c.twomm, c.r_twomm), Va, rVa);
        const Num lift5 = div_r(CLrSV * Va * sp, c.twomm, c.r_twomm);
        const Num dx5 = W ? div_r(-(vc3 - lift5), Vacg, rVacg) : div_r(-(-lift5), Vacg, rVacg);
        f[0] = val(s1[0] - vx * dt - s0[0]);
        f[1] = val(s1[1] - vy * dt - s0[1]);
        f[2] = val(s1[2] - vz * dt - s0[2]);
        f[3] = val(s1[3] - dx3 * dt - s0[3]);
        f[4] = val(s1[4] - dx4 * dt - s0[4]);
        f[5] = val(s1[5] - dx5 * dt - s0[5]);
        f[6] = val(s1[6] - dphi * dt - s0[6]);
        f[7] = val(s1[7] - dCL * dt - s0[7]);
    }
    ts_out.dmax = 0.0, ts_out.dssq = 0.0;
    if (mode_has_summary(MODE)) {
        double m = 0.0, q = 0.0;
        if (active) {
#pragma unroll
            for (int i = 0; i < PF; i++) {
                m = max_nan(m, fabs(f[i]));
                q += f[i] * f[i];
            }
        }
        ts_out.dmax = m, ts_out.dssq = q;
    }
    __syncwarp();  // every lane has read its window: the slice is dead, sx becomes the staging area
    if (dep_wait) pdl_wait();  // nothing has been stored so far

    if (needF && !OP) {
        double *fs = sx + F_LD * lane;
        st2(fs + 0, f[0], f[1]);
        st2(fs + 2, f[2], f[3]);
        st2(fs + 4, f[4], f[5]);
        st2(fs + 6, f[6], f[7]);
        __syncwarp();
        double *dst = Fb + 1 + PF * k0;
#pragma unroll
        for (int it = 0; it < PF; it++) {
            const int i = lane + 32 * it;  // i-th defect of the warp: window i/8, state i%8
            if (i < PF * nk) dst[i] = sx[F_LD * (i >> 3) + (i & 7)];
        }
        __syncwarp();
    }
    if (mode_is_fonly(MODE) || !needG) return;

    if (OP) {
    } else if (S10) {
        // objective row [dt, (x, y, T) of every node]: this warp's 3*nk (+3) entries
        if (active) {
            sx[3 * lane] = val(r0x);
            sx[3 * lane + 1] = val(r0y);
            sx[3 * lane + 2] = val(c.kT * T);
        }
        if (last_window) {
            sx[3 * lane + 3] = val(rex);
            sx[3 * lane + 4] = val(rey);
            sx[3 * lane + 5] = val(c.kT * Te);
        }
        __syncwarp();
        const int cnt0 = 3 * nk + ((k0 + nk == ts) ? 3 : 0);
        double *dst = Gb + 1 + 3 * k0;
        for (int i = lane; i < cnt0; i += 32) dst[i] = sx[i];
    } else {
        // G7 objective row [dt, x_0, y_0, T_0 .. T_{ts-1}, x_ts, y_ts, T_ts], src/problemG7.cpp:343-380
        if (active) Gb[3 + k] = val(c.kT * T);
        if (last_window) Gb[ts + 5] = val(c.kT * Te);
    }

    // ---- Jacobian rows, src/problem.cpp:1074-1192 ----
    Num v[NVAR];
    v[0] = -vx;  // F1 :1084-1088
    v[1] = mdt * cc * cg;
    v[2] = Vadt * cc * sg;
    v[3] = Vadt * cg * sc;
    v[4] = -vy;  // F2 :1098-1102
    v[5] = mdt * cg * sc;
    v[6] = Vadt * sc * sg;
    v[7] = -(Vadt * cc * cg);
    v[8] = Vasg;  // F3 :1112-1115
    v[9] = dt * sg;
    v[10] = Vadt * cg;
    {  // F4 :1125-1130
        const Num dragv = div_r(rSV * CdT, c.mm, c.r_mm);
        const Num drag11 = div_r(c.rhoSS * Va2 * CdT, c.twomm, c.r_twomm);
        v[11] = W ? va3 - Tmm + gsg + drag11 : -Tmm + gsg + drag11;
        v[12] = X3 ? dt * (ccg * ax - sg * az + cgsc * ay + dragv) - 1.0
                   : (W ? dt * (-(sg * az) + dragv) - 1.0 : dt * dragv - 1.0);
        v[13] = X3 ? mdt * (n4 + Vacg * az + Vaccsg * ax + Vascsg * ay) : (W ? mdt * (n4 + Vacg * az) : mdt * n4);
        v[14] = X3 ? dt * (ex * vx + vy * ey + ez * vz + Vacccg * ay - vy * ax) : (W ? dt * (ez * vz) : 0.0);
        v[15] = div_r(CLrS * Va2 * dt, c.ARpieemm, c.r_ARpieemm);
        v[16] = div_r(mdt, c.mm, c.r_mm);
    }
    {  // F5 :1140-1145
        const Num rVa2 = 1.0 / Va2;
        const Num S5 = n4 + div_r(CLrS * Va2 * cp, c.twomm, c.r_twomm);
        const Num liftv = div_r(CLrSV * cp, c.mm, c.r_mm);
        v[17] = div_r(-S5, Va, rVa);
        v[18] = X3 ? div_r(dt * S5, Va2, rVa2) - div_r(dt * (ccg * bx - sg * bz + cgsc * by + liftv), Va, rVa)
                : W ? div_r(dt * S5, Va2, rVa2) - div_r(dt * (-(sg * bz) + liftv), Va, rVa)
                  : div_r(dt * S5, Va2, rVa2) - div_r(dt * liftv, Va, rVa);
        v[19] = X3 ? div_r(-(dt * (va3 + gsg - Vacg * bz - Vaccsg * bx - Vascsg * by)), Va, rVa) - 1.0
                : W ? div_r(-(dt * (va3 + gsg - Vacg * bz)), Va, rVa) - 1.0 : div_r(-(dt * gsg), Va, rVa) - 1.0;
        v[20] = X3 ? div_r(-(dt * (fx * vx + vy * fy + fz * vz + Vacccg * by - vy * bx)), Va, rVa)
                : W ? div_r(-(dt * (fz * vz)), Va, rVa) : 0.0;
        v[21] = div_r(CLrSV * dt * sp, c.twomm, c.r_twomm);
        v[22] = div_r(-(rSV * dt * cp), c.twomm, c.r_twomm);
    }
    {  // F6 :1155-1160
        const Num lift6 = div_r(CLrS * Va2 * sp, c.twomm, c.r_twomm);
        const Num Q = W ? vc3 - lift6 : -lift6;
        const Num sidev = div_r(CLrSV * sp, c.mm, c.r_mm);
        const Num Va2cg = Va2 * cg, Vacg2 = Va * (cg * cg), tmcg = c.twomm * cg;
        const Num rVa2cg = 1.0 / Va2cg, rVacg2 = 1.0 / Vacg2, rtmcg = 1.0 / tmcg;
        v[23] = div_r(Q, Vacg, rVacg);
        v[24] = X3 ? div_r(-(dt * (sg * cz - ccg * cx - cgsc * cy + sidev)), Vacg, rVacg) - div_r(dt * Q, Va2cg, rVa2cg)
                : W ? div_r(-(dt * (sg * cz + sidev)), Vacg, rVacg) - div_r(dt * Q, Va2cg, rVa2cg)
                  : div_r(-(dt * sidev), Vacg, rVacg) - div_r(dt * Q, Va2cg, rVa2cg);
        v[25] = X3 ? div_r(dt * sg * Q, Vacg2, rVacg2) - div_r(dt * (Vacg * cz + Vaccsg * cx + Vascsg * cy), Vacg, rVacg)
                : W ? div_r(dt * sg * Q, Vacg2, rVacg2) - div_r(dt * (Vacg * cz), Vacg, rVacg)
                  : div_r(dt * sg * Q, Vacg2, rVacg2);
        v[26] = X3 ? div_r(-(dt * (vz * dz + dxw * vx + vy * dyw - Vacccg * cy + vy * cx)), Vacg, rVacg) - 1.0
                : W ? div_r(-(dt * (vz * dz)), Vacg, rVacg) - 1.0 : -1.0;
        v[27] = div_r(-(CLrSV * dt * cp), tmcg, rtmcg);
        v[28] = div_r(-(rSV * dt * sp), tmcg, rtmcg);
    }
    v[29] = -dphi;  // F7 :1172
    v[30] = -dCL;   // F8 :1184
    if constexpr (OP && MODE != MODE_HVP) {
        // the 31 entries meet in registers before the products consume them: left free, ptxas interleaves their
        // arithmetic with the dot products and spills at the 128-register cap
#pragma unroll
        for (int i = 0; i < NVAR; i++) asm volatile("" : "+d"(v[i]));
    }

    if constexpr (MODE == MODE_JVP) {
        // y = J d for this warp's rows: the window's 8 defect rows (src/problem.cpp:1074-1192 entries times the
        // matching d components, columns in ascending order) leave like F; the objective row's share of this
        // tile (src/problemS10.cpp:340-372, src/problemG7.cpp:370) goes back through sumT
        cp_async_wait<0>();
        __syncwarp();
        const double *d0 = tile + 1 + PX * (active ? lane : 0);
        double dv[12], y[PF];
#pragma unroll
        for (int j = 0; j < PX; j++) dv[1 + j] = d0[j];
        dv[0] = __ldg(Gb);
        const double dTe = d0[PX + 10], dxe = d0[PX], dye = d0[PX + 1];
        double part = 0.0;
        if (active) part = S10 ? r0x * dv[1] + r0y * dv[2] + (c.kT * T) * dv[11] : (c.kT * T) * dv[11];
        if (last_window) part += S10 ? rex * dxe + rey * dye + (c.kT * Te) * dTe : (c.kT * Te) * dTe;
        sumT = part;
        // the last column of row s multiplies component s of node k+1
        double acc[PF];
        rec_times_vec(v, mdt, dv, acc, std::make_integer_sequence<int, PF>());
#pragma unroll
        for (int s2 = 0; s2 < PF; s2++) y[s2] = acc[s2] + d0[PX + s2];
        __syncwarp();
        double *fs = sx + F_LD * lane;
        st2(fs + 0, y[0], y[1]);
        st2(fs + 2, y[2], y[3]);
        st2(fs + 4, y[4], y[5]);
        st2(fs + 6, y[6], y[7]);
        __syncwarp();
        double *dst = Fb + 1 + PF * k0;
#pragma unroll
        for (int it = 0; it < PF; it++) {
            const int i = lane + 32 * it;
            if (i < PF * nk) dst[i] = sx[F_LD * (i >> 3) + (i & 7)];
        }
        __syncwarp();
        return;
    }
    if constexpr (MODE == MODE_VJP || MODE == MODE_HVP) {
        // z = J^T lambda for this warp's nodes: node k collects its own window's columns, the +1 entries of
        // window k-1 (component c of node k appears in row c of window k-1 with value 1), the objective row's
        // entries times lambda_0, and -- nodes 0 and ts only -- the boundary rows' share prepared in aux.
        // MODE_HVP: the same in dual arithmetic; the derivative parts are w (no share from window k-1: its +1
        // entries are constants), the value parts z
        const Num *auxn = reinterpret_cast<const Num *>(aux);
        const double *lamrow = Fb;
        const double lam0 = __ldg(lamrow);
        cp_async_wait<0>();
        __syncwarp();
        const double *lprev = tile + LAM_OFF + PF * lane;  // multipliers of window k-1, then of window k
        double lam[PF];
        Num z[12];
#pragma unroll
        for (int s2 = 0; s2 < PF; s2++) lam[s2] = active ? lprev[PF + s2] : 0.0;
        rec_transposed_times_vec(v, mdt, lam, z, std::make_integer_sequence<int, 12>());
        sumT = active ? val(z[0]) : 0.0;  // d/d dt column: summed over the trajectory
        if (MODE == MODE_HVP) sump = active ? der(z[0]) : 0.0;
        if (S10) {
            z[1] += lam0 * r0x;
            z[2] += lam0 * r0y;
        }
        z[11] += lam0 * (c.kT * T);
        double *zst = tile + ZST_OFF;  // MODE_HVP: z is staged here, w in sx
        if (active) {
            double *zs = sx + 1 + PX * lane;
#pragma unroll
            for (int j = 0; j < PX; j++) {
                Num zz = z[1 + j];
                if (j < PF && k > 0) zz += lprev[j];
                if (k == 0) zz += auxn[j];
                if constexpr (MODE == MODE_HVP) zs[j] = der(zz), zst[1 + PX * lane + j] = val(zz);
                else zs[j] = zz;
            }
        }
        if (last_window) {
            double *ze = sx + 1 + PX * (lane + 1);
#pragma unroll
            for (int j = 0; j < PX; j++) {
                Num zz = j < PF ? lam[j < PF ? j : 0] : 0.0;
                if (S10 && j == 0) zz += lam0 * rex;
                if (S10 && j == 1) zz += lam0 * rey;
                if (j == 10) zz += lam0 * (c.kT * Te);
                if constexpr (MODE == MODE_HVP) {
                    const Num ze_j = zz + auxn[PX + j];
                    ze[j] = der(ze_j), zst[1 + PX * (lane + 1) + j] = val(ze_j);
                } else {
                    ze[j] = zz + aux[PX + j];
                }
            }
        }
        __syncwarp();
        const int cntz = PX * nk + ((k0 + nk == ts) ? PX : 0);
        double *dst = Gb + 1 + (size_t)PX * k0;
        for (int i = lane; i < cntz; i += 32) dst[i] = sx[1 + i];
        if (MODE == MODE_HVP && Zb) {
            double *zdst = Zb + 1 + (size_t)PX * k0;
            for (int i = lane; i < cntz; i += 32) zdst[i] = zst[1 + i];
        }
        __syncwarp();
        return;
    }

    if constexpr (MODE == MODE_COMPACT) {
        // compact G: the warp's windows as NVAR doubles each, contiguous at Gb + R0 + NVAR*k; staged in the
        // tile half a warp at a time (lane stride 31 doubles: conflict-free) and sent as one bulk copy
        double *Gc = Gb + c.R0 + (size_t)NVAR * k0;
#pragma unroll 1
        for (int hf = 0; hf < 2; hf++) {
            if (16 * hf >= nk) break;
            if ((lane >> 4) == hf) {
                double *q = tile + (lane & 15) * NVAR;
#pragma unroll
                for (int i = 0; i < NVAR; i++) q[i] = v[i];
            }
            const int cnt = min(16, nk - 16 * hf) * NVAR;
            double *dst = Gc + (size_t)NVAR * 16 * hf;
            const bool bulkc = ((reinterpret_cast<uintptr_t>(dst) & 15) == 0) && ((cnt & 1) == 0);
            if (bulkc) {
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncwarp();
                if (lane == 0) {
                    bulk_store(dst, tile_s, cnt * 8);
                    bulk_wait_read<0>();
                }
                __syncwarp();
            } else {
                __syncwarp();
                for (int i = lane; i < cnt; i += 32) dst[i] = tile[i];
                __syncwarp();
            }
        }
        return;
    }

    if constexpr (mode_has_records(MODE)) tile_drain(c, tile, tile_s, k0, nk, lane, Gb, tile_mis, v, mdt);
}

// ---- end of a trajectory: F[0], boundary rows, objective-row ends --------------------------------------
//
// Executed by one whole warp.  tT, tp: the trajectory's cost sums; n0 / ne: lane c < 11 holds state c of
// node 0 / node ts.  gl: the trajectory's goal.
template <int FORM, class GoalT>
__device__ __forceinline__ void traj_epilogue(const FgConst &c, const GoalT gl, const int lane, const double dt,
                                              const double tT, const double tp, const double n0,
                                              const double ne, double *__restrict__ Fb,
                                              double *__restrict__ Gb, const int needF, const int needG,
                                              const double dmax, const double dssq, double *__restrict__ Sb,
                                              const int recw = REC) {
    constexpr bool S10 = (FORM == TOLCUDA_FORM_S10);
    const int ts = c.ts;
    double f0 = 0.0, bval = 0.0;  // objective (lane 0) and this lane's boundary-row value
    double *Fbnd = Fb + (c.neF - c.nb);
    double *Gbnd = Gb + c.R0 + (size_t)recw * ts;  // recw = NVAR in the compact layout
    if (recw != REC && needG && lane == 0) Gbnd[c.nbG] = -dt;  // compact rows end with the records' -dt entry
    if constexpr (S10) {
        if (needF) {
            if (lane == 0) Fb[0] = c.half_kT * tT + c.half_kp * tp + c.kdt * dt;  // src/problemS10.cpp:264
            if (lane < PX) {  // src/problemS10.cpp:292-303
                double d = ne - n0;
                if (lane == 5) d = d - 2.0 * M_PI;
                Fbnd[lane] = d;
            }
        }
        if (Sb) {
            f0 = c.half_kT * tT + c.half_kp * tp + c.kdt * dt;
            if (lane < PX) bval = lane == 5 ? ne - n0 - 2.0 * M_PI : ne - n0;
        }
        if (needG) {
            if (lane == 0) Gb[0] = c.kdt;  // src/problemS10.cpp:378-381
            // boundary rows [dt, (0,c), (ts,c)]: the dt entry is uninitialised in the reference
            // (src/problemS10.cpp:397,414) and DEFINED as 0.0 here
            for (int i = lane; i < 3 * PX; i += 32) {
                const int m = i % 3;
                Gbnd[i] = m == 0 ? 0.0 : (m == 1 ? -1.0 : 1.0);
            }
        }
    } else {
        const double x0 = __shfl_sync(0xffffffffu, n0, 0), y0 = __shfl_sync(0xffffffffu, n0, 1);
        const double xf = __shfl_sync(0xffffffffu, ne, 0), yf = __shfl_sync(0xffffffffu, ne, 1);
        const double ddx = xf - x0, ddy = yf - y0;
        const double dist = sqrt(ddx * ddx + ddy * ddy);
        if (needF) {
            if (lane == 0) {
                Fb[0] = c.half_kT * tT + c.kv_ts * dt / dist;  // src/problemG7.cpp:249
                const double gx = gl.xg(c) - x0, gy = gl.yg(c) - y0;   // src/problemG7.cpp:276-294
                const double dmax = sqrt(gx * gx + gy * gy);
                Fbnd[0] = ddx - dist * gl.cos_chid(c);
                Fbnd[1] = ddy - dist * gl.sin_chid(c);
                Fbnd[11] = dist - dmax;
            }
            if (lane >= 2 && lane < PX) Fbnd[lane] = ne - n0;
        }
        if (Sb) {
            const double gx = gl.xg(c) - x0, gy = gl.yg(c) - y0;
            f0 = c.half_kT * tT + c.kv_ts * dt / dist;
            if (lane >= 2 && lane < PX) bval = ne - n0;
            if (lane == 0) bval = ddx - dist * gl.cos_chid(c);
            if (lane == 1) bval = ddy - dist * gl.sin_chid(c);
            if (lane == PX) bval = max_nan(dist - sqrt(gx * gx + gy * gy), 0.0);  // dist <= dmax: only excess counts
        }
        if (needG && lane == 0) {
            // objective row ends, src/problemG7.cpp:343-380 (sic: kp, where cost() uses kv)
            const double d3 = dist * dist * dist;
            const double gx0 = c.kp_ts * dt * ddx / d3, gy0 = c.kp_ts * dt * ddy / d3;
            Gb[0] = c.kp_ts / dist;
            Gb[1] = gx0;
            Gb[2] = gy0;
            Gb[ts + 3] = -gx0;
            Gb[ts + 4] = -gy0;
            // boundary rows, src/problemG7.cpp:404-511
            const double ex = ddx / dist, ey = ddy / dist;
            const double cd = gl.cos_chid(c), sd = gl.sin_chid(c);
            double *p = Gbnd;
            p[0] = 0.0, p[1] = -1.0 + ex * cd, p[2] = ey * cd;
            p[3] = 1.0 - ex * cd, p[4] = -(ey * cd);
            p += 5;
            p[0] = 0.0, p[1] = ex * sd, p[2] = -1.0 + ey * sd;
            p[3] = -(ex * sd), p[4] = 1.0 - ey * sd;
            p += 5;
#pragma unroll
            for (int cidx = 2; cidx < PX; cidx++) {
                p[0] = 0.0, p[1] = -1.0, p[2] = 1.0;
                p += 3;
            }
            p[0] = 0.0, p[1] = -ex, p[2] = -ey, p[3] = ex, p[4] = ey;
        }
    }
    if (Sb) {  // [objective, max |defect|, max |boundary violation|, sum of defect^2]
        const double bmax = warp_max(fabs(bval));
        if (lane == 0) {
            Sb[0] = f0;
            Sb[1] = dmax;
            Sb[2] = bmax;
            Sb[3] = dssq;
        }
    }
}

// ---- matrix-free operators: the rows / columns of J that touch only dt, node 0 and node ts ------------------------
//
// G7's objective-row ends and boundary rows (src/problemG7.cpp:343-380, 404-511) from node 0 / node ts held by
// lanes < 11 of a whole warp, with the expressions of traj_epilogue
template <class Num>
struct G7Ends {
    Num dist, gx0, gy0, ex, ey;
};
template <class Num>
__device__ __forceinline__ G7Ends<Num> g7_ends(const FgConst &c, const Num dt, const Num n0, const Num ne) {
    const Num x0 = shfl(n0, 0), y0 = shfl(n0, 1);
    const Num xf = shfl(ne, 0), yf = shfl(ne, 1);
    const Num ddx = xf - x0, ddy = yf - y0;
    G7Ends<Num> e;
    e.dist = sqrt(ddx * ddx + ddy * ddy);
    const Num d3 = e.dist * e.dist * e.dist;
    e.gx0 = c.kp_ts * dt * ddx / d3, e.gy0 = c.kp_ts * dt * ddy / d3;
    e.ex = ddx / e.dist, e.ey = ddy / e.dist;
    return e;
}

// the trajectory's dt, node 0 and node ts (lanes < 11) as operands of MODE_HVP: with the components of d at the
// same places (the trajectory's row Db)
template <class Num>
struct EndNodes {
    Num dt, n0, ne;
};
template <class Num>
__device__ __forceinline__ EndNodes<Num> end_nodes(const FgConst &c, const int lane, const double dt, const double n0,
                                                   const double ne, const double *__restrict__ Db) {
    if constexpr (std::is_same_v<Num, Dual>) {
        double dn0 = 0.0, dne = 0.0;
        if (lane < PX) dn0 = __ldg(Db + 1 + lane), dne = __ldg(Db + 1 + (size_t)PX * c.ts + lane);
        return {Dual(dt, __ldg(Db)), Dual(n0, dn0), Dual(ne, dne)};
    } else {
        return {dt, n0, ne};
    }
}

// MODE_VJP, before a tile that owns node 0 or node ts: what lambda_0 (G7 objective-row ends) and the boundary rows'
// multipliers add to z at node 0 (aux[0..10]) and node ts (aux[11..21]); executed by the tile's whole warp, aux is
// the warp's own (otherwise unused) record buffer.  Num = Dual (MODE_HVP): the same terms and their derivatives
// along d, as 22 Duals
template <int FORM, class Num = double>
__device__ __forceinline__ void op_aux(const FgConst &c, const int lane, const double dt_in, const double n0_in,
                                       const double ne_in, const double *__restrict__ lamrow, double *aux_out,
                                       const double *__restrict__ Db = nullptr) {
    const EndNodes<Num> en = end_nodes<Num>(c, lane, dt_in, n0_in, ne_in, Db);
    const Num dt = en.dt, n0 = en.n0, ne = en.ne;
    Num *aux = reinterpret_cast<Num *>(aux_out);
    const double lb = lane < c.nb ? __ldg(lamrow + (c.neF - c.nb) + lane) : 0.0;
    Num a0 = -lb, a1 = lb;  // rows [dt: 0, (0,c): -1, (ts,c): +1], src/problemS10.cpp:395-415, src/problemG7.cpp:404-511
    if (FORM == TOLCUDA_FORM_G7) {
        const double lam0 = __ldg(lamrow);
        const G7Ends<Num> e = g7_ends(c, dt, n0, ne);
        const double lb0 = __shfl_sync(0xffffffffu, lb, 0), lb1 = __shfl_sync(0xffffffffu, lb, 1);
        const double lb11 = __shfl_sync(0xffffffffu, lb, 11);
        const double cd = c.cos_chid, sd = c.sin_chid;
        if (lane == 0) {
            a0 = lam0 * e.gx0 + lb0 * (-1.0 + e.ex * cd) + lb1 * (e.ex * sd) + lb11 * (-e.ex);
            a1 = lam0 * (-e.gx0) + lb0 * (1.0 - e.ex * cd) + lb1 * (-(e.ex * sd)) + lb11 * e.ex;
        } else if (lane == 1) {
            a0 = lam0 * e.gy0 + lb0 * (e.ey * cd) + lb1 * (-1.0 + e.ey * sd) + lb11 * (-e.ey);
            a1 = lam0 * (-e.gy0) + lb0 * (-(e.ey * cd)) + lb1 * (1.0 - e.ey * sd) + lb11 * e.ey;
        }
    }
    if (lane < PX) aux[lane] = a0, aux[PX + lane] = a1;
}

// end of a trajectory in the operator modes, one whole warp; tot: the trajectory's sum of the tiles' shares
// (MODE_JVP: objective-row entries times d; MODE_VJP, MODE_HVP: the d/d dt column times lambda; MODE_HVP: totd, the
// derivative of that sum)
template <int FORM, int MODE>
__device__ __forceinline__ void op_epilogue(const FgConst &c, const int lane, const double dt, const double tot,
                                            const double n0, const double ne, double *__restrict__ Fb,
                                            double *__restrict__ Gb, const double totd = 0.0,
                                            const double *__restrict__ Db = nullptr, double *__restrict__ Zb = nullptr) {
    constexpr bool S10 = (FORM == TOLCUDA_FORM_S10);
    const int ts = c.ts;
    if (MODE == MODE_JVP) {  // Fb: y (out), Gb: d (in)
        const double ddt = __ldg(Gb);
        double d0 = 0.0, de = 0.0;
        if (lane < PX) d0 = __ldg(Gb + 1 + lane), de = __ldg(Gb + 1 + (size_t)PX * ts + lane);
        double *ybnd = Fb + (c.neF - c.nb);
        if (S10) {
            if (lane == 0) Fb[0] = c.kdt * ddt + tot;
            if (lane < PX) ybnd[lane] = de - d0;
        } else {
            const G7Ends<double> e = g7_ends(c, dt, n0, ne);
            const double d0x = __shfl_sync(0xffffffffu, d0, 0), d0y = __shfl_sync(0xffffffffu, d0, 1);
            const double dex = __shfl_sync(0xffffffffu, de, 0), dey = __shfl_sync(0xffffffffu, de, 1);
            const double cd = c.cos_chid, sd = c.sin_chid;
            if (lane == 0) {
                Fb[0] = (c.kp_ts / e.dist) * ddt + e.gx0 * d0x + e.gy0 * d0y + tot + (-e.gx0) * dex + (-e.gy0) * dey;
                ybnd[0] = (-1.0 + e.ex * cd) * d0x + (e.ey * cd) * d0y + (1.0 - e.ex * cd) * dex + (-(e.ey * cd)) * dey;
                ybnd[1] = (e.ex * sd) * d0x + (-1.0 + e.ey * sd) * d0y + (-(e.ex * sd)) * dex + (1.0 - e.ey * sd) * dey;
                ybnd[11] = (-e.ex) * d0x + (-e.ey) * d0y + e.ex * dex + e.ey * dey;
            }
            if (lane >= 2 && lane < PX) ybnd[lane] = de - d0;
        }
    } else if constexpr (MODE == MODE_VJP) {  // Fb: lambda (in), Gb: z (out)
        const double lam0 = __ldg(Fb);
        double row0dt = c.kdt;
        if (!S10) row0dt = c.kp_ts / g7_ends(c, dt, n0, ne).dist;
        if (lane == 0) Gb[0] = tot + lam0 * row0dt;
    } else {  // Fb: lambda (in), Gb: w (out), Zb: z (out, optional)
        const EndNodes<Dual> en = end_nodes<Dual>(c, lane, dt, n0, ne, Db);
        const double lam0 = __ldg(Fb);
        Dual row0dt = c.kdt;
        if (!S10) row0dt = c.kp_ts / g7_ends(c, en.dt, en.n0, en.ne).dist;
        const Dual r = Dual(tot, totd) + lam0 * row0dt;
        if (lane == 0) {
            Gb[0] = r.d;
            if (Zb) Zb[0] = r.v;
        }
    }
}

// ---- kernel A: one CTA per run of `per` consecutive trajectories ------------------------------------------------
//
// blockDim.x = 32*ceil(ts/32) (<= MAXT).  Warp w owns windows 32w..32w+31 of every trajectory of the run and
// works on its own after start-up; the cost sums of a trajectory cross warps through shared memory and an
// arrival counter, and the last warp to arrive runs that trajectory's epilogue.  The warp's two x-slice buffers
// form a ring: the slices of the first two trajectories are requested at start-up, the slice of trajectory
// t+2 as soon as trajectory t has left its buffer, so from the second trajectory on neither the CTA launch nor
// the x load is on the critical path, and the record slots' constants are written once per run.  Measured
// (S10 ts=200, B=65,536): per = 1 2.174 ms, 2 2.068, 3 2.098, 4 2.113, 6 2.156, 8 2.185 (longer runs leave a
// longer tail at the end of the grid); per = 2 is the default (tolcuda_set_option "per").
// The body is shared by the instances with the context's goal (fg_cta_kernel) and those with a goal table
// (fg_cta_goals_kernel, GOALS: goals = row 0 of the launch's rows of the table).
constexpr int MAXPER = 4;
// MODE_HVP instances of kernel A: CTAs of 128 threads per SM (256 threads: half as many).  Measured on one B200
// (1,000 W; profiles/r4_opbench_hvp.txt): 4 (128 registers, 130-1,030 bytes of spill) 1.91 ms on S10 ts=200 at
// B=65,536 and 80 us on G7 ts=100 at B=4,096; 3 (168 / 255 registers) 2.34 ms / 90.5 us; 2 (255 registers, no
// spill but 8 warps per SM) 2.34 ms / 109 us: the dual arithmetic wants warps more than registers
constexpr int HVP_MINB = 4;
template <int FORM, int WIND, int MAXT, int MINB, int MODE, bool LOOP, bool GOALS>
__device__ __forceinline__ void fg_cta_body(const FgConst &c, int nrun, int per_arg, const double *__restrict__ x, long ldx,
                                            double *__restrict__ F, long ldF, double *__restrict__ G, long ldG, int needF,
                                            int needG, int flow, double *__restrict__ S, long ldS,
                                            const double *__restrict__ goals, const double *__restrict__ dm = nullptr,
                                            long ldd = 0, double *__restrict__ zm = nullptr, long ldz = 0) {
    pdl_release();
    constexpr bool SUMM = mode_has_summary(MODE);
    extern __shared__ __align__(16) double smem[];
    constexpr bool OP = mode_is_op(MODE);
    constexpr bool HVP = MODE == MODE_HVP;
    __shared__ double red[MAXPER][SUMM ? 4 : 2][32];
    __shared__ int arrivals[MAXPER];
    const int ts = c.ts;
    const int tid = thread_index();
    // the warp index through a shuffle from lane 0: provably warp-uniform, so everything derived from it
    // (k0, slice and record addresses, the bulk copies' operands) can live on the uniform datapath
    const int lane = tid & 31, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), nwarps = blockDim.x >> 5;
    // what __launch_bounds__ tells the kernel; the body is optimised before it is inlined there, and without this
    // the loops over the warps would be compiled for any block size
    __builtin_assume(blockDim.x <= MAXT);
    // LOOP = false is the straight-line instance for runs of one trajectory (small batches): ptxas then
    // hoists the address arithmetic the loop form has to re-derive per trajectory (7 % fewer instructions)
    const int per = LOOP ? per_arg : 1;
    const int nslice = per > 1 ? 2 : 1;  // slice buffers per warp (the host sizes the dynamic shared memory alike)
    double *wsm = smem + (size_t)warp * (nslice * SX_LEN + tile_len_of(MODE));
    double *tile = wsm + nslice * SX_LEN;
    const uint32_t wsm_s = smem_addr(wsm), tile_s = wsm_s + 8 * nslice * SX_LEN;
    // CTAs [0, nrun) own runs of `per` consecutive trajectories, the CTAs behind them one trajectory each: the grid
    // ends on short CTAs, so its tail drains in half the time (launch_cta_as sizes the two parts)
    const int bid = blockIdx.x;
    const bool run = LOOP && bid < nrun;
    const size_t b0 = LOOP ? (run ? (size_t)per * bid : (size_t)per * nrun + (size_t)(bid - nrun)) : (size_t)bid;
    const int ntraj = run ? per : 1;
    const int k0 = 32 * warp;
    const int nk = min(32, ts - k0);
    const int cnt = 1 + PX * (nk + 1);           // doubles of a slice
    const double *xw = x + b0 * ldx + (size_t)PX * k0;  // this warp's slice of the run's first trajectory
    slice_prefetch(wsm_s, xw, cnt, lane);
    if (GOALS) goal_prefetch<FORM>(wsm_s, goals + TOLCUDA_GOAL_LD * b0, lane);
    cp_async_commit();
    // dt, node 0 and node ts of a trajectory are requested one trajectory ahead, like its slice
    double dt_nx = __ldg(xw - (size_t)PX * k0), n0_nx = 0.0, ne_nx = 0.0;
    if (lane < PX) {
        n0_nx = __ldg(xw - (size_t)PX * k0 + 1 + lane);
        ne_nx = __ldg(xw - (size_t)PX * k0 + (size_t)PX * ts + 1 + lane);
    }
    // alignment of this warp's records in the run's first trajectory (tile_eval re-initialises the slots if a
    // later trajectory's differs: odd leading dimension)
    int tile_mis = 0;
    if (mode_has_records(MODE)) {
        tile_mis = (int)(reinterpret_cast<uintptr_t>(G + b0 * ldG + c.R0 + (size_t)REC * k0) >> 3) & 1;
        if (needG) tile_init(tile, lane, tile_mis);
    }
    if (tid < MAXPER) arrivals[tid] = 0;
    __syncthreads();
#pragma unroll 1
    for (int t = 0; t < ntraj; t++) {
        const size_t b = b0 + t;
        const int slot = t & 1;
        const double dt = dt_nx, n0 = n0_nx, ne = ne_nx;
        // the next trajectory's slice goes to the other buffer (whose previous user, trajectory t-1, is done)
        if (t + 1 < ntraj) {
            const double *xn = xw + (t + 1) * ldx;
            slice_prefetch(wsm_s + 8 * (slot ^ 1) * SX_LEN, xn, cnt, lane);
            if (GOALS) {
                // G7: the epilogue of trajectory t-1 (lane 0 alone, without G) has read its goal values in that buffer
                if (FORM != TOLCUDA_FORM_S10) __syncwarp();
                goal_prefetch<FORM>(wsm_s + 8 * (slot ^ 1) * SX_LEN, goals + TOLCUDA_GOAL_LD * (b + 1), lane);
            }
            dt_nx = __ldg(xn - (size_t)PX * k0);
            if (lane < PX) {
                n0_nx = __ldg(xn - (size_t)PX * k0 + 1 + lane);
                ne_nx = __ldg(xn - (size_t)PX * k0 + (size_t)PX * ts + 1 + lane);
            }
        }
        cp_async_commit();
        cp_async_wait<1>();
        __syncwarp();
        double *Fb = F + b * ldF, *Gb = G + b * ldG;
        const double *Db = HVP ? dm + b * ldd : nullptr;
        double *Zb = HVP && zm ? zm + b * ldz : nullptr;
        TileSums tsum;
        if ((MODE == MODE_VJP || HVP) && (k0 == 0 || k0 + nk == ts)) {  // the warps that own node 0 / node ts (warp-uniform)
            op_aux<FORM, std::conditional_t<HVP, Dual, double>>(c, lane, dt, n0, ne, Fb, tile, Db);
            __syncwarp();
        }
        tile_eval<FORM, WIND, MODE, GOALS>(c, wsm + slot * SX_LEN, tile, tile_s, dt, k0, nk, lane, Fb, Gb, needF, needG, tsum,
                                    !OP && t == 0 && (flow & FLOW_WAIT), tile_mis, OP ? tile : nullptr, Db, Zb);
        __syncwarp();
        const double sumT = warp_sum(tsum.sumT);
        const double sump = FORM == TOLCUDA_FORM_S10 || HVP ? warp_sum(tsum.sump) : 0.0;
        const double wdmax = SUMM ? warp_max(tsum.dmax) : 0.0, wdssq = SUMM ? warp_sum(tsum.dssq) : 0.0;
        int last = 0;
        if (lane == 0) {
            red[t][0][warp] = sumT;
            red[t][1][warp] = sump;
            if (SUMM) {
                red[t][SUMM ? 2 : 0][warp] = wdmax;
                red[t][SUMM ? 3 : 0][warp] = wdssq;
            }
            __threadfence_block();
            last = (atomicAdd(&arrivals[t], 1) == nwarps - 1);
        }
        last = __shfl_sync(0xffffffffu, last, 0);
        if (last) {
            __threadfence_block();
            const volatile double *vred = &red[t][0][0];
            double tT = 0.0, tp = 0.0, dmax = 0.0, dssq = 0.0;
            for (int w = 0; w < nwarps; w++) {  // fixed order: deterministic
                tT += vred[w];
                tp += vred[32 + w];
                if (SUMM) {
                    dmax = max_nan(dmax, vred[64 + w]);
                    dssq += vred[96 + w];
                }
            }
            if (OP)
                op_epilogue<FORM, MODE>(c, lane, dt, tT, n0, ne, Fb, Gb, tp, Db, Zb);
            else
                traj_epilogue<FORM>(c, Goal<FORM, GOALS>{wsm + slot * SX_LEN + GOAL_SX}, lane, dt, tT, tp, n0, ne, Fb,
                                           Gb, needF, mode_is_fonly(MODE) ? 0 : needG, dmax, dssq,
                                           SUMM ? S + b * ldS : nullptr, MODE == MODE_COMPACT ? NVAR : REC);
        }
    }
    cp_async_wait<0>();
}

template <int FORM, int WIND, int MAXT, int MINB, int MODE, bool LOOP>
__global__ void __launch_bounds__(MAXT, MINB)
fg_cta_kernel(const __grid_constant__ FgConst c, int nrun, int per_arg, const double *__restrict__ x, long ldx,
               double *__restrict__ F, long ldF, double *__restrict__ G, long ldG, int needF, int needG, int flow,
               double *__restrict__ S, long ldS) {
    fg_cta_body<FORM, WIND, MAXT, MINB, MODE, LOOP, false>(c, nrun, per_arg, x, ldx, F, ldF, G, ldG, needF, needG, flow, S,
                                                           ldS, nullptr);
}

// MODE_HVP: lam / w in the F / G places, then d and the optional z
template <int FORM, int WIND, int MAXT, int MINB, bool LOOP>
__global__ void __launch_bounds__(MAXT, MINB)
fg_cta_hvp_kernel(const __grid_constant__ FgConst c, int nrun, int per_arg, const double *__restrict__ x, long ldx,
                  double *__restrict__ lam, long ldl, double *__restrict__ w, long ldw, const double *__restrict__ d,
                  long ldd, double *__restrict__ z, long ldz) {
    fg_cta_body<FORM, WIND, MAXT, MINB, MODE_HVP, LOOP, false>(c, nrun, per_arg, x, ldx, lam, ldl, w, ldw, 1, 1, 0, nullptr, 0,
                                                               nullptr, d, ldd, z, ldz);
}

template <int FORM, int WIND, int MAXT, int MINB, int MODE, bool LOOP>
__global__ void __launch_bounds__(MAXT, MINB)
fg_cta_goals_kernel(const __grid_constant__ FgConst c, int nrun, int per_arg, const double *__restrict__ x, long ldx,
                    double *__restrict__ F, long ldF, double *__restrict__ G, long ldG, int needF, int needG, int flow,
                    double *__restrict__ S, long ldS, const double *__restrict__ goals) {
    fg_cta_body<FORM, WIND, MAXT, MINB, MODE, LOOP, true>(c, nrun, per_arg, x, ldx, F, ldF, G, ldG, needF, needG, flow, S,
                                                          ldS, goals);
}

// ---- kernel L: one CTA per trajectory of any length -------------------------------------------------------------
//
// Up to 8 warps (the host picks the count that balances the tiles); warp w walks tiles w, w+W, w+2W, ... of the trajectory, keeping its share of the cost
// sums in registers, while the slice of its next tile is already in flight into the other slice buffer; the sums
// cross warps once per trajectory as in kernel A.  Serves trajectories longer than 256 windows (and any
// trajectory with tolcuda_set_option(h, "kernel", 2)).  All warps of a CTA write the same G row, as in kernel A: the earlier
// persistent-warp kernel (one whole trajectory per warp, 16 x 148 rows being written at a time) reached 0.82 of
// the roofline on S10 ts=200 where kernel A reaches 0.98.
// The body is shared by fg_long_kernel and fg_long_goals_kernel, as kernel A's.
constexpr int LWARPS = 8;
template <int FORM, int WIND, int MODE, bool GOALS>
__device__ __forceinline__ void fg_long_body(const FgConst &c, const double *__restrict__ x, long ldx,
                                             double *__restrict__ F, long ldF, double *__restrict__ G, long ldG, int needF,
                                             int needG, int flow, double *__restrict__ S, long ldS,
                                             const double *__restrict__ goals, const double *__restrict__ dm = nullptr,
                                             long ldd = 0, double *__restrict__ zm = nullptr, long ldz = 0) {
    pdl_release();
    constexpr bool SUMM = mode_has_summary(MODE);
    extern __shared__ __align__(16) double smem[];
    constexpr bool OP = mode_is_op(MODE);
    constexpr bool HVP = MODE == MODE_HVP;
    __shared__ double red[SUMM ? 4 : 2][32];
    __shared__ int arrivals;
    const int ts = c.ts;
    const int nt = (ts + 31) >> 5;
    const int tid = thread_index();
    const int lane = tid & 31, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), nwarps = blockDim.x >> 5;
    __builtin_assume(blockDim.x <= LWARPS * 32);  // as in fg_cta_body
    double *wsm = smem + (size_t)warp * WARP_SMEM_B;
    double *tile = wsm + 2 * SX_LEN;
    const uint32_t wsm_s = smem_addr(wsm), tile_s = wsm_s + 8 * 2 * SX_LEN;
    const size_t b = blockIdx.x;
    const double *xb = x + b * ldx;
    double *Fb = F + b * ldF, *Gb = G + b * ldG;
    const double *Db = HVP ? dm + b * ldd : nullptr;
    double *Zb = HVP && zm ? zm + b * ldz : nullptr;
    slice_prefetch(wsm_s, xb + (size_t)PX * 32 * warp, 1 + PX * (min(32, ts - 32 * warp) + 1), lane);
    // S10: the goal values go into both slice buffers with the first slice; the later slices leave them alone
    if (GOALS && FORM == TOLCUDA_FORM_S10) {
        goal_prefetch<FORM>(wsm_s, goals + TOLCUDA_GOAL_LD * b, lane);
        goal_prefetch<FORM>(wsm_s + 8 * SX_LEN, goals + TOLCUDA_GOAL_LD * b, lane);
    }
    cp_async_commit();
    const double dt = __ldg(xb);
    double n0 = 0.0, ne = 0.0;
    if (lane < PX) {
        n0 = __ldg(xb + 1 + lane);
        ne = __ldg(xb + (size_t)PX * ts + 1 + lane);
    }
    int tile_mis = 0;
    if (mode_has_records(MODE)) {
        tile_mis = (int)(reinterpret_cast<uintptr_t>(Gb + c.R0) >> 3) & 1;  // REC*k0 is even
        if (needG) tile_init(tile, lane, tile_mis);
    }
    if (tid == 0) arrivals = 0;
    __syncthreads();
    double accT = 0.0, accp = 0.0, accm = 0.0, accq = 0.0;
    int slot = 0;
#pragma unroll 1
    for (int j = warp; j < nt; j += nwarps) {
        const int jn = j + nwarps;
        if (jn < nt)
            slice_prefetch(wsm_s + 8 * (slot ^ 1) * SX_LEN, xb + (size_t)PX * 32 * jn, 1 + PX * (min(32, ts - 32 * jn) + 1), lane);
        cp_async_commit();
        cp_async_wait<1>();
        __syncwarp();
        TileSums tsum;
        if ((MODE == MODE_VJP || HVP) && (j == 0 || j == nt - 1)) {  // the tiles that own node 0 / node ts (warp-uniform)
            op_aux<FORM, std::conditional_t<HVP, Dual, double>>(c, lane, dt, n0, ne, Fb, tile, Db);
            __syncwarp();
        }
        tile_eval<FORM, WIND, MODE, GOALS>(c, wsm + slot * SX_LEN, tile, tile_s, dt, 32 * j, min(32, ts - 32 * j), lane, Fb, Gb,
                                    needF, needG, tsum, !OP && j == warp && (flow & FLOW_WAIT), tile_mis, OP ? tile : nullptr,
                                    Db, Zb);
        __syncwarp();
        accT += tsum.sumT;
        accp += tsum.sump;
        accm = max_nan(accm, tsum.dmax);
        accq += tsum.dssq;
        slot ^= 1;
    }
    cp_async_wait<0>();
    const double sumT = warp_sum(accT);
    const double sump = FORM == TOLCUDA_FORM_S10 || HVP ? warp_sum(accp) : 0.0;
    const double wdmax = SUMM ? warp_max(accm) : 0.0, wdssq = SUMM ? warp_sum(accq) : 0.0;
    int last = 0;
    if (lane == 0) {
        red[0][warp] = sumT;
        red[1][warp] = sump;
        if (SUMM) {
            red[SUMM ? 2 : 0][warp] = wdmax;
            red[SUMM ? 3 : 0][warp] = wdssq;
        }
        __threadfence_block();
        last = (atomicAdd(&arrivals, 1) == nwarps - 1);
    }
    last = __shfl_sync(0xffffffffu, last, 0);
    if (!last) return;
    __threadfence_block();
    const volatile double *vred = &red[0][0];
    double tT = 0.0, tp = 0.0, dmax = 0.0, dssq = 0.0;
    for (int w = 0; w < nwarps; w++) {  // fixed order: deterministic
        tT += vred[w];
        tp += vred[32 + w];
        if (SUMM) {
            dmax = max_nan(dmax, vred[64 + w]);
            dssq += vred[96 + w];
        }
    }
    if (OP)
        op_epilogue<FORM, MODE>(c, lane, dt, tT, n0, ne, Fb, Gb, tp, Db, Zb);
    else
        traj_epilogue<FORM>(c, Goal<FORM, GOALS, true>{GOALS ? goals + TOLCUDA_GOAL_LD * b : nullptr}, lane, dt, tT, tp, n0, ne, Fb, Gb, needF,
                                   mode_is_fonly(MODE) ? 0 : needG, dmax, dssq, SUMM ? S + b * ldS : nullptr,
                                   MODE == MODE_COMPACT ? NVAR : REC);
}

template <int FORM, int WIND, int MODE>
__global__ void __launch_bounds__(LWARPS * 32, 2)
fg_long_kernel(const __grid_constant__ FgConst c, const double *__restrict__ x, long ldx,
               double *__restrict__ F, long ldF, double *__restrict__ G, long ldG, int needF, int needG, int flow,
               double *__restrict__ S, long ldS) {
    fg_long_body<FORM, WIND, MODE, false>(c, x, ldx, F, ldF, G, ldG, needF, needG, flow, S, ldS, nullptr);
}

// MODE_HVP, as fg_cta_hvp_kernel
constexpr int HVP_LMINB = 1;
template <int FORM, int WIND>
__global__ void __launch_bounds__(LWARPS * 32, HVP_LMINB)
fg_long_hvp_kernel(const __grid_constant__ FgConst c, const double *__restrict__ x, long ldx, double *__restrict__ lam,
                   long ldl, double *__restrict__ w, long ldw, const double *__restrict__ d, long ldd,
                   double *__restrict__ z, long ldz) {
    fg_long_body<FORM, WIND, MODE_HVP, false>(c, x, ldx, lam, ldl, w, ldw, 1, 1, 0, nullptr, 0, nullptr, d, ldd, z, ldz);
}

template <int FORM, int WIND, int MODE>
__global__ void __launch_bounds__(LWARPS * 32, 2)
fg_long_goals_kernel(const __grid_constant__ FgConst c, const double *__restrict__ x, long ldx,
                     double *__restrict__ F, long ldF, double *__restrict__ G, long ldG, int needF, int needG, int flow,
                     double *__restrict__ S, long ldS, const double *__restrict__ goals) {
    fg_long_body<FORM, WIND, MODE, true>(c, x, ldx, F, ldF, G, ldG, needF, needG, flow, S, ldS, goals);
}

// one launch, optionally as a programmatic dependent of the launch before it on the stream (FgLaunch::pdl)
template <class Kern, class... Args>
cudaError_t launch_kernel(Kern kern, const int grid, const int nthr, const size_t smem, const FgLaunch &L, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid), cfg.blockDim = dim3((unsigned)nthr);
    cfg.dynamicSmemBytes = smem, cfg.stream = L.stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at, cfg.numAttrs = L.pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, args...);
}

// lets KERN use smem bytes of dynamic shared memory on the launch's device.  The attribute is per device, so the cache of
// what has been set is too (tolbatch drives one device per thread), and one per kernel instance (KERN).
template <auto KERN>
cudaError_t reserve_smem(const FgLaunch &L, const size_t smem) {
    static std::atomic<size_t> configured[MAX_DEVICES];
    std::atomic<size_t> &done = configured[L.device & (MAX_DEVICES - 1)];
    if (smem > done.load(std::memory_order_acquire)) {
        cudaError_t e = cudaFuncSetAttribute(KERN, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        done.store(smem, std::memory_order_release);
    }
    return cudaSuccess;
}

template <int FORM, int WIND, int MAXT, int MINB, int MODE, bool LOOP, bool GOALS>
cudaError_t launch_cta_as(const FgLaunch &L, const int per, const int nsingle) {
    constexpr auto kern = [] {
        if constexpr (MODE == MODE_HVP) return fg_cta_hvp_kernel<FORM, WIND, MAXT, MINB, LOOP>;
        else if constexpr (GOALS) return fg_cta_goals_kernel<FORM, WIND, MAXT, MINB, MODE, LOOP>;
        else return fg_cta_kernel<FORM, WIND, MAXT, MINB, MODE, LOOP>;
    }();
    const int nthr = 32 * ((L.c->ts + 31) / 32);
    const size_t smem = sizeof(double) * (size_t)(nthr / 32) * ((per > 1 ? 2 : 1) * SX_LEN + tile_len_of(MODE));
    if (cudaError_t e = reserve_smem<kern>(L, smem)) return e;
    const int nrun = LOOP ? (L.B - nsingle) / per : 0;  // nsingle makes this exact (launch_cta)
    const int grid = LOOP ? nrun + nsingle : L.B;
    if constexpr (MODE == MODE_HVP)
        return launch_kernel(kern, grid, nthr, smem, L, *L.c, nrun, per, L.x, L.ldx, L.F, L.ldF, L.G, L.ldG, L.D, L.ldD,
                             L.Z, L.ldZ);
    else if constexpr (GOALS)
        return launch_kernel(kern, grid, nthr, smem, L, *L.c, nrun, per, L.x, L.ldx, L.F, L.ldF, L.G, L.ldG, L.needF,
                             L.needG, L.pdl == 1 ? FLOW_WAIT : 0, L.S, L.ldS, L.goals);
    else
        return launch_kernel(kern, grid, nthr, smem, L, *L.c, nrun, per, L.x, L.ldx, L.F, L.ldF, L.G, L.ldG, L.needF,
                             L.needG, L.pdl == 1 ? FLOW_WAIT : 0, L.S, L.ldS);
}

// Runs of `per` trajectories per CTA pay off once the grid is many waves deep (the x load and the CTA launch
// leave the critical path, the slots' constants are written once per run); small batches keep one trajectory
// per CTA (more CTAs to spread over the SMs, and the cheaper straight-line instance).  A grid of runs ends on
// `tail` waves of single-trajectory CTAs: when the runs are exhausted the SMs' CTA slots free up over one run's
// duration, and short CTAs fill them to a common end instead of leaving half of them idle for a whole run.
template <int FORM, int WIND, int MAXT, int MINB, int MODE, bool GOALS>
cudaError_t launch_cta(const FgLaunch &L) {
    int per = L.per < 1 ? 1 : (L.per > MAXPER ? MAXPER : L.per);
    if (L.per_auto && L.B < L.per_min_waves * MINB * L.sm_count) per = 1;
    if (per == 1) return launch_cta_as<FORM, WIND, MAXT, MINB, MODE, false, GOALS>(L, 1, 0);
    long nsingle = (long)(L.tail_waves_x4 * MINB * L.sm_count) / 4;
    if (nsingle > L.B) nsingle = L.B;
    nsingle += (L.B - nsingle) % per;
    return launch_cta_as<FORM, WIND, MAXT, MINB, MODE, true, GOALS>(L, per, (int)nsingle);
}

template <int FORM, int WIND, int MODE, bool GOALS>
cudaError_t launch_long(const FgLaunch &L) {
    constexpr auto kern = [] {
        if constexpr (MODE == MODE_HVP) return fg_long_hvp_kernel<FORM, WIND>;
        else if constexpr (GOALS) return fg_long_goals_kernel<FORM, WIND, MODE>;
        else return fg_long_kernel<FORM, WIND, MODE>;
    }();
    // as many warps (<= 8) as give every warp the same number of tiles, give or take one: 10 tiles -> 5 warps x 2
    const int nt = (L.c->ts + 31) / 32;
    const int rounds = (nt + LWARPS - 1) / LWARPS;
    int nthr = 32 * ((nt + rounds - 1) / rounds);
    if (L.lwarps > 0) nthr = 32 * (L.lwarps < nt ? L.lwarps : nt);  // tolcuda_set_option "lwarps"
    const size_t smem = sizeof(double) * (size_t)(nthr / 32) * WARP_SMEM_B;
    if (cudaError_t e = reserve_smem<kern>(L, smem)) return e;
    if constexpr (MODE == MODE_HVP)
        return launch_kernel(kern, L.B, nthr, smem, L, *L.c, L.x, L.ldx, L.F, L.ldF, L.G, L.ldG, L.D, L.ldD, L.Z, L.ldZ);
    else if constexpr (GOALS)
        return launch_kernel(kern, L.B, nthr, smem, L, *L.c, L.x, L.ldx, L.F, L.ldF, L.G, L.ldG, L.needF, L.needG,
                             L.pdl == 1 ? FLOW_WAIT : 0, L.S, L.ldS, L.goals);
    else
        return launch_kernel(kern, L.B, nthr, smem, L, *L.c, L.x, L.ldx, L.F, L.ldF, L.G, L.ldG, L.needF, L.needG,
                             L.pdl == 1 ? FLOW_WAIT : 0, L.S, L.ldS);
}


template <int FORM, int WIND, int MODE, bool GOALS>
cudaError_t launch_sel(const FgLaunch &L) {
    const int ts = L.c->ts;
    if constexpr (mode_is_fonly(MODE)) {
        // kernel A only (launch_any sends ts <= 256 here).  64 registers: 32 warps / SM at ts <= 128, 28 at ts = 200
        if (ts <= 128) return launch_cta<FORM, WIND, 128, 8, MODE, GOALS>(L);
        return launch_cta<FORM, WIND, 256, 4, MODE, GOALS>(L);
    } else {
        // Kernel A needs the whole trajectory in one CTA with one tile per warp: ts <= 256.  Longer trajectories,
        // and L.kernel == 2, take kernel L, whose warps walk several tiles each (any ts).
        if (L.kernel == 2 || ts > 256) return launch_long<FORM, WIND, MODE, GOALS>(L);
        if constexpr (MODE == MODE_HVP) {
            if (ts <= 128) return launch_cta<FORM, WIND, 128, HVP_MINB, MODE, GOALS>(L);
            return launch_cta<FORM, WIND, 256, HVP_MINB / 2, MODE, GOALS>(L);
        } else {
            if (ts <= 128) return launch_cta<FORM, WIND, 128, 4, MODE, GOALS>(L);         // 128 registers, 16 warps / SM
            return launch_cta<FORM, WIND, 256, 2, MODE, GOALS>(L);                      // 128 registers, 14-16 warps / SM
        }
    }
}

// the per-trajectory summary is a separate instantiation so that plain F/G launches pay nothing for it; so is a
// goal table (GOALS), and the matrix-free modes have no instances with one
template <int FORM, int WIND, bool GOALS>
cudaError_t launch_flavour(const FgLaunch &L) {
    if (L.compact) return launch_sel<FORM, WIND, MODE_COMPACT, GOALS>(L);
    if (!L.needG && L.kernel != 2 && L.c->ts <= 256)
        return L.S ? launch_sel<FORM, WIND, MODE_FSUMM, GOALS>(L) : launch_sel<FORM, WIND, MODE_FONLY, GOALS>(L);
    return L.S ? launch_sel<FORM, WIND, MODE_SUMMARY, GOALS>(L) : launch_sel<FORM, WIND, MODE_PLAIN, GOALS>(L);
}

template <int FORM, int WIND>
cudaError_t launch_any(const FgLaunch &L) {
    if (L.op && L.goals) return cudaErrorInvalidValue;
    if (L.op == 1) return launch_sel<FORM, WIND, MODE_JVP, false>(L);
    if (L.op == 2) return launch_sel<FORM, WIND, MODE_VJP, false>(L);
    if (L.op == 3) return launch_sel<FORM, WIND, MODE_HVP, false>(L);
    return L.goals ? launch_flavour<FORM, WIND, true>(L) : launch_flavour<FORM, WIND, false>(L);
}

}  // namespace

cudaError_t fg_launch(const FgLaunch &L) {
    if (L.B <= 0) return cudaSuccess;
    if (!L.c || L.c->ts < 1) return cudaErrorInvalidValue;
    if (L.c->form == TOLCUDA_FORM_S10) {
        if (L.c->wind == 1) return launch_any<TOLCUDA_FORM_S10, 1>(L);
        if (L.c->wind == 0) return launch_any<TOLCUDA_FORM_S10, 0>(L);
        if (L.c->wind == 3) return launch_any<TOLCUDA_FORM_S10, 3>(L);
    } else if (L.c->form == TOLCUDA_FORM_G7) {
        if (L.c->wind == 1) return launch_any<TOLCUDA_FORM_G7, 1>(L);
        if (L.c->wind == 0) return launch_any<TOLCUDA_FORM_G7, 0>(L);
        if (L.c->wind == 3) return launch_any<TOLCUDA_FORM_G7, 3>(L);
    }
    return cudaErrorInvalidValue;
}
