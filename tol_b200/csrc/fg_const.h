// Constants of one tolcuda context, built once at create time.  Every launch hands them to the kernel
// as a `const __grid_constant__` parameter, i.e. they live in the constant bank and are used as
// immediate constant operands (no registers, no loads).
//
// They replace the reference's `aircraft ac`, `gain gn`, `snopt sn` members and goal fields that
// every gradient call re-reads (reference include/problem.h:50-53,81-83, include/parameters.h:22-74).
// Products of constants are stored pre-multiplied ONLY where the reference's own left-to-right
// association forms exactly that product (e.g. `rho*ac.SS*Va...` starts with (rho*SS)), so the
// kernels reproduce the reference's rounding sequence.
#ifndef TOLCUDA_FG_CONST_H_
#define TOLCUDA_FG_CONST_H_

#define TOLCUDA_PX 11      /* numinp,    problems/<M>/snopt.param line 3 */
#define TOLCUDA_PF 8       /* numstates, problems/<M>/snopt.param line 4 */
#define TOLCUDA_REC 104    /* G values per collocation window: 8 defect rows x 13 columns */
#define TOLCUDA_NVAR 31    /* of which depend on x (two more are -dt, the rest 0 or +-1) */
/* doubles per row of a context's goal table (tolcuda_set_goals): xg, yg, rg, cos_chid, sin_chid, 3 unused; 64 bytes */
#define TOLCUDA_GOAL_LD 8

#ifdef __CUDACC__
#define TOLCUDA_HD __host__ __device__
#else
#define TOLCUDA_HD
#endif

// THE table of a window's Jacobian record (row s = p / 13 of the 8 defect rows, column j = p % 13: 0 = dt,
// 1..11 = component j-1 of node k, 12 = component s of node k+1; reference src/problem.cpp:1074-1192, 1204).
// What record position p holds: >= 0: index into the window's TOLCUDA_NVAR x-dependent values, in coordinate
// order; -1: 0.0; -2: +1.0; -3: -1.0; -4: -dt.  Every user -- the kernels' record slots (fg_kernels.cu), the
// host expansion of compact rows (compact.cpp) and the device expansion (expand_kernel.cu) -- derives its
// layout from this one function.
TOLCUDA_HD constexpr int tolcuda_rec_kind(int p) {
    constexpr int pos[TOLCUDA_NVAR] = {0,  4,  5,  6,  13, 17, 18, 19, 26, 30, 31, 39, 43, 44, 45, 47,
                                       50, 52, 56, 57, 58, 59, 60, 65, 69, 70, 71, 72, 73, 78, 91};
    for (int i = 0; i < TOLCUDA_NVAR; i++)
        if (pos[i] == p) return i;
    if (p == 1 || p == 15 || p == 29 || p == 85 || p == 99) return -3;  // d/d(own state) of rows F1-F3, F7, F8
    if (p % 13 == 12) return -2;                                        // d/d(state s at node k+1)
    if (p == 87 || p == 101) return -4;                                 // d/d(dphi), d/d(dCL) of rows F7, F8
    return -1;
}

struct FgConst {
    int form, ts, wind, nb;
    int n, neF, neG;
    int R0;    // length of the objective-row block = G offset of window 0's record
    int nbG;   // length of the boundary block (33 for S10, 42 for G7)
    int pad_;
    double mm;       // ac.mm
    double SS;       // ac.SS
    double rho;      // include/problem.h:73
    double g;        // include/problem.h:72
    double Cd0;      // ac.Cd0
    double rhoSS;    // rho*ac.SS
    double ARpiee;   // ac.AR*M_PI*ac.ee
    double ARpieemm; // ac.AR*M_PI*ac.ee*ac.mm
    double twomm;    // 2.0*ac.mm
    double r_mm, r_twomm, r_ARpiee, r_ARpieemm;  // correctly rounded reciprocals of the four above
    double kT, kp, kdt;
    double half_kT;  // 0.5*gn.kT (== gn.kT*0.5)
    double half_kp;  // 0.5*gn.kp
    double kv_ts;    // gn.kv*sn.ts
    double kp_ts;    // gn.kp*sn.ts
    double xg, yg, rg;
    double cos_chid, sin_chid; // cos/sin of chi_d = atan2(yg - yi, xg - xi), src/problemG7.cpp:524
    double wind_Wxz;           // dWx_dz = -dv_dz = -(-Vref/href), src/problem.cpp:524,975
    // wind model 3: the cached wind cube (device pointers), src/problem.cpp:443-459, 544-695
    int grid_ne, grid_nn, grid_nu, pad2_;
    const double *grid_x, *grid_y, *grid_z;  // cache[i][0][0].x, cache[0][j][0].y, cache[0][0][k].z
    const double *grid_v;                    // cache[i][j][k].v, i-major
    double datum[3];                         // EastFromDatum, NorthFromDatum, UpFromDatum
    double spacing[3];                       // xspacing, yspacing, zspacing
};

#endif
