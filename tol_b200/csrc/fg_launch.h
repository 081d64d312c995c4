// Host-side launch interface of fg_kernels.cu (internal to libtolcuda).
#ifndef TOLCUDA_FG_LAUNCH_H_
#define TOLCUDA_FG_LAUNCH_H_

#include <cuda_runtime.h>

#include "fg_const.h"

#define TOLCUDA_FORM_G7 7
#define TOLCUDA_FORM_S10 10

struct FgLaunch {
    const FgConst *c;  // the context's constants; passed by value as a __grid_constant__ parameter
    int B;
    const double *x;
    long ldx;
    double *F;
    long ldF;
    double *G;
    long ldG;
    int needF, needG;
    double *S;  // optional per-trajectory summary [B][ldS >= 4]: objective, max|defect|, max|boundary|, sum defect^2
    long ldS;
    int op;  // 0: F/G; 1: y = J d (F receives y [neF], G holds d [n]); 2: z = J^T lambda (F holds lambda [neF], G receives z [n]);
             // 3: w = D_x[J^T lambda] d (F holds lambda [neF], G receives w [n], D holds d [n], Z receives z [n] or is NULL)
    const double *D;  // op 3: d
    long ldD;
    double *Z;        // op 3: z = J^T lambda, optional
    long ldZ;
    int compact;  // G/ldG address the compact layout [R0 | 31 per window | boundary block] (host-pointer path)
    int kernel;    // 0/1 = kernel A (CTA per run of trajectories), 2 = kernel L (CTA per trajectory, tile loop; any ts)
    int lwarps;    // kernel L: warps per CTA (0: the count that balances the tiles)
    int per;       // kernel A: trajectories per CTA (1..4)
    int per_auto;  // 1: small batches (fewer than per_min_waves waves of CTAs) use 1 regardless of `per`
    int per_min_waves;   // kernel A: batches below this many waves of single-trajectory CTAs run one trajectory per CTA
    int tail_waves_x4;   // kernel A with runs: quarter-waves of single-trajectory CTAs the grid ends on
    int pdl;       // 0: ordinary launch; 1: programmatic dependent launch, the kernel waits for the preceding launch on
                   // the stream before its first store; 2: the same without the wait (outputs disjoint from the
                   // preceding launch's reads and writes).  Never set for op != 0 (d / lambda are read early).
    const double *goals;  // NULL: every trajectory has the context's goal; else trajectory b's goal is the row
                          // goals + TOLCUDA_GOAL_LD*b of a device goal table (op == 0 only)
    int sm_count;  // SMs of the device
    int device;    // CUDA device ordinal the launch goes to (the current device)
    cudaStream_t stream;
};

// enqueue one batched F/G evaluation; device pointers
cudaError_t fg_launch(const FgLaunch &L);

// enqueue the expansion of B compact G rows into rows in coordinate order (expand_kernel.cu); device pointers
cudaError_t expand_launch(int form, int ts, int R0, int nbG, long B, const double *Gc, long ldGc, double *G,
                          long ldG, cudaStream_t stream);

// enqueue out[b][p] = G[b][perm[p]] for B rows (coordinate order -> column-compressed order); device pointers
cudaError_t repack_launch(int neG, const int *perm, long B, const double *G, long ldG, double *out, long ldo,
                          cudaStream_t stream);

#endif
