// libtolcuda C ABI (include/tolcuda.h): contexts, constant upload, streams, pinned staging and the
// host/device batch paths around the sm_100a kernels of fg_kernels.cu.  No CPU evaluation path
// exists in this library: if CUDA is unavailable every evaluation call fails with the CUDA error.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <new>

#include "fg_launch.h"
#include "tolcuda_internal.h"

#define TOLCUDA_VERSION "0.1.0"

namespace tolcuda {

static thread_local std::string g_err;
void set_error(const std::string &msg) { g_err = msg; }

static int cuda_fail(cudaError_t e, const char *what) {
    set_error(std::string(what) + ": " + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ")");
    return (int)e;
}

#define CU(call)                                          \
    do {                                                  \
        cudaError_t e_ = (call);                          \
        if (e_ != cudaSuccess) return cuda_fail(e_, #call); \
    } while (0)

}  // namespace tolcuda

using namespace tolcuda;

int tolcuda::tolcuda_copy_raw(int device, void *dst, const void *src, size_t bytes, int kind) {
    if ((!dst || !src) && bytes) return TOLCUDA_EINVAL;
    CU(cudaSetDevice(device));
    CU(cudaMemcpy(dst, src, bytes, kind == 1 ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToHost));
    return 0;
}

// One staging lane of the host-pointer batch path: device buffers for a chunk of trajectories and
// the stream that carries H2D -> kernel -> D2H for that chunk.
struct BatchLane {
    cudaStream_t stream = nullptr;
    cudaEvent_t done = nullptr;  // the lane's last D2H has landed
    double *d_x = nullptr, *d_F = nullptr, *d_G = nullptr, *d_S = nullptr;
    double *h_Gc = nullptr;  // pinned landing area of compact G rows, expanded from here into the caller's G
    int cap = 0;             // trajectories
    long ldG = 0;            // row length d_G was allocated for (full or compact rows)
    long ldGc = 0;           // row length h_Gc was allocated for (0: none)
};
constexpr int NLANES = 3;

struct tolcuda_ctx {
    tolcuda_config cfg;
    FgConst c;
    int kernel = 0;
    // launch shape (fg_kernels.cu launch_sel / launch_cta), set through tolcuda_set_option only
    int per = 2;             // trajectories per CTA for large batches
    int per_auto = 1;        // ... and one per CTA below per_min_waves waves of CTAs
    int per_min_waves = -1;  // -1: 24 (8 for launches that overlap their predecessor: tools/sweep.py, profiles/r2_sweep.txt)
    int tail_waves_x4 = -1;  // quarter-waves of single-trajectory CTAs a grid of runs ends on; -1: 2, and 0 for
                             // TOLCUDA_OVERLAP_DISJOINT launches (the next grid fills the tail anyway)
    int lwarps = 0;  // kernel L: warps per CTA override (0 = automatic)
    int zero_copy = 1;  // single-trajectory path: kernel works on the mapped pinned block (0: staged copies)
    int chunk_mb = 32;  // host-pointer path: device bytes per lane (measured: 8..64 MB equally good, tools/expandbw.py)
    int sm_count = 148;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    std::vector<int> iG, jG;
    // single-trajectory path: pinned host staging + device buffers, allocated once
    double *h_one = nullptr;  // [n | neF | neG], pinned
    double *d_one = nullptr;  // same layout on the device
    long ox = 0, oF = 0, oG = 0;
    // host-pointer batch path
    BatchLane lane[NLANES];
    int compact_host = 1;  // host-pointer path: compact G across PCIe, expanded by host threads (0: full rows)
    int full_rows_pct = 0;  // ... with this share of the chunks (0..100) sent as full rows all the same: the copy engines
                            // carry them while the cores expand the others (what the host can take is box-dependent)
    int host_threads = 0;  // 0: HostPool::default_threads()
    std::unique_ptr<HostPool> pool;
    long launches = 0;
    double *d_grid = nullptr;  // wind cube: gx | gy | gz | v
    int *d_perm = nullptr;     // CSC position -> coordinate-order position, uploaded at first use
    double *d_goals = nullptr;  // goal table (tolcuda_set_goals): ngoals rows of TOLCUDA_GOAL_LD doubles (goal_row)
    long ngoals = 0;
    std::string dump_dir;      // DEFINEGusrfg_: the reference's per-call dump files go here (empty: none)
    bool dump_warned = false;
};

namespace {

std::mutex g_mu;
tolcuda_ctx *g_bound = nullptr;

long round_up(long v, long m) { return (v + m - 1) / m * m; }

// A goal (tolcuda_config.goal: xg, yg, zg, rg in NED) as the kernels read it: one row of a goal table, xg, yg, rg,
// cos_chid, sin_chid.  chi_d = atan2(yg - yi, xg - xi) with the hard-coded xi = yi = 0 of the reference constructor
// (src/problemG7.cpp:524, src/problem.cpp:111-112); host libm, as in the reference.  tolcuda_create and
// tolcuda_set_goals both derive the values here, so a table row and a context created with the same goal give the
// kernels the same bits.
void goal_row(const double *goal, double row[TOLCUDA_GOAL_LD]) {
    const double chi_d = std::atan2(goal[1] - 0.0, goal[0] - 0.0);
    row[0] = goal[0], row[1] = goal[1], row[2] = goal[3];
    row[3] = std::cos(chi_d), row[4] = std::sin(chi_d);
    for (int i = 5; i < TOLCUDA_GOAL_LD; i++) row[i] = 0.0;
}

// goals: NULL, or the device goal-table row of the launch's first trajectory
int launch(tolcuda_ctx *h, cudaStream_t st, int B, const double *x, long ldx, double *F, long ldF,
           double *G, long ldG, int needF, int needG, double *S = nullptr, long ldS = 0, int compact = 0, int op = 0,
           int pdl = 0, const double *goals = nullptr, const double *D = nullptr, long ldD = 0, double *Z = nullptr,
           long ldZ = 0) {
    FgLaunch L{};
    L.goals = goals;
    L.D = D, L.ldD = ldD, L.Z = Z, L.ldZ = ldZ;
    L.S = S, L.ldS = ldS;
    L.compact = compact;
    L.op = op;
    L.c = &h->c;
    L.B = B;
    L.x = x, L.ldx = ldx, L.F = F, L.ldF = ldF, L.G = G, L.ldG = ldG;
    L.needF = needF, L.needG = needG;
    L.kernel = h->kernel;
    L.per = h->per;
    L.lwarps = h->lwarps;
    L.per_auto = h->per_auto;
    L.pdl = op ? 0 : pdl;
    L.per_min_waves = h->per_min_waves >= 0 ? h->per_min_waves : (L.pdl == 2 ? 8 : 24);
    L.tail_waves_x4 = h->tail_waves_x4 >= 0 ? h->tail_waves_x4 : (L.pdl == 2 ? 0 : 2);
    L.sm_count = h->sm_count;
    L.device = h->cfg.device;
    L.stream = st;
    cudaError_t e = fg_launch(L);
    if (e != cudaSuccess) return cuda_fail(e, "fg_launch");
    h->launches++;
    return 0;
}

void free_lane(BatchLane &l) {
    if (l.d_x) cudaFree(l.d_x);
    if (l.d_F) cudaFree(l.d_F);
    if (l.d_G) cudaFree(l.d_G);
    if (l.d_S) cudaFree(l.d_S);
    if (l.h_Gc) cudaFreeHost(l.h_Gc);
    if (l.done) cudaEventDestroy(l.done);
    if (l.stream) cudaStreamDestroy(l.stream);
    l = BatchLane();
}

// device buffers for `cap` trajectories with G rows of ldG doubles; ldGc > 0: plus the pinned landing area
int ensure_lane(tolcuda_ctx *h, BatchLane &l, int cap, long ldG, long ldGc) {
    if (!l.stream) CU(cudaStreamCreateWithFlags(&l.stream, cudaStreamNonBlocking));
    if (!l.done) CU(cudaEventCreateWithFlags(&l.done, cudaEventDisableTiming));
    if (l.cap < cap || l.ldG < ldG) {
        if (l.d_x) cudaFree(l.d_x);
        if (l.d_F) cudaFree(l.d_F);
        if (l.d_G) cudaFree(l.d_G);
        if (l.d_S) cudaFree(l.d_S);
        l.d_x = l.d_F = l.d_G = l.d_S = nullptr;
        const int ncap = std::max(cap, l.cap);
        const long nldG = std::max(ldG, l.ldG);
        l.cap = 0, l.ldG = 0;
        const long ldx = tolcuda_padded_ld(h->c.n), ldF = tolcuda_padded_ld(h->c.neF);
        CU(cudaMalloc(&l.d_x, sizeof(double) * ldx * ncap));
        CU(cudaMalloc(&l.d_F, sizeof(double) * ldF * ncap));
        CU(cudaMalloc(&l.d_G, sizeof(double) * nldG * ncap));
        CU(cudaMalloc(&l.d_S, sizeof(double) * 4 * ncap));
        if (l.h_Gc) cudaFreeHost(l.h_Gc);  // sized with cap
        l.h_Gc = nullptr, l.ldGc = 0;
        l.cap = ncap, l.ldG = nldG;
    }
    if (ldGc > 0 && l.ldGc < ldGc) {
        if (l.h_Gc) cudaFreeHost(l.h_Gc);
        l.h_Gc = nullptr, l.ldGc = 0;
        CU(cudaMallocHost(&l.h_Gc, sizeof(double) * ldGc * l.cap));
        l.ldGc = ldGc;
    }
    return 0;
}

}  // namespace

extern "C" {

const char *tolcuda_last_error(void) { return g_err.c_str(); }
const char *tolcuda_version(void) { return TOLCUDA_VERSION; }

long tolcuda_padded_ld(long len) { return round_up(len, 16); }

int tolcuda_host_alloc(size_t bytes, void **ptr) {
    if (!ptr) return TOLCUDA_EINVAL;
    CU(cudaMallocHost(ptr, bytes));
    return 0;
}

int tolcuda_host_free(void *ptr) {
    if (ptr) CU(cudaFreeHost(ptr));
    return 0;
}

int tolcuda_device_count(int *count) {
    if (!count) return TOLCUDA_EINVAL;
    CU(cudaGetDeviceCount(count));
    return 0;
}

// ---- result buffers written by peer GPUs over NVLink (include/tolcuda.h) ----

int tolcuda_device_alloc(int device, size_t bytes, void **ptr) {
    if (!ptr) return TOLCUDA_EINVAL;
    *ptr = nullptr;
    CU(cudaSetDevice(device));
    CU(cudaMalloc(ptr, bytes));
    return 0;
}

int tolcuda_device_free(int device, void *ptr) {
    if (!ptr) return 0;
    CU(cudaSetDevice(device));
    CU(cudaFree(ptr));
    return 0;
}

static_assert(sizeof(cudaIpcMemHandle_t) == TOLCUDA_IPC_HANDLE_BYTES, "CUDA IPC handle size");

int tolcuda_ipc_export(int device, const void *ptr, unsigned char *handle) {
    if (!ptr || !handle) return TOLCUDA_EINVAL;
    CU(cudaSetDevice(device));
    cudaIpcMemHandle_t hd;
    CU(cudaIpcGetMemHandle(&hd, const_cast<void *>(ptr)));
    std::memcpy(handle, &hd, sizeof hd);
    return 0;
}

int tolcuda_ipc_open(int device, const unsigned char *handle, void **ptr) {
    if (!handle || !ptr) return TOLCUDA_EINVAL;
    *ptr = nullptr;
    CU(cudaSetDevice(device));
    cudaIpcMemHandle_t hd;
    std::memcpy(&hd, handle, sizeof hd);
    CU(cudaIpcOpenMemHandle(ptr, hd, cudaIpcMemLazyEnablePeerAccess));
    return 0;
}

int tolcuda_ipc_close(int device, void *ptr) {
    if (!ptr) return 0;
    CU(cudaSetDevice(device));
    CU(cudaIpcCloseMemHandle(ptr));
    return 0;
}

int tolcuda_enable_peer(int device, int peer) {
    if (device == peer) return 0;
    int can = 0;
    CU(cudaDeviceCanAccessPeer(&can, device, peer));
    if (!can) {
        set_error("tolcuda_enable_peer: no peer access between the two devices");
        return TOLCUDA_EUNSUPPORTED;
    }
    CU(cudaSetDevice(device));
    cudaError_t e = cudaDeviceEnablePeerAccess(peer, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) {
        cudaGetLastError();
        return 0;
    }
    if (e != cudaSuccess) return cuda_fail(e, "cudaDeviceEnablePeerAccess");
    return 0;
}

// cuStreamWriteValue32 / cuStreamWaitValue32 through the runtime's driver entry point lookup (libtolcuda links the
// static runtime only)
namespace {
typedef int (*StreamMemOp32)(cudaStream_t, unsigned long long, unsigned int, unsigned int);
int stream_memop(tolcuda_ctx *h, std::atomic<void *> &cached, const char *symbol, const void *flag, unsigned int value,
                 unsigned int opflags) {
    if (!h || !flag || (reinterpret_cast<uintptr_t>(flag) & 3)) return TOLCUDA_EINVAL;
    CU(cudaSetDevice(h->cfg.device));
    void *fn = cached.load(std::memory_order_acquire);
    if (!fn) {  // looked up once per process
        cudaDriverEntryPointQueryResult qr;
        CU(cudaGetDriverEntryPoint(symbol, &fn, cudaEnableDefault, &qr));
        if (!fn || qr != cudaDriverEntryPointSuccess) {
            set_error(std::string(symbol) + ": not provided by this driver");
            return TOLCUDA_EUNSUPPORTED;
        }
        cached.store(fn, std::memory_order_release);
    }
    const int rc = reinterpret_cast<StreamMemOp32>(fn)(h->stream, (unsigned long long)reinterpret_cast<uintptr_t>(flag), value, opflags);
    if (rc != 0) {
        set_error(std::string(symbol) + " failed with CUresult " + std::to_string(rc));
        return rc;
    }
    return 0;
}
}  // namespace

int tolcuda_stream_signal(tolcuda_handle h, void *flag, unsigned int value) {
    static std::atomic<void *> fn{nullptr};
    return stream_memop(h, fn, "cuStreamWriteValue32", flag, value, 0 /* CU_STREAM_WRITE_VALUE_DEFAULT: fence before the write */);
}

int tolcuda_stream_wait(tolcuda_handle h, const void *flag, unsigned int value) {
    static std::atomic<void *> fn{nullptr};
    return stream_memop(h, fn, "cuStreamWaitValue32", flag, value, 0 /* CU_STREAM_WAIT_VALUE_GEQ */);
}

int tolcuda_read_params(const char *path, double *values, int cap, int *count) {
    if (!path || !count) return TOLCUDA_EINVAL;
    std::vector<double> v;
    int e = read_params(path, v);
    if (e) {
        set_error(std::string("cannot open parameter file ") + path);
        return e;
    }
    *count = (int)v.size();
    for (int i = 0; i < cap && i < (int)v.size(); i++) values[i] = v[i];
    return 0;
}

int tolcuda_create(const tolcuda_config *cfg, tolcuda_handle *out) {
    if (!cfg || !out) return TOLCUDA_EINVAL;
    *out = nullptr;
    if (cfg->formulation != TOLCUDA_G7 && cfg->formulation != TOLCUDA_S10) {
        set_error("formulation must be TOLCUDA_G7 or TOLCUDA_S10");
        return TOLCUDA_EUNSUPPORTED;
    }
    if (cfg->wind_model != TOLCUDA_WIND_NONE && cfg->wind_model != TOLCUDA_WIND_LINEAR_LAYER) {
        set_error("wind model not built (0 = none, 1 = linear boundary layer)");
        return TOLCUDA_EUNSUPPORTED;
    }
    if (cfg->ts < 1 || cfg->ts > 1000000) {
        set_error("ts must be in 1..1000000");
        return TOLCUDA_EUNSUPPORTED;
    }
    tolcuda_ctx *h = new (std::nothrow) tolcuda_ctx();
    if (!h) return TOLCUDA_ENOMEM;
    h->cfg = *cfg;
    FgConst &c = h->c;
    std::memset(&c, 0, sizeof c);
    c.form = cfg->formulation;
    c.ts = cfg->ts;
    c.wind = cfg->wind_model;
    c.nb = c.form == TOLCUDA_G7 ? 12 : 11;
    pattern_dims(c.form, c.ts, &c.n, &c.neF, &c.neG, &c.R0, &c.nbG);
    const double *ac = cfg->aircraft, *gn = cfg->gains;
    const double mm = ac[0], SS = ac[2], ee = ac[3], AR = ac[4], Cd0 = ac[5];
    c.mm = mm, c.SS = SS, c.Cd0 = Cd0;
    c.rho = 1.2682;  // reference include/problem.h:73
    c.g = 9.81;      // reference include/problem.h:72
    c.rhoSS = c.rho * SS;
    c.ARpiee = AR * M_PI * ee;
    c.ARpieemm = AR * M_PI * ee * mm;
    c.twomm = 2.0 * mm;
    c.r_mm = 1.0 / c.mm, c.r_twomm = 1.0 / c.twomm;
    c.r_ARpiee = 1.0 / c.ARpiee, c.r_ARpieemm = 1.0 / c.ARpieemm;
    c.kT = gn[0], c.kp = gn[1], c.kdt = gn[4];
    c.half_kT = 0.5 * gn[0];
    c.half_kp = 0.5 * gn[1];
    c.kv_ts = gn[2] * c.ts;
    c.kp_ts = gn[1] * c.ts;
    double grow[TOLCUDA_GOAL_LD];
    goal_row(cfg->goal, grow);
    c.xg = grow[0], c.yg = grow[1], c.rg = grow[2], c.cos_chid = grow[3], c.sin_chid = grow[4];
    {
        const double Vref = 2.4, href = 10;  // src/problem.cpp:504-505
        const double dv_dz = -Vref / href;   // :524
        c.wind_Wxz = -dv_dz;                 // :975
    }
    pattern_build(c.form, c.ts, h->iG, h->jG);

    if (const char *env = std::getenv("TOLCUDA_DUMP_DIR")) h->dump_dir = env;

    int rc = 0;
    do {
        cudaError_t e = cudaSetDevice(cfg->device);
        if (e != cudaSuccess) { rc = cuda_fail(e, "cudaSetDevice"); break; }
        int sms = 0;
        e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, cfg->device);
        if (e != cudaSuccess) { rc = cuda_fail(e, "cudaDeviceGetAttribute"); break; }
        h->sm_count = sms;
        e = cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking);
        if (e != cudaSuccess) { rc = cuda_fail(e, "cudaStreamCreate"); break; }
        h->stream = h->own_stream;
        h->ox = 0;
        h->oF = tolcuda_padded_ld(c.n);
        h->oG = h->oF + tolcuda_padded_ld(c.neF);
        const size_t bytes = sizeof(double) * (h->oG + tolcuda_padded_ld(c.neG));
        e = cudaMallocHost(&h->h_one, bytes);
        if (e != cudaSuccess) { rc = cuda_fail(e, "cudaMallocHost"); break; }
        e = cudaMalloc(&h->d_one, bytes);
        if (e != cudaSuccess) { rc = cuda_fail(e, "cudaMalloc"); break; }
    } while (0);
    if (rc) {
        tolcuda_destroy(h);
        return rc;
    }
    *out = h;
    return 0;
}

int tolcuda_config_from_files(const char *root, const char *aircraft, const char *mission,
                              double east, double north, double up, double east_goal,
                              double north_goal, double up_goal, double radius_goal,
                              int ts_override, int device, tolcuda_config *out) {
    (void)east, (void)north, (void)up;  // stored by the reference, unused on the evaluation path
    if (!root || !aircraft || !mission || !out) return TOLCUDA_EINVAL;
    tolcuda_config cfg;
    std::memset(&cfg, 0, sizeof cfg);
    const std::string ms(mission);
    if (ms == "G7") cfg.formulation = TOLCUDA_G7;
    else if (ms == "S10") cfg.formulation = TOLCUDA_S10;
    else {
        set_error("Problem " + ms + " not recognized.");  // reference src/problem.cpp:361
        return TOLCUDA_EUNSUPPORTED;
    }
    int e;
    if ((e = read_aircraft(root, aircraft, cfg.aircraft))) return e;
    if ((e = read_gains(root, ms, cfg.gains))) return e;
    double sn[6];
    if ((e = read_snopt(root, ms, sn))) return e;
    if ((e = read_limits(root, ms, cfg.limits))) return e;
    cfg.solver_tol[0] = sn[4];
    cfg.solver_tol[1] = sn[5];
    const int nb = cfg.formulation == TOLCUDA_G7 ? 12 : 11;
    if ((int)sn[1] != TOLCUDA_PX || (int)sn[2] != TOLCUDA_PF || (int)sn[3] != nb) {
        set_error("snopt.param: numinp/numstates/numbounds differ from the built formulation");
        return TOLCUDA_EUNSUPPORTED;
    }
    cfg.ts = ts_override > 0 ? ts_override : (int)sn[0];
    cfg.wind_model = TOLCUDA_WIND_LINEAR_LAYER;  // what the reference falls back to, src/problem.cpp:77
    cfg.device = device;
    // ENU -> NED, reference src/problem.cpp:24-27
    cfg.goal[0] = north_goal;
    cfg.goal[1] = east_goal;
    cfg.goal[2] = -up_goal;
    cfg.goal[3] = radius_goal;
    *out = cfg;
    return 0;
}

int tolcuda_create_from_files(const char *root, const char *aircraft, const char *mission,
                              double east, double north, double up, double east_goal,
                              double north_goal, double up_goal, double radius_goal,
                              int ts_override, int device, tolcuda_handle *out) {
    if (!out) return TOLCUDA_EINVAL;
    *out = nullptr;
    tolcuda_config cfg;
    int e = tolcuda_config_from_files(root, aircraft, mission, east, north, up, east_goal, north_goal, up_goal,
                                      radius_goal, ts_override, device, &cfg);
    if (e) return e;
    return tolcuda_create(&cfg, out);
}

int tolcuda_set_wind_grid(tolcuda_handle h, int ne, int nn, int nu, const double *gx, const double *gy,
                          const double *gz, const double *v, const double *datum, const double *spacing) {
    if (!h || ne < 2 || nn < 2 || nu < 2 || !gx || !gy || !gz || !v || !datum || !spacing) {
        set_error("tolcuda_set_wind_grid: need at least 2 grid points per axis and non-null arrays");
        return TOLCUDA_EINVAL;
    }
    CU(cudaSetDevice(h->cfg.device));
    CU(cudaStreamSynchronize(h->stream));
    if (h->d_grid) CU(cudaFree(h->d_grid));
    h->d_grid = nullptr;
    const size_t nv = (size_t)ne * nn * nu, tot = (size_t)ne + nn + nu + nv;
    CU(cudaMalloc(&h->d_grid, sizeof(double) * tot));
    double *d = h->d_grid;
    CU(cudaMemcpy(d, gx, sizeof(double) * ne, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d + ne, gy, sizeof(double) * nn, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d + ne + nn, gz, sizeof(double) * nu, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d + ne + nn + nu, v, sizeof(double) * nv, cudaMemcpyHostToDevice));
    FgConst &c = h->c;
    c.grid_ne = ne, c.grid_nn = nn, c.grid_nu = nu;
    c.grid_x = d, c.grid_y = d + ne, c.grid_z = d + ne + nn, c.grid_v = d + ne + nn + nu;
    for (int i = 0; i < 3; i++) c.datum[i] = datum[i], c.spacing[i] = spacing[i];
    c.wind = TOLCUDA_WIND_CUBE;
    h->cfg.wind_model = TOLCUDA_WIND_CUBE;
    return 0;
}

int tolcuda_destroy(tolcuda_handle h) {
    if (!h) return 0;
    {
        std::lock_guard<std::mutex> lk(g_mu);
        if (g_bound == h) g_bound = nullptr;
    }
    cudaSetDevice(h->cfg.device);
    if (h->own_stream) cudaStreamSynchronize(h->own_stream);
    for (BatchLane &l : h->lane) {
        if (l.stream) cudaStreamSynchronize(l.stream);
        free_lane(l);
    }
    if (h->h_one) cudaFreeHost(h->h_one);
    if (h->d_one) cudaFree(h->d_one);
    if (h->d_grid) cudaFree(h->d_grid);
    if (h->d_perm) cudaFree(h->d_perm);
    if (h->d_goals) cudaFree(h->d_goals);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    delete h;
    return 0;
}

int tolcuda_dims(tolcuda_handle h, int *n, int *neF, int *neG) {
    if (!h) return TOLCUDA_EINVAL;
    if (n) *n = h->c.n;
    if (neF) *neF = h->c.neF;
    if (neG) *neG = h->c.neG;
    return 0;
}

int tolcuda_pattern(tolcuda_handle h, int *iGfun, int *jGvar) {
    if (!h || !iGfun || !jGvar) return TOLCUDA_EINVAL;
    std::memcpy(iGfun, h->iG.data(), sizeof(int) * h->iG.size());
    std::memcpy(jGvar, h->jG.data(), sizeof(int) * h->jG.size());
    return 0;
}

int tolcuda_problem_dims(int formulation, int ts, int *n, int *neF, int *neG) {
    if ((formulation != TOLCUDA_G7 && formulation != TOLCUDA_S10) || ts < 1) return TOLCUDA_EINVAL;
    pattern_dims(formulation, ts, n, neF, neG, nullptr, nullptr);
    return 0;
}

int tolcuda_problem_pattern(int formulation, int ts, int *iGfun, int *jGvar) {
    if ((formulation != TOLCUDA_G7 && formulation != TOLCUDA_S10) || ts < 1 || !iGfun || !jGvar)
        return TOLCUDA_EINVAL;
    std::vector<int> iG, jG;
    pattern_build(formulation, ts, iG, jG);
    std::memcpy(iGfun, iG.data(), sizeof(int) * iG.size());
    std::memcpy(jGvar, jG.data(), sizeof(int) * jG.size());
    return 0;
}

static bool config_ok(const tolcuda_config *cfg) {
    return cfg && (cfg->formulation == TOLCUDA_G7 || cfg->formulation == TOLCUDA_S10) && cfg->ts >= 1;
}

int tolcuda_problem_initial_guess(const tolcuda_config *cfg, double *x0) {
    if (!config_ok(cfg) || !x0) return TOLCUDA_EINVAL;
    initial_guess(*cfg, x0);
    return 0;
}

int tolcuda_problem_bounds(const tolcuda_config *cfg, double *xlow, double *xupp, double *Flow,
                           double *Fupp) {
    if (!config_ok(cfg) || !xlow || !xupp || !Flow || !Fupp) return TOLCUDA_EINVAL;
    bounds(*cfg, xlow, xupp, Flow, Fupp);
    return 0;
}

int tolcuda_write_results_json(const tolcuda_config *cfg, const char *aircraft, const char *mission, double east,
                               double north, double up, const double *x, double final_cost, const char *path) {
    if (!config_ok(cfg) || !aircraft || !mission || !x || !path) return TOLCUDA_EINVAL;
    return write_results_json(*cfg, aircraft, mission, east, north, up, x, final_cost, path);
}

int tolcuda_write_results_txt(const tolcuda_config *cfg, const double *x, double final_cost, const char *path) {
    if (!config_ok(cfg) || !x || !path) return TOLCUDA_EINVAL;
    return write_results_txt(*cfg, x, final_cost, path);
}

int tolcuda_get_config(tolcuda_handle h, tolcuda_config *cfg) {
    if (!h || !cfg) return TOLCUDA_EINVAL;
    *cfg = h->cfg;
    return 0;
}

int tolcuda_set_stream(tolcuda_handle h, void *cuda_stream) {
    if (!h) return TOLCUDA_EINVAL;
    h->stream = (cudaStream_t)cuda_stream;
    return 0;
}

int tolcuda_use_own_stream(tolcuda_handle h) {
    if (!h) return TOLCUDA_EINVAL;
    h->stream = h->own_stream;
    return 0;
}

int tolcuda_synchronize(tolcuda_handle h) {
    if (!h) return TOLCUDA_EINVAL;
    CU(cudaSetDevice(h->cfg.device));
    CU(cudaStreamSynchronize(h->stream));
    return 0;
}

long tolcuda_launch_count(tolcuda_handle h) { return h ? h->launches : 0; }

int tolcuda_eval(tolcuda_handle h, const double *x, int needF, double *F, int needG, double *G) {
    if (!h || !x || (needF > 0 && !F) || (needG > 0 && !G)) return TOLCUDA_EINVAL;
    if (needF <= 0 && needG <= 0) return 0;
    const FgConst &c = h->c;
    CU(cudaSetDevice(h->cfg.device));
    cudaStream_t st = h->stream;
    std::memcpy(h->h_one + h->ox, x, sizeof(double) * c.n);
    // G crosses PCIe as a compact row (a third of the bytes) and is expanded straight into the caller's array
    // with ordinary stores -- SNOPT reads it next (option "compact_host" = 0: the full row is copied instead)
    const int compact = needG > 0 && h->compact_host;
    const long lenG = compact ? compact_len(c.form, c.ts) : (long)c.neG;
    if (h->zero_copy) {
        // One launch, no copy commands: the pinned staging block is mapped into the device's address
        // space (UVA), so the kernel reads x from it and writes F/G into it across PCIe directly.
        int rc = launch(h, st, 1, h->h_one + h->ox, c.n, h->h_one + h->oF, c.neF, h->h_one + h->oG, lenG,
                        needF > 0, needG > 0, nullptr, 0, compact);
        if (rc) return rc;
        CU(cudaStreamSynchronize(st));
    } else {
        CU(cudaMemcpyAsync(h->d_one + h->ox, h->h_one + h->ox, sizeof(double) * c.n, cudaMemcpyHostToDevice, st));
        int rc = launch(h, st, 1, h->d_one + h->ox, c.n, h->d_one + h->oF, c.neF, h->d_one + h->oG, lenG,
                        needF > 0, needG > 0, nullptr, 0, compact);
        if (rc) return rc;
        if (needF > 0)
            CU(cudaMemcpyAsync(h->h_one + h->oF, h->d_one + h->oF, sizeof(double) * c.neF, cudaMemcpyDeviceToHost, st));
        if (needG > 0)
            CU(cudaMemcpyAsync(h->h_one + h->oG, h->d_one + h->oG, sizeof(double) * lenG, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
    }
    if (needF > 0) std::memcpy(F, h->h_one + h->oF, sizeof(double) * c.neF);
    if (needG > 0) {
        if (compact) expand_row_cached(c.form, c.ts, h->h_one + h->oG, G);
        else std::memcpy(G, h->h_one + h->oG, sizeof(double) * c.neG);
    }
    return 0;
}

int tolcuda_eval_batch(tolcuda_handle h, int B, const double *x, long ldx, double *F, long ldF,
                       double *G, long ldG, int flags) {
    return tolcuda_eval_batch_summary(h, B, x, ldx, F, ldF, G, ldG, nullptr, 0, flags);
}

// The body of tolcuda_eval_batch_summary and tolcuda_eval_batch_goals.  goals: NULL (every trajectory has the
// context's goal), or the device goal-table row of trajectory 0 of this call.
static int eval_batch(tolcuda_handle h, int B, const double *x, long ldx, double *F, long ldF, double *G, long ldG,
                      double *summary, long lds, int flags, const double *goals) {
    if (!h || B < 0 || (summary && lds < 4)) return TOLCUDA_EINVAL;
    const int needF = (flags & TOLCUDA_NEED_F) != 0;
    if (flags & ~TOLCUDA_FLAGS_ALL) {
        set_error("tolcuda_eval_batch: unknown flag bits");
        return TOLCUDA_EINVAL;
    }
    const int needG = (flags & TOLCUDA_NEED_G) != 0;
    if (B == 0 || (!needF && !needG && !summary)) return 0;
    const FgConst &c = h->c;
    const long lenGc = compact_len(c.form, c.ts);
    const bool compact_rows = (flags & TOLCUDA_COMPACT_G) != 0;  // the CALLER's G holds compact rows
    if (compact_rows && summary) {
        set_error("tolcuda_eval_batch_summary: TOLCUDA_COMPACT_G cannot be combined with a summary");
        return TOLCUDA_EUNSUPPORTED;
    }
    if (!x || ldx < c.n || (needF && (!F || ldF < c.neF)) ||
        (needG && (!G || ldG < (compact_rows ? lenGc : (long)c.neG)))) {
        set_error("tolcuda_eval_batch: null pointer or leading dimension shorter than the row");
        return TOLCUDA_EINVAL;
    }
    CU(cudaSetDevice(h->cfg.device));
    bool host = (flags & TOLCUDA_HOST_PTRS) != 0;
    if (!host && !(flags & TOLCUDA_DEVICE_PTRS)) {
        cudaPointerAttributes at;
        cudaError_t e = cudaPointerGetAttributes(&at, x);
        if (e != cudaSuccess) {
            cudaGetLastError();
            host = true;
        } else {
            host = !(at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged);
        }
    }
    const int pdl = (flags & TOLCUDA_OVERLAP_DISJOINT) ? 2 : ((flags & TOLCUDA_OVERLAP) ? 1 : 0);
    if (pdl && (host || !(flags & TOLCUDA_NO_SYNC))) {
        set_error("tolcuda_eval_batch: TOLCUDA_OVERLAP needs device pointers and TOLCUDA_NO_SYNC");
        return TOLCUDA_EINVAL;
    }
    if (!host) {
        int rc = launch(h, h->stream, B, x, ldx, F, ldF, G, ldG, needF, needG, summary, lds, compact_rows, 0, pdl, goals);
        if (rc) return rc;
        if (!(flags & TOLCUDA_NO_SYNC)) CU(cudaStreamSynchronize(h->stream));
        return 0;
    }

    // Host pointers: chunks of trajectories rotate over NLANES lanes; a lane's stream carries
    // H2D(x) -> kernel -> D2H(F, G) for its chunk, so one lane's copies overlap another's kernel.
    // G normally crosses PCIe as compact rows (31 of a window's 104 values, compact.cpp) into the lane's
    // pinned landing area and is expanded from there into the caller's G by the host thread pool while
    // the next lanes are in flight; TOLCUDA_FULL_G_COPY (or option "compact_host" = 0, or a summary request)
    // copies full rows straight into the caller's G instead.
    const bool via_compact = needG && !compact_rows && !summary && h->compact_host && !(flags & TOLCUDA_FULL_G_COPY);
    const bool dev_compact = via_compact || compact_rows;  // layout of the lane's d_G
    const long dldx = tolcuda_padded_ld(c.n), dldF = tolcuda_padded_ld(c.neF);
    const long dldG = tolcuda_padded_ld(dev_compact ? lenGc : (long)c.neG);
    const long rowG = dev_compact ? lenGc : (long)c.neG;  // doubles of a G row that cross PCIe
    // Mixed mode: a share of the chunks crosses PCIe as full rows (DMA straight into the caller's G) while the others
    // go as compact rows and are expanded by the host threads -- the copy engines and the cores are different
    // resources, and which of them a host has to spare differs from box to box (DESIGN.md 6a).  Chunk ci is a
    // full-row chunk when the running share crosses an integer (evenly spread over the call).
    const int mix = via_compact ? h->full_rows_pct : 0;
    const long dldGfull = tolcuda_padded_ld((long)c.neG);
    auto full_chunk = [&](int ci) { return mix > 0 && ((long)(ci + 1) * mix) / 100 != ((long)ci * mix) / 100; };
    const size_t per_traj = sizeof(double) * (size_t)(dldx + dldF + dldG);
    // device bytes per lane: at most chunk_mb, and small enough for ~160 chunks per call (never below 1 MB) -- the
    // first chunk's copies and kernel and the last chunk's expansion are not overlapped with anything, which costs
    // 10-15 % of a call made of 21 chunks (8,192 rows, one GPU's shard of 8) and nothing at 160
    // (tools/e2e_sweep.py, profiles/r2_e2e_sweep_8gpu.jsonl)
    const size_t cap = (size_t)h->chunk_mb << 20;
    const size_t budget = std::min(cap, std::max<size_t>((size_t)1 << 20, per_traj * (size_t)B / 160));
    int chunk = (int)std::max<size_t>(1, budget / per_traj);
    chunk = std::min(chunk, B);
    if (B > chunk && B < NLANES * chunk) chunk = (B + NLANES - 1) / NLANES;
    const int nchunks = (B + chunk - 1) / chunk;
    const int nlanes = std::min(NLANES, nchunks);
    for (int l = 0; l < nlanes; l++) {
        int rc = ensure_lane(h, h->lane[l], chunk, mix > 0 ? dldGfull : dldG, via_compact ? dldG : 0);
        if (rc) return rc;
    }
    if (via_compact && !h->pool)
        h->pool.reset(new HostPool(h->host_threads > 0 ? h->host_threads : HostPool::default_threads()));

    auto enqueue = [&](int ci) -> int {
        BatchLane &l = h->lane[ci % NLANES];
        const int b0 = ci * chunk, nb = std::min(chunk, B - b0);
        CU(cudaMemcpy2DAsync(l.d_x, sizeof(double) * dldx, x + (size_t)b0 * ldx, sizeof(double) * ldx,
                             sizeof(double) * c.n, nb, cudaMemcpyHostToDevice, l.stream));
        const bool fullc = full_chunk(ci);
        int rc = launch(h, l.stream, nb, l.d_x, dldx, l.d_F, dldF, l.d_G, fullc ? dldGfull : dldG, needF, needG,
                        summary ? l.d_S : nullptr, 4, dev_compact && !fullc, 0, 0,
                        goals ? goals + (size_t)TOLCUDA_GOAL_LD * b0 : nullptr);
        if (rc) return rc;
        if (needF)
            CU(cudaMemcpy2DAsync(F + (size_t)b0 * ldF, sizeof(double) * ldF, l.d_F, sizeof(double) * dldF,
                                 sizeof(double) * c.neF, nb, cudaMemcpyDeviceToHost, l.stream));
        if (summary)
            CU(cudaMemcpy2DAsync(summary + (size_t)b0 * lds, sizeof(double) * lds, l.d_S, sizeof(double) * 4,
                                 sizeof(double) * 4, nb, cudaMemcpyDeviceToHost, l.stream));
        if (needG && fullc)
            CU(cudaMemcpy2DAsync(G + (size_t)b0 * ldG, sizeof(double) * ldG, l.d_G, sizeof(double) * dldGfull,
                                 sizeof(double) * c.neG, nb, cudaMemcpyDeviceToHost, l.stream));
        else if (needG && via_compact)
            CU(cudaMemcpyAsync(l.h_Gc, l.d_G, sizeof(double) * dldG * nb, cudaMemcpyDeviceToHost, l.stream));
        else if (needG)
            CU(cudaMemcpy2DAsync(G + (size_t)b0 * ldG, sizeof(double) * ldG, l.d_G, sizeof(double) * dldG,
                                 sizeof(double) * rowG, nb, cudaMemcpyDeviceToHost, l.stream));
        CU(cudaEventRecord(l.done, l.stream));
        return 0;
    };
    auto drain = [&]() {  // error exit: nothing of this call may still be writing into the caller's arrays
        for (int l = 0; l < nlanes; l++) cudaStreamSynchronize(h->lane[l].stream);
    };
    int rc = 0;
    for (int ci = 0; ci < nlanes && !rc; ci++) rc = enqueue(ci);
    for (int ci = 0; ci < nchunks && !rc; ci++) {
        BatchLane &l = h->lane[ci % NLANES];
        cudaError_t e = cudaEventSynchronize(l.done);
        if (e != cudaSuccess) {
            rc = cuda_fail(e, "cudaEventSynchronize");
            break;
        }
        if (via_compact && !full_chunk(ci)) {
            const int b0 = ci * chunk, nb = std::min(chunk, B - b0);
            expand_rows(*h->pool, c.form, c.ts, nb, l.h_Gc, dldG, G + (size_t)b0 * ldG, ldG);
        }
        if (ci + NLANES < nchunks) rc = enqueue(ci + NLANES);
    }
    if (rc) drain();
    return rc;
}

int tolcuda_eval_batch_summary(tolcuda_handle h, int B, const double *x, long ldx, double *F, long ldF,
                               double *G, long ldG, double *summary, long lds, int flags) {
    return eval_batch(h, B, x, ldx, F, ldF, G, ldG, summary, lds, flags, nullptr);
}

int tolcuda_set_goals(tolcuda_handle h, long count, const double *goal, long ldg) {
    if (!h) {
        set_error("tolcuda_set_goals: null handle");
        return TOLCUDA_EINVAL;
    }
    if (count < 0 || (count > 0 && (!goal || ldg < 4))) {
        set_error("tolcuda_set_goals: negative count, null goal array or ldg < 4");
        return TOLCUDA_EINVAL;
    }
    std::vector<double> rows((size_t)count * TOLCUDA_GOAL_LD);
    for (long b = 0; b < count; b++) goal_row(goal + (size_t)b * ldg, rows.data() + (size_t)b * TOLCUDA_GOAL_LD);
    CU(cudaSetDevice(h->cfg.device));
    CU(cudaStreamSynchronize(h->stream));  // launches still reading the old table
    if (h->d_goals) CU(cudaFree(h->d_goals));
    h->d_goals = nullptr, h->ngoals = 0;
    if (count == 0) return 0;
    CU(cudaMalloc(&h->d_goals, sizeof(double) * rows.size()));
    CU(cudaMemcpy(h->d_goals, rows.data(), sizeof(double) * rows.size(), cudaMemcpyHostToDevice));
    h->ngoals = count;
    return 0;
}

int tolcuda_eval_batch_goals(tolcuda_handle h, long row0, int B, const double *x, long ldx, double *F, long ldF,
                             double *G, long ldG, double *summary, long lds, int flags) {
    if (!h) {
        set_error("tolcuda_eval_batch_goals: null handle");
        return TOLCUDA_EINVAL;
    }
    if (!h->d_goals) {
        set_error("tolcuda_eval_batch_goals: no goal table (tolcuda_set_goals)");
        return TOLCUDA_EINVAL;
    }
    if (row0 < 0 || B < 0 || row0 + B > h->ngoals) {
        set_error("tolcuda_eval_batch_goals: rows [" + std::to_string(row0) + ", " + std::to_string(row0 + B) +
                  ") outside the goal table's " + std::to_string(h->ngoals) + " rows");
        return TOLCUDA_EINVAL;
    }
    return eval_batch(h, B, x, ldx, F, ldF, G, ldG, summary, lds, flags, h->d_goals + (size_t)TOLCUDA_GOAL_LD * row0);
}

long tolcuda_compact_len(int formulation, int ts) {
    if ((formulation != TOLCUDA_G7 && formulation != TOLCUDA_S10) || ts < 1) return TOLCUDA_EINVAL;
    return compact_len(formulation, ts);
}

int tolcuda_expand_compact_g(int formulation, int ts, long B, const double *Gc, long ldGc, double *G, long ldG,
                             int threads) {
    if ((formulation != TOLCUDA_G7 && formulation != TOLCUDA_S10) || ts < 1 || B < 0) return TOLCUDA_EINVAL;
    int neG;
    pattern_dims(formulation, ts, nullptr, nullptr, &neG, nullptr, nullptr);
    if (B > 0 && (!Gc || !G || ldGc < compact_len(formulation, ts) || ldG < neG)) {
        set_error("tolcuda_expand_compact_g: null pointer or leading dimension shorter than the row");
        return TOLCUDA_EINVAL;
    }
    HostPool pool(threads > 0 ? threads : HostPool::default_threads());
    expand_rows(pool, formulation, ts, B, Gc, ldGc, G, ldG);
    return 0;
}

int tolcuda_expand_compact_g_device(tolcuda_handle h, long B, const double *Gc, long ldGc, double *G, long ldG,
                                    int flags) {
    if (!h || B < 0) return TOLCUDA_EINVAL;
    const FgConst &c = h->c;
    if (B > 0 && (!Gc || !G || ldGc < compact_len(c.form, c.ts) || ldG < c.neG)) {
        set_error("tolcuda_expand_compact_g_device: null pointer or leading dimension shorter than the row");
        return TOLCUDA_EINVAL;
    }
    CU(cudaSetDevice(h->cfg.device));
    cudaError_t e = expand_launch(c.form, c.ts, c.R0, c.nbG, B, Gc, ldGc, G, ldG, h->stream);
    if (e != cudaSuccess) return cuda_fail(e, "expand_launch");
    h->launches += B > 0 ? (B + 65534) / 65535 : 0;
    if (!(flags & TOLCUDA_NO_SYNC)) CU(cudaStreamSynchronize(h->stream));
    return 0;
}

// y = J(x) d and z = J(x)^T lambda without materialising G (fg_kernels.cu, MODE_JVP / MODE_VJP)
static int jac_op(tolcuda_handle h, int op, int B, const double *x, long ldx, const double *in, long ldin, long len_in,
                  double *out, long ldout, long len_out, int flags, const char *who) {
    if (!h || B < 0) return TOLCUDA_EINVAL;
    if (B == 0) return 0;
    const FgConst &c = h->c;
    if (!x || !in || !out || ldx < c.n || ldin < len_in || ldout < len_out) {
        set_error(std::string(who) + ": null pointer or leading dimension shorter than the row");
        return TOLCUDA_EINVAL;
    }
    if (flags & TOLCUDA_HOST_PTRS) {
        set_error(std::string(who) + ": device pointers only");
        return TOLCUDA_EUNSUPPORTED;
    }
    CU(cudaSetDevice(h->cfg.device));
    // op 1: the F pointer receives y, the G pointer holds d; op 2: the F pointer holds lambda, the G pointer receives z
    double *Fp = op == 1 ? out : const_cast<double *>(in), *Gp = op == 1 ? const_cast<double *>(in) : out;
    const long ldFp = op == 1 ? ldout : ldin, ldGp = op == 1 ? ldin : ldout;
    int rc = launch(h, h->stream, B, x, ldx, Fp, ldFp, Gp, ldGp, 1, 1, nullptr, 0, 0, op);
    if (rc) return rc;
    if (!(flags & TOLCUDA_NO_SYNC)) CU(cudaStreamSynchronize(h->stream));
    return 0;
}

int tolcuda_jac_vec(tolcuda_handle h, int B, const double *x, long ldx, const double *d, long ldd, double *y, long ldy,
                    int flags) {
    return jac_op(h, 1, B, x, ldx, d, ldd, h ? h->c.n : 0, y, ldy, h ? h->c.neF : 0, flags, "tolcuda_jac_vec");
}

int tolcuda_jac_tvec(tolcuda_handle h, int B, const double *x, long ldx, const double *lambda, long ldl, double *z,
                     long ldz, int flags) {
    return jac_op(h, 2, B, x, ldx, lambda, ldl, h ? h->c.neF : 0, z, ldz, h ? h->c.n : 0, flags, "tolcuda_jac_tvec");
}

// w = D_x[J(x)^T lambda] d and optionally z = J(x)^T lambda (fg_kernels.cu, MODE_HVP)
int tolcuda_lag_hess_vec(tolcuda_handle h, int B, const double *x, long ldx, const double *lambda, long ldl,
                         const double *d, long ldd, double *w, long ldw, double *z, long ldz, int flags) {
    if (!h || B < 0) return TOLCUDA_EINVAL;
    if (B == 0) return 0;
    const FgConst &c = h->c;
    if (!x || !lambda || !d || !w || ldx < c.n || ldl < c.neF || ldd < c.n || ldw < c.n || (z && ldz < c.n)) {
        set_error("tolcuda_lag_hess_vec: null pointer or leading dimension shorter than the row");
        return TOLCUDA_EINVAL;
    }
    if (flags & TOLCUDA_HOST_PTRS) {
        set_error("tolcuda_lag_hess_vec: device pointers only");
        return TOLCUDA_EUNSUPPORTED;
    }
    CU(cudaSetDevice(h->cfg.device));
    int rc = launch(h, h->stream, B, x, ldx, const_cast<double *>(lambda), ldl, w, ldw, 1, 1, nullptr, 0, 0, 3, 0, nullptr,
                    d, ldd, z, z ? ldz : 0);
    if (rc) return rc;
    if (!(flags & TOLCUDA_NO_SYNC)) CU(cudaStreamSynchronize(h->stream));
    return 0;
}

int tolcuda_problem_pattern_csc(int formulation, int ts, int *colptr, int *rowidx, int *perm) {
    if ((formulation != TOLCUDA_G7 && formulation != TOLCUDA_S10) || ts < 1 || !colptr || !rowidx) return TOLCUDA_EINVAL;
    std::vector<int> cp, ri, pm;
    pattern_csc(formulation, ts, cp, ri, pm);
    std::memcpy(colptr, cp.data(), sizeof(int) * cp.size());
    std::memcpy(rowidx, ri.data(), sizeof(int) * ri.size());
    if (perm) std::memcpy(perm, pm.data(), sizeof(int) * pm.size());
    return 0;
}

int tolcuda_repack_csc_device(tolcuda_handle h, long B, const double *G, long ldG, double *Gcsc, long ldC, int flags) {
    if (!h || B < 0) return TOLCUDA_EINVAL;
    const FgConst &c = h->c;
    if (B > 0 && (!G || !Gcsc || ldG < c.neG || ldC < c.neG)) {
        set_error("tolcuda_repack_csc_device: null pointer or leading dimension shorter than the row");
        return TOLCUDA_EINVAL;
    }
    CU(cudaSetDevice(h->cfg.device));
    if (!h->d_perm) {
        std::vector<int> cp, ri, pm;
        pattern_csc(c.form, c.ts, cp, ri, pm);
        CU(cudaMalloc(&h->d_perm, sizeof(int) * pm.size()));
        CU(cudaMemcpy(h->d_perm, pm.data(), sizeof(int) * pm.size(), cudaMemcpyHostToDevice));
    }
    cudaError_t e = repack_launch(c.neG, h->d_perm, B, G, ldG, Gcsc, ldC, h->stream);
    if (e != cudaSuccess) return cuda_fail(e, "repack_launch");
    h->launches += B > 0 ? (B + 65534) / 65535 : 0;
    if (!(flags & TOLCUDA_NO_SYNC)) CU(cudaStreamSynchronize(h->stream));
    return 0;
}

int tolcuda_set_host_threads(tolcuda_handle h, int threads) {
    if (!h || threads < 0) return TOLCUDA_EINVAL;
    h->host_threads = threads;
    h->pool.reset();  // rebuilt with the new size by the next host-pointer batch call
    return 0;
}

// Execution-strategy options: every value of every option produces the same bits in F and G.
int tolcuda_set_option(tolcuda_handle h, const char *name, long value) {
    if (!h || !name) return TOLCUDA_EINVAL;
    const std::string k(name);
    auto in = [&](long lo, long hi) { return value >= lo && value <= hi; };
    bool ok = true;
    if (k == "kernel") ok = in(0, 2), h->kernel = ok ? (int)value : h->kernel;
    else if (k == "per") {
        ok = in(0, 4);
        if (ok && value == 0) h->per = 2, h->per_auto = 1;
        else if (ok) h->per = (int)value, h->per_auto = 0;
    } else if (k == "per_min_waves") ok = in(-1, 1 << 20), h->per_min_waves = ok ? (int)value : h->per_min_waves;
    else if (k == "tail_x4") ok = in(-1, 64), h->tail_waves_x4 = ok ? (int)value : h->tail_waves_x4;
    else if (k == "lwarps") ok = in(0, 8), h->lwarps = ok ? (int)value : h->lwarps;
    else if (k == "zero_copy") ok = in(0, 1), h->zero_copy = ok ? (int)value : h->zero_copy;
    else if (k == "compact_host") ok = in(0, 1), h->compact_host = ok ? (int)value : h->compact_host;
    else if (k == "chunk_mb") ok = in(1, 4096), h->chunk_mb = ok ? (int)value : h->chunk_mb;
    else if (k == "full_rows_pct") ok = in(0, 100), h->full_rows_pct = ok ? (int)value : h->full_rows_pct;
    else {
        set_error("tolcuda_set_option: unknown option " + k);
        return TOLCUDA_EINVAL;
    }
    if (!ok) {
        set_error("tolcuda_set_option: value out of range for " + k);
        return TOLCUDA_EINVAL;
    }
    return 0;
}

int tolcuda_set_dump_dir(tolcuda_handle h, const char *dir) {
    if (!h) return TOLCUDA_EINVAL;
    h->dump_dir = dir ? dir : "";
    h->dump_warned = false;
    return 0;
}

int tolcuda_write_dump(const char *path, const double *values, long count) {
    if (!path || count < 0 || (count > 0 && !values)) return TOLCUDA_EINVAL;
    return write_value_dump(path, values, count);
}

int tolcuda_write_wind_dump(const char *path, int wind_model, int ts, const double *x) {
    if (!path || ts < 1 || !x) return TOLCUDA_EINVAL;
    return write_wind_dump(path, wind_model, ts, x);
}

int tolcuda_bind_global(tolcuda_handle h) {
    std::lock_guard<std::mutex> lk(g_mu);
    g_bound = h;
    return 0;
}

void DEFINEGusrfg_(int *Status, int *n, double x[], int *needF, int *neF, double F[], int *needG,
                   int *neG, double G[], char *cu, int *lencu, int iu[], int *leniu, double ru[],
                   int *lenru) {
    (void)cu, (void)lencu, (void)iu, (void)leniu, (void)ru, (void)lenru;  // unused, as in the reference
    tolcuda_ctx *h;
    {
        std::lock_guard<std::mutex> lk(g_mu);
        h = g_bound;
    }
    int rc;
    if (!h) {
        set_error("DEFINEGusrfg_: no context bound (call tolcuda_bind_global first)");
        rc = TOLCUDA_ENOCTX;
    } else if ((n && *n != h->c.n) || (neF && *needF > 0 && *neF != h->c.neF) ||
               (neG && *needG > 0 && *neG != h->c.neG)) {
        set_error("DEFINEGusrfg_: n/neF/neG differ from the bound context's problem");
        rc = TOLCUDA_EINVAL;
    } else {
        // the reference's dump files, in its order: X before anything is evaluated, W inside modelWind, F and G
        // after they have been computed (src/DefineFG.cpp:16-46).  A file that cannot be written is reported once
        // and does not stop the solve.
        const bool dump = !h->dump_dir.empty();
        auto dumped = [&](int e) {
            if (e && !h->dump_warned) {
                std::fprintf(stderr, "tolcuda: dump files: %s\n", tolcuda_last_error());
                h->dump_warned = true;
            }
        };
        const std::string dir = dump ? h->dump_dir + "/" : std::string();
        if (dump) {
            dumped(write_value_dump(dir + "Xoutput.txt", x, h->c.n));
            if (h->c.wind != TOLCUDA_WIND_CUBE) dumped(write_wind_dump(dir + "Woutput.txt", h->c.wind, h->c.ts, x));
        }
        rc = tolcuda_eval(h, x, *needF, F, *needG, G);
        if (dump && !rc) {
            if (*needF > 0) dumped(write_value_dump(dir + "Foutput.txt", F, h->c.neF));
            if (*needG > 0) dumped(write_value_dump(dir + "Goutput.txt", G, h->c.neG));
        }
    }
    if (rc) {
        std::fprintf(stderr, "tolcuda: user function failed (%d): %s\n", rc, tolcuda_last_error());
        if (Status) *Status = -2;  // SNOPT: terminate
    }
}

}  // extern "C"
