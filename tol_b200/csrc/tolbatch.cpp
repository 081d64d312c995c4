// tolbatch -- batch driver over libtolcuda: the counterpart of the reference's CLI `tol E N U Eg Ng Ug Rg
// aircraft mission` (src/tol.cpp:38-53, src/arguments.cpp:32-46), which builds ONE problem and hands it to
// SNOPT.  tolbatch builds the same problem from the same positional arguments and the same .param files,
// takes the reference's initial guess, spreads B perturbed copies of it (or B trajectories read from a
// file) over the GPUs of the box by trajectory index, evaluates F and G for all of them through
// tolcuda_eval_batch, gathers the rows in one pinned host buffer and reports throughput plus a
// per-trajectory summary.  It uses nothing but the C ABI of include/tolcuda.h.
//
//   tolbatch E N U Eg Ng Ug Rg aircraft mission [--root DIR/] [--ts N] [--batch B] [--gpus G]
//            [--seed S] [--perturb REL,ABS] [--x-file raw_f64] [--steps K] [--json out.json]
//            [--results DIR [--nresults K]]   the reference's snopt_results.json (src/problem.cpp:1247-1365)
//                                             for the first K trajectories, as DIR/snopt_results_<b>.json
//            [--summary-only]                 screening mode: only x goes to the GPUs and only the per-trajectory
//                                             summary the kernels compute on the fly comes back
//                                             (tolcuda_eval_batch_summary without F or G: objective, worst defect,
//                                             worst boundary violation), no F/G rows on the host
//            [--host-path compact|full|auto|P]  how G reaches the host rows: compact rows across PCIe + expansion by host
//                                             threads (default), every G value across PCIe, P % of the chunks as full
//                                             rows and the rest compact (copy engines and cores side by side), or
//                                             whatever calibration calls find fastest on this box (the answer depends
//                                             on the host: its DMA ingest rate against its cores' store rate)
//            [--gather-gpu D]                 after the host gather: the same batch once more with every GPU's shard
//                                             written straight into GPU D's memory by the shards' own kernels
//                                             (tolcuda_gather_*: NVLink peer stores, no host in between), timed, and
//                                             compared bit for bit with the rows of the host gather
//            [--goals FILE]                   one goal per trajectory: line b of FILE is `Eg Ng Ug Rg` (arguments 4-7 of
//                                             the reference CLI) for trajectory b, whose initial guess is then the
//                                             reference's for that goal; B = the line count (--batch, if given, must
//                                             equal it).  One launch per device for all goals (tolcuda_eval_batch_goals);
//                                             --results writes each trajectory's own goal.  Not with --gather-gpu.
#include <chrono>
#include <cctype>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "../../include/tolcuda.h"

namespace {

struct Args {
    double enu[3] = {0, 0, 0}, goal[4] = {0, 0, 0, 0};
    std::string aircraft, mission, root = "./", xfile, json, results, host_path = "compact", goals_file;
    std::vector<double> goals;  // --goals: 4 per trajectory, xg, yg, zg, rg in NED (tolcuda_config.goal)
    int ts = 0, batch = 4096, gpus = 0, steps = 3, nresults = 4, gather_gpu = -1;
    bool summary_only = false;
    uint64_t seed = 1;
    double rel = 0.05, abs_ = 0.01;
};

// splitmix64: one independent stream per trajectory index, so the batch does not depend on the sharding
struct Rng {
    uint64_t s;
    explicit Rng(uint64_t seed) : s(seed) {}
    uint64_t next() {
        uint64_t z = (s += 0x9e3779b97f4a7c15ULL);
        z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ULL;
        z = (z ^ (z >> 27)) * 0x94d049bb133111ebULL;
        return z ^ (z >> 31);
    }
    double sym() { return 2.0 * ((next() >> 11) * (1.0 / 9007199254740992.0)) - 1.0; }  // U(-1, 1)
};

void die(const std::string &msg) {
    std::fprintf(stderr, "tolbatch: %s\n", msg.c_str());
    std::exit(2);
}

void check(int rc, const char *what) {
    if (rc) die(std::string(what) + " failed (" + std::to_string(rc) + "): " + tolcuda_last_error());
}

// --goals FILE: every line `Eg Ng Ug Rg` (ENU, radius), stored as the NED goal tolcuda_config_from_files makes of the
// same command-line arguments (reference src/problem.cpp:24-27); anything else in the file is refused
void read_goals(const std::string &path, std::vector<double> &out) {
    FILE *f = std::fopen(path.c_str(), "r");
    if (!f) die("cannot open goal file " + path);
    std::string text;
    char buf[4096];
    for (size_t got; (got = std::fread(buf, 1, sizeof buf, f)) > 0;) text.append(buf, got);
    std::fclose(f);
    size_t pos = 0;
    for (long line = 1; pos < text.size(); line++) {
        size_t end = text.find('\n', pos);
        if (end == std::string::npos) end = text.size();
        const std::string ln = text.substr(pos, end - pos);
        pos = end + 1;
        double v[4];
        const char *p = ln.c_str();
        for (int i = 0; i < 4; i++) {
            char *q;
            v[i] = std::strtod(p, &q);
            if (q == p || !std::isfinite(v[i])) die(path + ":" + std::to_string(line) + ": want `Eg Ng Ug Rg`");
            p = q;
        }
        while (std::isspace((unsigned char)*p)) p++;
        if (*p) die(path + ":" + std::to_string(line) + ": want `Eg Ng Ug Rg`, found more");
        out.insert(out.end(), {v[1], v[0], -v[2], v[3]});
    }
    if (out.empty()) die(path + ": no goals");
}

Args parse(int argc, char **argv) {
    if (argc < 10)
        die("usage: tolbatch E N U Eg Ng Ug Rg aircraft mission [--root DIR/] [--ts N] [--batch B] [--gpus G] "
            "[--seed S] [--perturb REL,ABS] [--x-file F] [--steps K] [--json OUT] [--results DIR [--nresults K]] [--summary-only] "
            "[--gather-gpu D] [--goals FILE]");
    Args a;
    bool batch_set = false;
    for (int i = 0; i < 3; i++) a.enu[i] = std::atof(argv[1 + i]);  // as src/arguments.cpp:35-41 (atof)
    for (int i = 0; i < 4; i++) a.goal[i] = std::atof(argv[4 + i]);
    a.aircraft = argv[8];
    a.mission = argv[9];
    for (int i = 10; i < argc; i++) {
        const std::string k = argv[i];
        auto val = [&]() -> const char * {
            if (i + 1 >= argc) die("missing value after " + k);
            return argv[++i];
        };
        if (k == "--root") a.root = val();
        else if (k == "--ts") a.ts = std::atoi(val());
        else if (k == "--batch") a.batch = std::atoi(val()), batch_set = true;
        else if (k == "--goals") a.goals_file = val();
        else if (k == "--gpus") a.gpus = std::atoi(val());
        else if (k == "--steps") a.steps = std::atoi(val());
        else if (k == "--seed") a.seed = std::strtoull(val(), nullptr, 10);
        else if (k == "--x-file") a.xfile = val();
        else if (k == "--json") a.json = val();
        else if (k == "--results") a.results = val();
        else if (k == "--nresults") a.nresults = std::atoi(val());
        else if (k == "--summary-only") a.summary_only = true;
        else if (k == "--gather-gpu") a.gather_gpu = std::atoi(val());
        else if (k == "--host-path") a.host_path = val();
        else if (k == "--perturb") {
            if (std::sscanf(val(), "%lf,%lf", &a.rel, &a.abs_) != 2) die("--perturb wants REL,ABS");
        } else die("unknown option " + k);
    }
    if (!a.root.empty() && a.root.back() != '/') a.root += '/';  // the reference concatenates paths
    if (a.batch < 1) die("--batch must be at least 1");
    if (a.steps < 1) die("--steps must be at least 1");
    if (a.nresults < 0) die("--nresults must not be negative");
    if (a.gpus < 0) die("--gpus must not be negative");
    if (a.ts < 0) die("--ts must not be negative");
    if (a.host_path != "compact" && a.host_path != "full" && a.host_path != "auto" &&
        !(std::isdigit((unsigned char)a.host_path[0]) && std::atoi(a.host_path.c_str()) <= 100))
        die("--host-path wants compact, full, auto or a percentage 0..100");
    if (a.gather_gpu >= 0 && a.summary_only) die("--gather-gpu gathers F and G rows: not available with --summary-only");
    if (!a.goals_file.empty()) {
        if (a.gather_gpu >= 0) die("--goals cannot be combined with --gather-gpu (the gather protocol has no goal table)");
        read_goals(a.goals_file, a.goals);
        const long lines = (long)a.goals.size() / 4;
        if (batch_set && lines != a.batch)
            die(a.goals_file + ": " + std::to_string(lines) + " goals for --batch " + std::to_string(a.batch));
        a.batch = (int)lines;
    }
    return a;
}

}  // namespace

int main(int argc, char **argv) {
    const Args a = parse(argc, argv);
    int ndev = 0;
    check(tolcuda_device_count(&ndev), "device query");
    const int G = a.gpus > 0 ? a.gpus : ndev;
    if (G < 1 || G > ndev) die("asked for " + std::to_string(G) + " GPUs, " + std::to_string(ndev) + " present");

    std::vector<tolcuda_handle> h(G, nullptr);
    for (int g = 0; g < G; g++)
        check(tolcuda_create_from_files(a.root.c_str(), a.aircraft.c_str(), a.mission.c_str(), a.enu[0], a.enu[1],
                                        a.enu[2], a.goal[0], a.goal[1], a.goal[2], a.goal[3], a.ts, g, &h[g]),
              "tolcuda_create_from_files");
    int n, neF, neG;
    check(tolcuda_dims(h[0], &n, &neF, &neG), "tolcuda_dims");
    tolcuda_config cfg;
    check(tolcuda_get_config(h[0], &cfg), "tolcuda_get_config");
    const int ts = cfg.ts, B = a.batch;
    const long ldx = tolcuda_padded_ld(n), ldF = tolcuda_padded_ld(neF), ldG = tolcuda_padded_ld(neG);
    std::printf("TOLBATCH: %s / %s, ts=%d, n=%d neF=%d neG=%d, %d trajectories on %d GPU(s)\n", a.mission.c_str(),
                a.aircraft.c_str(), ts, n, neF, neG, B, G);

    double *X, *F = nullptr, *Gv = nullptr, *S = nullptr;
    check(tolcuda_host_alloc(sizeof(double) * ldx * B, (void **)&X), "pinned x");
    if (a.summary_only) {
        check(tolcuda_host_alloc(sizeof(double) * 4 * B, (void **)&S), "pinned summary");
    } else {
        check(tolcuda_host_alloc(sizeof(double) * ldF * B, (void **)&F), "pinned F");
        check(tolcuda_host_alloc(sizeof(double) * ldG * B, (void **)&Gv), "pinned G");
    }

    // inputs: the reference's initial trajectory, perturbed per trajectory index, or a raw float64 file
    std::vector<double> x0(n);
    check(tolcuda_problem_initial_guess(&cfg, x0.data()), "initial guess");
    if (!a.xfile.empty()) {
        FILE *f = std::fopen(a.xfile.c_str(), "rb");
        if (!f) die("cannot open " + a.xfile);
        for (int b = 0; b < B; b++)
            if (std::fread(X + (size_t)b * ldx, sizeof(double), n, f) != (size_t)n) die("short read from " + a.xfile);
        std::fclose(f);
    } else {
        for (int b = 0; b < B; b++) {
            Rng r(a.seed * 0x100000001b3ULL + (uint64_t)b);
            double *xb = X + (size_t)b * ldx;
            if (!a.goals.empty()) {  // the reference's initial guess for this trajectory's goal (G7's rotates by chi_d)
                tolcuda_config cb = cfg;
                for (int i = 0; i < 4; i++) cb.goal[i] = a.goals[4 * (size_t)b + i];
                check(tolcuda_problem_initial_guess(&cb, x0.data()), "initial guess");
            }
            // with --goals and --perturb 0,0 every row is its goal's x0 itself (x0 + 0*u would turn -0.0 into +0.0), so
            // its result file is the one a single-goal run writes for trajectory 0
            const bool copy = b == 0 || (!a.goals.empty() && a.rel == 0.0 && a.abs_ == 0.0);
            for (int i = 0; i < n; i++) {
                const double u = r.sym(), up = r.sym();
                xb[i] = copy ? x0[i] : x0[i] * (1.0 + a.rel * u) + a.abs_ * up;  // trajectory 0 is x0 itself
            }
        }
    }

    // evaluate: one host thread per device, contiguous block of trajectory indices each, no collective
    const int per_dev = (B + G - 1) / G;
    for (int g = 0; g < G && !a.goals.empty(); g++) {  // each device's context holds its shard's rows of the goal table
        const int b0 = std::min(B, g * per_dev), b1 = std::min(B, b0 + per_dev);
        check(tolcuda_set_goals(h[g], b1 - b0, a.goals.data() + 4 * (size_t)b0, 4), "tolcuda_set_goals");
    }
    std::vector<double> secs(G, 0.0);
    double best = 1e300;
    // share of the chunks that cross PCIe as full rows (tolcuda_set_option "full_rows_pct"; 100 = all of them)
    auto set_share = [&](int pct) {
        for (int g = 0; g < G; g++) {
            check(tolcuda_set_option(h[g], "compact_host", pct == 100 ? 0 : 1), "tolcuda_set_option");
            check(tolcuda_set_option(h[g], "full_rows_pct", pct == 100 ? 0 : pct), "tolcuda_set_option");
        }
    };
    int share = a.host_path == "full" ? 100 : (std::isdigit((unsigned char)a.host_path[0]) ? std::atoi(a.host_path.c_str()) : 0);
    // --host-path auto: untimed calls (two per candidate, the first one allocates) of all compact, all full, then the
    // share t_c / (t_c + t_f) that would balance copy engines and cores; the fastest wins, compact unless 3 % faster
    std::vector<std::pair<int, double>> cal;
    int ncal = (a.host_path == "auto" && !a.summary_only) ? 6 : 0;
    for (int step = -ncal; step < a.steps; step++) {
        if (step < 0) {
            const int k = (step + ncal) / 2;
            if (k == 0) share = 0;
            else if (k == 1) share = 100;
            else share = (int)std::lround(100.0 * cal[0].second / (cal[0].second + cal[1].second));
        }
        if (step == 0 && ncal) {
            share = 0;
            double tb = cal[0].second;
            std::printf("TOLBATCH: host path calibration:");
            for (auto &c : cal) {
                std::printf(" %d %% full rows %.3f ms;", c.first, 1e3 * c.second);
                if (c.second < 0.97 * cal[0].second && c.second < tb) tb = c.second, share = c.first;
            }
            std::printf(" -> %d %% full rows\n", share);
        }
        if (step <= 0) set_share(share);
        std::vector<std::thread> th;
        const auto t0 = std::chrono::steady_clock::now();
        for (int g = 0; g < G; g++)
            th.emplace_back([&, g]() {
                const int b0 = std::min(B, g * per_dev), b1 = std::min(B, b0 + per_dev);
                const auto s0 = std::chrono::steady_clock::now();
                if (b1 > b0 && !a.goals.empty())
                    check(a.summary_only
                              ? tolcuda_eval_batch_goals(h[g], 0, b1 - b0, X + (size_t)b0 * ldx, ldx, nullptr, 0, nullptr, 0,
                                                         S + (size_t)b0 * 4, 4, TOLCUDA_HOST_PTRS)
                              : tolcuda_eval_batch_goals(h[g], 0, b1 - b0, X + (size_t)b0 * ldx, ldx, F + (size_t)b0 * ldF,
                                                         ldF, Gv + (size_t)b0 * ldG, ldG, nullptr, 0,
                                                         TOLCUDA_NEED_F | TOLCUDA_NEED_G | TOLCUDA_HOST_PTRS),
                          "tolcuda_eval_batch_goals");
                else if (b1 > b0 && a.summary_only)
                    check(tolcuda_eval_batch_summary(h[g], b1 - b0, X + (size_t)b0 * ldx, ldx, nullptr, 0, nullptr, 0,
                                                     S + (size_t)b0 * 4, 4, TOLCUDA_HOST_PTRS),
                          "tolcuda_eval_batch_summary");
                else if (b1 > b0)
                    check(tolcuda_eval_batch(h[g], b1 - b0, X + (size_t)b0 * ldx, ldx, F + (size_t)b0 * ldF, ldF,
                                             Gv + (size_t)b0 * ldG, ldG, TOLCUDA_NEED_F | TOLCUDA_NEED_G | TOLCUDA_HOST_PTRS),
                          "tolcuda_eval_batch");
                secs[g] = std::chrono::duration<double>(std::chrono::steady_clock::now() - s0).count();
            });
        for (auto &t : th) t.join();
        const double wall = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        if (step < 0) {
            if ((step + ncal) % 2) cal.emplace_back(share, wall);  // the second call of a candidate counts
            continue;
        }
        best = std::min(best, wall);
        std::printf("TOLBATCH: step %d: %.3f ms wall, %.4g node-evals/s end to end (host x -> host %s)\n", step,
                    1e3 * wall, (double)B * ts / wall, a.summary_only ? "summary" : "F,G");
    }

    // per-trajectory summary: objective, worst defect, worst boundary violation, finiteness
    const int nb = cfg.formulation == TOLCUDA_G7 ? 12 : 11;
    long nonfinite = 0;
    double worst_defect = 0.0;
    std::vector<double> obj(B), defect(B), bnd(B);
    for (int b = 0; b < B && a.summary_only; b++) {
        // what the kernels reduced on the fly: [objective, max |defect|, max boundary violation, sum defect^2]
        const double *Sb = S + (size_t)b * 4;
        for (int i = 0; i < 4; i++) nonfinite += !std::isfinite(Sb[i]);
        obj[b] = Sb[0], defect[b] = Sb[1], bnd[b] = Sb[2];
        worst_defect = std::fmax(worst_defect, Sb[1]);
    }
    for (int b = 0; b < B && !a.summary_only; b++) {
        const double *Fb = F + (size_t)b * ldF, *Gb = Gv + (size_t)b * ldG;
        double d = 0.0, e = 0.0;
        // NaN if a row is NaN, as the summary's maxima (tolcuda.h): std::fmax would drop it
        const auto max_nan = [](double u, double v) { return (u > v || u != u) ? u : v; };
        for (int i = 1; i < neF - nb; i++) d = max_nan(d, std::fabs(Fb[i]));
        for (int i = neF - nb; i < neF; i++) e = max_nan(e, std::fabs(Fb[i]));
        for (int i = 0; i < neF; i++) nonfinite += !std::isfinite(Fb[i]);
        for (int i = 0; i < neG; i++) nonfinite += !std::isfinite(Gb[i]);
        obj[b] = Fb[0], defect[b] = d, bnd[b] = e;
        worst_defect = std::fmax(worst_defect, d);
    }
    std::printf("TOLBATCH: best %.3f ms, %.4g node-evals/s; F[0] of trajectory 0 = %.17g; worst defect %.6g; "
                "non-finite values %ld\n",
                1e3 * best, (double)B * ts / best, obj[0], worst_defect, nonfinite);

    // ---- the same batch gathered on ONE GPU by the shards' own kernels (tolcuda_gather_*), against the host gather
    bool gather_same = true;
    if (a.gather_gpu >= 0) {
        const int D = a.gather_gpu;
        if (D >= G) die("--gather-gpu " + std::to_string(D) + ": only " + std::to_string(G) + " GPU(s) in use");
        const int per = (B + G - 1) / G;
        std::vector<double *> dx(G, nullptr);
        for (int g = 0; g < G; g++) {
            const int b0 = std::min(B, g * per), b1 = std::min(B, b0 + per);
            if (b1 <= b0) continue;
            check(tolcuda_device_alloc(g, sizeof(double) * ldx * (b1 - b0), (void **)&dx[g]), "device x");
            check(tolcuda_copy_to_device(g, dx[g], X + (size_t)b0 * ldx, sizeof(double) * ldx * (b1 - b0)), "x to device");
        }
        std::vector<tolcuda_gather_handle> gh(G, nullptr);
        check(tolcuda_gather_create(h[D], B, G, D, &gh[D], nullptr), "tolcuda_gather_create");
        for (int g = 0; g < G; g++)
            if (g != D) check(tolcuda_gather_attach(h[g], B, G, g, D, gh[D], nullptr, &gh[g]), "tolcuda_gather_attach");
        double *dF = nullptr, *dG = nullptr;
        long gldF = 0, gldG = 0;
        double gbest = 1e300;
        for (int step = 0; step < a.steps + 1; step++) {  // one thread enqueues for every device: all calls are asynchronous
            const auto t0 = std::chrono::steady_clock::now();
            for (int g = 0; g < G; g++)
                if (g != D && dx[g]) check(tolcuda_gather_send(gh[g], dx[g], ldx, 4), "tolcuda_gather_send");
            check(tolcuda_gather_collect(gh[D], dx[D], ldx, 4, &dF, &gldF, &dG, &gldG), "tolcuda_gather_collect");
            for (int g = 0; g < G; g++)
                if (g != D) check(tolcuda_synchronize(h[g]), "tolcuda_synchronize");
            const double wall = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
            if (step > 0) gbest = std::min(gbest, wall);
        }
        // rows on GPU D against the rows of the host gather, bit for bit, in slabs of 256 trajectories
        const int slab = 256;
        std::vector<double> tF((size_t)slab * gldF), tG((size_t)slab * gldG);
        for (int b0 = 0; b0 < B; b0 += slab) {
            const int nbk = std::min(slab, B - b0);
            check(tolcuda_copy_to_host(D, tF.data(), dF + (size_t)b0 * gldF, sizeof(double) * gldF * nbk), "F rows to host");
            check(tolcuda_copy_to_host(D, tG.data(), dG + (size_t)b0 * gldG, sizeof(double) * gldG * nbk), "G rows to host");
            for (int b = 0; b < nbk; b++) {
                gather_same = gather_same && !std::memcmp(tF.data() + (size_t)b * gldF, F + (size_t)(b0 + b) * ldF, sizeof(double) * neF);
                gather_same = gather_same && !std::memcmp(tG.data() + (size_t)b * gldG, Gv + (size_t)(b0 + b) * ldG, sizeof(double) * neG);
            }
        }
        std::printf("TOLBATCH: gather on GPU %d (device x -> F,G rows of all %d trajectories in its memory): best %.3f ms, "
                    "%.4g node-evals/s; rows bit-identical to the host gather: %s\n",
                    D, B, 1e3 * gbest, (double)B * ts / gbest, gather_same ? "yes" : "NO");
        for (int g = 0; g < G; g++)
            if (g != D) tolcuda_gather_close(gh[g]);
        tolcuda_gather_close(gh[D]);
        for (int g = 0; g < G; g++) tolcuda_device_free(g, dx[g]);
    }

    if (!a.json.empty()) {
        FILE *f = std::fopen(a.json.c_str(), "w");
        if (!f) die("cannot write " + a.json);
        std::fprintf(f, "{\n \"mission\": \"%s\", \"aircraft\": \"%s\", \"ts\": %d, \"n\": %d, \"neF\": %d, \"neG\": %d,\n",
                     a.mission.c_str(), a.aircraft.c_str(), ts, n, neF, neG);
        std::fprintf(f, " \"batch\": %d, \"gpus\": %d, \"best_ms\": %.6f, \"node_evals_per_s\": %.6g, \"nonfinite\": %ld,\n", B, G,
                     1e3 * best, (double)B * ts / best, nonfinite);
        // summary-only: max_abs_boundary is the worst boundary VIOLATION (G7's dist <= dmax row counts only when exceeded)
        std::fprintf(f, " \"summary_only\": %s,\n", a.summary_only ? "true" : "false");
        std::fprintf(f, " \"trajectories\": [\n");
        for (int b = 0; b < B; b++)
            std::fprintf(f, "  {\"b\": %d, \"objective\": %.17g, \"max_abs_defect\": %.17g, \"max_abs_boundary\": %.17g}%s\n", b,
                         obj[b], defect[b], bnd[b], b + 1 < B ? "," : "");
        std::fprintf(f, " ]\n}\n");
        std::fclose(f);
    }
    if (!a.results.empty() && a.summary_only) die("--results needs the F rows: not available with --summary-only");
    if (!a.results.empty())
        for (int b = 0; b < std::min(B, a.nresults); b++) {
            const std::string path = a.results + "/snopt_results_" + std::to_string(b) + ".json";
            tolcuda_config cb = cfg;  // "args" holds the trajectory's own goal
            for (int i = 0; i < 4 && !a.goals.empty(); i++) cb.goal[i] = a.goals[4 * (size_t)b + i];
            check(tolcuda_write_results_json(&cb, a.aircraft.c_str(), a.mission.c_str(), a.enu[0], a.enu[1], a.enu[2],
                                             X + (size_t)b * ldx, obj[b], path.c_str()),
                  "tolcuda_write_results_json");
        }
    for (int g = 0; g < G; g++) tolcuda_destroy(h[g]);
    tolcuda_host_free(X), tolcuda_host_free(F), tolcuda_host_free(Gv), tolcuda_host_free(S);
    return (nonfinite || !gather_same) ? 1 : 0;
}
