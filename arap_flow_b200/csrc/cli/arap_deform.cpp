// arap_deform -- command-line front end with the argv / list-file / environment contract of the reference's
// ARAP/deformation/src/main.cpp:162-241, as driven by para_gen.py:178-214, run_arap.py:10-15 and generate.py:
//   arap_deform RGB MASK CSTR FLO_out WRGB_out WMASK_out [BFLO_out OCC_out]      or      arap_deform LISTFILE
// The two optional outputs (8 tokens instead of 6, in argv or on a list line) are the backward flow (.flo) and the
// occlusion of frame 1 (PNG, 255 = occluded; DESIGN.md 4.3); lines of 6 tokens run and write exactly what they always did.
// Differences from the reference are on the inside only: consecutive list entries of one image size are
// solved together (several problems per cooperative launch), nothing is interpreted from $ARAP_PLAN.
//
// Resident worker (SURVEY.md 8f N2, second half).  para_gen.py spawns one solver process per dispatch
// (para_gen.py:178-200), and every process pays CUDA context creation + buffer allocation (0.6-4 s) before
// its first pair -- more than the GPU work of a handful of pairs.  Two extra invocations remove that cost
// without touching the driver's calling convention:
//   arap_deform --serve SPOOLDIR [--warm WxH]
//                                    one long-lived process per GPU: keeps the context, the plan and the
//                                    device buffers, and runs every list file dropped into SPOOLDIR; --warm
//                                    builds plan + buffers for that image size at start-up
//   ARAP_SERVER=SPOOLDIR arap_deform LISTFILE | RGB MASK CSTR FLO WRGB WMASK [BFLO OCC]
//                                    thin client: same argv contract, same "Saved" lines, same exit code;
//                                    the work is done by the server that watches SPOOLDIR
// Protocol: the client writes SPOOLDIR/<id>.job.tmp (the 6- or 8-tuples, one per line), renames it to <id>.job and
// waits for <id>.done (first line = exit code); the server renames <id>.job to <id>.run while it works.
// SPOOLDIR/stop makes the server exit.
#include "../../../include/Opt.h"
#include "../../../include/arapb200.h"
#include "image_io.h"

#include <chrono>
#include <csignal>
#include <cstdio>
#include <cstring>
#include <dirent.h>
#include <sys/stat.h>
#include <thread>
#include <unistd.h>
#include <cstdlib>
#include <fstream>
#include <algorithm>
#include <deque>
#include <future>
#include <memory>
#include <sstream>
#include <string>
#include <vector>

using namespace arapcli;

struct InputPaths {
    std::string rgb, mask, cstr, flo, wrgb, wmask;
    std::string bflo, occ; // both empty = a 6-token line: no backward flow / occlusion
    bool extras() const { return !bflo.empty(); }
};

static void usage()
{
    puts("Usage:\n");
    puts("./arap_deform RGB Mask Constraint Flow warped_RGB warped_Mask\n");
    puts("Deform the object of an image as rigidly as possible so that the given point matches are met,");
    puts("and write the dense flow, the warped image and the warped mask.\n");
    puts("RGB \t\t [input]  path to an input RGB image (.png only)");
    puts("Mask\t\t [input]  path to an input mask image (.png only), red channel 0 for object, non-zero for background");
    puts("Constraint \t [input]  path to list of constraints, text file: n, then n lines x1 y1 x2 y2");
    puts("Flow \t\t [output] path to optical flow (.flo only)");
    puts("warped_RGB \t [output] path to output warped image (.png), all intermediate directories must exist");
    puts("warped_Mask \t [output] path to output warped mask (.png), all intermediate directories must exist");
    puts("\n./arap_deform RGB Mask Constraint Flow warped_RGB warped_Mask Backward_Flow Occlusion\n");
    puts("also writes, from the same solve and warp:");
    puts("Backward_Flow \t [output] path to the backward flow (.flo): from each frame-2 pixel to its frame-1 source point, 0 where nothing landed");
    puts("Occlusion \t [output] path to the occlusion of frame 1 (.png): 255 where a pixel is not visible in frame 2, else 0");
    puts("\n./arap_deform LISTFILE   (one such 6- or 8-tuple per line, both kinds may be mixed; further tokens are ignored)");
    puts("./arap_deform --serve SPOOLDIR [--warm WxH]   (resident worker: runs the list files that clients with ARAP_SERVER=SPOOLDIR");
    puts("                                               submit; --warm pre-builds the plan and buffers for that image size)");
    puts("Environment: ARAP_PLAN = path of the ARAP energy file (default ./arap_plan.t); CUDA_VISIBLE_DEVICES selects the GPU;");
    puts("             ARAP_BATCH = problems solved together (default 8: two cooperative launches of four)");
    puts("             ARAP_PCG_RTOL = opt-in relative PCG tolerance, e.g. 1e-3 (default 0: fixed 400 iterations)");
    puts("             ARAP_SOLVER = gaussNewtonGPU (default) | LMGPU (opt-in: trust region + Q-based exit of the linear loops)");
    puts("             ARAP_GN_RTOL = opt-in relative cost-decrease tolerance of the Gauss-Newton steps (default 0: fixed 8 steps)");
    puts("             ARAP_SERVER = spool directory of a running `arap_deform --serve`: hand the work to it instead of solving here");
}

struct Loaded {
    ImageRGB rgb;
    std::vector<uint8_t> mask_red;
    std::vector<int32_t> cstr;
    std::vector<float> flow;
    std::vector<uint8_t> wrgb, wmask;
    std::vector<float> bflow;  // only for 8-token lines
    std::vector<uint8_t> occ;
};

// the GPU context that outlives a list file (and, in --serve mode, every client request)
struct Context {
    arapb200_batch* ctx = NULL;
    int W = 0, H = 0;
    long saved = 0;
    ~Context() { if (ctx) arapb200_batch_destroy(ctx); }
};

static bool read_list(const char* path, std::vector<InputPaths>& lines)
{
    std::ifstream infile(path);
    if (!infile) return false;
    std::string line;
    while (getline(infile, line)) {
        std::stringstream s(line);
        InputPaths p;
        if (s >> p.rgb >> p.mask >> p.cstr >> p.flo >> p.wrgb >> p.wmask) {
            std::string b, o;
            if (s >> b >> o) { p.bflo = b; p.occ = o; }
            lines.push_back(p);
        }
    }
    return true;
}

struct Settings {
    // the solver budget is a compile-time constant of the reference: main.cpp:215-221
    int nCont = 19, nGN = 8, nPCG = 400;
    int batch = 8;
    // opt-in, off by default: convergence-aware PCG loops (changes results; include/arapb200.h)
    double pcg_rtol = 0.0, gn_rtol = 0.0;
    bool lm = false;     // ARAP_SOLVER=LMGPU: the reference's other solver kind (o.t:121-124), default gaussNewtonGPU
    bool timing = false; // ARAP_TIMING=1: per-stage wall times on stderr
    Settings()
    {
        if (getenv("ARAP_BATCH")) batch = atoi(getenv("ARAP_BATCH"));
        if (batch < 1) batch = 1;
        if (getenv("ARAP_PCG_RTOL")) pcg_rtol = atof(getenv("ARAP_PCG_RTOL"));
        if (getenv("ARAP_GN_RTOL")) gn_rtol = atof(getenv("ARAP_GN_RTOL"));
        timing = getenv("ARAP_TIMING") != NULL;
        if (const char* k = getenv("ARAP_SOLVER")) {
            if (strcmp(k, "LMGPU") == 0) lm = true;
            else if (strcmp(k, "gaussNewtonGPU") != 0) {
                fprintf(stderr, "ARAP_SOLVER must be gaussNewtonGPU or LMGPU\n");
                exit(1);
            }
        }
    }
};

// (re)build the batch context -- the "plan" of the reference -- for images of W x H; 0 = ok
static int ensure_context(Context& C, const Settings& S, int W, int H)
{
    if (C.ctx && W == C.W && H == C.H) return 0;
    if (C.ctx) {
        printf("Warning: Input image has different size to one in the prebuilt plan.\n"
               "To avoid re-building the plan and to save time, put images of the "
               "same size in the same list.\nStarting to re-build plan...\n");
        arapb200_batch_destroy(C.ctx);
        C.ctx = NULL;
    }
    C.ctx = arapb200_batch_create(W, H, S.batch, S.nCont, S.nGN, S.nPCG, ARAPB200_BACKEND_AUTO);
    if (!C.ctx) return 1;
    if (S.pcg_rtol > 0.0 && arapb200_batch_set_option(C.ctx, "pcg_rtol", S.pcg_rtol)) {
        fprintf(stderr, "ARAP_PCG_RTOL must be in [0, 1)\n");
        return 1;
    }
    if (S.gn_rtol > 0.0 && arapb200_batch_set_option(C.ctx, "gn_rtol", S.gn_rtol)) {
        fprintf(stderr, "ARAP_GN_RTOL must be in [0, 1)\n");
        return 1;
    }
    if (S.lm && arapb200_batch_set_option(C.ctx, "lm", 1.0)) return 1;
    C.W = W; C.H = H;
    return 0;
}

// deformSingle for every entry (ARAP/deformation/src/main.cpp:223-238), batched and pipelined
static int process(const std::vector<InputPaths>& lines, Context& C)
{
    const Settings S;
    const int batch = S.batch;
    const bool timing = S.timing;
    const auto t_begin = std::chrono::steady_clock::now();
    auto since = [&](std::chrono::steady_clock::time_point t0) {
        return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    };
    double t_decode = 0, t_gpu_wait = 0, t_encode = 0, t_create = 0;

    // Three overlapped stages (SURVEY.md 8f, N2): the main thread decodes group k+1 and encodes group k-1 while
    // a worker thread runs group k on the GPU.  Output order and the "Saved" lines stay in list order.
    struct Group {
        size_t first = 0;
        int W = 0, H = 0;
        std::vector<Loaded> items;
    };
    auto gpu_stage = [&](std::shared_ptr<Group> g) -> int {
        if (!C.ctx || g->W != C.W || g->H != C.H) {
            const auto t0 = std::chrono::steady_clock::now();
            const int rc = ensure_context(C, S, g->W, g->H);
            t_create += since(t0);
            if (rc) return rc;
        }
        for (size_t k = 0; k < g->items.size(); ++k) {
            Loaded& L = g->items[k];
            const bool ex = !L.occ.empty();
            if (arapb200_batch_submit_ex(C.ctx, (int)k, g->W, g->H, L.rgb.px.data(), L.mask_red.data(), L.cstr.data(),
                                         (int)(L.cstr.size() / 4), L.flow.data(), L.wrgb.data(), L.wmask.data(), NULL,
                                         ex ? L.bflow.data() : NULL, ex ? L.occ.data() : NULL))
                return 1;
        }
        return arapb200_batch_run(C.ctx);
    };
    // decode / encode run one task per list entry (zlib dominates: ~0.1 s of CPU per pair at 854x480)
    auto save_one = [&](const Group& g, size_t k) -> bool {
        const Loaded& L = g.items[k];
        const InputPaths& p = lines[g.first + k];
        auto gray3 = [](const std::vector<uint8_t>& m) { // a mask as an RGB image (README.md:25-32)
            std::vector<uint8_t> m3(3 * m.size());
            for (size_t q = 0; q < m.size(); ++q) m3[3 * q] = m3[3 * q + 1] = m3[3 * q + 2] = m[q];
            return m3;
        };
        if (!save_png_rgb(p.wrgb, g.W, g.H, L.wrgb.data()) || !save_png_rgb(p.wmask, g.W, g.H, gray3(L.wmask).data()) ||
            !write_flo(p.flo, g.W, g.H, L.flow.data()))
            return false;
        return !p.extras() ||
               (write_flo(p.bflo, g.W, g.H, L.bflow.data()) && save_png_rgb(p.occ, g.W, g.H, gray3(L.occ).data()));
    };
    auto save_stage = [&](const Group& g) -> bool {
        std::vector<std::future<bool>> jobs;
        for (size_t k = 0; k < g.items.size(); ++k) jobs.push_back(std::async(std::launch::async, save_one, std::cref(g), k));
        bool ok = true;
        for (auto& j : jobs) {
            if (j.get()) { printf("Saved\n"); ++C.saved; } // list order
            else ok = false;
        }
        return ok;
    };
    auto load_one = [&](size_t idx, Loaded* out) -> bool {
        Loaded& L = *out;
        ImageRGB m;
        if (!read_constraints(lines[idx].cstr, L.cstr) || !load_png_rgb(lines[idx].rgb, L.rgb) || !load_png_rgb(lines[idx].mask, m))
            return false;
        if (m.W != L.rgb.W || m.H != L.rgb.H) {
            fprintf(stderr, "mask %s and image %s differ in size\n", lines[idx].mask.c_str(), lines[idx].rgb.c_str());
            return false;
        }
        const size_t N = (size_t)m.W * m.H;
        L.mask_red.resize(N);
        for (size_t q = 0; q < N; ++q) L.mask_red[q] = m.px[3 * q]; // red channel only
        L.flow.resize(2 * N);
        L.wrgb.resize(3 * N);
        L.wmask.resize(N);
        if (lines[idx].extras()) {
            L.bflow.resize(2 * N);
            L.occ.resize(N);
        }
        return true;
    };

    std::future<int> running;
    std::shared_ptr<Group> in_flight, done;
    std::deque<Loaded> ready; // decoded, not yet grouped (a size change leaves the tail for the next group)
    size_t decoded = 0, grouped = 0;
    while (grouped < lines.size() || in_flight) {
        // ---- decode ahead: keep up to `batch` entries ready, all of them in parallel ----
        std::shared_ptr<Group> next;
        if (grouped < lines.size()) {
            const size_t want = std::min(lines.size() - grouped, (size_t)batch);
            if (ready.size() < want) {
                const auto t0 = std::chrono::steady_clock::now();
                const size_t n_new = want - ready.size();
                std::vector<Loaded> fresh(n_new);
                std::vector<std::future<bool>> jobs;
                for (size_t k = 0; k < n_new; ++k) jobs.push_back(std::async(std::launch::async, load_one, decoded + k, &fresh[k]));
                bool ok = true;
                for (auto& j : jobs) ok = j.get() && ok;
                if (!ok) return 1;
                for (auto& L : fresh) ready.push_back(std::move(L));
                decoded += n_new;
                t_decode += since(t0);
            }
            // ---- the next group: consecutive entries of one image size ----
            next = std::make_shared<Group>();
            next->first = grouped;
            next->W = ready.front().rgb.W;
            next->H = ready.front().rgb.H;
            while (!ready.empty() && (int)next->items.size() < batch && ready.front().rgb.W == next->W &&
                   ready.front().rgb.H == next->H) {
                next->items.push_back(std::move(ready.front()));
                ready.pop_front();
                ++grouped;
            }
        }
        // ---- wait for the group on the GPU, start the next one, then encode the finished one ----
        if (in_flight) {
            const auto t0 = std::chrono::steady_clock::now();
            const int rc = running.get();
            t_gpu_wait += since(t0);
            if (rc) {
                fprintf(stderr, "arap_deform: solver failed (%d)\n", rc);
                return rc;
            }
            done = in_flight;
            in_flight.reset();
        }
        if (next) {
            in_flight = next;
            running = std::async(std::launch::async, gpu_stage, next);
        }
        if (done) {
            const auto t0 = std::chrono::steady_clock::now();
            if (!save_stage(*done)) return 1;
            t_encode += since(t0);
            done.reset();
        }
    }
    if (timing)
        fprintf(stderr, "arap_deform timing: total %.3f s | decode %.3f | waiting for the GPU %.3f (context + buffers %.3f) | "
                        "encode %.3f\n", since(t_begin), t_decode, t_gpu_wait, t_create, t_encode);
    return 0;
}

static bool plan_ok(const char* planPath)
{
    Opt_InitializationParameters ip = {0, 0, 0, 0};
    Opt_State* st = Opt_NewState(ip);
    Opt_Problem* pr = st ? Opt_ProblemDefine(st, planPath, "gaussNewtonGPU") : NULL;
    if (!pr) return false;
    Opt_ProblemDelete(st, pr);
    return true;
}

static bool exists(const std::string& p)
{
    struct stat sb;
    return stat(p.c_str(), &sb) == 0;
}

static volatile sig_atomic_t g_stop = 0;
static void on_signal(int) { g_stop = 1; }

// ---- resident worker ----------------------------------------------------------------------------------
static int serve(const std::string& dir, int warmW, int warmH)
{
    mkdir(dir.c_str(), 0777);
    signal(SIGTERM, on_signal);
    signal(SIGINT, on_signal);
    // a worker pays every one-time cost at start-up, not on the first request: all kernels are loaded with the context
    // (the default is lazy loading at first launch) ...
    setenv("CUDA_MODULE_LOADING", "EAGER", 0);
    Context C;
    {
        int sm = 0;
        if (arapb200_device_info(&sm, NULL, NULL, NULL)) return 1;
    }
    if (warmW > 0 && warmH > 0) {
        // ... and, when the image size is known (--warm WxH: para_gen's --size), so are the device and pinned buffers and
        // the first launch: one empty problem (no object pixel) through the whole path
        const Settings S;
        if (ensure_context(C, S, warmW, warmH)) return 1;
        const size_t N = (size_t)warmW * warmH;
        std::vector<uint8_t> rgb(3 * N, 0), mask(N, 255), wrgb(3 * N), wmask(N);
        std::vector<float> flow(2 * N);
        if (arapb200_batch_submit(C.ctx, 0, warmW, warmH, rgb.data(), mask.data(), NULL, 0, flow.data(), wrgb.data(), wmask.data(), NULL) ||
            arapb200_batch_run(C.ctx))
            return 1;
    }
    {   // tell clients (and the driver that started us) that the worker is up
        std::ofstream r(dir + "/ready.tmp");
        r << getpid() << "\n";
        r.close();
        rename((dir + "/ready.tmp").c_str(), (dir + "/ready").c_str());
    }
    fprintf(stderr, "arap_deform: serving %s (pid %d)\n", dir.c_str(), (int)getpid());
    while (!g_stop) {
        if (exists(dir + "/stop")) break;
        std::vector<std::string> jobs;
        if (DIR* d = opendir(dir.c_str())) {
            while (dirent* e = readdir(d)) {
                const std::string n = e->d_name;
                if (n.size() > 4 && n.compare(n.size() - 4, 4, ".job") == 0) jobs.push_back(n.substr(0, n.size() - 4));
            }
            closedir(d);
        }
        if (jobs.empty()) {
            std::this_thread::sleep_for(std::chrono::milliseconds(2));
            continue;
        }
        std::sort(jobs.begin(), jobs.end()); // ids start with a timestamp: oldest first
        for (const std::string& id : jobs) {
            const std::string job = dir + "/" + id + ".job", run = dir + "/" + id + ".run";
            if (rename(job.c_str(), run.c_str()) != 0) continue; // somebody else took it
            std::vector<InputPaths> lines;
            int rc = 1;
            C.saved = 0;
            if (read_list(run.c_str(), lines) && !lines.empty()) rc = process(lines, C);
            fflush(stdout);
            std::ofstream o(dir + "/" + id + ".done.tmp");
            o << rc << "\n" << C.saved << "\n";
            o.close();
            rename((dir + "/" + id + ".done.tmp").c_str(), (dir + "/" + id + ".done").c_str());
            unlink(run.c_str());
        }
    }
    unlink((dir + "/ready").c_str());
    return 0;
}

// ---- thin client --------------------------------------------------------------------------------------
static int submit(const std::string& dir, const std::vector<InputPaths>& lines)
{
    if (!exists(dir + "/ready")) {
        fprintf(stderr, "arap_deform: no server is watching %s (start one with: arap_deform --serve %s)\n", dir.c_str(), dir.c_str());
        return 1;
    }
    char id[128];
    const long long now = std::chrono::duration_cast<std::chrono::microseconds>(
                              std::chrono::system_clock::now().time_since_epoch()).count();
    snprintf(id, sizeof(id), "%020lld_%d", now, (int)getpid());
    const std::string base = dir + "/" + id;
    {
        std::ofstream o(base + ".job.tmp");
        for (const InputPaths& p : lines) {
            o << p.rgb << " " << p.mask << " " << p.cstr << " " << p.flo << " " << p.wrgb << " " << p.wmask;
            if (p.extras()) o << " " << p.bflo << " " << p.occ;
            o << "\n";
        }
        if (!o) return 1;
    }
    if (rename((base + ".job.tmp").c_str(), (base + ".job").c_str()) != 0) return 1;
    while (!exists(base + ".done")) {
        if (!exists(dir + "/ready") && !exists(base + ".done")) {
            fprintf(stderr, "arap_deform: the server watching %s went away\n", dir.c_str());
            unlink((base + ".job").c_str());
            return 1;
        }
        std::this_thread::sleep_for(std::chrono::milliseconds(1));
    }
    int rc = 1;
    long saved = 0;
    {
        std::ifstream in(base + ".done");
        in >> rc >> saved;
    }
    unlink((base + ".done").c_str());
    for (long k = 0; k < saved; ++k) printf("Saved\n");
    return rc;
}

int main(int argc, const char* argv[])
{
    const char* planPath = getenv("ARAP_PLAN") == NULL ? "arap_plan.t" : getenv("ARAP_PLAN");
    if ((argc == 3 || argc == 5) && strcmp(argv[1], "--serve") == 0) {
        int ww = 0, wh = 0;
        if (argc == 5 && (strcmp(argv[3], "--warm") != 0 || sscanf(argv[4], "%dx%d", &ww, &wh) != 2 || ww <= 0 || wh <= 0)) {
            printf("Invalid Input!\n");
            usage();
            return 1;
        }
        printf("Optimization plan at %s\n", planPath);
        if (!plan_ok(planPath)) {
            printf(" Not found! Please run export ARAP_PLAN=/path/to/plan.t or copy "
                   "the file to the running folder with name arap_plan.t");
            return 1;
        }
        return serve(argv[2], ww, wh);
    }
    std::vector<InputPaths> lines;
    if (argc == 7 || argc == 9) {
        lines.push_back({argv[1], argv[2], argv[3], argv[4], argv[5], argv[6], argc == 9 ? argv[7] : "",
                         argc == 9 ? argv[8] : ""});
    } else if (argc == 2) { // a list file: main.cpp:182-193
        read_list(argv[1], lines);
    } else {
        printf("Invalid Input!\n");
        usage();
        return 1;
    }
    if (lines.empty()) {
        printf("No file to be processed");
        return 1;
    }
    printf("Optimization plan at %s\n", planPath);
    if (!plan_ok(planPath)) {
        printf(" Not found! Please run export ARAP_PLAN=/path/to/plan.t or copy "
               "the file to the running folder with name arap_plan.t");
        return 1;
    }
    if (const char* srv = getenv("ARAP_SERVER")) {
        if (*srv) return submit(srv, lines);
    }
    Context C;
    return process(lines, C);
}
