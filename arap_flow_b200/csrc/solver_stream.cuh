// solver_stream.cuh -- the streaming Gauss-Newton/PCG back-end (state in L2/HBM, two kernels per
// PCG iteration, a whole GN step captured in one CUDA graph).  Used for problems whose PCG state
// does not fit on chip (1920x1080, SURVEY.md C4) and as the general-size path behind Opt.h.
#pragma once
#include "common.cuh"
#include "kernel_timer.cuh"
#include <vector>

namespace arapb200 {

constexpr int ST_TILE = 32;                 // 32 x 32 pixel tiles
constexpr int ST_THREADS = 256;             // thread = one aligned vertical quad (contract C3 group)
constexpr unsigned FLAG_FIT = 0x10u;        // bits 0..3: neighbour n valid (order +x,-x,+y,-y)
constexpr unsigned FLAG_ACTIVE = 0x20u;

struct StreamScalars {
    float num, den, bnum, cost;
    unsigned bad_u; // number of pixels whose UrShape is not the pixel grid
    // opt-in early exit of the PCG loop (SURVEY.md 8f N4): threshold on r.z, set once per Gauss-Newton step, and the sticky
    // "converged" flag that turns the remaining k_step_a / k_step_b launches of the captured graph into no-ops
    float stop;
    unsigned conv;
    // opt-in early exit of the Gauss-Newton steps: once a step lowers the cost by less than gn_rtol (relative), gn_done makes
    // every later step of the same Opt_ProblemSolve a no-op (k_prep raises conv, delta stays 0, the cost repeats)
    unsigned gn_done;
    float gn_prev;
    unsigned pad[3];
};

// Accumulator sets (common.cuh: wide fixed-point accumulators).  r.z of PCG iteration j lives in set (j + 3) % 3
// (j = -1: the initial r.p of PCGInit1), p.q of iteration j in set 3 + (j & 1); set 5 is the cost.
constexpr int ST_ACC_D0 = 3;
constexpr int ST_ACC_COST = 5;
constexpr int ST_ACC_SETS = 6;

// Solver-owned state is stored TILE-INTERLEAVED: for every 32 x 32 tile one contiguous block of ST_NPL planes of 1024
// floats (r, p ping, p pong, q, delta, cos/sin, preconditioner, flags as bytes).  A thread then reaches every value of
// its pixels as [one base register + compile-time immediate]: no per-load address arithmetic, 4 KB contiguous per plane
// and tile in DRAM.  Pixels of edge tiles that lie outside the image exist in storage and always hold zeros.
constexpr int ST_TILE_PX = ST_TILE * ST_TILE;
constexpr int PL_R = 0;      // 3 planes
constexpr int PL_P = 3;      // 2 x 3 planes: search direction, ping-ponged per PCG iteration (buffer it & 1)
constexpr int PL_Q = 9;      // 3
constexpr int PL_D = 12;     // 3
constexpr int PL_CS = 15;    // cos, sin of Angle, refreshed per GN step
constexpr int PL_PRE = 17;   // guarded-inverted diagonal: X part (both comps), angle part
constexpr int PL_FLAGS = 19; // first 1024 BYTES of this plane
constexpr int PL_EDGE = 20;  // [13 halo-relevant planes][column 0, column 31][32 rows]: mirrors of the tile's outer
                             // columns, so that a neighbour reads its ring column as ONE contiguous 128-byte run
                             // instead of 32 strided sectors
constexpr int ST_NPL = 21;
constexpr size_t ST_TILE_FLOATS = (size_t)ST_NPL * ST_TILE_PX;

// What the solver owns, fixed for its lifetime: passed to the kernels BY VALUE (constant bank), so that no block starts
// with a chain of dependent pointer loads.
struct StreamPlanes {
    int W, H, tx, ty, ntiles;
    float* planes;              // [ntiles][ST_NPL][32][32]
    unsigned char* tile_active; // per tile: any object pixel (set by k_prep)
    unsigned long long* acc;    // [ST_ACC_SETS][WA_COPIES][WA_LIMBS]
    StreamScalars* sc;
};

// Plus what the caller binds (Opt_ProblemInit/Step re-bind on every call: ARAP/API/src/util.t:664-692).  This part is
// read through a pointer to a device copy, so that a captured graph stays valid across re-binds.
struct StreamDev : StreamPlanes {
    float2* X;            // Offset  (in/out)
    float* A;             // Angle   (in/out)
    const float2* U;      // UrShape
    const float2* C;      // Constraints
    const float* M;       // Mask
    float wf, wr, wf2, wr2;
    float* trace;         // optional: (den, num, bnum) per PCG iteration of the current GN step
    float gn_rtol;        // 0 = every Gauss-Newton step runs; > 0: see StreamScalars::gn_done
    float pcg_rtol2;      // 0 = fixed budget (reference behaviour); > 0: the PCG loop ends once r.z <= pcg_rtol2 * (r.z at PCGInit1)
};

class StreamSolver {
public:
    StreamSolver(int W, int H);
    ~StreamSolver();
    StreamSolver(const StreamSolver&) = delete;
    StreamSolver& operator=(const StreamSolver&) = delete;

    // bind the caller's device images + weights (== util.initParameters in the reference)
    void bind(float2* X, float* A, const float2* U, const float2* C, const float* M, float wf, float wr,
              cudaStream_t stream);
    // flags + cos/sin + UrShape check, then cost.  Enqueue only.
    void enqueue_init(cudaStream_t stream);
    // one Gauss-Newton step: PCGInit, nPCG iterations, update, cos/sin refresh, cost.  Enqueue only.
    // trace (device, 3*nPCG floats) may be null; tracing bypasses the graph.
    void enqueue_gn_step(int nPCG, cudaStream_t stream, float* d_trace = nullptr);
    // blocking read of (cost, bad_u) after the enqueued work
    void read_back(cudaStream_t stream, float* cost, unsigned* bad_u);
    // unit-level pieces for the parity tests (enqueue only)
    void enqueue_prep(cudaStream_t stream);
    void enqueue_pcg_init(cudaStream_t stream);
    void enqueue_step_a(bool first, int it, cudaStream_t stream); // also decodes p.q into scalars().den
    // UrShape is not the pixel grid: use the general-d kernels (slower; same arithmetic contract)
    void set_general(bool general);
    // opt-in (never on the parity path): relative tolerance of the PCG loops; takes effect with the next bind()
    void set_pcg_rtol(float rtol);
    void set_gn_rtol(float rtol);
    // per-kernel timing (Opt_InitializationParameters.collectPerKernelTimingInfo): every launch of a Gauss-Newton step is
    // bracketed by an event pair under the reference's kernel name; bypasses the graph.  Null = off.
    void set_timer(KernelTimer* t) { timer_ = t; }
    bool general() const { return general_; }
    const StreamDev& host_view() const { return h_; }
    // debug / parity tests: one plane (PL_*) <-> a row-major host image; blocking
    void download_plane(int plane, float* dst) const;
    void upload_plane(int plane, const float* src);
    void download_flags(unsigned char* dst) const;
    StreamScalars* d_scalars() const { return h_.sc; }
    long long launches() const { return launches_; }
    int W() const { return h_.W; }
    int H() const { return h_.H; }

private:
    void upload(cudaStream_t stream);
    void launch_gn_body(int nPCG, cudaStream_t stream, bool tracing);
    void launch_step_a(bool first, int it, cudaStream_t stream);
    void launch_step_b(int it, cudaStream_t stream);
    bool general_ = false;
    KernelTimer* timer_ = nullptr;
    float pcg_rtol_ = 0.0f, gn_rtol_ = 0.0f;
    bool rt() const { return (pcg_rtol_ > 0.0f || gn_rtol_ > 0.0f) && !general_; } // the early-exit kernel instantiations
    StreamDev h_{};
    StreamDev* d_ = nullptr;
    cudaGraphExec_t graph_ = nullptr;
    int graph_npcg_ = -1;
    long long graph_nodes_ = 0;
    long long launches_ = 0;
};

} // namespace arapb200
