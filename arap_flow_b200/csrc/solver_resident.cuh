// solver_resident.cuh -- the resident Gauss-Newton/PCG back-end: ONE persistent cooperative kernel runs
// whole Gauss-Newton solves (optionally whole 19-step continuation schedules) with the PCG state
// (r, delta, p, cos/sin, flags) held in registers and the search direction shared through shared-memory
// tiles.  Nothing but tile-boundary values and two 16-byte partial sums per CTA cross L2 per PCG iteration.
// See DESIGN.md section 4 for the decomposition, the barrier and the halo protocol.
#pragma once
#include "common.cuh"
#include <vector>

namespace arapb200 {

constexpr int RS_STRIP_W = 32;   // a strip is 32 x RS_STRIP_H pixels: one warp, lane = column
constexpr int RS_STRIP_H = 8;    // two contract-C3 groups per lane
constexpr int RS_MAX_WARPS = 16; // strips per CTA
constexpr int RS_MAX_CTAS = 160; // CTAs per problem (8-bit arrival count per barrier word)
constexpr int RS_PROF_SLOTS = 16; // u64 per CTA of the optional cycle accounting (arapb200_debug_resident_profile)
constexpr int RS_OUTBOX_ENTRIES = 64 + 2 * RS_STRIP_H; // top row, bottom row, left column, right column; 32 bytes each

// One problem as the kernel sees it (device memory, one per blockIdx.y)
struct ResProb {
    int W, H, SX, SY;
    int n_strips;          // active strips
    int G;                 // CTAs working on this problem (blockIdx.x >= G exits)
    float2* X;             // Offset (in/out)
    float* A;              // Angle (in/out)
    const float2* C;       // Constraints image, or (lerp_mode) per-pixel match target, (<0) = none
    const float* M;        // Mask (0 = active)
    int lerp_mode;         // 1: C holds targets; constraint = (1-a)*pixel + a*target, a = (t+1)/nCont
    float wf, wr, wf2, wr2;
    const int2* strip_xy;      // [n_strips] strip coordinates (sx, sy), column-major order
    const int* slot_of_strip;  // [SY*SX] -> slot or -1
    uint4* outbox;             // [n_strips][RS_OUTBOX_ENTRIES][2]: four (float, tag) words per boundary pixel
    unsigned long long* bar;   // [2][4] barrier words: 16-bit arrival count | 48-bit fixed-point limb sum
    float* costs;              // [nCont][nGN+1]
    float* trace;              // optional [nCont*nGN][nPCG][3]
    int* status;               // [0] abort flag, [1] error code
    int nCont, nGN, nPCG;
    float gn_rtol;             // 0 = every GN step runs; > 0: a continuation step ends once a GN step gains less than this (relative)
    float pcg_rtol2;           // 0 = fixed budget (reference behaviour); > 0: leave a PCG loop once r.z <= rtol^2 * r0.z0
    unsigned long long* prof;  // optional [G][RS_PROF_SLOTS] cycle counters (debug)
};

class ResidentSolver {
public:
    // capacity: largest image handled, number of problem slots that can be prepared / launched together
    explicit ResidentSolver(int maxW, int maxH, int max_slots = 1);
    ~ResidentSolver();
    ResidentSolver(const ResidentSolver&) = delete;
    ResidentSolver& operator=(const ResidentSolver&) = delete;

    // ---- single-problem convenience (slot 0) ----
    // Build the strip tables for mask M (device, float[N], 0 = active).  Blocking (4-byte read-back).
    // Returns false when the problem does not fit on chip (caller falls back to the streaming back-end).
    bool prepare(int W, int H, const float* d_M, cudaStream_t stream);
    // Enqueue a launch: nCont continuation steps x nGN Gauss-Newton steps x nPCG iterations; costs
    // (device, nCont*(nGN+1) floats) receives the cost before the first and after every GN step.
    void enqueue(float2* X, float* A, const float2* C, int lerp_mode, float wf, float wr, int nCont, int nGN,
                 int nPCG, float* d_costs, float* d_trace, cudaStream_t stream);

    // ---- batched interface: several independent problems share ONE cooperative launch (blockIdx.y) ----
    void prepare_enqueue(int slot, int W, int H, const float* d_M, cudaStream_t stream); // kernels + async read-back
    bool prepare_finish(int slot);                                                       // after a stream sync
    void set_problem(int slot, float2* X, float* A, const float2* C, int lerp_mode, float wf, float wr,
                     float* d_costs, float* d_trace);
    // how many of the prepared slots first, first+1, ... can be co-resident in one launch (>= 1)
    int group_size(int first, int limit) const;
    void enqueue_group(int first, int count, int nCont, int nGN, int nPCG, cudaStream_t stream);
    // small problems (each fits one thread-block cluster): cluster-scope barrier through distributed shared memory, any
    // number of problems per launch.  cluster_run = how many consecutive prepared slots qualify (0: use enqueue_group).
    int cluster_run(int first, int limit) const;
    void enqueue_cluster(int first, int count, int nCont, int nGN, int nPCG, cudaStream_t stream);
    void set_cluster_barrier(bool on) { cluster_barrier_ = on; }
    int cluster_ctas(int slot = 0) const { return slots_[slot].cluster_ctas; }

    // after the stream has been synchronised: non-zero = the kernel bailed out (watchdog)
    int status(cudaStream_t stream);
    long long launches() const { return launches_; }
    int n_strips(int slot = 0) const { return slots_[slot].n_strips; }
    int ctas(int slot = 0) const { return slots_[slot].G; }
    int warps(int slot = 0) const { return slots_[slot].NW; }
    int max_slots() const { return (int)slots_.size(); }
    int last_variant() const { return last_variant_; }
    // shape of the last cooperative launch: {max threads, min CTAs per SM of the kernel variant, grid.x, grid.y, threads}
    void last_launch_shape(int out[5]) const { for (int i = 0; i < 5; ++i) out[i] = last_shape_[i]; }
    // debug: per-CTA cycle accounting of the next launches into d_prof ([ctas()][RS_PROF_SLOTS] u64), or null to disable
    void set_profile(unsigned long long* d_prof) { d_prof_ = d_prof; }
    // opt-in convergence-aware schedule (SURVEY.md 8f N4); 0 restores the reference's fixed iteration budget
    void set_pcg_rtol(float rtol) { pcg_rtol_ = rtol > 0.0f ? rtol : 0.0f; }
    void set_gn_rtol(float rtol) { gn_rtol_ = rtol > 0.0f ? rtol : 0.0f; }

private:
    struct Slot {
        int W = 0, H = 0, SX = 0, SY = 0, n_strips = 0, G = 0, NW = 0;
        int cluster_ctas = 0; // > 0: the problem fits one cluster of that many CTAs
        bool fits = false;
        const float* d_M = nullptr;
        int2* d_strip_xy = nullptr;
        int* d_slot_of_strip = nullptr;
        int* d_count = nullptr;
        uint4* d_outbox = nullptr;
        unsigned long long* d_bar = nullptr;
        ResProb prob{};
    };
    int maxW_, maxH_;
    size_t strip_cap_ = 0;
    std::vector<Slot> slots_;
    int* h_counts_ = nullptr;   // pinned
    int* d_status_ = nullptr;   // shared by all slots
    ResProb* d_probs_ = nullptr;
    int sm_count_ = 0;
    long long launches_ = 0;
    unsigned long long* d_prof_ = nullptr;
    int last_variant_ = -1;
    int last_shape_[5] = {0, 0, 0, 0, 0};
    float pcg_rtol_ = 0.0f, gn_rtol_ = 0.0f;
    bool cluster_barrier_ = false; // measured slower than the L2 barrier with co-residency (DESIGN.md 4.1): opt-in
    bool cluster_schedulable(int cs);
    signed char cluster_ok_[17] = {0}; // per cluster size: 0 unknown, 1 yes, -1 no
};

} // namespace arapb200
