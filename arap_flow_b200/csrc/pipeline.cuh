// pipeline.cuh -- per-image path of arap_deform on the device, batched: what CombinedSolver (ARAP/
// deformation/src/CombinedSolver.h:139-242, 280-366) and CombinedSolverBase::singleSolve (ARAP/shared/
// CombinedSolverBase.h:99-120) do around the solver, for many independent (image, segment) problems at once,
// with every host<->device hop removed except the upload of the inputs and the download of the outputs.
#pragma once
#include "blur.cuh"
#include "devmem.cuh"
#include "plan.cuh"
#include "warp.cuh"
#include <vector>

namespace arapb200 {

struct HostProblem {
    int W = 0, H = 0;
    const unsigned char* rgb = nullptr;      // uint8x3[N]
    const unsigned char* mask_red = nullptr; // uint8[N]
    const int* matches = nullptr;            // int32[4*n], without border pins
    int n_matches = 0;
    float* out_flow = nullptr;               // float2[N]
    unsigned char* out_rgb = nullptr;        // uint8x3[N]
    unsigned char* out_mask = nullptr;       // uint8[N]
    float* out_costs = nullptr;              // float[nCont*(nGN+1)] or null
    float* out_bflow = nullptr;              // float2[N] backward flow or null (opt-in, DESIGN.md 4.3)
    unsigned char* out_occ = nullptr;        // uint8[N] occlusion of frame 1 or null (opt-in)
    // opt-in frame sequence (DESIGN.md 4.4): continuation steps t_1 < ... < t_K, and per frame k the outputs of
    // enqueue_warp_seq, each [K][N][...] or null; out_rgb / out_mask are required when steps is not empty
    std::vector<int> steps;
    unsigned char *seq_rgb = nullptr, *seq_mask = nullptr, *seq_occ = nullptr;
    float *seq_flow = nullptr, *seq_bflow = nullptr, *seq_flow0 = nullptr;
    // a layer of a HostScene: backward flow, occlusion and frames are computed and stay on the device; of the outputs
    // above only out_costs is copied out
    bool scene = false;
    // a layer of a blurred scene: the continuation steps whose X its sub-frames read (sorted; DESIGN.md 4.8)
    std::vector<int> blur_states;
};

// A scene (DESIGN.md 4.6): problems first .. first + n - 1 of a run are its layers in segment order (same W x H and rgb),
// composited on the device over a moving background.  maps: the composite_coeffs of the pair (motion_from = identity),
// then of frame k = 1 .. K (A_{k-1} -> A_k), K = the layers' step count.  Host buffers; outputs as
// arapb200_batch_submit_scene describes them.
struct HostScene {
    int first = 0, n = 0, W = 0, H = 0;
    const unsigned char* background = nullptr; // uint8x3[bgW*bgH]
    int bgW = 0, bgH = 0, bg_x = 0, bg_y = 0;
    std::vector<float> maps;                   // [1 + K][18]
    float* out_flow = nullptr;
    unsigned char *out_rgb = nullptr, *out_mask = nullptr, *out_occ = nullptr, *out_rgb0 = nullptr;
    float* out_bflow = nullptr;
    unsigned char *seq_rgb = nullptr, *seq_mask = nullptr, *seq_occ = nullptr;
    float *seq_flow = nullptr, *seq_bflow = nullptr;
    std::vector<double> motions; // [1 + K][6]: A, then A_1 .. A_K, as submitted
    // opt-in motion blur (DESIGN.md 4.8, arapb200_batch_scene_blur): blur_S sub-frames per image (0 = none); blur[(image
    // + 1) * blur_S + j] is sub-frame j of image -1 (frame 0), 0 (the pair) or k (frame k), filled for the images asked
    // for; blur_states: the continuation steps those sub-frames read, sorted
    int blur_S = 0;
    std::vector<BlurSub> blur;
    std::vector<int> blur_states;
    unsigned char *blur_rgb = nullptr, *blur_rgb0 = nullptr, *seq_blur_rgb = nullptr;
};

// compact constraint record: source pixel index and the match, after the reference's filtering
// (mask(src) == 0, later entries override earlier ones, border pins appended: main.cpp:130-136,
// CombinedSolver.h:223-242)
struct MatchRec {
    int idx;
    float x1, y1, x2, y2;
};

// host-side: filter + dedupe the match list exactly like setConstraintImage would resolve it
void build_match_records(int W, int H, const unsigned char* mask_red, const int* matches, int n_matches,
                         std::vector<MatchRec>& out);

class BatchPipeline {
public:
    // up to max_problems problems of at most maxW x maxH in flight
    BatchPipeline(int maxW, int maxH, int max_problems, int nCont, int nGN, int nPCG, int backend);
    ~BatchPipeline();
    BatchPipeline(const BatchPipeline&) = delete;
    BatchPipeline& operator=(const BatchPipeline&) = delete;
    // upload, solve (all continuation steps), flow, warp, download -- for every problem given; then the composite of every
    // scene, whose layers are among the problems.  Blocking.
    int run(const HostProblem* problems, int count, const HostScene* scenes = nullptr, int n_scenes = 0);
    long long launches() const { return launches_; }
    float last_ms_total() const { return ms_total_; }
    float last_ms_solve() const { return ms_solve_; }
    float last_ms_warp() const { return ms_warp_; }
    int last_resident_count() const { return n_resident_; }
    int last_group_size() const { return group_size_; }
    // {problems in the largest cooperative launch, variant max threads, variant min CTAs/SM, grid.x, grid.y, threads} of
    // the last resident launch of the last run (zeros if everything streamed)
    void last_launch_info(int out[6]) const
    {
        out[0] = group_size_;
        int sh[5] = {0, 0, 0, 0, 0};
        if (resident_ && n_resident_ > 0) resident_->last_launch_shape(sh);
        for (int i = 0; i < 5; ++i) out[1 + i] = sh[i];
    }
    int max_problems() const { return (int)dev_.size(); }
    // opt-in early exits of the PCG loops / of the Gauss-Newton steps (both back-ends)
    void set_pcg_rtol(float rtol);
    void set_gn_rtol(float rtol);
    // opt-in: every Opt_ProblemSolve of the schedule runs the reference's other solver kind, "LMGPU" (solver_lm.cuh:
    // trust region + Q-based exit of the linear loops) with its default parameters, one problem at a time
    void set_lm(bool on) { lm_on_ = on; }

private:
    struct Dev { // device + pinned staging of one problem slot
        DevBuf<float2> X, U, C, flow;
        DevBuf<float> A, M, costs;
        DevBuf<unsigned char> rgb, mask, orgb, omask;
        DevBuf<unsigned> z;
        GrowBuf h_in{GrowBuf::Pinned}, h_out{GrowBuf::Pinned};
        GrowBuf matches; // MatchRec[], grown with headroom for a longer list
        // opt-in extras, allocated the first time the slot asks for them: [bflow | occ] on the device and pinned
        GrowBuf extras, h_extras{GrowBuf::Pinned};
        // opt-in frame sequence, allocated the first time the slot asks and regrown for a longer list
        GrowBuf frames;
        // X after each of the blur states of a blurred scene's layer (8 B/px per state), regrown for a longer list
        GrowBuf blur;
        // placed in the buffers above for the current run
        float2* bflow = nullptr;
        unsigned char* occ = nullptr;
        float2* seq_pos = nullptr; // X after each requested continuation step
        float2* blur_pos = nullptr; // X after each blur state
        unsigned* seq_z = nullptr; // two z-buffers
        SeqOut seq{};
        std::vector<MatchRec> recs;
        bool resident = false;
        const MatchRec* recs_dev() const { return (const MatchRec*)matches.data(); }
    };
    void solve_streaming(const HostProblem& hp, Dev& d);
    void solve_lm(const HostProblem& hp, Dev& d);
    // the resident problems first .. first + count - 1 in one cooperative launch per schedule, or per continuation step
    // when one of them asks for frames or blur states
    void solve_resident(const HostProblem* problems, int first, int count);
    // X -> frame buffer if step t is one of hp's frames, and -> blur buffer if it is one of its blur states
    void snapshot(const HostProblem& hp, Dev& d, int t);
    // device buffer of the j-th scene of a run, allocated the first time and grown for a larger scene: the background,
    // frame 0 and the composited pair and frames (21 B/px each), laid out by SceneLayout (pipeline.cu)
    std::vector<GrowBuf> scene_dev_;
    void enqueue_scene(const HostScene& sc, unsigned char* buf); // the scene's kernels (DESIGN.md 4.6)
    // the blurred scene at the j-th scene position, its scratch allocated the first time and grown for a larger scene:
    // the layers' z-buffers (4 B/px each), the accumulator (8 B/px) and the blurred images (3 B/px each), laid out by
    // BlurLayout (pipeline.cu)
    std::vector<GrowBuf> blur_dev_;
    void enqueue_scene_blur(const HostScene& sc, const unsigned char* scene_buf, unsigned char* buf); // DESIGN.md 4.8
    LmSolver* lm_ = nullptr;
    int lmW_ = 0, lmH_ = 0;
    bool lm_on_ = false;
    std::vector<float> lm_costs_;
    int maxW_, maxH_, nCont_, nGN_, nPCG_, backend_;
    std::vector<Dev> dev_;
    StreamSolver* solver_ = nullptr;
    int solverW_ = 0, solverH_ = 0;
    ResidentSolver* resident_ = nullptr;
    cudaStream_t stream_ = nullptr;
    cudaEvent_t ev_[4] = {nullptr, nullptr, nullptr, nullptr};
    long long launches_ = 0;
    float ms_total_ = 0, ms_solve_ = 0, ms_warp_ = 0;
    int n_resident_ = 0, group_size_ = 0;
    float pcg_rtol_ = 0.0f, gn_rtol_ = 0.0f;
};

// shared small kernels
void enqueue_reset_state(int W, int H, const unsigned char* d_mask_red, float2* d_X, float2* d_U, float* d_A,
                         float* d_M, cudaStream_t stream);
// resident back-end: per-pixel match target image ((-1e30, -1e30) = none); the kernel does the lerp
void enqueue_target_image(int W, int H, const MatchRec* d_matches, int n, float2* d_C, cudaStream_t stream);
void enqueue_constraint_image(int W, int H, const MatchRec* d_matches, int n, float alpha, float2* d_C,
                              cudaStream_t stream);

} // namespace arapb200
