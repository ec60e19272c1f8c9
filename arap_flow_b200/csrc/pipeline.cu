// pipeline.cu -- see pipeline.cuh
#include "pipeline.cuh"
#include "composite.cuh"
#include <algorithm>
#include <cmath>
#include <cstring>
#include <unordered_map>

namespace arapb200 {

void build_match_records(int W, int H, const unsigned char* mask_red, const int* matches, int n_matches,
                         std::vector<MatchRec>& out)
{
    out.clear();
    std::unordered_map<int, int> where; // pixel -> position in out (later entries override earlier)
    auto add = [&](int x1, int y1, int x2, int y2) {
        if (x1 < 0 || x1 >= W || y1 < 0 || y1 >= H) return; // the reference would index out of bounds
        const int idx = y1 * W + x1;
        if (mask_red[idx] != 0) return; // CombinedSolver.h:234
        MatchRec r{idx, (float)x1, (float)y1, (float)x2, (float)y2};
        auto it = where.find(idx);
        if (it == where.end()) {
            where.emplace(idx, (int)out.size());
            out.push_back(r);
        } else {
            out[it->second] = r;
        }
    };
    for (int k = 0; k < n_matches; ++k) add(matches[4 * k], matches[4 * k + 1], matches[4 * k + 2], matches[4 * k + 3]);
    // border pins in row-major order (main.cpp:130-136); they come last, so they override
    for (int y = 0; y < H; ++y) {
        if (y == 0 || y == H - 1) {
            for (int x = 0; x < W; ++x) add(x, y, x, y);
        } else {
            add(0, y, 0, y);
            if (W > 1) add(W - 1, y, W - 1, y);
        }
    }
}

namespace {

// resetGPU (CombinedSolver.h:207-221): UrShape = X = pixel grid, Angle = 0, Mask = float(red)
__global__ void __launch_bounds__(256) k_reset(int W, int H, const unsigned char* __restrict__ mask_red,
                                                float2* __restrict__ X, float2* __restrict__ U,
                                                float* __restrict__ A, float* __restrict__ M)
{
    const size_t N = (size_t)W * H;
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const float2 g = make_float2((float)(int)(i % W), (float)(int)(i / W));
    X[i] = g;
    U[i] = g;
    A[i] = 0.f;
    M[i] = (float)mask_red[i];
}

__global__ void __launch_bounds__(256) k_fill_c(size_t N, float2* __restrict__ C)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N) C[i] = make_float2(-1.f, -1.f);
}

// setConstraintImage (CombinedSolver.h:223-242) on the compact, already filtered match list
__global__ void __launch_bounds__(256) k_scatter_c(const MatchRec* __restrict__ m, int n, float alpha,
                                                    float2* __restrict__ C)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const MatchRec r = m[k];
    const float om = 1.0f - alpha;
    C[r.idx] = make_float2(om * r.x1 + alpha * r.x2, om * r.y1 + alpha * r.y2);
}

// resident back-end: per-pixel match TARGET image; the kernel applies the continuation lerp itself
__global__ void __launch_bounds__(256) k_fill_t(size_t N, float2* __restrict__ C)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N) C[i] = make_float2(-1e30f, -1e30f);
}
__global__ void __launch_bounds__(256) k_scatter_t(const MatchRec* __restrict__ m, int n, float2* __restrict__ C)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const MatchRec r = m[k];
    C[r.idx] = make_float2(r.x2, r.y2);
}

__global__ void k_copy_cost(const StreamScalars* __restrict__ sc, float* __restrict__ dst) { *dst = sc->cost; }

// a scene's device buffer: [background][rgb0][flow][rgb][mask][bflow][occ], the last five holding the pair (index 0) and
// frames 1 .. K, so that each frame output leaves in one copy
struct SceneLayout {
    size_t bg, rgb0, flow, rgb, mask, bflow, occ, bytes;
    explicit SceneLayout(const HostScene& sc)
    {
        const size_t N = (size_t)sc.W * sc.H, F = N * (sc.maps.size() / 18);
        Layout l;
        bg = l.take(3 * (size_t)sc.bgW * sc.bgH);
        rgb0 = l.take(sc.out_rgb0 ? 3 * N : 0);
        flow = l.take(8 * F);
        rgb = l.take(3 * F);
        mask = l.take(F);
        bflow = l.take(8 * F);
        occ = l.take(F);
        bytes = l.bytes();
    }
};

// a blurred scene's scratch: [z: one z-buffer per layer][acc: ushort4 per pixel][rgb][rgb0][seq: K frames], the last
// three the blurred images asked for (DESIGN.md 4.8)
struct BlurLayout {
    size_t z, acc, rgb, rgb0, seq, bytes;
    explicit BlurLayout(const HostScene& sc)
    {
        const size_t N = (size_t)sc.W * sc.H, K = sc.maps.size() / 18 - 1;
        Layout l;
        z = l.take(4 * N * sc.n);
        acc = l.take(sizeof(ushort4) * N);
        rgb = l.take(3 * N);
        rgb0 = l.take(sc.blur_rgb0 ? 3 * N : 0);
        seq = l.take(sc.seq_blur_rgb ? 3 * N * K : 0);
        bytes = l.bytes();
    }
};

} // namespace

void enqueue_reset_state(int W, int H, const unsigned char* d_mask_red, float2* d_X, float2* d_U, float* d_A,
                         float* d_M, cudaStream_t stream)
{
    const size_t N = (size_t)W * H;
    k_reset<<<(unsigned)((N + 255) / 256), 256, 0, stream>>>(W, H, d_mask_red, d_X, d_U, d_A, d_M);
}

void enqueue_constraint_image(int W, int H, const MatchRec* d_matches, int n, float alpha, float2* d_C,
                              cudaStream_t stream)
{
    const size_t N = (size_t)W * H;
    k_fill_c<<<(unsigned)((N + 255) / 256), 256, 0, stream>>>(N, d_C);
    if (n > 0) k_scatter_c<<<(n + 255) / 256, 256, 0, stream>>>(d_matches, n, alpha, d_C);
}

void enqueue_target_image(int W, int H, const MatchRec* d_matches, int n, float2* d_C, cudaStream_t stream)
{
    const size_t N = (size_t)W * H;
    k_fill_t<<<(unsigned)((N + 255) / 256), 256, 0, stream>>>(N, d_C);
    if (n > 0) k_scatter_t<<<(n + 255) / 256, 256, 0, stream>>>(d_matches, n, d_C);
}

BatchPipeline::BatchPipeline(int maxW, int maxH, int max_problems, int nCont, int nGN, int nPCG, int backend)
    : maxW_(maxW), maxH_(maxH), nCont_(nCont), nGN_(nGN), nPCG_(nPCG), backend_(backend)
{
    const size_t N = (size_t)maxW * maxH;
    ARAP_CUDA_CHECK(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking));
    for (auto& e : ev_) ARAP_CUDA_CHECK(cudaEventCreate(&e));
    dev_.resize(max_problems > 0 ? max_problems : 1);
    const size_t cbytes = (size_t)nCont * (nGN + 1) * sizeof(float);
    for (Dev& d : dev_) {
        d.X = DevBuf<float2>(N);
        d.U = DevBuf<float2>(N);
        d.C = DevBuf<float2>(N);
        d.flow = DevBuf<float2>(N);
        d.A = DevBuf<float>(N);
        d.M = DevBuf<float>(N);
        d.costs = DevBuf<float>((size_t)nCont * (nGN + 1));
        d.rgb = DevBuf<unsigned char>(3 * N);
        d.mask = DevBuf<unsigned char>(N);
        d.orgb = DevBuf<unsigned char>(3 * N);
        d.omask = DevBuf<unsigned char>(N);
        d.z = DevBuf<unsigned>(N);
        d.h_in.reserve(4 * N);
        d.h_out.reserve(12 * N + cbytes);
    }
    if (backend_ != ARAPB200_BACKEND_STREAM) resident_ = new ResidentSolver(maxW, maxH, (int)dev_.size());
}

BatchPipeline::~BatchPipeline()
{
    cudaStreamSynchronize(stream_);
    delete solver_;
    delete resident_;
    delete lm_;
    for (auto& e : ev_) cudaEventDestroy(e);
    cudaStreamDestroy(stream_);
}

void BatchPipeline::snapshot(const HostProblem& hp, Dev& d, int t)
{
    const size_t N = (size_t)hp.W * hp.H;
    auto copy = [&](const std::vector<int>& list, float2* dst) {
        const auto it = std::lower_bound(list.begin(), list.end(), t);
        if (it == list.end() || *it != t) return;
        ARAP_CUDA_CHECK(cudaMemcpyAsync(dst + (size_t)(it - list.begin()) * N, d.X.p, N * sizeof(float2),
                                        cudaMemcpyDeviceToDevice, stream_));
    };
    copy(hp.steps, d.seq_pos);
    copy(hp.blur_states, d.blur_pos);
}

// the streaming back-end: one graph launch per Gauss-Newton step (problems too large for the chip)
void BatchPipeline::solve_streaming(const HostProblem& hp, Dev& d)
{
    const int W = hp.W, H = hp.H;
    if (!solver_ || solverW_ != W || solverH_ != H) { // re-plan on a size change (CombinedSolver.h:149-160)
        if (solver_) launches_ += solver_->launches();
        delete solver_;
        solver_ = new StreamSolver(W, H);
        solverW_ = W;
        solverH_ = H;
    }
    const long long l0 = solver_->launches();
    const float wf = sqrtf(100.0f), wr = sqrtf(0.01f); // CombinedSolver.h:172-177
    solver_->set_pcg_rtol(pcg_rtol_);
    solver_->set_gn_rtol(gn_rtol_);
    solver_->bind(d.X.p, d.A.p, d.U.p, d.C.p, d.M.p, wf, wr, stream_);
    for (int t = 0; t < nCont_; ++t) {
        const float alpha = (float)(t + 1) / (float)nCont_; // CombinedSolver.h:199-201
        enqueue_constraint_image(W, H, d.recs_dev(), (int)d.recs.size(), alpha, d.C.p, stream_);
        launches_ += d.recs.empty() ? 1 : 2;
        solver_->enqueue_init(stream_);
        k_copy_cost<<<1, 1, 0, stream_>>>(solver_->d_scalars(), d.costs.p + (size_t)t * (nGN_ + 1));
        for (int g = 0; g < nGN_; ++g) {
            solver_->enqueue_gn_step(nPCG_, stream_);
            k_copy_cost<<<1, 1, 0, stream_>>>(solver_->d_scalars(), d.costs.p + (size_t)t * (nGN_ + 1) + g + 1);
        }
        launches_ += 1 + nGN_;
        snapshot(hp, d, t);
    }
    launches_ += solver_->launches() - l0;
}

// the "LMGPU" solver kind: per continuation step one Opt_ProblemSolve = init + up to nGN steps (o.t:2548-2551), the host
// deciding acceptance after each (solver_lm.cu).  Cost log: prevCost after init and after every step; entries of steps the
// solver did not take repeat the last one.
void BatchPipeline::solve_lm(const HostProblem& hp, Dev& d)
{
    const int W = hp.W, H = hp.H;
    if (!lm_ || lmW_ != W || lmH_ != H) {
        if (lm_) launches_ += lm_->launches();
        delete lm_;
        lm_ = nullptr;
        lm_ = new LmSolver(W, H);
        lmW_ = W;
        lmH_ = H;
    }
    const long long l0 = lm_->launches();
    const float wf = sqrtf(100.0f), wr = sqrtf(0.01f); // CombinedSolver.h:172-177
    lm_->bind(d.X.p, d.A.p, d.U.p, d.C.p, d.M.p, wf, wr);
    lm_costs_.assign((size_t)nCont_ * (nGN_ + 1), 0.0f);
    for (int t = 0; t < nCont_; ++t) {
        const float alpha = (float)(t + 1) / (float)nCont_; // CombinedSolver.h:199-201
        enqueue_constraint_image(W, H, d.recs_dev(), (int)d.recs.size(), alpha, d.C.p, stream_);
        launches_ += d.recs.empty() ? 1 : 2;
        float* c = lm_costs_.data() + (size_t)t * (nGN_ + 1);
        float prev = lm_->init(stream_);
        c[0] = prev;
        int g = 0;
        while (g < nGN_) {
            const int more = lm_->step(nPCG_, stream_, &prev);
            c[++g] = prev;
            if (!more) break;
        }
        for (int k = g + 1; k <= nGN_; ++k) c[k] = prev;
        snapshot(hp, d, t);
    }
    ARAP_CUDA_CHECK(cudaMemcpyAsync(d.costs.p, lm_costs_.data(), lm_costs_.size() * sizeof(float), cudaMemcpyHostToDevice, stream_));
    ARAP_CUDA_CHECK(cudaStreamSynchronize(stream_)); // lm_costs_ is reused by the next problem
    launches_ += lm_->launches() - l0;
}

void BatchPipeline::solve_resident(const HostProblem* problems, int first, int count)
{
    const float wf = sqrtf(100.0f), wr = sqrtf(0.01f); // CombinedSolver.h:172-177
    bool frames = false;
    for (int j = 0; j < count; ++j)
        frames = frames || !problems[first + j].steps.empty() || !problems[first + j].blur_states.empty();
    if (!frames) { // the whole schedule in one launch; the kernel lerps the constraints itself (lerp_mode 1)
        for (int j = 0; j < count; ++j) {
            Dev& dj = dev_[first + j];
            const HostProblem& hp = problems[first + j];
            enqueue_target_image(hp.W, hp.H, dj.recs_dev(), (int)dj.recs.size(), dj.C.p, stream_);
            launches_ += dj.recs.empty() ? 1 : 2;
            resident_->set_problem(first + j, dj.X.p, dj.A.p, dj.C.p, 1, wf, wr, dj.costs.p, nullptr);
        }
        resident_->enqueue_group(first, count, nCont_, nGN_, nPCG_, stream_);
        return;
    }
    // Frames and blur need X after individual continuation steps: one launch per step, on the constraint image of that
    // step as the streaming path builds it (lerp_mode 0), the same bits as the single launch (DESIGN.md 4.4)
    for (int t = 0; t < nCont_; ++t) {
        const float alpha = (float)(t + 1) / (float)nCont_; // CombinedSolver.h:199-201
        for (int j = 0; j < count; ++j) {
            Dev& dj = dev_[first + j];
            const HostProblem& hp = problems[first + j];
            enqueue_constraint_image(hp.W, hp.H, dj.recs_dev(), (int)dj.recs.size(), alpha, dj.C.p, stream_);
            launches_ += dj.recs.empty() ? 1 : 2;
            resident_->set_problem(first + j, dj.X.p, dj.A.p, dj.C.p, 0, wf, wr, dj.costs.p + (size_t)t * (nGN_ + 1),
                                   nullptr);
        }
        resident_->enqueue_group(first, count, 1, nGN_, nPCG_, stream_);
        for (int j = 0; j < count; ++j) snapshot(problems[first + j], dev_[first + j], t);
    }
}

// frame 0, the pair, then frame k = 1 .. K with the layers' frame k and as source masks the input masks (k = 1) or the
// warped masks of frame k - 1 (DESIGN.md 4.6)
void BatchPipeline::enqueue_scene(const HostScene& sc, unsigned char* buf)
{
    const SceneLayout o(sc);
    const size_t N = (size_t)sc.W * sc.H;
    const int K = (int)(sc.maps.size() / 18) - 1;
    const unsigned char* bg = buf + o.bg;
    Layers L{};
    L.n = sc.n;
    for (int s = 0; s < sc.n; ++s) {
        const Dev& d = dev_[sc.first + s];
        L.flow[s] = d.flow.p;
        L.rgb[s] = d.orgb.p;
        L.mask[s] = d.omask.p;
        L.bflow[s] = d.bflow;
        L.src[s] = d.mask.p;
    }
    if (sc.out_rgb0) {
        enqueue_scene_input(sc.W, sc.H, L, dev_[sc.first].rgb.p, bg, sc.bgW, sc.bgH, sc.bg_x, sc.bg_y, buf + o.rgb0,
                            stream_);
        launches_ += 1;
    }
    for (int k = 0; k <= K; ++k) {
        if (k > 0)
            for (int s = 0; s < sc.n; ++s) {
                const SeqOut& q = dev_[sc.first + s].seq;
                const size_t f = (size_t)(k - 1) * N;
                L.flow[s] = q.flow + f;
                L.rgb[s] = q.rgb + 3 * f;
                L.mask[s] = q.mask + f;
                L.bflow[s] = q.bflow + f;
                L.src[s] = k == 1 ? dev_[sc.first + s].mask.p : q.mask + f - N;
            }
        const size_t f = (size_t)k * N;
        enqueue_composite(sc.W, sc.H, L, k >= 2, bg, sc.bgW, sc.bgH, sc.bg_x, sc.bg_y, sc.maps.data() + 18 * k,
                          (float2*)(buf + o.flow) + f, buf + o.rgb + 3 * f, buf + o.mask + f,
                          (float2*)(buf + o.bflow) + f, buf + o.occ + f, stream_);
        launches_ += 2;
    }
}

// per image asked for (frame 0, the pair, frames 1 .. K) its S sub-frames, each lerping every layer between two of its
// blur snapshots (DESIGN.md 4.8); w == 0 and w == 1 read one state, which then stands for both
void BatchPipeline::enqueue_scene_blur(const HostScene& sc, const unsigned char* scene_buf, unsigned char* buf)
{
    const BlurLayout o(sc);
    const size_t N = (size_t)sc.W * sc.H;
    const int K = (int)(sc.maps.size() / 18) - 1, S = sc.blur_S;
    const unsigned char* bg = scene_buf + SceneLayout(sc).bg;
    auto state = [&](int s, int t) -> const float2* { // null = the pixel grid
        if (t < 0) return nullptr;
        const auto it = std::lower_bound(sc.blur_states.begin(), sc.blur_states.end(), t);
        return dev_[sc.first + s].blur_pos + (size_t)(it - sc.blur_states.begin()) * N;
    };
    BlurLayers L{};
    L.n = sc.n;
    for (int s = 0; s < sc.n; ++s) L.mask_red[s] = dev_[sc.first + s].mask.p;
    for (int image = -1; image <= K; ++image) {
        unsigned char* out = image < 0    ? (sc.blur_rgb0 ? buf + o.rgb0 : nullptr)
                             : image == 0 ? buf + o.rgb
                                          : (sc.seq_blur_rgb ? buf + o.seq + 3 * N * (image - 1) : nullptr);
        if (!out) continue;
        for (int j = 0; j < S; ++j) {
            const BlurSub& b = sc.blur[(size_t)(image + 1) * S + j];
            for (int s = 0; s < sc.n; ++s) {
                L.qa[s] = b.w == 1.f ? state(s, b.j0 + 1) : state(s, b.j0);
                L.qb[s] = b.w == 0.f ? L.qa[s] : state(s, b.j0 + 1);
            }
            launches_ += enqueue_blur_subframe(sc.W, sc.H, L, b.w, b.smap, dev_[sc.first].rgb.p, bg, sc.bgW, sc.bgH,
                                               sc.bg_x, sc.bg_y, (unsigned*)(buf + o.z), (ushort4*)(buf + o.acc), j,
                                               S, out, stream_);
        }
    }
}

void BatchPipeline::set_pcg_rtol(float rtol)
{
    pcg_rtol_ = rtol > 0.0f ? rtol : 0.0f;
    if (resident_) resident_->set_pcg_rtol(rtol);
}

void BatchPipeline::set_gn_rtol(float rtol)
{
    gn_rtol_ = rtol > 0.0f ? rtol : 0.0f;
    if (resident_) resident_->set_gn_rtol(rtol);
}

int BatchPipeline::run(const HostProblem* problems, int count, const HostScene* scenes, int n_scenes)
{
    if (count <= 0) return 0;
    if (count > (int)dev_.size()) {
        fprintf(stderr, "arapb200: %d problems submitted, pipeline holds %d\n", count, (int)dev_.size());
        return 1;
    }
    const size_t cbytes = (size_t)nCont_ * (nGN_ + 1) * sizeof(float);
    const long long r0 = resident_ ? resident_->launches() : 0;
    const size_t Nmax = (size_t)maxW_ * maxH_;
    Layout xl; // a slot's opt-in extras, on the device and in pinned staging: [bflow | occ] of maxW x maxH
    const size_t x_bflow = xl.take(8 * Nmax), x_occ = xl.take(Nmax);
    // ---- stage + upload every problem, reset its state (resetGPU), build its strip tables ----
    for (int i = 0; i < count; ++i) {
        const HostProblem& hp = problems[i];
        Dev& d = dev_[i];
        if (hp.W <= 0 || hp.H <= 0 || (size_t)hp.W * hp.H > (size_t)maxW_ * maxH_) {
            fprintf(stderr, "arapb200: problem %dx%d does not fit the pipeline (%dx%d)\n", hp.W, hp.H, maxW_, maxH_);
            return 1;
        }
        const size_t N = (size_t)hp.W * hp.H;
        build_match_records(hp.W, hp.H, hp.mask_red, hp.matches, hp.n_matches, d.recs);
        if (d.recs.size() * sizeof(MatchRec) > d.matches.capacity())
            d.matches.reserve((d.recs.size() * 2 + 1024) * sizeof(MatchRec));
        if (hp.out_bflow || hp.out_occ || hp.scene) {
            unsigned char* x = d.extras.reserve(xl.bytes());
            d.bflow = (float2*)(x + x_bflow);
            d.occ = x + x_occ;
        }
        if (hp.out_bflow || hp.out_occ) d.h_extras.reserve(xl.bytes());
        if (!hp.steps.empty()) { // [pos][z][rgb][mask][flow][bflow][occ][flow0]: z two z-buffers, the rest K frames each
            const size_t F = Nmax * hp.steps.size();
            Layout l;
            const size_t pos = l.take(8 * F), z = l.take(2 * 4 * Nmax), rgb = l.take(3 * F), mask = l.take(F),
                         flow = l.take(8 * F), bflow = l.take(8 * F), occ = l.take(F), flow0 = l.take(8 * F);
            unsigned char* f = d.frames.reserve(l.bytes());
            d.seq_pos = (float2*)(f + pos);
            d.seq_z = (unsigned*)(f + z);
            d.seq = SeqOut{f + rgb, f + mask, (float2*)(f + flow), (float2*)(f + bflow), f + occ, (float2*)(f + flow0)};
        }
        if (!hp.blur_states.empty()) d.blur_pos = (float2*)d.blur.reserve(8 * N * hp.blur_states.size());
        memcpy(d.h_in.data(), hp.rgb, 3 * N);
        memcpy(d.h_in.data() + 3 * N, hp.mask_red, N);
    }
    if (n_scenes > (int)scene_dev_.size()) scene_dev_.resize(n_scenes);
    for (int j = 0; j < n_scenes; ++j) scene_dev_[j].reserve(SceneLayout(scenes[j]).bytes);
    if (n_scenes > (int)blur_dev_.size()) blur_dev_.resize(n_scenes);
    for (int j = 0; j < n_scenes; ++j)
        if (scenes[j].blur_S) blur_dev_[j].reserve(BlurLayout(scenes[j]).bytes);
    ARAP_CUDA_CHECK(cudaEventRecord(ev_[0], stream_));
    for (int i = 0; i < count; ++i) {
        const HostProblem& hp = problems[i];
        Dev& d = dev_[i];
        const size_t N = (size_t)hp.W * hp.H;
        ARAP_CUDA_CHECK(cudaMemcpyAsync(d.rgb.p, d.h_in.data(), 3 * N, cudaMemcpyHostToDevice, stream_));
        ARAP_CUDA_CHECK(cudaMemcpyAsync(d.mask.p, d.h_in.data() + 3 * N, N, cudaMemcpyHostToDevice, stream_));
        if (!d.recs.empty())
            ARAP_CUDA_CHECK(cudaMemcpyAsync(d.matches.data(), d.recs.data(), d.recs.size() * sizeof(MatchRec),
                                            cudaMemcpyHostToDevice, stream_));
        enqueue_reset_state(hp.W, hp.H, d.mask.p, d.X.p, d.U.p, d.A.p, d.M.p, stream_);
        launches_ += 1;
        d.resident = false;
        if (resident_ && !lm_on_) resident_->prepare_enqueue(i, hp.W, hp.H, d.M.p, stream_);
    }
    for (int j = 0; j < n_scenes; ++j) {
        const HostScene& sc = scenes[j];
        ARAP_CUDA_CHECK(cudaMemcpyAsync(scene_dev_[j].data(), sc.background, 3 * (size_t)sc.bgW * sc.bgH,
                                        cudaMemcpyHostToDevice, stream_));
    }
    n_resident_ = 0;
    if (resident_ && !lm_on_) {
        ARAP_CUDA_CHECK(cudaStreamSynchronize(stream_)); // strip counts are needed to size the launches
        for (int i = 0; i < count; ++i) {
            dev_[i].resident = resident_->prepare_finish(i);
            if (!dev_[i].resident && backend_ == ARAPB200_BACKEND_RESIDENT) {
                fprintf(stderr, "arapb200: problem %dx%d (%d strips) does not fit the resident back-end\n", problems[i].W,
                        problems[i].H, resident_->n_strips(i));
                return 3;
            }
            n_resident_ += dev_[i].resident ? 1 : 0;
        }
    }
    ARAP_CUDA_CHECK(cudaEventRecord(ev_[1], stream_));
    // ---- solve.  Resident problems: whole continuation schedules, several problems per cooperative launch ----
    group_size_ = 0;
    for (int i = 0; i < count;) {
        Dev& d = dev_[i];
        if (lm_on_) {
            solve_lm(problems[i], d);
            ++i;
            continue;
        }
        if (!d.resident) {
            solve_streaming(problems[i], d);
            ++i;
            continue;
        }
        int run_len = 0; // consecutive resident problems
        while (i + run_len < count && dev_[i + run_len].resident) ++run_len;
        int gsz = resident_->group_size(i, run_len);
        if (gsz < run_len) { // several launches: split the run evenly instead of one full launch and a small remainder
            const int ngroups = (run_len + gsz - 1) / gsz;
            gsz = std::min(gsz, (run_len + ngroups - 1) / ngroups);
        }
        solve_resident(problems, i, gsz);
        if (gsz > group_size_) group_size_ = gsz;
        i += gsz;
    }
    ARAP_CUDA_CHECK(cudaEventRecord(ev_[2], stream_));
    // ---- flow extraction + forward warp + download ----
    for (int i = 0; i < count; ++i) {
        const HostProblem& hp = problems[i];
        Dev& d = dev_[i];
        enqueue_pos_to_flow(hp.W, hp.H, d.X.p, d.flow.p, stream_);
        const bool extras = hp.out_bflow || hp.out_occ || hp.scene;
        enqueue_warp(hp.W, hp.H, d.X.p, d.rgb.p, d.mask.p, d.z.p, d.orgb.p, d.omask.p, stream_,
                     extras ? d.bflow : nullptr);
        launches_ += 1 + warp_launches_per_call();
        if (extras) {
            enqueue_occlusion(hp.W, hp.H, d.mask.p, d.flow.p, d.z.p, d.bflow, d.occ, stream_);
            launches_ += 1;
        }
        if (!hp.steps.empty())
            launches_ += enqueue_warp_seq(hp.W, hp.H, (int)hp.steps.size(), d.seq_pos, d.rgb.p, d.mask.p, d.seq_z, d.seq,
                                          stream_);
    }
    for (int j = 0; j < n_scenes; ++j) {
        enqueue_scene(scenes[j], scene_dev_[j].data());
        if (scenes[j].blur_S) enqueue_scene_blur(scenes[j], scene_dev_[j].data(), blur_dev_[j].data());
    }
    ARAP_CUDA_CHECK(cudaEventRecord(ev_[3], stream_));
    for (int i = 0; i < count; ++i) {
        const HostProblem& hp = problems[i];
        Dev& d = dev_[i];
        const size_t N = (size_t)hp.W * hp.H;
        unsigned char* o = d.h_out.data();
        if (!hp.scene) {
            ARAP_CUDA_CHECK(cudaMemcpyAsync(o, d.flow.p, N * sizeof(float2), cudaMemcpyDeviceToHost, stream_));
            ARAP_CUDA_CHECK(cudaMemcpyAsync(o + 8 * N, d.orgb.p, 3 * N, cudaMemcpyDeviceToHost, stream_));
            ARAP_CUDA_CHECK(cudaMemcpyAsync(o + 11 * N, d.omask.p, N, cudaMemcpyDeviceToHost, stream_));
        }
        if (!hp.scene || hp.out_costs)
            ARAP_CUDA_CHECK(cudaMemcpyAsync(o + 12 * N, d.costs.p, cbytes, cudaMemcpyDeviceToHost, stream_));
        if (hp.out_bflow || hp.out_occ) {
            unsigned char* h = d.h_extras.data();
            ARAP_CUDA_CHECK(cudaMemcpyAsync(h + x_bflow, d.bflow, N * sizeof(float2), cudaMemcpyDeviceToHost, stream_));
            ARAP_CUDA_CHECK(cudaMemcpyAsync(h + x_occ, d.occ, N, cudaMemcpyDeviceToHost, stream_));
        }
        // frames go straight to the caller's buffers: K of them would need K times the pinned staging
        const size_t F = N * hp.steps.size();
        const struct { void* dst; const void* src; size_t bytes; } seq[] = {
            {hp.seq_rgb, d.seq.rgb, 3 * F}, {hp.seq_mask, d.seq.mask, F}, {hp.seq_flow, d.seq.flow, 8 * F},
            {hp.seq_bflow, d.seq.bflow, 8 * F}, {hp.seq_occ, d.seq.occ, F}, {hp.seq_flow0, d.seq.flow0, 8 * F}};
        for (const auto& c : seq)
            if (c.dst && F) ARAP_CUDA_CHECK(cudaMemcpyAsync(c.dst, c.src, c.bytes, cudaMemcpyDeviceToHost, stream_));
    }
    // scene outputs go straight to the caller's buffers: the pair is frame index 0 of each block, frames 1 .. K follow
    for (int j = 0; j < n_scenes; ++j) {
        const HostScene& sc = scenes[j];
        const SceneLayout l(sc);
        const unsigned char* b = scene_dev_[j].data();
        const size_t N = (size_t)sc.W * sc.H, F = N * (sc.maps.size() / 18 - 1);
        const struct { void* dst; size_t off, bytes; } out[] = {
            {sc.out_flow, l.flow, 8 * N}, {sc.out_rgb, l.rgb, 3 * N}, {sc.out_mask, l.mask, N},
            {sc.out_bflow, l.bflow, 8 * N}, {sc.out_occ, l.occ, N}, {sc.out_rgb0, l.rgb0, 3 * N},
            {sc.seq_flow, l.flow + 8 * N, 8 * F}, {sc.seq_rgb, l.rgb + 3 * N, 3 * F}, {sc.seq_mask, l.mask + N, F},
            {sc.seq_bflow, l.bflow + 8 * N, 8 * F}, {sc.seq_occ, l.occ + N, F}};
        for (const auto& c : out)
            if (c.dst && c.bytes)
                ARAP_CUDA_CHECK(cudaMemcpyAsync(c.dst, b + c.off, c.bytes, cudaMemcpyDeviceToHost, stream_));
        if (!sc.blur_S) continue;
        const BlurLayout bl(sc);
        const unsigned char* bb = blur_dev_[j].data();
        const struct { void* dst; size_t off, bytes; } blurred[] = {
            {sc.blur_rgb, bl.rgb, 3 * N}, {sc.blur_rgb0, bl.rgb0, 3 * N}, {sc.seq_blur_rgb, bl.seq, 3 * F}};
        for (const auto& c : blurred)
            if (c.dst && c.bytes)
                ARAP_CUDA_CHECK(cudaMemcpyAsync(c.dst, bb + c.off, c.bytes, cudaMemcpyDeviceToHost, stream_));
    }
    ARAP_CUDA_CHECK(cudaStreamSynchronize(stream_));
    if (resident_ && n_resident_ > 0) {
        if (int st = resident_->status(stream_)) {
            fprintf(stderr, "arapb200: resident solver aborted (watchdog, code %d)\n", st);
            return 4;
        }
    }
    if (solver_ && n_resident_ < count) {
        unsigned bad = 0;
        solver_->read_back(stream_, nullptr, &bad);
        if (bad) {
            fprintf(stderr, "arapb200: internal error: UrShape check failed\n");
            return 2;
        }
    }
    for (int i = 0; i < count; ++i) {
        const HostProblem& hp = problems[i];
        Dev& d = dev_[i];
        const size_t N = (size_t)hp.W * hp.H;
        const unsigned char* o = d.h_out.data();
        if (hp.out_flow) memcpy(hp.out_flow, o, N * sizeof(float2));
        if (hp.out_rgb) memcpy(hp.out_rgb, o + 8 * N, 3 * N);
        if (hp.out_mask) memcpy(hp.out_mask, o + 11 * N, N);
        if (hp.out_costs) memcpy(hp.out_costs, o + 12 * N, cbytes);
        if (hp.out_bflow) memcpy(hp.out_bflow, d.h_extras.data() + x_bflow, N * sizeof(float2));
        if (hp.out_occ) memcpy(hp.out_occ, d.h_extras.data() + x_occ, N);
    }
    if (resident_) launches_ += resident_->launches() - r0;
    cudaEventElapsedTime(&ms_total_, ev_[0], ev_[3]);
    cudaEventElapsedTime(&ms_solve_, ev_[1], ev_[2]);
    cudaEventElapsedTime(&ms_warp_, ev_[2], ev_[3]);
    return 0;
}

} // namespace arapb200
