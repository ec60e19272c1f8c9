// plan.cu -- see plan.cuh
#include "plan.cuh"
#include <cstring>

namespace arapb200 {

namespace {
constexpr int kMaxCostLog = 4096;
// the resident and streaming kernels are specialised for UrShape == pixel grid: verify it
// out[0] = number of active pixels whose UrShape is not the pixel grid; out[1..2] = an order-free 64-bit fingerprint of
// the active set (sum and xor of a mixed pixel index), used to recognise "same mask as the previous call" so that the
// strip tables of the resident back-end are rebuilt only when the mask really changed (one image = 19 Opt_ProblemSolve
// calls with the same Mask pointer, CombinedSolverBase.h:108-117).
__device__ __forceinline__ unsigned long long mix64(unsigned long long x)
{
    x ^= x >> 33; x *= 0xff51afd7ed558ccdull; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull; x ^= x >> 33;
    return x;
}
__global__ void __launch_bounds__(256) k_check_grid(int W, int H, const float2* __restrict__ U,
                                                     const float* __restrict__ M, unsigned long long* __restrict__ out)
{
    const size_t N = (size_t)W * H;
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long h = 0, bad = 0;
    if (i < N && M[i] == 0.0f) {
        const float2 u = U[i];
        bad = (u.x != (float)(int)(i % W) || u.y != (float)(int)(i / W)) ? 1ull : 0ull;
        h = mix64(i + 0x9E3779B97F4A7C15ull);
    }
    unsigned long long hx = h;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        h += __shfl_xor_sync(0xffffffffu, h, o);
        hx ^= __shfl_xor_sync(0xffffffffu, hx, o);
        bad += __shfl_xor_sync(0xffffffffu, bad, o);
    }
    if ((threadIdx.x & 31) == 0) {
        if (bad) atomicAdd(out, bad);
        if (h) { atomicAdd(out + 1, h); atomicXor(out + 2, hx); }
    }
}
} // namespace

GnPlan::GnPlan(int W, int H, int verbosity, int backend, bool lm, bool collect_timing)
    : W_(W), H_(H), verbosity_(verbosity), backend_(backend), collect_timing_(collect_timing)
{
    if (lm) lm_.reset(new LmSolver(W, H));
    stream_h_ = make_stream();
    d_costs_ = DevBuf<float>(kMaxCostLog);
    d_check_ = DevBuf<unsigned long long>(3);
    h_check_ = DevBuf<unsigned long long>(3, GrowBuf::Pinned);
}

// The caller works on the default stream (the reference host: cudaMemset of Angle on the legacy stream,
// ARAP/deformation/src/CombinedSolver.h:220, pageable cudaMemcpy uploads whose last DMA may still be in flight when
// the call returns, ARAP/shared/OptImage.h:50); upstream Opt ran on that same stream and was ordered behind it for free.
// This library runs on its own non-blocking stream, so every Opt_* entry that touches the images first waits for both
// flavours of the default stream.
void GnPlan::order_after_caller()
{
    ARAP_CUDA_CHECK(cudaStreamSynchronize(cudaStreamLegacy));
    ARAP_CUDA_CHECK(cudaStreamSynchronize(cudaStreamPerThread));
}

long long GnPlan::launches() const
{
    return (stream_ ? stream_->launches() : 0) + (resident_ ? resident_->launches() : 0) + (lm_ ? lm_->launches() : 0);
}

GnPlan::~GnPlan()
{
    cudaStreamSynchronize(stream_h_.get());
}

bool GnPlan::set_parameter(const char* name, const void* value)
{
    if (strcmp(name, "nIterations") == 0) { n_iterations_ = *(const int*)value; return true; }
    if (strcmp(name, "lIterations") == 0) { l_iterations_ = *(const int*)value; return true; }
    // extension (SURVEY.md 8f N4): float, relative PCG tolerance; 0 (default) = the reference's fixed budget
    // ("gn_rtol": the same one level up; both are range-checked: 0 <= v < 1, anything else is ignored with a message)
    if (strcmp(name, "pcg_rtol") == 0 || strcmp(name, "gn_rtol") == 0) {
        const float v = *(const float*)value;
        if (!(v >= 0.0f) || v >= 1.0f) {
            fprintf(stderr, "arapb200: %s = %g is outside [0, 1): ignored\n", name, (double)v);
            return true;
        }
        (name[0] == 'p' ? pcg_rtol_ : gn_rtol_) = v;
        return true;
    }
    if (lm_ && lm_->set_parameter(name, value)) return true;
    // Levenberg-Marquardt knobs of SolverParameters (:26-39): valid names, unused by gaussNewtonGPU
    static const char* lm[] = {"residual_reset_period", "min_relative_decrease", "min_trust_region_radius",
                               "max_trust_region_radius", "q_tolerance", "function_tolerance",
                               "trust_region_radius", "radius_decrease_factor", "min_lm_diagonal",
                               "max_lm_diagonal"};
    for (const char* k : lm)
        if (strcmp(name, k) == 0) return true;
    return false;
}

// AUTO: resident when the active part of the image fits on chip, else streaming.  An UrShape image other than the pixel
// grid (never bound by the ARAP app, CombinedSolver.h:207-221, but legal for an Opt.h caller) takes the streaming
// back-end's general-d kernels.
void GnPlan::choose_backend(void** pp)
{
    order_after_caller();
    const size_t N = (size_t)W_ * H_;
    cudaStream_t s = stream_h_.get();
    ARAP_CUDA_CHECK(cudaMemsetAsync(d_check_.p, 0, 3 * sizeof(unsigned long long), s));
    k_check_grid<<<(unsigned)((N + 255) / 256), 256, 0, s>>>(W_, H_, (const float2*)pp[2], (const float*)pp[4],
                                                             d_check_.p);
    ARAP_CUDA_CHECK(cudaMemcpyAsync(h_check_.p, d_check_.p, 3 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
    ARAP_CUDA_CHECK(cudaStreamSynchronize(s));
    const unsigned long long* chk = h_check_.p;
    general_ = chk[0] != 0;
    const bool same_mask = have_mask_key_ && mask_ptr_ == pp[4] && mask_key_[0] == chk[1] && mask_key_[1] == chk[2];
    mask_ptr_ = pp[4]; mask_key_[0] = chk[1]; mask_key_[1] = chk[2]; have_mask_key_ = true;
    const bool was_resident = use_resident_;
    use_resident_ = false;
    // per-kernel timing needs kernels to time: the streaming back-end (same results bit for bit), launched eagerly
    if (backend_ != ARAPB200_BACKEND_STREAM && !general_ && !collect_timing_) {
        if (!resident_) resident_.reset(new ResidentSolver(W_, H_));
        // same Mask image as the previous call: the strip tables are still valid
        use_resident_ = (same_mask && was_resident) ? true : resident_->prepare(W_, H_, (const float*)pp[4], s);
        if (!use_resident_ && backend_ == ARAPB200_BACKEND_RESIDENT)
            arap_fail(1, "problem %dx%d (%d strips) does not fit the resident back-end", W_, H_, resident_->n_strips());
    }
    if (!use_resident_) {
        if (!stream_) stream_.reset(new StreamSolver(W_, H_));
        stream_->set_general(general_);
        stream_->set_timer(collect_timing_ ? timer_.get() : nullptr);
        stream_->set_pcg_rtol(general_ ? 0.0f : pcg_rtol_);
        stream_->set_gn_rtol(general_ ? 0.0f : gn_rtol_);
        if (general_ && (gn_rtol_ > 0.0f || pcg_rtol_ > 0.0f) && !warned_rtol_) { // never silently
            warned_rtol_ = true;
            fprintf(stderr, "arapb200: warning: pcg_rtol / gn_rtol are not honoured for a non-grid UrShape (general-d kernels): "
                            "this %dx%d problem runs the fixed budget\n", W_, H_);
        }
    }
}

// resident launch: cost before and after each of nGN Gauss-Newton steps; returns the last cost
float GnPlan::run_resident(void** pp, int nGN, float* trace)
{
    if (nGN + 1 > kMaxCostLog) arap_fail(1, "nIterations too large");
    resident_->set_pcg_rtol(pcg_rtol_);
    resident_->set_gn_rtol(gn_rtol_);
    resident_->enqueue((float2*)pp[0], (float*)pp[1], (const float2*)pp[3], 0, *(const float*)pp[5],
                       *(const float*)pp[6], 1, nGN, l_iterations_, d_costs_.p, trace, stream_h_.get());
    float c = 0.f;
    ARAP_CUDA_CHECK(cudaMemcpyAsync(&c, d_costs_.p + nGN, sizeof(float), cudaMemcpyDeviceToHost, stream_h_.get()));
    ARAP_CUDA_CHECK(cudaStreamSynchronize(stream_h_.get()));
    if (int st = resident_->status(stream_h_.get())) arap_fail(3, "resident solver aborted (watchdog, code %d)", st);
    return c;
}

void GnPlan::bind(void** pp)
{
    // arap_plan.t:2-8: Offset, Angle, UrShape, Constraints, Mask, w_fitSqrt, w_regSqrt
    // (scalars are dereferenced on the host at init AND at every step: util.t:664-692)
    stream_->bind((float2*)pp[0], (float*)pp[1], (const float2*)pp[2], (const float2*)pp[3], (const float*)pp[4],
                  *(const float*)pp[5], *(const float*)pp[6], stream_h_.get());
}

void GnPlan::timer_begin()
{
    timer_.reset();
    if (verbosity_ > 0 || collect_timing_) {
        timer_.reset(new KernelTimer);
        overall_idx_ = timer_->start("overall", stream_h_.get());
    }
    if (lm_) lm_->set_timer(collect_timing_ ? timer_.get() : nullptr);
}

// solverGPUGaussNewton.t:1009-1014: end of a solve -- "final cost", then the timer table
void GnPlan::cleanup()
{
    if (verbosity_ > 0) printf("final cost=%f\n", prev_cost_);
    if (!timer_) return;
    timer_->stop_at(overall_idx_, stream_h_.get());
    timing_report_ = KernelTimer::format(timer_->aggregate());
    if (verbosity_ > 0) fputs(timing_report_.c_str(), stdout); // Timer:evaluate prints under verbosity only (util.t:452)
    if (stream_) stream_->set_timer(nullptr);
    if (lm_) lm_->set_timer(nullptr);
    timer_.reset();
}

void GnPlan::lm_bind(void** pp)
{
    lm_->bind((float2*)pp[0], (float*)pp[1], (const float2*)pp[2], (const float2*)pp[3], (const float*)pp[4],
              *(const float*)pp[5], *(const float*)pp[6]);
}

void GnPlan::init(void** pp)
{
    timer_begin();
    if (lm_) {
        order_after_caller();
        lm_bind(pp);
        n_iter_ = 0;
        prev_cost_ = lm_->init(stream_h_.get());
        return;
    }
    choose_backend(pp);
    n_iter_ = 0;
    if (use_resident_) {
        prev_cost_ = run_resident(pp, 0, nullptr);
        return;
    }
    bind(pp);
    stream_->enqueue_init(stream_h_.get());
    stream_->read_back(stream_h_.get(), &prev_cost_, nullptr);
}

int GnPlan::step(void** pp)
{
    if (n_iter_ >= n_iterations_) { cleanup(); return 0; }
    order_after_caller();
    if (lm_) {
        lm_bind(pp);
        const float before = prev_cost_;
        const int more = lm_->step(l_iterations_, stream_h_.get(), &prev_cost_);
        if (verbosity_ > 0) {
            const LmStepInfo& st = lm_->last_step();
            printf("cost: %f -> %f (model %f, %d linear iterations, %s, trust_region_radius=%f)\n", before, st.new_cost,
                   st.model_cost, st.pcg_iterations,
                   st.verdict == 1 ? "accepted" : st.verdict == 0 ? "REVERT" : st.verdict == 2 ? "function tolerance reached"
                                                                                              : "radius below the minimum",
                   st.radius_after);
        }
        if (!more) { cleanup(); return 0; } // tolerance / minimum radius: nIter does not advance (:1129-1133, :1149-1153)
        ++n_iter_;
        return 1;
    }
    float* tr = d_trace_ ? d_trace_ + (size_t)3 * l_iterations_ * n_iter_ : nullptr;
    float c;
    if (use_resident_) {
        c = run_resident(pp, 1, tr);
    } else {
        bind(pp);
        stream_->enqueue_gn_step(l_iterations_, stream_h_.get(), tr);
        stream_->read_back(stream_h_.get(), &c, nullptr);
    }
    if (verbosity_ > 0) printf("cost: %f -> %f\n", prev_cost_, c); // :1158-1163
    prev_cost_ = c;
    ++n_iter_;
    return 1;
}

void GnPlan::solve(void** pp)
{
    if (verbosity_ > 0 || lm_ || collect_timing_) { // per-step prints / host decisions / per-kernel events: the stepwise path
        init(pp);
        while (step(pp)) {}
        return;
    }
    choose_backend(pp);
    n_iter_ = 0;
    if (use_resident_) {
        prev_cost_ = run_resident(pp, n_iterations_, d_trace_); // ONE launch for the whole Opt_ProblemSolve
        n_iter_ = n_iterations_;
        return;
    }
    bind(pp);
    stream_->enqueue_init(stream_h_.get());
    for (; n_iter_ < n_iterations_; ++n_iter_) {
        float* tr = d_trace_ ? d_trace_ + (size_t)3 * l_iterations_ * n_iter_ : nullptr;
        stream_->enqueue_gn_step(l_iterations_, stream_h_.get(), tr);
    }
    stream_->read_back(stream_h_.get(), &prev_cost_, nullptr);
}

} // namespace arapb200
