// plan.cuh -- the object behind Opt_Plan: solver parameters, iteration state and the back-end.
// Mirrors the plan vtable {init, step, cost, setsolverparameter, free} of ARAP/API/src/o.t:126-133 as
// filled by ARAP/API/src/solverGPUGaussNewton.t:1254-1284.
#pragma once
#include "../../include/arapb200.h"
#include "solver_stream.cuh"
#include "solver_resident.cuh"
#include "solver_lm.cuh"
#include <memory>
#include <string>

namespace arapb200 {

class GnPlan {
public:
    // lm: the "LMGPU" solver kind (Levenberg-Marquardt, solver_lm.cuh) instead of "gaussNewtonGPU"
    // collect_timing: Opt_InitializationParameters.collectPerKernelTimingInfo (kernel_timer.cuh)
    GnPlan(int W, int H, int verbosity, int backend, bool lm = false, bool collect_timing = false);
    ~GnPlan();
    // solverGPUGaussNewton.t:1205-1221.  false = unknown name.
    bool set_parameter(const char* name, const void* value);
    void init(void** problemparams);  // :956-1007
    int step(void** problemparams);   // :1016-1177
    void solve(void** problemparams); // o.t:2548-2551, with a single host sync at the end
    double current_cost() const { return (double)prev_cost_; }
    // sticky error of the Opt_* entry points (they have no error return): 0 = fine
    int error() const { return error_; }
    void set_error(int code) { error_ = code ? code : 1; prev_cost_ = __builtin_nanf(""); }
    long long launches() const;
    bool using_resident() const { return use_resident_; }
    bool general_urshape() const { return general_; }
    bool is_lm() const { return lm_ != nullptr; }
    const LmStepInfo* lm_last_step() const { return lm_ ? &lm_->last_step() : nullptr; }
    // parity/debug: device buffer of 3*lIterations floats per GN step, or null
    void set_trace(float* d_trace) { d_trace_ = d_trace; }
    // the table the reference prints at the end of a solve (util.t:469-508), of the last finished solve; empty if none
    const std::string& timing_report() const { return timing_report_; }

private:
    void bind(void** problemparams);
    int W_, H_, verbosity_, backend_;
    int n_iterations_ = 10, l_iterations_ = 10; // solver_parameter_defaults, :26-39
    float pcg_rtol_ = 0.0f, gn_rtol_ = 0.0f;    // extensions, 0 = off
    bool warned_rtol_ = false;
    int n_iter_ = 0;
    int error_ = 0;
    float prev_cost_ = 0.f;
    StreamHandle stream_h_;                     // declared before the solvers: destroyed after them
    std::unique_ptr<StreamSolver> stream_;      // created on first use
    std::unique_ptr<ResidentSolver> resident_;  // created on first use
    std::unique_ptr<LmSolver> lm_;              // "LMGPU" plans only
    bool collect_timing_ = false;
    std::unique_ptr<KernelTimer> timer_;        // verbosity > 0 or collect_timing_: "overall" (+ per-kernel) events
    size_t overall_idx_ = 0;
    std::string timing_report_;
    void timer_begin();                         // init: Timer:init + startEvent("overall") (:958-960)
    void cleanup();                             // :1009-1014
    void lm_bind(void** problemparams);
    bool use_resident_ = false;
    bool general_ = false;                      // UrShape is not the pixel grid
    void** last_params_ = nullptr;
    DevBuf<float> d_costs_;                     // resident: cost log of the current launch
    DevBuf<unsigned long long> d_check_;        // [0] non-grid UrShape count, [1..2] fingerprint of the active set
    DevBuf<unsigned long long> h_check_;        // pinned copy
    const void* mask_ptr_ = nullptr;            // Mask image + fingerprint the resident strip tables were built for
    unsigned long long mask_key_[2] = {0, 0};
    bool have_mask_key_ = false;
    void order_after_caller();
    float* d_trace_ = nullptr;
    void choose_backend(void** problemparams);
    float run_resident(void** problemparams, int nGN, float* trace);
};

} // namespace arapb200
