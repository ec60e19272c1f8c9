// solver_lm.cuh -- the reference's dormant "LMGPU" solver kind (SURVEY.md 8f N4): Levenberg-Marquardt around the same
// Jacobi-preconditioned PCG, ARAP/API/src/solverGPUGaussNewton.t with problemSpec:UsesLambda() == true
// (:616-680 kernels, :956-1007 init, :1016-1177 step).  Opt-in through Opt_ProblemDefine(..., "LMGPU"); the ARAP app
// never asks for it (CombinedSolverBase.h:76), so this back-end is written for clarity, any UrShape, plain row-major
// planes, one kernel per reference kernel -- same arithmetic contract and exact sums as the tuned back-ends, checked
// bit for bit against oracle/arap_oracle.c (arap_oracle_lm_solve).
#pragma once
#include "common.cuh"
#include "devmem.cuh"
#include "kernel_timer.cuh"

namespace arapb200 {

// SolverParameters of solverGPUGaussNewton.t:140-157 with the defaults of :26-39 (all binary32 in the reference)
struct LmParameters {
    float min_relative_decrease = (float)1e-3;
    float min_trust_region_radius = (float)1e-32;
    float max_trust_region_radius = (float)1e16;
    float q_tolerance = (float)0.0001;
    float function_tolerance = (float)0.000001;
    float trust_region_radius = (float)1e4;
    float radius_decrease_factor = (float)2.0;
    float min_lm_diagonal = (float)1e-6;
    float max_lm_diagonal = (float)1e32;
    int residual_reset_period = 10;
};

struct LmScalars {
    float num, alpha, beta, q0;  // r.z, PCG step sizes, Q of the previous iteration
    float cost, model, q_last;   // results of a step
    unsigned conv;               // zeta < q_tolerance reached: the rest of the PCG loop is a no-op
    int iters;                   // PCG iterations run in this step
    int pad[3];
};

// what one step did, for callers that want more than the cost (parity tests): oracle lm_step's stat[]
struct LmStepInfo {
    float radius_after;
    int pcg_iterations;
    int verdict; // 1 accepted, 0 reverted, 2 function tolerance reached, 3 radius below minimum
    float model_cost, new_cost, q_last;
};

class LmSolver {
public:
    LmSolver(int W, int H);
    LmSolver(const LmSolver&) = delete;
    LmSolver& operator=(const LmSolver&) = delete;

    // false = not one of the LM names
    bool set_parameter(const char* name, const void* value);
    void bind(float2* X, float* A, const float2* U, const float2* C, const float* M, float wf, float wr);
    // :956-1007 -- run-time radius / diagonal bounds from the solver parameters, prevCost = cost(X)
    float init(cudaStream_t s);
    // :1016-1177 -- returns 1 to continue, 0 when the solver stopped (tolerance / minimum radius)
    int step(int lIterations, cudaStream_t s, float* prev_cost);
    const LmStepInfo& last_step() const { return info_; }
    long long launches() const { return launches_; }
    void set_timer(KernelTimer* t) { timer_ = t; } // per-kernel timing under the reference's kernel names; null = off
    struct Dev { // the argument block of the kernels in solver_lm.cu
        int W, H;
        size_t N;
        float2* X;
        float* A;
        const float2* U;
        const float2* C;
        const float* M;
        float wf, wr, wf2, wr2;
        float* pl;
        unsigned char* flags;
        unsigned long long* acc;
        LmScalars* sc;
    };

private:
    void enqueue_cost(cudaStream_t s, int acc);
    int W_, H_;
    LmParameters sp_;                       // solver parameters (what set_parameter writes)
    float radius_ = 0.f, decrease_ = 0.f;   // pd.parameters.trust_region_radius / radius_decrease_factor (run time)
    float min_diag_ = 0.f, max_diag_ = 0.f;
    bool first_ = true;                     // nIter == 0: save the Jacobi scaling (ONCE_PER_SOLVE)
    Dev d_{};                               // host copy of the kernel argument block
    DevBuf<float> planes_;
    DevBuf<unsigned char> flags_;
    DevBuf<unsigned long long> acc_;
    DevBuf<LmScalars> sc_;
    DevBuf<LmScalars> h_sc_;                // pinned
    LmStepInfo info_{};
    long long launches_ = 0;
    KernelTimer* timer_ = nullptr;
};

} // namespace arapb200
