// opt_api.cu -- the 10 Opt_* entry points of include/Opt.h over the hand-written solver back-ends.
//
// Reference behaviour being replaced: ARAP/API/src/createwrapper.t:124-220 (thunks),
// ARAP/API/src/o.t:2521-2558 (API bodies), ARAP/API/src/solverGPUGaussNewton.t:956-1007 (init),
// :1016-1177 (step), :1179-1182 (cost), :1205-1221 (setSolverParameter), :1223-1284 (free/makePlan).
#include "../../include/Opt.h"
#include "../../include/arapb200.h"
#include "plan.cuh"

#include <cstring>
#include <memory>
#include <string>

using namespace arapb200;

struct Opt_State {
    Opt_InitializationParameters params;
};

struct Opt_Problem {
    std::string filename;
    bool lm = false; // solver kind "LMGPU"
};

struct Opt_Plan {
    std::unique_ptr<GnPlan> plan;
};

// These three have no error return in the ABI.  A failure (CUDA error, watchdog) is printed, recorded on the plan
// (arapb200_plan_error, below) and makes Opt_ProblemCurrentCost return NaN; Opt_ProblemStep reports "finished" so that
// a stepping caller's loop ends.  The reference exits the process instead (solverGPUGaussNewton.t:59-73).
template <class F>
static void plan_guard(Opt_Plan* plan, F&& f)
{
    if (!plan || !plan->plan) return;
    try {
        f();
    } catch (const ArapError& e) {
        plan->plan->set_error(e.code);
    } catch (...) {
        plan->plan->set_error(2);
    }
}

extern "C" {

Opt_State* Opt_NewState(Opt_InitializationParameters params)
{
    if (params.doublePrecision) {
        fprintf(stderr, "arapb200: doublePrecision is not supported (the ARAP app never enables it: "
                        "CombinedSolverParameters.h:14)\n");
        return nullptr;
    }
    Opt_State* s = new Opt_State;
    s->params = params;
    return s;
}

// The energy file is identified, not interpreted: it must exist and declare the ARAP unknowns.
static bool looks_like_arap_plan(const char* filename)
{
    FILE* f = fopen(filename, "rb");
    if (!f) return false;
    std::string txt;
    char buf[4096];
    size_t n;
    while ((n = fread(buf, 1, sizeof(buf), f)) > 0 && txt.size() < (1u << 20)) txt.append(buf, n);
    fclose(f);
    const char* need[] = {"Offset", "Angle", "UrShape", "Constraints", "Mask", "w_fitSqrt", "w_regSqrt", "Rotate2D"};
    for (const char* k : need)
        if (txt.find(k) == std::string::npos) return false;
    return true;
}

Opt_Problem* Opt_ProblemDefine(Opt_State* state, const char* filename, const char* solverkind)
{
    if (!state || !filename || !solverkind) return nullptr;
    // o.t:121-124 asserts gaussNewtonGPU or LMGPU; the app only ever asks for the former (CombinedSolverBase.h:76)
    const bool lm = strcmp(solverkind, "LMGPU") == 0;
    if (!lm && strcmp(solverkind, "gaussNewtonGPU") != 0) {
        fprintf(stderr, "arapb200: solver kind '%s' not supported (gaussNewtonGPU or LMGPU)\n", solverkind);
        return nullptr;
    }
    if (!looks_like_arap_plan(filename)) {
        fprintf(stderr, "arapb200: '%s' is missing or is not the ARAP energy (arap_plan.t)\n", filename);
        return nullptr;
    }
    Opt_Problem* p = new Opt_Problem;
    p->filename = filename;
    p->lm = lm;
    return p;
}

void Opt_ProblemDelete(Opt_State*, Opt_Problem* problem) { delete problem; }

Opt_Plan* Opt_ProblemPlan(Opt_State* state, Opt_Problem* problem, unsigned int* dimensions)
{
    if (!state || !problem || !dimensions) return nullptr;
    const unsigned W = dimensions[0], H = dimensions[1];
    if (W == 0 || H == 0 || W > 65535u || H > 65535u) {
        fprintf(stderr, "arapb200: bad plan dimensions %u x %u\n", W, H);
        return nullptr;
    }
    // failure => NULL, which the reference caller asserts on (ARAP/shared/OptSolver.h:54-56)
    try {
        std::unique_ptr<GnPlan> plan(new GnPlan((int)W, (int)H, state->params.verbosityLevel, ARAPB200_BACKEND_AUTO,
                                                problem->lm, state->params.collectPerKernelTimingInfo != 0));
        return new Opt_Plan{std::move(plan)};
    } catch (...) {
        fprintf(stderr, "arapb200: Opt_ProblemPlan failed for %u x %u\n", W, H);
        return nullptr;
    }
}

void Opt_PlanFree(Opt_State*, Opt_Plan* plan) { delete plan; }

void Opt_SetSolverParameter(Opt_State* state, Opt_Plan* plan, const char* name, void* value)
{
    if (!plan || !name || !value) return;
    if (!plan->plan->set_parameter(name, value) && state && state->params.verbosityLevel > 0)
        fprintf(stderr, "Warning: tried to set nonexistent solver parameter %s\n", name); // :1220
}

void Opt_ProblemInit(Opt_State*, Opt_Plan* plan, void** problemparams)
{
    plan_guard(plan, [&] { plan->plan->init(problemparams); });
}

int Opt_ProblemStep(Opt_State*, Opt_Plan* plan, void** problemparams)
{
    int more = 0;
    plan_guard(plan, [&] { more = plan->plan->step(problemparams); });
    return (plan && plan->plan && plan->plan->error()) ? 0 : more;
}

void Opt_ProblemSolve(Opt_State*, Opt_Plan* plan, void** problemparams)
{
    // o.t:2548-2551: init, then step until it reports completion
    plan_guard(plan, [&] { plan->plan->solve(problemparams); });
}

double Opt_ProblemCurrentCost(Opt_State*, Opt_Plan* plan) { return plan->plan->current_cost(); }

// extension (not in the reference's Opt.h): 0, or the code of the first failure since the plan was made
int arapb200_plan_error(Opt_Plan* plan) { return (plan && plan->plan) ? plan->plan->error() : 1; }

// extension: the kernel-timing table of the last finished solve of a plan whose state was created with
// collectPerKernelTimingInfo (or verbosityLevel > 0: then only the "overall" row) -- the text the reference prints at the
// end of a solve (util.t:469-508).  Copies at most cap - 1 characters, returns the full length.
size_t arapb200_plan_timing_report(Opt_Plan* plan, char* buf, size_t cap)
{
    if (!plan || !plan->plan) return 0;
    const std::string& r = plan->plan->timing_report();
    if (buf && cap) {
        const size_t n = r.size() < cap - 1 ? r.size() : cap - 1;
        memcpy(buf, r.data(), n);
        buf[n] = 0;
    }
    return r.size();
}

// extension: what the last Opt_ProblemStep of an "LMGPU" plan did.  info6 = trust-region radius after the step, linear
// iterations run, verdict (1 accepted, 0 reverted, 2 function tolerance reached, 3 radius below minimum), model cost,
// cost at the trial point, last Q.  Returns 0, or 1 when the plan is not an LM plan.
int arapb200_plan_lm_info(Opt_Plan* plan, float info6[6])
{
    const LmStepInfo* st = (plan && plan->plan) ? plan->plan->lm_last_step() : nullptr;
    if (!st || !info6) return 1;
    info6[0] = st->radius_after; info6[1] = (float)st->pcg_iterations; info6[2] = (float)st->verdict;
    info6[3] = st->model_cost; info6[4] = st->new_cost; info6[5] = st->q_last;
    return 0;
}

} // extern "C"
