// solver_lm.cu -- see solver_lm.cuh.  One kernel per kernel of the reference's LM path; a thread owns one contract-C3
// group (an aligned vertical quad of pixels), a warp 32 neighbouring columns, so every plane access is coalesced and
// the per-thread partial IS the group term.  Grid-wide sums go through the fence-free wide accumulators of common.cuh
// and are rounded once by a one-warp scalar kernel -- the PCG loop runs without a host round trip (the reference
// fetches Q with a blocking cudaMemcpy every iteration, solverGPUGaussNewton.t:829-833, :1093); its q_tolerance exit
// is a sticky device flag that turns the remaining launches into no-ops and that the host polls every 16 iterations.
#include "solver_lm.cuh"
#include "grid_math.cuh"
#include <cmath>
#include <cstring>

namespace arapb200 {

namespace {
using Dev = LmSolver::Dev;

constexpr int LM_THREADS = 128;
constexpr int LM_RING = 64; // PCG iterations whose accumulators are live at a time (accumulator sets: LmSolver::LmSolver)
// planes of N floats each
enum : int {
    L_CS = 0,    // cos, sin of the angle the current linearisation uses
    L_R = 2,     // residual
    L_P = 5,     // direction
    L_Q = 8,     // (J^T J + CtC) p
    L_PRE = 11,  // preconditioner: position entry, angle entry
    L_D = 13,    // delta
    L_CTC = 16,  // clamped C^T C: position entry, angle entry
    L_B = 18,    // right-hand side (r at PCGFinalizeDiagonal)
    L_SSQ = 21,  // Jacobi scaling saved at the first iteration of a solve
    L_AD = 23,   // (J^T J + CtC) delta, residual refresh
    L_PREV = 26, // unknowns before the speculative update
    L_PLANES = 29
};
enum : unsigned { LF_ACTIVE = 16u, LF_FIT = 32u }; // bits 0..3: neighbour n valid (+x, -x, +y, -y)

__device__ __forceinline__ float* plane(const Dev& d, int k) { return d.pl + (size_t)k * d.N; }
__device__ __forceinline__ unsigned long long* acc_set(const Dev& d, int set) { return d.acc + (size_t)set * WA_WORDS; }
__device__ __forceinline__ void publish(const Dev& d, int set, HL v)
{
    const unsigned copy = blockIdx.y * gridDim.x + blockIdx.x;
    if (threadIdx.x == 0) wide_add(acc_set(d, set), copy, v.h);
    if (threadIdx.x == 1) wide_add(acc_set(d, set), copy, v.l);
}
// one warp: the rounded values of two accumulators (lane 0 / lane 16 hold them after the call; returned to every lane)
__device__ __forceinline__ void decode2(const Dev& d, int set_a, int set_b, float& a, float& b)
{
    const int lane = threadIdx.x & 31;
    const float v = wide_round(wide_fetch(acc_set(d, lane < 16 ? set_a : set_b), lane & 15));
    a = __shfl_sync(0xffffffffu, v, 0);
    b = __shfl_sync(0xffffffffu, v, 16);
}
__device__ __forceinline__ size_t nb_index(const Dev& d, size_t i, int n)
{
    return n == 0 ? i + 1 : n == 1 ? i - 1 : n == 2 ? i + d.W : i - d.W;
}

// the quad of pixels a thread owns
struct Quad {
    int x, y0;
    bool on;
};
__device__ __forceinline__ Quad my_quad(const Dev& d)
{
    Quad q;
    q.x = blockIdx.x * 32 + (threadIdx.x & 31);
    q.y0 = (blockIdx.y * 4 + (threadIdx.x >> 5)) * 4;
    q.on = q.x < d.W;
    return q;
}

__global__ void __launch_bounds__(256) k_lm_flags(const Dev d)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= d.N) return;
    const int x = (int)(i % d.W), y = (int)(i / d.W);
    unsigned f = 0;
    if (d.M[i] == 0.0f) { // arap_plan.t:11
        f = LF_ACTIVE;
        if (x + 1 < d.W && d.M[i + 1] == 0.0f) f |= 1u;
        if (x > 0 && d.M[i - 1] == 0.0f) f |= 2u;
        if (y + 1 < d.H && d.M[i + d.W] == 0.0f) f |= 4u;
        if (y > 0 && d.M[i - d.W] == 0.0f) f |= 8u;
        const float2 c = d.C[i];
        if (c.x >= 0.0f && c.y >= 0.0f) f |= LF_FIT; // arap_plan.t:22
    }
    d.flags[i] = (unsigned char)f;
}

__global__ void __launch_bounds__(256) k_lm_cs(const Dev d)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= d.N || !(d.flags[i] & LF_ACTIVE)) return;
    float s, c;
    contract_sincos(d.A[i], s, c);
    plane(d, L_CS)[i] = c;
    plane(d, L_CS + 1)[i] = s;
}

// computeCost (:580-592)
__global__ void __launch_bounds__(LM_THREADS) k_lm_cost(const Dev d, int set)
{
    __shared__ double red[64];
    const Quad q = my_quad(d);
    const float *cs0 = plane(d, L_CS), *cs1 = plane(d, L_CS + 1);
    float g = 0.0f;
    if (q.on) {
        for (int r = 0; r < 4; ++r) {
            const int y = q.y0 + r;
            if (y >= d.H) break;
            const size_t i = (size_t)y * d.W + q.x;
            const unsigned f = d.flags[i];
            if (!(f & LF_ACTIVE)) continue;
            const float2 Xi = d.X[i], ui = d.U[i];
            float acc = 0.0f;
#pragma unroll
            for (int n = 0; n < 4; ++n) {
                if (!(f & (1u << n))) continue;
                const size_t j = nb_index(d, i, n);
                const float2 Xj = d.X[j], uj = d.U[j];
                acc = cost_nb_gen(acc, Xi.x, Xi.y, cs0[i], cs1[i], Xj.x, Xj.y, ui.x - uj.x, ui.y - uj.y, d.wr);
            }
            if (f & LF_FIT) {
                const float2 c = d.C[i];
                acc = cost_fit(acc, Xi.x, Xi.y, c.x, c.y, d.wf);
            }
            g = g + acc;
        }
    }
    publish(d, set, block_exact_sum(g, red));
}

// PCGInit1 (:361-397) + PCGSaveSSq (:624-629) + PCGComputeCtC (:616-622) + PCGFinalizeDiagonal (:631-664)
__device__ __forceinline__ void lm_diagonal(float D, bool first, float radius, float inv_radius, float min_diag,
                                            float max_diag, float& ssq, float& ctc, float& pre)
{
    if (first) ssq = guarded_invert(D); // jacobiScaling ONCE_PER_SOLVE (:18-24)
    const float u = D * inv_radius;     // o.t:2277-2279
    const float invS = 1.0f / ssq;
    const float mult = invS / radius;
    const float lo = min_diag * mult, hi = max_diag * mult;
    ctc = fminf(fmaxf(u, lo), hi);
    pre = 1.0f / (ctc + radius * u);
}

__global__ void __launch_bounds__(LM_THREADS) k_lm_init(const Dev d, int first, float radius, float inv_radius,
                                                        float min_diag, float max_diag, int set_num, int set_q)
{
    __shared__ double red[64];
    __shared__ double red2[64];
    const Quad q = my_quad(d);
    const float *cs0 = plane(d, L_CS), *cs1 = plane(d, L_CS + 1);
    float g = 0.0f, gq = 0.0f;
    if (q.on) {
        for (int r = 0; r < 4; ++r) {
            const int y = q.y0 + r;
            if (y >= d.H) break;
            const size_t i = (size_t)y * d.W + q.x;
            const unsigned f = d.flags[i];
            if (!(f & LF_ACTIVE)) continue;
            const float2 Xi = d.X[i], ui = d.U[i];
            const float ci = cs0[i], si = cs1[i];
            JtfAcc a;
            jtf_zero(a);
#pragma unroll
            for (int n = 0; n < 4; ++n) {
                if (!(f & (1u << n))) continue;
                const size_t j = nb_index(d, i, n);
                const float2 Xj = d.X[j], uj = d.U[j];
                jtf_nb_gen(a, Xi.x, Xi.y, ci, si, Xj.x, Xj.y, cs0[j], cs1[j], ui.x - uj.x, ui.y - uj.y);
            }
            const bool fit = (f & LF_FIT) != 0;
            float2 c = make_float2(0.f, 0.f);
            if (fit) c = d.C[i];
            float g0, g1, ga, DX, DA;
            jtf_finish(a, Xi.x, Xi.y, fit, c.x, c.y, d.wr2, d.wf2, g0, g1, ga, DX, DA);
            float sX = plane(d, L_SSQ)[i], sA = plane(d, L_SSQ + 1)[i], cX, cA, pX, pA;
            lm_diagonal(DX, first != 0, radius, inv_radius, min_diag, max_diag, sX, cX, pX);
            lm_diagonal(DA, first != 0, radius, inv_radius, min_diag, max_diag, sA, cA, pA);
            if (first) { plane(d, L_SSQ)[i] = sX; plane(d, L_SSQ + 1)[i] = sA; }
            plane(d, L_CTC)[i] = cX; plane(d, L_CTC + 1)[i] = cA;
            plane(d, L_PRE)[i] = pX; plane(d, L_PRE + 1)[i] = pA;
            const float r0 = -g0, r1 = -g1, r2 = -ga;
            const float p0 = pX * r0, p1 = pX * r1, p2 = pA * r2;
            plane(d, L_R)[i] = r0; plane(d, L_R + 1)[i] = r1; plane(d, L_R + 2)[i] = r2;
            plane(d, L_B)[i] = r0; plane(d, L_B + 1)[i] = r1; plane(d, L_B + 2)[i] = r2;
            plane(d, L_P)[i] = p0; plane(d, L_P + 1)[i] = p1; plane(d, L_P + 2)[i] = p2;
            plane(d, L_D)[i] = 0.f; plane(d, L_D + 1)[i] = 0.f; plane(d, L_D + 2)[i] = 0.f;
            g = g + dot3(r0, r1, r2, p0, p1, p2);
            gq = gq + 0.5f * dot3(0.f, 0.f, 0.f, r0 + r0, r1 + r1, r2 + r2); // Q with delta = 0 (:658-660)
        }
    }
    publish(d, set_num, block_exact_sum(g, red));
    publish(d, set_q, block_exact_sum(gq, red2));
}

// scalars of PCGInit: r.z and Q0
__global__ void __launch_bounds__(32) k_lm_begin(const Dev d, int set_num, int set_q)
{
    float num, q0;
    decode2(d, set_num, set_q, num, q0);
    if (threadIdx.x == 0) {
        d.sc->num = num; d.sc->q0 = q0; d.sc->q_last = q0;
        d.sc->alpha = 0.f; d.sc->beta = 0.f; d.sc->conv = 0u; d.sc->iters = 0;
    }
}

// PCGStep1 (:421-434) for MODE 0 (v = p, out = q, sum p.q) / computeAdelta (:566-571) for MODE 1 (v = delta, out = Adelta)
template <int MODE>
__global__ void __launch_bounds__(LM_THREADS) k_lm_apply(const Dev d, int set_den)
{
    __shared__ double red[64];
    if (d.sc->conv) return;
    const Quad q = my_quad(d);
    const float *cs0 = plane(d, L_CS), *cs1 = plane(d, L_CS + 1);
    const float* v = plane(d, MODE == 0 ? L_P : L_D);
    float* out = plane(d, MODE == 0 ? L_Q : L_AD);
    const size_t N = d.N;
    float g = 0.0f;
    if (q.on) {
        for (int r = 0; r < 4; ++r) {
            const int y = q.y0 + r;
            if (y >= d.H) break;
            const size_t i = (size_t)y * d.W + q.x;
            const unsigned f = d.flags[i];
            if (!(f & LF_ACTIVE)) continue;
            const float2 ui = d.U[i];
            const float v0 = v[i], v1 = v[i + N], va = v[i + 2 * N];
            JtjAcc a;
            jtj_zero(a);
#pragma unroll
            for (int n = 0; n < 4; ++n) {
                if (!(f & (1u << n))) continue;
                const size_t j = nb_index(d, i, n);
                const float2 uj = d.U[j];
                jtj_nb_gen(a, v0, v1, v[j], v[j + N], v[j + 2 * N], cs0[j], cs1[j], ui.x - uj.x, ui.y - uj.y);
            }
            float q0, q1, qa;
            jtj_finish(a, cs0[i], cs1[i], v0, v1, va, (f & LF_FIT) != 0, d.wr2, d.wf2, q0, q1, qa);
            const float cX = plane(d, L_CTC)[i], cA = plane(d, L_CTC + 1)[i];
            q0 = fmaf(cX, v0, q0); // o.t:2076-2082
            q1 = fmaf(cX, v1, q1);
            qa = fmaf(cA, va, qa);
            out[i] = q0; out[i + N] = q1; out[i + 2 * N] = qa;
            if (MODE == 0) g = g + dot3(v0, v1, va, q0, q1, qa);
        }
    }
    if (MODE == 0) publish(d, set_den, block_exact_sum(g, red));
}

__global__ void __launch_bounds__(32) k_lm_alpha(const Dev d, int set_den)
{
    if (d.sc->conv) return;
    float den, unused;
    decode2(d, set_den, set_den, den, unused);
    if (threadIdx.x == 0) d.sc->alpha = (den > 0.0f) ? d.sc->num / den : 0.0f; // :456-459
}

// PCGStep2_1stHalf (:491-503)
__global__ void __launch_bounds__(256) k_lm_axpy(const Dev d)
{
    if (d.sc->conv) return;
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= d.N || !(d.flags[i] & LF_ACTIVE)) return;
    const float alpha = d.sc->alpha;
    const float* p = plane(d, L_P);
    float* dl = plane(d, L_D);
#pragma unroll
    for (int k = 0; k < 3; ++k) dl[i + k * d.N] = fmaf(alpha, p[i + k * d.N], dl[i + k * d.N]);
}

// PCGStep2 (:446-489) / PCGStep2_2ndHalf (:505-534) when the residual is refreshed
template <bool RESET>
__global__ void __launch_bounds__(LM_THREADS) k_lm_step2(const Dev d, int set_b, int set_q)
{
    __shared__ double red[64];
    __shared__ double red2[64];
    if (d.sc->conv) return;
    const Quad q = my_quad(d);
    const float alpha = d.sc->alpha;
    const size_t N = d.N;
    float g = 0.0f, gq = 0.0f;
    if (q.on) {
        for (int r = 0; r < 4; ++r) {
            const int y = q.y0 + r;
            if (y >= d.H) break;
            const size_t i = (size_t)y * d.W + q.x;
            if (!(d.flags[i] & LF_ACTIVE)) continue;
            float rr[3], dl[3], z[3], rb[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const float b = plane(d, L_B)[i + k * N];
                if (RESET) {
                    dl[k] = plane(d, L_D)[i + k * N];
                    rr[k] = b - plane(d, L_AD)[i + k * N];
                } else {
                    dl[k] = fmaf(alpha, plane(d, L_P)[i + k * N], plane(d, L_D)[i + k * N]);
                    rr[k] = fmaf(-alpha, plane(d, L_Q)[i + k * N], plane(d, L_R)[i + k * N]);
                    plane(d, L_D)[i + k * N] = dl[k];
                }
                plane(d, L_R)[i + k * N] = rr[k];
                z[k] = plane(d, L_PRE)[i + (k == 2 ? N : 0)] * rr[k];
                rb[k] = rr[k] + b;
            }
            g = g + dot3(z[0], z[1], z[2], rr[0], rr[1], rr[2]);
            gq = gq + 0.5f * dot3(dl[0], dl[1], dl[2], rb[0], rb[1], rb[2]); // computeQ (:479-484)
        }
    }
    publish(d, set_b, block_exact_sum(g, red));
    publish(d, set_q, block_exact_sum(gq, red2));
}

// scalars after PCGStep2: beta (:537-547), r.z hand-over (:1091), the Q test (:1093-1101)
__global__ void __launch_bounds__(32) k_lm_beta(const Dev d, int set_b, int set_q, int it, float q_tolerance)
{
    if (d.sc->conv) return;
    float bnum, q1;
    decode2(d, set_b, set_q, bnum, q1);
    if (threadIdx.x == 0) {
        const float num = d.sc->num;
        d.sc->beta = (num > 0.0f) ? bnum / num : 0.0f;
        d.sc->num = bnum;
        d.sc->iters = it + 1;
        d.sc->q_last = q1;
        const float zeta = ((float)(it + 1) * (q1 - d.sc->q0)) / q1;
        if (zeta < q_tolerance) d.sc->conv = 1u;
        else d.sc->q0 = q1;
    }
}

// PCGStep3 (:537-550)
__global__ void __launch_bounds__(256) k_lm_step3(const Dev d)
{
    if (d.sc->conv) return;
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= d.N || !(d.flags[i] & LF_ACTIVE)) return;
    const float beta = d.sc->beta;
    float* p = plane(d, L_P);
    const float* r = plane(d, L_R);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const float z = plane(d, L_PRE)[i + (k == 2 ? d.N : 0)] * r[i + k * d.N];
        p[i + k * d.N] = fmaf(beta, p[i + k * d.N], z);
    }
}

// computeModelCost (:666-679): sum over the pixel's residuals of (F + J delta)^2 (o.t:2174-2202)
__global__ void __launch_bounds__(LM_THREADS) k_lm_model(const Dev d, int set)
{
    __shared__ double red[64];
    const Quad q = my_quad(d);
    const float *cs0 = plane(d, L_CS), *cs1 = plane(d, L_CS + 1);
    const float* dl = plane(d, L_D);
    const size_t N = d.N;
    float g = 0.0f;
    if (q.on) {
        for (int r = 0; r < 4; ++r) {
            const int y = q.y0 + r;
            if (y >= d.H) break;
            const size_t i = (size_t)y * d.W + q.x;
            const unsigned f = d.flags[i];
            if (!(f & LF_ACTIVE)) continue;
            const float2 Xi = d.X[i], ui = d.U[i];
            const float ci = cs0[i], si = cs1[i];
            const float di0 = dl[i], di1 = dl[i + N], dai = dl[i + 2 * N];
            float acc = 0.0f;
#pragma unroll
            for (int n = 0; n < 4; ++n) {
                if (!(f & (1u << n))) continue;
                const size_t j = nb_index(d, i, n);
                const float2 Xj = d.X[j], uj = d.U[j];
                const float dx = ui.x - uj.x, dy = ui.y - uj.y;
                const float dX0 = Xi.x - Xj.x, dX1 = Xi.y - Xj.y;
                const float Ri0 = ci * dx - si * dy, Ri1 = si * dx + ci * dy;
                const float e0 = dX0 - Ri0, e1 = dX1 - Ri1;
                const float dd0 = di0 - dl[j], dd1 = di1 - dl[j + N];
                const float Q0 = (-(si * dx)) - ci * dy, Q1 = ci * dx - si * dy; // R'(a_i) d
                const float m0 = (e0 + dd0) - Q0 * dai, m1 = (e1 + dd1) - Q1 * dai;
                const float w0 = d.wr * m0, w1 = d.wr * m1;
                acc = fmaf(w0, w0, acc);
                acc = fmaf(w1, w1, acc);
            }
            if (f & LF_FIT) {
                const float2 c = d.C[i];
                const float f0 = d.wf * ((Xi.x - c.x) + di0), f1 = d.wf * ((Xi.y - c.y) + di1);
                acc = fmaf(f0, f0, acc);
                acc = fmaf(f1, f1, acc);
            }
            g = g + acc;
        }
    }
    publish(d, set, block_exact_sum(g, red));
}

// savePreviousUnknowns (:573-578) + PCGLinearUpdate (:552-557)
__global__ void __launch_bounds__(256) k_lm_update(const Dev d)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= d.N || !(d.flags[i] & LF_ACTIVE)) return;
    const float2 X = d.X[i];
    const float a = d.A[i];
    plane(d, L_PREV)[i] = X.x; plane(d, L_PREV + 1)[i] = X.y; plane(d, L_PREV + 2)[i] = a;
    d.X[i] = make_float2(X.x + plane(d, L_D)[i], X.y + plane(d, L_D + 1)[i]);
    d.A[i] = a + plane(d, L_D + 2)[i];
}

// revertUpdate (:559-564)
__global__ void __launch_bounds__(256) k_lm_revert(const Dev d)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= d.N || !(d.flags[i] & LF_ACTIVE)) return;
    d.X[i] = make_float2(plane(d, L_PREV)[i], plane(d, L_PREV + 1)[i]);
    d.A[i] = plane(d, L_PREV + 2)[i];
}

__global__ void __launch_bounds__(32) k_lm_finish(const Dev d, int set_model, int set_cost)
{
    float m, c;
    decode2(d, set_model, set_cost, m, c);
    if (threadIdx.x == 0) { d.sc->model = 0.5f * m; d.sc->cost = 0.5f * c; }
}

} // namespace

LmSolver::LmSolver(int W, int H) : W_(W), H_(H)
{
    const size_t N = (size_t)W * H;
    d_.W = W; d_.H = H; d_.N = N;
    planes_ = DevBuf<float>((size_t)L_PLANES * N);
    ARAP_CUDA_CHECK(cudaMemset(planes_.p, 0, (size_t)L_PLANES * N * sizeof(float)));
    flags_ = DevBuf<unsigned char>(N);
    ARAP_CUDA_CHECK(cudaMemset(flags_.p, 0, N));
    sc_ = DevBuf<LmScalars>(1);
    ARAP_CUDA_CHECK(cudaMemset(sc_.p, 0, sizeof(LmScalars)));
    h_sc_ = DevBuf<LmScalars>(1, GrowBuf::Pinned);
    ARAP_CUDA_CHECK(cudaDeviceSynchronize()); // the memsets ran on the legacy stream; the solver runs on its own
    d_.pl = planes_.p; d_.flags = flags_.p; d_.sc = sc_.p;
    // Accumulator sets: 0 / 1 = r.z and Q of PCGInit, then a ring of LM_RING iterations x (p.q, r.z, Q), then model cost
    // and cost.  A ring slot is cleared (stream-ordered memset) before its second use, so the footprint does not grow
    // with lIterations.
    acc_ = DevBuf<unsigned long long>((size_t)(2 + 3 * LM_RING + 2) * WA_WORDS);
    d_.acc = acc_.p;
}

bool LmSolver::set_parameter(const char* name, const void* value)
{
    typedef float LmParameters::*Field;
    struct F { const char* n; Field m; };
    static const F fl[] = {{"min_relative_decrease", &LmParameters::min_relative_decrease},
                           {"min_trust_region_radius", &LmParameters::min_trust_region_radius},
                           {"max_trust_region_radius", &LmParameters::max_trust_region_radius},
                           {"q_tolerance", &LmParameters::q_tolerance},
                           {"function_tolerance", &LmParameters::function_tolerance},
                           {"trust_region_radius", &LmParameters::trust_region_radius},
                           {"radius_decrease_factor", &LmParameters::radius_decrease_factor},
                           {"min_lm_diagonal", &LmParameters::min_lm_diagonal},
                           {"max_lm_diagonal", &LmParameters::max_lm_diagonal}};
    for (const F& f : fl)
        if (strcmp(name, f.n) == 0) { sp_.*(f.m) = *(const float*)value; return true; }
    if (strcmp(name, "residual_reset_period") == 0) {
        const int v = *(const int*)value;
        sp_.residual_reset_period = v < 1 ? 1 : v; // the reference would divide by zero
        return true;
    }
    return false;
}

void LmSolver::bind(float2* X, float* A, const float2* U, const float2* C, const float* M, float wf, float wr)
{
    d_.X = X; d_.A = A; d_.U = U; d_.C = C; d_.M = M;
    d_.wf = wf; d_.wr = wr; d_.wf2 = wf * wf; d_.wr2 = wr * wr;
}

void LmSolver::enqueue_cost(cudaStream_t s, int acc)
{
    const unsigned nb = (unsigned)((d_.N + 255) / 256);
    const dim3 grid((W_ + 31) / 32, (H_ + 15) / 16);
    ARAP_TIMED(timer_, "precompute", s, (k_lm_cs<<<nb, 256, 0, s>>>(d_)));
    ARAP_TIMED(timer_, "computeCost", s, (k_lm_cost<<<grid, LM_THREADS, 0, s>>>(d_, acc)));
    launches_ += 2;
}

float LmSolver::init(cudaStream_t s)
{
    // :996-1001: the run-time trust region restarts from the solver parameters
    radius_ = sp_.trust_region_radius;
    decrease_ = sp_.radius_decrease_factor;
    min_diag_ = sp_.min_lm_diagonal;
    max_diag_ = sp_.max_lm_diagonal;
    first_ = true;
    const unsigned nb = (unsigned)((d_.N + 255) / 256);
    ARAP_CUDA_CHECK(cudaMemsetAsync(acc_.p, 0, (size_t)2 * WA_WORDS * sizeof(unsigned long long), s));
    k_lm_flags<<<nb, 256, 0, s>>>(d_);
    enqueue_cost(s, 1);
    k_lm_finish<<<1, 32, 0, s>>>(d_, 0, 1);
    launches_ += 2;
    ARAP_CUDA_CHECK(cudaGetLastError());
    ARAP_CUDA_CHECK(cudaMemcpyAsync(h_sc_.p, sc_.p, sizeof(LmScalars), cudaMemcpyDeviceToHost, s));
    ARAP_CUDA_CHECK(cudaStreamSynchronize(s));
    return h_sc_.p->cost;
}

int LmSolver::step(int L, cudaStream_t s, float* prev_cost)
{
    if (L < 0) L = 0;
    const Dev& d = d_;
    const unsigned nb = (unsigned)((d.N + 255) / 256);
    const dim3 grid((W_ + 31) / 32, (H_ + 15) / 16);
    const int set_model = 2 + 3 * LM_RING, set_cost = set_model + 1;
    ARAP_CUDA_CHECK(cudaMemsetAsync(acc_.p, 0, (size_t)(set_cost + 1) * WA_WORDS * sizeof(unsigned long long), s));
    k_lm_flags<<<nb, 256, 0, s>>>(d);
    ARAP_TIMED(timer_, "precompute", s, (k_lm_cs<<<nb, 256, 0, s>>>(d)));
    // PCGInit1 + PCGSaveSSq + PCGComputeCtC + PCGFinalizeDiagonal in one kernel
    ARAP_TIMED(timer_, "PCGInit1", s,
               (k_lm_init<<<grid, LM_THREADS, 0, s>>>(d, first_ ? 1 : 0, radius_, 1.0f / radius_, min_diag_, max_diag_, 0, 1)));
    k_lm_begin<<<1, 32, 0, s>>>(d, 0, 1);
    launches_ += 4;
    first_ = false;
    for (int it = 0; it < L; ++it) {
        const int base = 2 + 3 * (it % LM_RING);
        if (it > 0 && it % LM_RING == 0) // the ring wraps: every consumer of these sets is behind us in the stream
            ARAP_CUDA_CHECK(cudaMemsetAsync(acc_.p + (size_t)2 * WA_WORDS, 0, (size_t)3 * LM_RING * WA_WORDS * sizeof(unsigned long long), s));
        ARAP_TIMED(timer_, "PCGStep1", s, (k_lm_apply<0><<<grid, LM_THREADS, 0, s>>>(d, base)));
        k_lm_alpha<<<1, 32, 0, s>>>(d, base);
        if (((it + 1) % sp_.residual_reset_period) == 0) { // :1077-1086
            ARAP_TIMED(timer_, "PCGStep2_1stHalf", s, (k_lm_axpy<<<nb, 256, 0, s>>>(d)));
            ARAP_TIMED(timer_, "computeAdelta", s, (k_lm_apply<1><<<grid, LM_THREADS, 0, s>>>(d, 0)));
            ARAP_TIMED(timer_, "PCGStep2_2ndHalf", s, (k_lm_step2<true><<<grid, LM_THREADS, 0, s>>>(d, base + 1, base + 2)));
            launches_ += 2;
        } else {
            ARAP_TIMED(timer_, "PCGStep2", s, (k_lm_step2<false><<<grid, LM_THREADS, 0, s>>>(d, base + 1, base + 2)));
        }
        k_lm_beta<<<1, 32, 0, s>>>(d, base + 1, base + 2, it, sp_.q_tolerance);
        ARAP_TIMED(timer_, "PCGStep3", s, (k_lm_step3<<<nb, 256, 0, s>>>(d)));
        launches_ += 5;
        if ((it & 15) == 15 && it + 1 < L) { // has the Q test ended the loop?  (the remaining launches would be no-ops)
            ARAP_CUDA_CHECK(cudaMemcpyAsync(&h_sc_.p->conv, &sc_.p->conv, sizeof(unsigned), cudaMemcpyDeviceToHost, s));
            ARAP_CUDA_CHECK(cudaStreamSynchronize(s));
            if (h_sc_.p->conv) break;
        }
    }
    ARAP_TIMED(timer_, "computeModelCost", s, (k_lm_model<<<grid, LM_THREADS, 0, s>>>(d, set_model))); // before the update (:1106-1112)
    ARAP_TIMED(timer_, "PCGLinearUpdate", s, (k_lm_update<<<nb, 256, 0, s>>>(d))); // + savePreviousUnknowns
    enqueue_cost(s, set_cost);
    k_lm_finish<<<1, 32, 0, s>>>(d, set_model, set_cost);
    launches_ += 3;
    ARAP_CUDA_CHECK(cudaGetLastError());
    ARAP_CUDA_CHECK(cudaMemcpyAsync(h_sc_.p, sc_.p, sizeof(LmScalars), cudaMemcpyDeviceToHost, s));
    ARAP_CUDA_CHECK(cudaStreamSynchronize(s));

    // the trust-region bookkeeping of :1106-1170, in the reference's types (binary32 fields, binary64 literals)
    const float prevCost = *prev_cost;
    const float model_cost = h_sc_.p->model, newCost = h_sc_.p->cost;
    const float model_cost_change = prevCost - model_cost;
    const float cost_change = prevCost - newCost;
    const float relative_decrease = cost_change / model_cost_change;
    info_.pcg_iterations = h_sc_.p->iters;
    info_.model_cost = model_cost;
    info_.new_cost = newCost;
    info_.q_last = h_sc_.p->q_last;
    int more = 1;
    if (cost_change >= 0.0f && relative_decrease > sp_.min_relative_decrease) {
        const float absolute_function_tolerance = prevCost * sp_.function_tolerance;
        if (cost_change <= absolute_function_tolerance) {
            info_.verdict = 2; // "Function tolerance reached": the update stays, prevCost is left as it was (:1129-1133)
            more = 0;
        } else {
            const double step_quality = (double)relative_decrease;
            const double min_factor = 1.0 / 3.0;
            const double tmp_factor = 1.0 - std::pow(2.0 * step_quality - 1.0, 3.0);
            radius_ = (float)((double)radius_ / std::fmax(min_factor, tmp_factor));
            radius_ = (float)std::fmin((double)radius_, (double)sp_.max_trust_region_radius);
            decrease_ = 2.0f;
            *prev_cost = newCost;
            info_.verdict = 1;
        }
    } else {
        ARAP_TIMED(timer_, "revertUpdate", s, (k_lm_revert<<<nb, 256, 0, s>>>(d)));
        ++launches_;
        ARAP_CUDA_CHECK(cudaGetLastError());
        ARAP_CUDA_CHECK(cudaStreamSynchronize(s));
        radius_ = radius_ / decrease_;
        decrease_ = (float)(2.0 * (double)decrease_);
        info_.verdict = 0;
        if (radius_ <= sp_.min_trust_region_radius) {
            info_.verdict = 3;
            more = 0;
        }
    }
    info_.radius_after = radius_;
    return more;
}

} // namespace arapb200
