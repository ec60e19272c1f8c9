// solver_stream.cu -- streaming Gauss-Newton / PCG back-end.
//
// Replaces the generated kernels PCGInit1 / PCGStep1 / PCGStep2 / PCGStep3 / PCGLinearUpdate /
// computeCost and the host loop of ARAP/API/src/solverGPUGaussNewton.t:361-397, 421-434, 446-489,
// 537-557, 580-592, 1016-1177 with:
//   k_prep    flags (validity of the 4 neighbours, fit, active), cos/sin table, UrShape check
//   k_init    r = -J^T F, pre, p = pre*r, delta = 0, sum r.p                    (PCGInit1)
//   k_step_a  p = pre*r + beta*p (recomputed on the halo), q = J^T J p, sum p.q  (PCGStep3 + PCGStep1)
//   k_step_b  alpha; delta += alpha p; r -= alpha q; sum (pre*r).r              (PCGStep2)
//   k_update  X += delta, refresh cos/sin                                        (PCGLinearUpdate)
//   k_cost    0.5 * sum residual^2                                               (computeCost)
// Scalars (alpha/beta numerators and denominators) never leave the device; every reduction is the
// deterministic exact sum of contract C3, accumulated without fences in wide fixed-point accumulators
// (common.cuh) and decoded by the blocks of the next kernel; a whole GN step (2*nPCG + 5 kernels) is one
// graph launch.  State layout: tile-interleaved planes (solver_stream.cuh).
#include "solver_stream.cuh"
#include "grid_math.cuh"

namespace arapb200 {

namespace {

constexpr int TS = ST_TILE + 2; // staged tile pitch (1-pixel halo)

__device__ __forceinline__ unsigned long long* acc_set(const StreamPlanes& pl, int set)
{
    return pl.acc + set * WA_WORDS;
}
__device__ __forceinline__ int bn_set(int j) // accumulator of r.z of PCG iteration j (j >= -2)
{
    return (j + 3) % 3;
}
// Block result (valid in warp 0) -> the grid-wide accumulator `set`.  Fire and forget: no fence, no counter; the
// consumers run in a later kernel.
__device__ __forceinline__ void publish(const StreamPlanes& pl, int set, HL blockval)
{
    if (threadIdx.x == 0) wide_add(acc_set(pl, set), blockIdx.x, blockval.h);
    if (threadIdx.x == 1) wide_add(acc_set(pl, set), blockIdx.x, blockval.l);
}
// Warp 0 of a block reads two accumulators at once: lanes 0..15 `set_lo`, lanes 16..31 `set_hi`.
__device__ __forceinline__ long long fetch2(const StreamPlanes& pl, int set_lo, int set_hi)
{
    const int lane = threadIdx.x & 31;
    return wide_fetch(acc_set(pl, lane < 16 ? set_lo : set_hi), lane & 15);
}
// ---- tile-interleaved addressing ----
__device__ __forceinline__ float* tile_ptr(const StreamPlanes& pl, int tile)
{
    return pl.planes + (size_t)tile * ST_TILE_FLOATS;
}
// float offset (plane 0) of image pixel (x, y)
__device__ __forceinline__ size_t tiled_off(const StreamPlanes& pl, int x, int y)
{
    return (size_t)((y >> 5) * pl.tx + (x >> 5)) * ST_TILE_FLOATS + (size_t)(((y & 31) << 5) + (x & 31));
}
// flags of the pixel whose plane-0 address is `px` inside the tile starting at `tb`
__device__ __forceinline__ unsigned char* flag_ptr(float* tb, int local)
{
    return reinterpret_cast<unsigned char*>(tb + PL_FLAGS * ST_TILE_PX) + local;
}
#define PLN(base, k) ((base)[(k) * ST_TILE_PX])
// read-only planes that every PCG kernel re-reads (cos/sin, preconditioner): ask L2 to keep them
__device__ __forceinline__ float ld_keep(const float* p)
{
    float v;
    asm volatile("{\n\t.reg .b64 pol;\n\tcreatepolicy.fractional.L2::evict_last.b64 pol, 1.0;\n\t"
                 "ld.global.L2::cache_hint.f32 %0, [%1], pol;\n\t}" : "=f"(v) : "l"(p));
    return v;
}
// edge mirrors (PL_EDGE): slot of a halo-relevant plane (r 0-2, p 3-8, cos/sin 15-16, pre 17-18)
__device__ __forceinline__ int edge_slot(int plane)
{
    return plane < 9 ? plane : plane - 6;
}
// to be called with every store to such a plane: pixels in column 0 / 31 also update their mirror
__device__ __forceinline__ void edge_put(float* tb, int plane, int lx, int row, float v)
{
    if (lx == 0 || lx == ST_TILE - 1)
        tb[PL_EDGE * ST_TILE_PX + (edge_slot(plane) * 2 + (lx != 0 ? 1 : 0)) * ST_TILE + row] = v;
}

// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(ST_THREADS) k_prep(const StreamDev* __restrict__ dpp)
{
    const StreamDev& dp = *dpp;
    const int W = dp.W, H = dp.H;
    const int lx = threadIdx.x & 31, lyb = (threadIdx.x >> 5) * 4;
    const int x = (blockIdx.x % dp.tx) * ST_TILE + lx;
    const int yb = (blockIdx.x / dp.tx) * ST_TILE + lyb;
    float* tb = tile_ptr(dp, blockIdx.x);
    unsigned bad = 0;
    int any = 0;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int y = yb + r;
        const int loc = (lyb + r) * ST_TILE + lx;
        unsigned f = 0;
        if (x < W && y < H) {
            const size_t i = (size_t)y * W + x;
            if (dp.M[i] == 0.0f) {
                f = FLAG_ACTIVE;
                any = 1;
                if (x + 1 < W && dp.M[i + 1] == 0.0f) f |= 1u;
                if (x > 0 && dp.M[i - 1] == 0.0f) f |= 2u;
                if (y + 1 < H && dp.M[i + W] == 0.0f) f |= 4u;
                if (y > 0 && dp.M[i - W] == 0.0f) f |= 8u;
                const float2 c = dp.C[i];
                if (c.x >= 0.0f && c.y >= 0.0f) f |= FLAG_FIT; // arap_plan.t:22
                float s, co;
                contract_sincos(dp.A[i], s, co);
                PLN(tb + loc, PL_CS) = co;
                PLN(tb + loc, PL_CS + 1) = s;
                edge_put(tb, PL_CS, lx, lyb + r, co);
                edge_put(tb, PL_CS + 1, lx, lyb + r, s);
                const float2 u = dp.U[i];
                if (u.x != (float)x || u.y != (float)y) bad = 1;
            }
        }
        *flag_ptr(tb, loc) = (unsigned char)f;
    }
    if (bad) atomicAdd(&dp.sc->bad_u, 1u);
    any = __syncthreads_or(any);
    if (threadIdx.x == 0) dp.tile_active[blockIdx.x] = any ? 1 : 0;
    // opt-in early exits: the PCG one is re-armed per Gauss-Newton step; a finished Gauss-Newton loop (gn_done) keeps the
    // step's PCG kernels switched off
    if (blockIdx.x == 0 && threadIdx.x == 0) { dp.sc->conv = dp.sc->gn_done ? 1u : 0u; dp.sc->stop = -1.0f; }
}

// Stage (X_x, X_y, cos, sin) of a tile + halo.  Inactive / out-of-image entries are never used.
__device__ __forceinline__ void stage_x_tile(const StreamDev& dp, float4 (*T)[TS], int x0, int y0)
{
    for (int e = threadIdx.x; e < TS * TS; e += ST_THREADS) {
        const int ly = e / TS, lx = e - ly * TS;
        const int x = x0 + lx - 1, y = y0 + ly - 1;
        float4 v = make_float4(0.f, 0.f, 1.f, 0.f);
        if (x >= 0 && x < dp.W && y >= 0 && y < dp.H) {
            const int tile = (y >> 5) * dp.tx + (x >> 5), loc = ((y & 31) << 5) + (x & 31);
            float* tb = tile_ptr(dp, tile);
            if (*flag_ptr(tb, loc) & FLAG_ACTIVE) {
                const float2 X = dp.X[(size_t)y * dp.W + x];
                v = make_float4(X.x, X.y, PLN(tb + loc, PL_CS), PLN(tb + loc, PL_CS + 1));
            }
        }
        T[ly][lx] = v;
    }
}

// PCGInit1 (solverGPUGaussNewton.t:361-397)
__global__ void __launch_bounds__(ST_THREADS) k_init(const StreamDev* __restrict__ dpp)
{
    __shared__ float4 T[TS][TS];
    __shared__ double red[64];
    const StreamDev& dp = *dpp;
    const int W = dp.W, H = dp.H;
    const int x0 = (blockIdx.x % dp.tx) * ST_TILE, y0 = (blockIdx.x / dp.tx) * ST_TILE;
    stage_x_tile(dp, T, x0, y0);
    __syncthreads();
    const int lx = threadIdx.x & 31, lyb = (threadIdx.x >> 5) * 4;
    const int x = x0 + lx;
    float* tb = tile_ptr(dp, blockIdx.x);
    float g = 0.0f;
    if (x < W) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int ly = lyb + r, y = y0 + ly;
            if (y >= H) break;
            const size_t i = (size_t)y * W + x;
            const int loc = ly * ST_TILE + lx;
            float* px = tb + loc;
            const unsigned f = *flag_ptr(tb, loc);
            if (!(f & FLAG_ACTIVE)) {
                // the branch-free PCG kernels rely on zeros here; a previous problem may have left values behind
#pragma unroll
                for (int k = 0; k < PL_FLAGS; ++k) PLN(px, k) = 0.f;
#pragma unroll
                for (int k = 0; k < PL_FLAGS; ++k)
                    if (k < PL_Q || k >= PL_CS) edge_put(tb, k, lx, ly, 0.f);
                continue;
            }
            const float4 Ei = T[ly + 1][lx + 1];
            JtfAcc a;
            jtf_zero(a);
            if (f & 1u) jtf_nb<0>(a, Ei.x, Ei.y, Ei.z, Ei.w, T[ly + 1][lx + 2]);
            if (f & 2u) jtf_nb<1>(a, Ei.x, Ei.y, Ei.z, Ei.w, T[ly + 1][lx]);
            if (f & 4u) jtf_nb<2>(a, Ei.x, Ei.y, Ei.z, Ei.w, T[ly + 2][lx + 1]);
            if (f & 8u) jtf_nb<3>(a, Ei.x, Ei.y, Ei.z, Ei.w, T[ly][lx + 1]);
            const bool fit = (f & FLAG_FIT) != 0;
            float2 c = make_float2(0.f, 0.f);
            if (fit) c = dp.C[i];
            float g0, g1, ga, DX, DA;
            jtf_finish(a, Ei.x, Ei.y, fit, c.x, c.y, dp.wr2, dp.wf2, g0, g1, ga, DX, DA);
            const float pX = guarded_invert(DX), pA = guarded_invert(DA);
            const float r0 = -g0, r1 = -g1, r2 = -ga;
            const float p0 = pX * r0, p1 = pX * r1, p2 = pA * r2;
            PLN(px, PL_PRE) = pX;
            PLN(px, PL_PRE + 1) = pA;
            PLN(px, PL_R) = r0; PLN(px, PL_R + 1) = r1; PLN(px, PL_R + 2) = r2;
            PLN(px, PL_P) = p0; PLN(px, PL_P + 1) = p1; PLN(px, PL_P + 2) = p2;
            edge_put(tb, PL_PRE, lx, ly, pX); edge_put(tb, PL_PRE + 1, lx, ly, pA);
            edge_put(tb, PL_R, lx, ly, r0); edge_put(tb, PL_R + 1, lx, ly, r1); edge_put(tb, PL_R + 2, lx, ly, r2);
            edge_put(tb, PL_P, lx, ly, p0); edge_put(tb, PL_P + 1, lx, ly, p1); edge_put(tb, PL_P + 2, lx, ly, p2);
            PLN(px, PL_D) = 0.f; PLN(px, PL_D + 1) = 0.f; PLN(px, PL_D + 2) = 0.f;
            g = g + dot3(r0, r1, r2, p0, p1, p2);
        }
    }
    publish(dp, bn_set(-1), block_exact_sum(g, red));
}

// PCGStep3 of the previous iteration fused with PCGStep1 (solverGPUGaussNewton.t:537-550, 421-434).
// Thread = one vertical quad of the tile (lane = column); threads 0..131 also own one pixel of the 1-pixel ring
// around the tile, whose NEW direction they recompute (the neighbouring tile is writing it in this very kernel, so p is
// ping-ponged).  Every global load of the block is issued before the first use; beta is decoded under them.
// RT (opt-in early exit, separate instantiation so that the default kernels compile exactly as before): once r.z of the
// previous iteration is <= sc->stop, this launch and every later k_step_a / k_step_b of the Gauss-Newton step return at
// once -- every block decodes the same scalar, so the decision is uniform; block 0 makes it sticky (sc->conv).
// SUB = rows per block, here and in k_step_b: two 128-thread blocks per tile beat one 256-thread block, because shorter
// blocks leave less idle time at the end of the grid.
constexpr int SUB = 16;
template <bool FIRST, bool RT = false>
__global__ void __launch_bounds__(SUB * 8) k_step_a(const __grid_constant__ StreamPlanes pl,
                                                    const StreamDev* __restrict__ dpp, int it)
{
    constexpr int NSUB = ST_TILE / SUB, TSY = SUB + 2;
    __shared__ float4 T[TSY][TS]; // (p_x, p_y, sin*p_a, cos*p_a) of the block's rows + ring
    __shared__ double red[64];
    __shared__ float s_beta;
    __shared__ int s_skip;
    const int tile = blockIdx.x / NSUB, sub = blockIdx.x % NSUB;
    const bool tile_on = pl.tile_active[tile] != 0; // tiles without object pixels have nothing to add
    if (!tile_on && blockIdx.x != 0) return;
    const int W = pl.W, H = pl.H;
    const int x0 = (tile % pl.tx) * ST_TILE, y0 = (tile / pl.tx) * ST_TILE + sub * SUB;
    const int lx = threadIdx.x & 31, lyb = (threadIdx.x >> 5) * 4; // row inside the block
    long long raw = 0;
    if (!FIRST && threadIdx.x < 32) raw = fetch2(pl, bn_set(it - 1), bn_set(it - 2));
    const float wr2 = dpp->wr2, wf2 = dpp->wf2;
    const int src = PL_P + 3 * (FIRST ? 0 : ((it - 1) & 1)), dst = PL_P + 3 * (it & 1);
    float* const tb = tile_ptr(pl, tile);
    float* const own = tb + (sub * SUB + lyb) * ST_TILE + lx; // plane 0, first row of the quad
    const float* const ps = own + src * ST_TILE_PX;

    // ---- loads: own quad (pixels outside the image exist in storage and hold zeros) ----
    float po[4][3], cs[4][2], pre[4][2], rr[4][3];
    unsigned fl[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const float* px = own + r * ST_TILE;
        if (FIRST) {
            po[r][0] = PLN(ps + r * ST_TILE, 0); po[r][1] = PLN(ps + r * ST_TILE, 1); po[r][2] = PLN(ps + r * ST_TILE, 2);
        } else { // the old direction is dead after this kernel
            po[r][0] = __ldcs(&PLN(ps + r * ST_TILE, 0)); po[r][1] = __ldcs(&PLN(ps + r * ST_TILE, 1)); po[r][2] = __ldcs(&PLN(ps + r * ST_TILE, 2));
        }
        cs[r][0] = ld_keep(&PLN(px, PL_CS)); cs[r][1] = ld_keep(&PLN(px, PL_CS + 1));
        if (!FIRST) {
            pre[r][0] = ld_keep(&PLN(px, PL_PRE)); pre[r][1] = ld_keep(&PLN(px, PL_PRE + 1));
            rr[r][0] = PLN(px, PL_R); rr[r][1] = PLN(px, PL_R + 1); rr[r][2] = PLN(px, PL_R + 2);
        }
        fl[r] = *flag_ptr(tb, (sub * SUB + lyb + r) * ST_TILE + lx);
    }
    // ---- loads: ring pixel of threads 0..131 (top row, bottom row, left column, right column) ----
    const int t = threadIdx.x;
    int hlx, hly;
    if (t < TS) { hlx = t; hly = 0; }
    else if (t < 2 * TS) { hlx = t - TS; hly = TSY - 1; }
    else if (t < 2 * TS + SUB) { hlx = 0; hly = t - 2 * TS + 1; }
    else { hlx = TS - 1; hly = t - 2 * TS - SUB + 1; }
    const int hx = x0 + hlx - 1, hy = y0 + hly - 1;
    const bool ring = t < 2 * TS + 2 * SUB;
    const bool hin = ring && hx >= 0 && hx < W && hy >= 0 && hy < H;
    // top / bottom ring pixels are read from the neighbour's planes (contiguous in x); left / right ring pixels from the
    // neighbour's edge mirrors (contiguous in y)
    const bool hedge = hin && (hlx == 0 || hlx == TS - 1);
    const float* hpx = own;
    if (hin) {
        hpx = hedge ? tile_ptr(pl, (hy >> 5) * pl.tx + (hx >> 5)) + PL_EDGE * ST_TILE_PX + ((hx & 31) != 0 ? ST_TILE : 0) + (hy & 31)
                    : pl.planes + tiled_off(pl, hx, hy);
    }
    auto hval = [&](int plane) { return hpx[hedge ? edge_slot(plane) * 2 * ST_TILE : plane * ST_TILE_PX]; };
    float hp[3], hcs[2], hpre[2], hr[3];
    hp[0] = hval(src); hp[1] = hval(src + 1); hp[2] = hval(src + 2);
    hcs[0] = hval(PL_CS); hcs[1] = hval(PL_CS + 1);
    if (!FIRST) {
        hpre[0] = hval(PL_PRE); hpre[1] = hval(PL_PRE + 1);
        hr[0] = hval(PL_R); hr[1] = hval(PL_R + 1); hr[2] = hval(PL_R + 2);
    }

    // ---- beta ----
    float beta = 0.0f;
    if (!FIRST) {
        if (threadIdx.x < 32) {
            const float v = wide_round(raw);
            const float bnum = __shfl_sync(0xffffffffu, v, 0), num = __shfl_sync(0xffffffffu, v, 16);
            if (threadIdx.x == 0) {
                s_beta = (num > 0.0f) ? bnum / num : 0.0f; // :544-547
                if (blockIdx.x == 0 && dpp->trace) dpp->trace[3 * (it - 1) + 2] = bnum;
                if (RT) {
                    const bool skip = pl.sc->conv != 0u || bnum <= pl.sc->stop;
                    s_skip = skip ? 1 : 0;
                    if (skip && blockIdx.x == 0) pl.sc->conv = 1u;
                }
            }
        }
        __syncthreads();
        if (RT && s_skip) return;
        beta = s_beta;
    }

    // ---- new direction: own quad (stored) and ring (kept in the tile only) ----
    // no activity test: every plane of an inactive pixel holds zeros, which flow through as zeros
    float* const pd = own + dst * ST_TILE_PX;
    float4 ent[4]; // the quad's own tile entries: vertical neighbours inside the quad come from registers
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        if (!FIRST) {
            po[r][0] = fmaf(beta, po[r][0], pre[r][0] * rr[r][0]);
            po[r][1] = fmaf(beta, po[r][1], pre[r][0] * rr[r][1]);
            po[r][2] = fmaf(beta, po[r][2], pre[r][1] * rr[r][2]);
            if (tile_on) {
                PLN(pd + r * ST_TILE, 0) = po[r][0]; PLN(pd + r * ST_TILE, 1) = po[r][1]; PLN(pd + r * ST_TILE, 2) = po[r][2];
                edge_put(tb, dst, lx, sub * SUB + lyb + r, po[r][0]);
                edge_put(tb, dst + 1, lx, sub * SUB + lyb + r, po[r][1]);
                edge_put(tb, dst + 2, lx, sub * SUB + lyb + r, po[r][2]);
            }
        }
        ent[r] = make_float4(po[r][0], po[r][1], cs[r][1] * po[r][2], cs[r][0] * po[r][2]);
        T[lyb + r + 1][lx + 1] = ent[r];
    }
    if (ring) {
        if (!FIRST) {
            hp[0] = fmaf(beta, hp[0], hpre[0] * hr[0]);
            hp[1] = fmaf(beta, hp[1], hpre[0] * hr[1]);
            hp[2] = fmaf(beta, hp[2], hpre[1] * hr[2]);
        }
        T[hly][hlx] = hin ? make_float4(hp[0], hp[1], hcs[1] * hp[2], hcs[0] * hp[2]) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    __syncthreads();

    // ---- q = J^T J p on the own quad ----
    float g = 0.0f;
    float* const pq = own + PL_Q * ST_TILE_PX;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const unsigned f = fl[r];
        if (!tile_on || !(f & FLAG_ACTIVE)) continue;
        const int ly = lyb + r;
        JtjAcc a;
        jtj_zero(a);
        jtj_nb_masked<0>(a, po[r][0], po[r][1], T[ly + 1][lx + 2], (f & 1u) ? 1.0f : 0.0f);
        jtj_nb_masked<1>(a, po[r][0], po[r][1], T[ly + 1][lx], (f & 2u) ? 1.0f : 0.0f);
        jtj_nb_masked<2>(a, po[r][0], po[r][1], r < 3 ? ent[r < 3 ? r + 1 : 3] : T[ly + 2][lx + 1], (f & 4u) ? 1.0f : 0.0f);
        jtj_nb_masked<3>(a, po[r][0], po[r][1], r > 0 ? ent[r > 0 ? r - 1 : 0] : T[ly][lx + 1], (f & 8u) ? 1.0f : 0.0f);
        float q0, q1, qa;
        jtj_finish(a, cs[r][0], cs[r][1], po[r][0], po[r][1], po[r][2], (f & FLAG_FIT) != 0, wr2, wf2, q0, q1, qa);
        PLN(pq + r * ST_TILE, 0) = q0; PLN(pq + r * ST_TILE, 1) = q1; PLN(pq + r * ST_TILE, 2) = qa;
        g = g + dot3(po[r][0], po[r][1], po[r][2], q0, q1, qa);
    }
    publish(pl, ST_ACC_D0 + (it & 1), block_exact_sum(g, red));
}

// PCGStep2 (solverGPUGaussNewton.t:446-489).  Branch-free: the planes of inactive pixels hold zeros (they are
// zero-initialised and never written), so they flow through as exact zeros and add +0 to the group term;
// every load of the four rows is issued before the first use.
template <bool RT = false>
__global__ void __launch_bounds__(SUB * 8) k_step_b(const __grid_constant__ StreamPlanes pl,
                                                    const StreamDev* __restrict__ dpp, int it)
{
    constexpr int NSUB = ST_TILE / SUB;
    __shared__ double red[64];
    __shared__ float s_alpha;
    __shared__ int s_skip;
    const int tile = blockIdx.x / NSUB, sub = blockIdx.x % NSUB;
    const bool tile_on = pl.tile_active[tile] != 0;
    if (!tile_on && blockIdx.x != 0) return;
    // warp 0: r.z of the previous iteration and this iteration's p.q; fetched before the planes, decoded after
    long long raw = 0;
    if (threadIdx.x < 32) raw = fetch2(pl, bn_set(it - 1), ST_ACC_D0 + (it & 1));
    float* const tbb = tile_ptr(pl, tile);
    float* const own = tbb + (sub * SUB + (threadIdx.x >> 5) * 4) * ST_TILE + (threadIdx.x & 31);
    const float* const pk = own + (PL_P + 3 * (it & 1)) * ST_TILE_PX;
    float pv[4][3], qv[4][3], rv[4][3], dv[4][3], pre[4][2];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const float* px = own + r * ST_TILE;
        pv[r][0] = PLN(pk + r * ST_TILE, 0); pv[r][1] = PLN(pk + r * ST_TILE, 1); pv[r][2] = PLN(pk + r * ST_TILE, 2);
        // q is dead after this read and delta is touched once per iteration: streaming hints keep L2 for r, p, pre
        qv[r][0] = __ldcs(&PLN(px, PL_Q)); qv[r][1] = __ldcs(&PLN(px, PL_Q + 1)); qv[r][2] = __ldcs(&PLN(px, PL_Q + 2));
        rv[r][0] = PLN(px, PL_R); rv[r][1] = PLN(px, PL_R + 1); rv[r][2] = PLN(px, PL_R + 2);
        dv[r][0] = __ldcs(&PLN(px, PL_D)); dv[r][1] = __ldcs(&PLN(px, PL_D + 1)); dv[r][2] = __ldcs(&PLN(px, PL_D + 2));
        pre[r][0] = ld_keep(&PLN(px, PL_PRE)); pre[r][1] = ld_keep(&PLN(px, PL_PRE + 1));
    }
    if (threadIdx.x < 32) {
        const float v = wide_round(raw);
        const float num = __shfl_sync(0xffffffffu, v, 0), den = __shfl_sync(0xffffffffu, v, 16);
        if (threadIdx.x == 0) {
            s_alpha = (den > 0.0f) ? num / den : 0.0f; // :456-459
            if (RT) {
                // it == 0: num is r.p of PCGInit1 -> the threshold of this Gauss-Newton step; later: num is r.z of iteration it-1
                if (it == 0) {
                    s_skip = pl.sc->conv != 0u ? 1 : 0; // set by k_prep: the Gauss-Newton loop has ended (gn_rtol)
                    if (blockIdx.x == 0 && !s_skip) pl.sc->stop = (dpp->pcg_rtol2 > 0.0f) ? dpp->pcg_rtol2 * num : -1.0f;
                }
                else s_skip = (pl.sc->conv != 0u || num <= pl.sc->stop) ? 1 : 0;
            }
            if (blockIdx.x == 0 && dpp->trace && !(RT && s_skip)) {
                dpp->trace[3 * it] = den;
                dpp->trace[3 * it + 1] = num;
            }
        }
    }
    if (RT) {
        __syncthreads();
        if (s_skip) return;
    }
    if (blockIdx.x == 0) { // recycle the accumulators nobody reads any more (their next writers are later kernels)
        for (int w = threadIdx.x; w < WA_WORDS; w += blockDim.x) {
            acc_set(pl, bn_set(it - 2))[w] = 0ULL;
            acc_set(pl, ST_ACC_D0 + ((it + 1) & 1))[w] = 0ULL;
        }
    }
    __syncthreads();
    const float alpha = s_alpha;
    float g = 0.0f;
    if (tile_on) {
        // pixels outside the image (edge tiles) hold zeros in every plane and stay zero: 0 + alpha * 0
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            float* px = own + r * ST_TILE;
            float rr[3], zz[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                __stcs(&PLN(px, PL_D + k), fmaf(alpha, pv[r][k], dv[r][k]));
                rr[k] = fmaf(-alpha, qv[r][k], rv[r][k]);
                PLN(px, PL_R + k) = rr[k];
                edge_put(tbb, PL_R + k, threadIdx.x & 31, sub * SUB + (threadIdx.x >> 5) * 4 + r, rr[k]);
                zz[k] = ((k < 2) ? pre[r][0] : pre[r][1]) * rr[k];
            }
            g = g + dot3(zz[0], zz[1], zz[2], rr[0], rr[1], rr[2]);
        }
    }
    publish(pl, bn_set(it), block_exact_sum(g, red));
}

// PCGLinearUpdate (solverGPUGaussNewton.t:552-557) + cos/sin refresh for the new angles
__global__ void __launch_bounds__(ST_THREADS) k_update(const StreamDev* __restrict__ dpp)
{
    const StreamDev& dp = *dpp;
    const int W = dp.W, H = dp.H;
    const int lx = threadIdx.x & 31, lyb = (threadIdx.x >> 5) * 4;
    const int x = (blockIdx.x % dp.tx) * ST_TILE + lx;
    const int yb = (blockIdx.x / dp.tx) * ST_TILE + lyb;
    if (x >= W) return;
    float* tb = tile_ptr(dp, blockIdx.x);
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int y = yb + r;
        if (y >= H) break;
        const size_t i = (size_t)y * W + x;
        const int loc = (lyb + r) * ST_TILE + lx;
        if (!(*flag_ptr(tb, loc) & FLAG_ACTIVE)) continue;
        float* px = tb + loc;
        float2 X = dp.X[i];
        X.x = X.x + PLN(px, PL_D);
        X.y = X.y + PLN(px, PL_D + 1);
        dp.X[i] = X;
        const float a = dp.A[i] + PLN(px, PL_D + 2);
        dp.A[i] = a;
        float s, c;
        contract_sincos(a, s, c);
        PLN(px, PL_CS) = c;
        PLN(px, PL_CS + 1) = s;
        edge_put(tb, PL_CS, lx, lyb + r, c);
        edge_put(tb, PL_CS + 1, lx, lyb + r, s);
    }
}

// computeCost (solverGPUGaussNewton.t:580-592, o.t:2375-2385)
__global__ void __launch_bounds__(ST_THREADS) k_cost(const StreamDev* __restrict__ dpp)
{
    __shared__ float4 T[TS][TS];
    __shared__ double red[64];
    const StreamDev& dp = *dpp;
    const int W = dp.W, H = dp.H;
    const int x0 = (blockIdx.x % dp.tx) * ST_TILE, y0 = (blockIdx.x / dp.tx) * ST_TILE;
    stage_x_tile(dp, T, x0, y0);
    __syncthreads();
    const int lx = threadIdx.x & 31, lyb = (threadIdx.x >> 5) * 4;
    const int x = x0 + lx;
    float* tb = tile_ptr(dp, blockIdx.x);
    float g = 0.0f;
    if (x < W) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int ly = lyb + r, y = y0 + ly;
            if (y >= H) break;
            const size_t i = (size_t)y * W + x;
            const unsigned f = *flag_ptr(tb, ly * ST_TILE + lx);
            if (!(f & FLAG_ACTIVE)) continue;
            const float4 Ei = T[ly + 1][lx + 1];
            float acc = 0.0f;
            if (f & 1u) acc = cost_nb<0>(acc, Ei.x, Ei.y, Ei.z, Ei.w, T[ly + 1][lx + 2], dp.wr);
            if (f & 2u) acc = cost_nb<1>(acc, Ei.x, Ei.y, Ei.z, Ei.w, T[ly + 1][lx], dp.wr);
            if (f & 4u) acc = cost_nb<2>(acc, Ei.x, Ei.y, Ei.z, Ei.w, T[ly + 2][lx + 1], dp.wr);
            if (f & 8u) acc = cost_nb<3>(acc, Ei.x, Ei.y, Ei.z, Ei.w, T[ly][lx + 1], dp.wr);
            if (f & FLAG_FIT) {
                const float2 c = dp.C[i];
                acc = cost_fit(acc, Ei.x, Ei.y, c.x, c.y, dp.wf);
            }
            g = g + acc;
        }
    }
    publish(dp, ST_ACC_COST, block_exact_sum(g, red));
}

// ---------------------------------------------------------------------------------------------
// General-UrShape variants of the three stencil kernels (Opt.h callers may bind any UrShape image; the ARAP app always
// binds the pixel grid, which takes the specialised kernels above).  Straightforward: thread = vertical quad, every
// neighbour value is read from global memory, the neighbour's new direction is recomputed in place.  Same arithmetic
// contract, bit-exact against the oracle; not tuned.
struct GenNb {
    const float* px; // neighbour's plane-0 address
    float dx, dy;    // u_i - u_j
    size_t j;        // neighbour's row-major index
};
__device__ __forceinline__ GenNb gen_nb(const StreamDev& dp, int x, int y, int n, float2 ui)
{
    const int xj = x + (n == 0 ? 1 : n == 1 ? -1 : 0), yj = y + (n == 2 ? 1 : n == 3 ? -1 : 0);
    GenNb r;
    r.j = (size_t)yj * dp.W + xj;
    r.px = dp.planes + tiled_off(dp, xj, yj);
    const float2 uj = dp.U[r.j];
    r.dx = ui.x - uj.x;
    r.dy = ui.y - uj.y;
    return r;
}

__global__ void __launch_bounds__(ST_THREADS) k_init_gen(const StreamDev* __restrict__ dpp)
{
    __shared__ double red[64];
    const StreamDev& dp = *dpp;
    const int W = dp.W, H = dp.H;
    const int lx = threadIdx.x & 31, lyb = (threadIdx.x >> 5) * 4;
    const int x = (blockIdx.x % dp.tx) * ST_TILE + lx, y0 = (blockIdx.x / dp.tx) * ST_TILE;
    float* tb = tile_ptr(dp, blockIdx.x);
    float g = 0.0f;
    if (x < W) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int ly = lyb + r, y = y0 + ly;
            if (y >= H) break;
            const size_t i = (size_t)y * W + x;
            const int loc = ly * ST_TILE + lx;
            float* px = tb + loc;
            const unsigned f = *flag_ptr(tb, loc);
            if (!(f & FLAG_ACTIVE)) {
#pragma unroll
                for (int k = 0; k < PL_FLAGS; ++k) PLN(px, k) = 0.f;
#pragma unroll
                for (int k = 0; k < PL_FLAGS; ++k)
                    if (k < PL_Q || k >= PL_CS) edge_put(tb, k, lx, ly, 0.f);
                continue;
            }
            const float2 Xi = dp.X[i], ui = dp.U[i];
            const float ci = PLN(px, PL_CS), si = PLN(px, PL_CS + 1);
            JtfAcc a;
            jtf_zero(a);
#pragma unroll
            for (int n = 0; n < 4; ++n) {
                if (!(f & (1u << n))) continue;
                const GenNb nb = gen_nb(dp, x, y, n, ui);
                const float2 Xj = dp.X[nb.j];
                jtf_nb_gen(a, Xi.x, Xi.y, ci, si, Xj.x, Xj.y, PLN(nb.px, PL_CS), PLN(nb.px, PL_CS + 1), nb.dx, nb.dy);
            }
            const bool fit = (f & FLAG_FIT) != 0;
            float2 c = make_float2(0.f, 0.f);
            if (fit) c = dp.C[i];
            float g0, g1, ga, DX, DA;
            jtf_finish(a, Xi.x, Xi.y, fit, c.x, c.y, dp.wr2, dp.wf2, g0, g1, ga, DX, DA);
            const float pX = guarded_invert(DX), pA = guarded_invert(DA);
            const float r0 = -g0, r1 = -g1, r2 = -ga;
            const float p0 = pX * r0, p1 = pX * r1, p2 = pA * r2;
            PLN(px, PL_PRE) = pX;
            PLN(px, PL_PRE + 1) = pA;
            PLN(px, PL_R) = r0; PLN(px, PL_R + 1) = r1; PLN(px, PL_R + 2) = r2;
            PLN(px, PL_P) = p0; PLN(px, PL_P + 1) = p1; PLN(px, PL_P + 2) = p2;
            edge_put(tb, PL_PRE, lx, ly, pX); edge_put(tb, PL_PRE + 1, lx, ly, pA);
            edge_put(tb, PL_R, lx, ly, r0); edge_put(tb, PL_R + 1, lx, ly, r1); edge_put(tb, PL_R + 2, lx, ly, r2);
            edge_put(tb, PL_P, lx, ly, p0); edge_put(tb, PL_P + 1, lx, ly, p1); edge_put(tb, PL_P + 2, lx, ly, p2);
            PLN(px, PL_D) = 0.f; PLN(px, PL_D + 1) = 0.f; PLN(px, PL_D + 2) = 0.f;
            g = g + dot3(r0, r1, r2, p0, p1, p2);
        }
    }
    publish(dp, bn_set(-1), block_exact_sum(g, red));
}

template <bool FIRST>
__global__ void __launch_bounds__(ST_THREADS) k_step_a_gen(const __grid_constant__ StreamPlanes pl,
                                                           const StreamDev* __restrict__ dpp, int it)
{
    __shared__ double red[64];
    __shared__ float s_beta;
    const StreamDev& dp = *dpp;
    const bool tile_on = pl.tile_active[blockIdx.x] != 0;
    if (!tile_on && blockIdx.x != 0) return;
    float beta = 0.0f;
    if (!FIRST) {
        if (threadIdx.x < 32) {
            const float v = wide_round(fetch2(pl, bn_set(it - 1), bn_set(it - 2)));
            const float bnum = __shfl_sync(0xffffffffu, v, 0), num = __shfl_sync(0xffffffffu, v, 16);
            if (threadIdx.x == 0) {
                s_beta = (num > 0.0f) ? bnum / num : 0.0f;
                if (blockIdx.x == 0 && dp.trace) dp.trace[3 * (it - 1) + 2] = bnum;
            }
        }
        __syncthreads();
        beta = s_beta;
    }
    const int W = pl.W, H = pl.H;
    const int src = PL_P + 3 * (FIRST ? 0 : ((it - 1) & 1)), dst = PL_P + 3 * (it & 1);
    const int lx = threadIdx.x & 31, lyb = (threadIdx.x >> 5) * 4;
    const int x = (blockIdx.x % pl.tx) * ST_TILE + lx, y0 = (blockIdx.x / pl.tx) * ST_TILE;
    float* tb = tile_ptr(pl, blockIdx.x);
    // the new direction of pixel at plane-0 address q (ping-pong: neighbours are recomputed, never read from dst)
    auto new_p = [&](const float* q, float& p0, float& p1, float& pa) {
        p0 = PLN(q, src); p1 = PLN(q, src + 1); pa = PLN(q, src + 2);
        if (!FIRST) {
            const float pX = PLN(q, PL_PRE), pA = PLN(q, PL_PRE + 1);
            p0 = fmaf(beta, p0, pX * PLN(q, PL_R));
            p1 = fmaf(beta, p1, pX * PLN(q, PL_R + 1));
            pa = fmaf(beta, pa, pA * PLN(q, PL_R + 2));
        }
    };
    float g = 0.0f;
    if (x < W && tile_on) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int ly = lyb + r, y = y0 + ly;
            if (y >= H) break;
            const int loc = ly * ST_TILE + lx;
            float* px = tb + loc;
            float p0, p1, pa;
            new_p(px, p0, p1, pa);
            if (!FIRST) {
                PLN(px, dst) = p0; PLN(px, dst + 1) = p1; PLN(px, dst + 2) = pa;
                edge_put(tb, dst, lx, ly, p0); edge_put(tb, dst + 1, lx, ly, p1); edge_put(tb, dst + 2, lx, ly, pa);
            }
            const unsigned f = *flag_ptr(tb, loc);
            if (!(f & FLAG_ACTIVE)) continue;
            const float2 ui = dp.U[(size_t)y * W + x];
            JtjAcc a;
            jtj_zero(a);
#pragma unroll
            for (int n = 0; n < 4; ++n) {
                if (!(f & (1u << n))) continue;
                const GenNb nb = gen_nb(dp, x, y, n, ui);
                float q0, q1, qa;
                new_p(nb.px, q0, q1, qa);
                jtj_nb_gen(a, p0, p1, q0, q1, qa, PLN(nb.px, PL_CS), PLN(nb.px, PL_CS + 1), nb.dx, nb.dy);
            }
            float q0, q1, qa;
            jtj_finish(a, PLN(px, PL_CS), PLN(px, PL_CS + 1), p0, p1, pa, (f & FLAG_FIT) != 0, dp.wr2, dp.wf2, q0, q1, qa);
            PLN(px, PL_Q) = q0; PLN(px, PL_Q + 1) = q1; PLN(px, PL_Q + 2) = qa;
            g = g + dot3(p0, p1, pa, q0, q1, qa);
        }
    }
    publish(pl, ST_ACC_D0 + (it & 1), block_exact_sum(g, red));
}

__global__ void __launch_bounds__(ST_THREADS) k_cost_gen(const StreamDev* __restrict__ dpp)
{
    __shared__ double red[64];
    const StreamDev& dp = *dpp;
    const int W = dp.W, H = dp.H;
    const int lx = threadIdx.x & 31, lyb = (threadIdx.x >> 5) * 4;
    const int x = (blockIdx.x % dp.tx) * ST_TILE + lx, y0 = (blockIdx.x / dp.tx) * ST_TILE;
    float* tb = tile_ptr(dp, blockIdx.x);
    float g = 0.0f;
    if (x < W) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int ly = lyb + r, y = y0 + ly;
            if (y >= H) break;
            const size_t i = (size_t)y * W + x;
            const int loc = ly * ST_TILE + lx;
            const unsigned f = *flag_ptr(tb, loc);
            if (!(f & FLAG_ACTIVE)) continue;
            const float2 Xi = dp.X[i], ui = dp.U[i];
            const float ci = PLN(tb + loc, PL_CS), si = PLN(tb + loc, PL_CS + 1);
            float acc = 0.0f;
#pragma unroll
            for (int n = 0; n < 4; ++n) {
                if (!(f & (1u << n))) continue;
                const GenNb nb = gen_nb(dp, x, y, n, ui);
                const float2 Xj = dp.X[nb.j];
                acc = cost_nb_gen(acc, Xi.x, Xi.y, ci, si, Xj.x, Xj.y, nb.dx, nb.dy, dp.wr);
            }
            if (f & FLAG_FIT) {
                const float2 c = dp.C[i];
                acc = cost_fit(acc, Xi.x, Xi.y, c.x, c.y, dp.wf);
            }
            g = g + acc;
        }
    }
    publish(dp, ST_ACC_COST, block_exact_sum(g, red));
}

// Cost accumulator -> scalars; with tracing, also the last iteration's r.z
// is_init: the cost of Opt_ProblemInit (a new Gauss-Newton loop starts); otherwise the cost after a step, which the opt-in
// gn_rtol rule compares with the previous one (same rule as the resident kernel and oracle/arap_oracle.c)
__global__ void __launch_bounds__(32) k_finish(const __grid_constant__ StreamPlanes pl, const StreamDev* __restrict__ dpp,
                                               int last_it, int is_init)
{
    const float v = wide_round(fetch2(pl, ST_ACC_COST, bn_set(last_it < 0 ? 0 : last_it)));
    if (threadIdx.x == 0) {
        const float c = 0.5f * v;
        StreamScalars* sc = pl.sc;
        sc->cost = c;
        if (is_init) { sc->gn_prev = c; sc->gn_done = 0u; }
        else if (dpp->gn_rtol > 0.0f && !sc->gn_done) {
            if (!((sc->gn_prev - c) > dpp->gn_rtol * sc->gn_prev)) sc->gn_done = 1u; // this step gained too little
            sc->gn_prev = c;
        }
    }
    if (threadIdx.x == 16 && last_it >= 0 && dpp->trace) dpp->trace[3 * last_it + 2] = v;
}

// debug: one accumulator -> a float
__global__ void __launch_bounds__(32) k_decode(const __grid_constant__ StreamPlanes pl, int set, float* dst)
{
    const float v = wide_round(fetch2(pl, set, set));
    if (threadIdx.x == 0) *dst = v;
}

} // namespace

// ------------------------------------------------------------------------------------------ host
static constexpr size_t ACC_BYTES = (size_t)ST_ACC_SETS * WA_WORDS * sizeof(unsigned long long);

StreamSolver::StreamSolver(int W, int H)
{
    h_.W = W;
    h_.H = H;
    h_.tx = (W + ST_TILE - 1) / ST_TILE;
    h_.ty = (H + ST_TILE - 1) / ST_TILE;
    h_.ntiles = h_.tx * h_.ty;
    const size_t bytes = (size_t)h_.ntiles * ST_TILE_FLOATS * sizeof(float);
    ARAP_CUDA_CHECK(cudaMalloc(&h_.planes, bytes));
    ARAP_CUDA_CHECK(cudaMemset(h_.planes, 0, bytes));
    ARAP_CUDA_CHECK(cudaMalloc(&h_.tile_active, (size_t)h_.ntiles));
    ARAP_CUDA_CHECK(cudaMemset(h_.tile_active, 1, (size_t)h_.ntiles));
    ARAP_CUDA_CHECK(cudaMalloc(&h_.acc, ACC_BYTES));
    ARAP_CUDA_CHECK(cudaMemset(h_.acc, 0, ACC_BYTES));
    ARAP_CUDA_CHECK(cudaMalloc(&h_.sc, sizeof(StreamScalars)));
    ARAP_CUDA_CHECK(cudaMemset(h_.sc, 0, sizeof(StreamScalars)));
    ARAP_CUDA_CHECK(cudaMalloc(&d_, sizeof(StreamDev)));
    // the memsets above ran on the legacy stream; the solver's kernels run on non-blocking streams that do not order
    // behind it, and the branch-free kernels rely on "inactive pixels hold zeros": finish the clears here
    ARAP_CUDA_CHECK(cudaDeviceSynchronize());
    h_.trace = nullptr;
}

StreamSolver::~StreamSolver()
{
    if (graph_) cudaGraphExecDestroy(graph_);
    cudaFree(h_.planes);
    cudaFree(h_.tile_active);
    cudaFree(h_.acc);
    cudaFree(h_.sc);
    cudaFree(d_);
}

// ---- debug access: row-major host image <-> one tile-interleaved plane ----
static size_t host_tiled_off(const StreamDev& h, int x, int y)
{
    return (size_t)((y >> 5) * h.tx + (x >> 5)) * ST_TILE_FLOATS + (size_t)(((y & 31) << 5) + (x & 31));
}

void StreamSolver::download_plane(int plane, float* dst) const
{
    std::vector<float> all((size_t)h_.ntiles * ST_TILE_FLOATS);
    ARAP_CUDA_CHECK(cudaMemcpy(all.data(), h_.planes, all.size() * sizeof(float), cudaMemcpyDeviceToHost));
    for (int y = 0; y < h_.H; ++y)
        for (int x = 0; x < h_.W; ++x) dst[(size_t)y * h_.W + x] = all[host_tiled_off(h_, x, y) + (size_t)plane * ST_TILE_PX];
}

void StreamSolver::upload_plane(int plane, const float* src)
{
    std::vector<float> all((size_t)h_.ntiles * ST_TILE_FLOATS);
    ARAP_CUDA_CHECK(cudaMemcpy(all.data(), h_.planes, all.size() * sizeof(float), cudaMemcpyDeviceToHost));
    for (int y = 0; y < h_.H; ++y)
        for (int x = 0; x < h_.W; ++x) {
            const float v = src[(size_t)y * h_.W + x];
            all[host_tiled_off(h_, x, y) + (size_t)plane * ST_TILE_PX] = v;
            const bool halo_plane = plane < PL_Q || (plane >= PL_CS && plane < PL_FLAGS);
            if (halo_plane && ((x & 31) == 0 || (x & 31) == 31)) { // keep the edge mirror in step (PL_EDGE)
                const size_t tile0 = (size_t)((y >> 5) * h_.tx + (x >> 5)) * ST_TILE_FLOATS;
                const int slot = plane < 9 ? plane : plane - 6;
                all[tile0 + (size_t)PL_EDGE * ST_TILE_PX + (size_t)(slot * 2 + ((x & 31) ? 1 : 0)) * ST_TILE + (y & 31)] = v;
            }
        }
    ARAP_CUDA_CHECK(cudaMemcpy(h_.planes, all.data(), all.size() * sizeof(float), cudaMemcpyHostToDevice));
}

void StreamSolver::download_flags(unsigned char* dst) const
{
    std::vector<float> all((size_t)h_.ntiles * ST_TILE_FLOATS);
    ARAP_CUDA_CHECK(cudaMemcpy(all.data(), h_.planes, all.size() * sizeof(float), cudaMemcpyDeviceToHost));
    for (int y = 0; y < h_.H; ++y)
        for (int x = 0; x < h_.W; ++x) {
            const size_t tile0 = (size_t)((y >> 5) * h_.tx + (x >> 5)) * ST_TILE_FLOATS;
            const unsigned char* fb = reinterpret_cast<const unsigned char*>(all.data() + tile0 + (size_t)PL_FLAGS * ST_TILE_PX);
            dst[(size_t)y * h_.W + x] = fb[((y & 31) << 5) + (x & 31)];
        }
}

void StreamSolver::upload(cudaStream_t stream)
{
    ARAP_CUDA_CHECK(cudaMemcpyAsync(d_, &h_, sizeof(StreamDev), cudaMemcpyHostToDevice, stream));
}

void StreamSolver::bind(float2* X, float* A, const float2* U, const float2* C, const float* M, float wf,
                        float wr, cudaStream_t stream)
{
    h_.X = X; h_.A = A; h_.U = U; h_.C = C; h_.M = M;
    h_.wf = wf; h_.wr = wr; h_.wf2 = wf * wf; h_.wr2 = wr * wr;
    h_.trace = nullptr;
    h_.pcg_rtol2 = pcg_rtol_ * pcg_rtol_;
    h_.gn_rtol = general_ ? 0.0f : gn_rtol_;
    upload(stream);
}

void StreamSolver::enqueue_prep(cudaStream_t stream)
{
    ARAP_CUDA_CHECK(cudaMemsetAsync(h_.acc, 0, ACC_BYTES, stream));
    k_prep<<<h_.ntiles, ST_THREADS, 0, stream>>>(d_);
    ++launches_;
}

void StreamSolver::enqueue_pcg_init(cudaStream_t stream)
{
    if (general_) k_init_gen<<<h_.ntiles, ST_THREADS, 0, stream>>>(d_);
    else k_init<<<h_.ntiles, ST_THREADS, 0, stream>>>(d_);
    ++launches_;
}

void StreamSolver::launch_step_a(bool first, int it, cudaStream_t stream)
{
    const StreamPlanes& pl = h_;
    if (general_) {
        if (first) k_step_a_gen<true><<<h_.ntiles, ST_THREADS, 0, stream>>>(pl, d_, it);
        else k_step_a_gen<false><<<h_.ntiles, ST_THREADS, 0, stream>>>(pl, d_, it);
    } else {
        const bool rt = this->rt(); // opt-in early exits: their own instantiations
        if (first) k_step_a<true><<<2 * h_.ntiles, 128, 0, stream>>>(pl, d_, it);
        else if (rt) k_step_a<false, true><<<2 * h_.ntiles, 128, 0, stream>>>(pl, d_, it);
        else k_step_a<false><<<2 * h_.ntiles, 128, 0, stream>>>(pl, d_, it);
    }
}

void StreamSolver::launch_step_b(int it, cudaStream_t stream)
{
    const StreamPlanes& pl = h_;
    if (rt()) k_step_b<true><<<2 * h_.ntiles, 128, 0, stream>>>(pl, d_, it);
    else k_step_b<false><<<2 * h_.ntiles, 128, 0, stream>>>(pl, d_, it);
}

void StreamSolver::set_pcg_rtol(float rtol)
{
    rtol = rtol > 0.0f ? rtol : 0.0f;
    const bool was = rt();
    pcg_rtol_ = rtol;
    if (rt() != was && graph_) { // other kernel instantiations: re-capture
        cudaGraphExecDestroy(graph_); graph_ = nullptr; graph_npcg_ = -1;
    }
}

void StreamSolver::set_gn_rtol(float rtol)
{
    rtol = rtol > 0.0f ? rtol : 0.0f;
    const bool was = rt();
    gn_rtol_ = rtol;
    if (rt() != was && graph_) {
        cudaGraphExecDestroy(graph_); graph_ = nullptr; graph_npcg_ = -1;
    }
}

void StreamSolver::set_general(bool general)
{
    if (general == general_) return;
    general_ = general;
    if (graph_) { cudaGraphExecDestroy(graph_); graph_ = nullptr; graph_npcg_ = -1; } // other kernels: re-capture
}

void StreamSolver::enqueue_step_a(bool first, int it, cudaStream_t stream)
{
    const StreamPlanes& pl = h_;
    launch_step_a(first, it, stream);
    k_decode<<<1, 32, 0, stream>>>(pl, ST_ACC_D0 + (it & 1), &h_.sc->den);
    launches_ += 2;
}

void StreamSolver::enqueue_init(cudaStream_t stream)
{
    const StreamPlanes& pl = h_;
    ARAP_CUDA_CHECK(cudaMemsetAsync(&h_.sc->bad_u, 0, sizeof(unsigned), stream));
    ARAP_TIMED(timer_, "precompute", stream, enqueue_prep(stream));
    if (general_) ARAP_TIMED(timer_, "computeCost", stream, (k_cost_gen<<<h_.ntiles, ST_THREADS, 0, stream>>>(d_)));
    else ARAP_TIMED(timer_, "computeCost", stream, (k_cost<<<h_.ntiles, ST_THREADS, 0, stream>>>(d_)));
    k_finish<<<1, 32, 0, stream>>>(pl, d_, -1, 1);
    launches_ += 2;
    ARAP_CUDA_CHECK(cudaGetLastError());
}

void StreamSolver::launch_gn_body(int nPCG, cudaStream_t stream, bool tracing)
{
    const StreamPlanes& pl = h_;
    KernelTimer* const tm = tracing ? timer_ : nullptr; // never inside a graph capture
    ARAP_CUDA_CHECK(cudaMemsetAsync(h_.acc, 0, ACC_BYTES, stream));
    // the caller may have changed the constraint image / mask between steps (Opt.h:58-60): refresh flags
    ARAP_TIMED(tm, "precompute", stream, (k_prep<<<h_.ntiles, ST_THREADS, 0, stream>>>(d_)));
    if (general_) ARAP_TIMED(tm, "PCGInit1", stream, (k_init_gen<<<h_.ntiles, ST_THREADS, 0, stream>>>(d_)));
    else ARAP_TIMED(tm, "PCGInit1", stream, (k_init<<<h_.ntiles, ST_THREADS, 0, stream>>>(d_)));
    for (int it = 0; it < nPCG; ++it) {
        // PCGStep3 of the previous iteration is fused into this kernel (k_step_a)
        ARAP_TIMED(tm, "PCGStep1", stream, launch_step_a(it == 0, it, stream));
        ARAP_TIMED(tm, "PCGStep2", stream, launch_step_b(it, stream));
    }
    ARAP_TIMED(tm, "PCGLinearUpdate", stream, (k_update<<<h_.ntiles, ST_THREADS, 0, stream>>>(d_)));
    if (general_) ARAP_TIMED(tm, "computeCost", stream, (k_cost_gen<<<h_.ntiles, ST_THREADS, 0, stream>>>(d_)));
    else ARAP_TIMED(tm, "computeCost", stream, (k_cost<<<h_.ntiles, ST_THREADS, 0, stream>>>(d_)));
    k_finish<<<1, 32, 0, stream>>>(pl, d_, nPCG - 1, 0);
}

void StreamSolver::enqueue_gn_step(int nPCG, cudaStream_t stream, float* d_trace)
{
    const long long nodes = 2LL * nPCG + 5;
    if (timer_ && !d_trace) { // per-kernel timing: eager launches, one event pair each
        launch_gn_body(nPCG, stream, true);
        ARAP_CUDA_CHECK(cudaGetLastError());
        launches_ += nodes;
        return;
    }
    if (d_trace) {
        h_.trace = d_trace;
        upload(stream);
        launch_gn_body(nPCG, stream, true);
        ARAP_CUDA_CHECK(cudaGetLastError());
        h_.trace = nullptr;
        upload(stream);
        launches_ += nodes;
        return;
    }
    if (!graph_ || graph_npcg_ != nPCG) {
        if (graph_) { cudaGraphExecDestroy(graph_); graph_ = nullptr; }
        cudaStream_t cap;
        ARAP_CUDA_CHECK(cudaStreamCreateWithFlags(&cap, cudaStreamNonBlocking));
        cudaGraph_t g;
        ARAP_CUDA_CHECK(cudaStreamBeginCapture(cap, cudaStreamCaptureModeThreadLocal));
        launch_gn_body(nPCG, cap, false);
        ARAP_CUDA_CHECK(cudaStreamEndCapture(cap, &g));
        ARAP_CUDA_CHECK(cudaGraphInstantiate(&graph_, g, 0));
        ARAP_CUDA_CHECK(cudaGraphDestroy(g));
        ARAP_CUDA_CHECK(cudaStreamDestroy(cap));
        graph_npcg_ = nPCG;
        graph_nodes_ = nodes;
    }
    ARAP_CUDA_CHECK(cudaGraphLaunch(graph_, stream));
    launches_ += graph_nodes_;
}

void StreamSolver::read_back(cudaStream_t stream, float* cost, unsigned* bad_u)
{
    StreamScalars s;
    ARAP_CUDA_CHECK(cudaMemcpyAsync(&s, h_.sc, sizeof(s), cudaMemcpyDeviceToHost, stream));
    ARAP_CUDA_CHECK(cudaStreamSynchronize(stream));
    if (cost) *cost = s.cost;
    if (bad_u) *bad_u = s.bad_u;
}

} // namespace arapb200
