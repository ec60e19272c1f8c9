// solver_resident.cu -- persistent, on-chip-resident Gauss-Newton / PCG solver (see solver_resident.cuh).
//
// Replaces the whole host loop of ARAP/API/src/solverGPUGaussNewton.t:1016-1177 (and, in lerp mode, the
// continuation loop of ARAP/shared/CombinedSolverBase.h:99-120 with CombinedSolver.h:223-242) by ONE
// kernel launch.  Arithmetic is the contract of DESIGN.md section 3, i.e. bit-identical to the streaming
// back-end and to oracle/arap_oracle.c.
//
// Decomposition: the active part of the image is cut into 32x8-pixel strips; a warp owns one strip, a lane
// one column of 8 pixels (two contract-C3 groups).  r, p_angle, cos/sin and the neighbour flags live in
// registers for the whole PCG loop, delta in shared memory; (p_x, p_y, sin*p_a, cos*p_a) of every pixel sits
// in a shared-memory tile with a one-pixel ring.  Strips of the same CTA read each other's tiles directly;
// strips of other CTAs exchange their boundary through a small global "outbox" per strip.
//
// Everything that crosses CTAs is FENCE-FREE (a __threadfence is MEMBAR.SC + CCTL.IVALL, > 1 us here):
//  * Grid barrier + all-reduce.  A dot product is accumulated in fixed point: every group term is split
//    against a common scale 2^S into four 24-bit limbs (exact for terms within 2^-67 of 2^S); a CTA adds its
//    limb sums into four 64-bit words with red.global.add.u64, the upper 16 bits of each contribution
//    counting the arrival (+ an overflow flag).  A word is complete when its count reaches G, so value and
//    "everybody arrived" travel in the same 8-byte word and integer addition makes the result independent
//    of arrival order.  Two buffers alternate; they are never reset inside a launch (readers subtract the
//    total they saw two barriers ago).  S is predicted from the previous result of the same reduction and
//    verified (overflow flag / magnitude of the result); a wrong guess costs one extra barrier.
//  * Halo.  Outbox words are (float, tag) pairs, each ONE 64-bit element of a st.relaxed.gpu.v2.b64; the receiver
//    spins with ld.relaxed.gpu.v2.b64 until the tag equals the publication sequence number, so the data
//    validates itself (64-bit elements are single-copy atomic: value and tag cannot tear).
//
// Per PCG iteration there are exactly two grid barriers (sum p.Ap, sum z.r).  The direction update
// p = z + beta p that follows the second one needs the neighbours' NEW p; instead of a third barrier every
// strip publishes (z, p_old) of its boundary pixels before the second barrier and the receiver applies beta.
#include "solver_resident.cuh"
#include "grid_math.cuh"
#include "solver_stream.cuh" // FLAG_* bit layout
#include <algorithm>

namespace arapb200 {
namespace {

constexpr int TW = RS_STRIP_W + 2, TH = RS_STRIP_H + 2;
constexpr int RS_THREADS_MAX = 384;
constexpr int OB_LEFT = 64, OB_RIGHT = 64 + RS_STRIP_H;
constexpr long long LIMB_BIAS = 1ll << 36;
constexpr int BAR_STRIDE = 128; // u64 words between barrier words (1 KiB): separate L2 slices, parallel atomics
constexpr int S_MIN = -100, S_MAX = 100;
// The barrier is ~55 % of a lone problem's PCG iteration, and its code is so latency-critical that harmless-looking
// changes move C1 by several percent either way.  Measure every alternative against this code (tools/build_variant.sh +
// tools/ab_sweep.sh); profiles/r2_barrier_ab.txt and DESIGN.md 4.1 record what was tried and removed.

struct __align__(16) StripSmem {
    float4 T[TH][TW];              // tile + ring: (p_x, p_y, sin*p_a, cos*p_a) or (X_x, X_y, cos, sin)
    float D[3][RS_STRIP_H][32];    // delta
    float2 rcs[RS_OUTBOX_ENTRIES]; // cos/sin of the ring pixels (remote sides only)
    float stage[RS_OUTBOX_ENTRIES][4]; // remote ring pixels: [0..2] fetched z (parked until beta is known), [3] their p_a
    float2 pre[RS_STRIP_H][32];        // (1/(1+sqrt(D_X))^2, 1/(1+sqrt(D_a))^2) per pixel, constant during a GN step
};

struct __align__(16) Ctl {
    int limb[RS_THREADS_MAX / 32][4];
    int ovf[RS_THREADS_MAX / 32];
    unsigned long long prev[2][4]; // totals last seen in each barrier buffer
    float bc;                      // broadcast result
    float stop;                    // opt-in early exit: leave the PCG loop once r.z <= stop (-1: never)
    float prev_cost;               // opt-in early exit of the Gauss-Newton loop: cost before the last step
    int bc_code;                   // 0 accept, 1 redo with bc_S
    int bc_S;
    int abort;
};

__device__ __forceinline__ unsigned long long ld_u64_volatile(const unsigned long long* p)
{
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void red_add_u64(unsigned long long* p, unsigned long long v)
{
    asm volatile("red.relaxed.gpu.global.add.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// An outbox entry is four (float, tag) words.  Each word is ONE 64-bit element (float in the low half, tag in the high
// half): 64-bit elements of a vector access are single-copy atomic in the PTX memory model, so a value can never be
// observed with another publication's tag, and a relaxed store paired with a relaxed load is a morally strong pair (no
// data race).  The uint4 view (x = float, y = tag, z = float, w = tag) is the same bytes.
__device__ __forceinline__ uint4 ld_entry_relaxed(const uint4* p)
{
    unsigned long long a, b;
    asm volatile("ld.relaxed.gpu.global.v2.b64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "l"(p) : "memory");
    return make_uint4((unsigned)a, (unsigned)(a >> 32), (unsigned)b, (unsigned)(b >> 32));
}
__device__ __forceinline__ void st_entry_relaxed(uint4* p, unsigned tag, float v0, float v1)
{
    const unsigned long long t = (unsigned long long)tag << 32;
    const unsigned long long a = t | __float_as_uint(v0), b = t | __float_as_uint(v1);
    asm volatile("st.relaxed.gpu.global.v2.b64 [%0], {%1, %2};" ::"l"(p), "l"(a), "l"(b) : "memory");
}
__device__ __forceinline__ double pow2_f64(int e) // 2^e, e in the normal range
{
    return __hiloint2double((e + 1023) << 20, 0);
}

// error-free a + b = s + e (Knuth)
__device__ __forceinline__ void two_sum(double a, double b, double& s, double& e)
{
    s = __dadd_rn(a, b);
    const double bb = __dadd_rn(s, -a);
    e = __dadd_rn(__dadd_rn(a, -__dadd_rn(s, -bb)), __dadd_rn(b, -bb));
}

// L0*2^72 + L1*2^48 + L2*2^24 + L3 (|Lj| < 2^45, units 2^e_unit) -> binary32 with ONE rounding: the four terms
// are exact doubles; they are added error-free (s + e), s + e is rounded to odd in binary64 (53 >= 24 + 2 bits)
// and only then to binary32.
__device__ __forceinline__ float limbs_to_float_rn(const long long L[4], int e_unit, bool& is_zero)
{
    const double a = __ll2double_rn(L[0]) * 4722366482869645213696.0; // 2^72
    const double b = __ll2double_rn(L[1]) * 281474976710656.0;        // 2^48
    const double c = __ll2double_rn(L[2]) * 16777216.0;               // 2^24
    const double d = __ll2double_rn(L[3]);
    double s1, e1, s2, e2, s3, e3;
    two_sum(c, d, s1, e1);   // low pair first: e1 is almost always 0
    two_sum(b, s1, s2, e2);
    two_sum(a, s2, s3, e3);
    const double e = __dadd_rn(__dadd_rn(e3, e2), e1); // |e| < ulp(s3); only its sign and non-zero-ness matter
    is_zero = (s3 == 0.0 && e == 0.0);
    // round (s3 + e) to odd: truncate toward zero and, when inexact, set the last bit
    const double zd = __dadd_rd(s3, e), zu = __dadd_ru(s3, e);
    double z = (zu > 0.0) ? zd : zu;
    if (zd != zu) z = __longlong_as_double(__double_as_longlong(z) | 1ll);
    e_unit = max(-900, min(900, e_unit));
    return (float)(z * pow2_f64(e_unit)); // exact scaling (barring binary32 underflow), single rounding
}

// Everything a warp needs to know about its strip
struct StripCtx {
    bool has;               // this warp owns a strip
    int x, y0;              // lane's column, first row
    float4* own;            // &T[0][0] of the own tile
    const float4* up_row;   // row y = -1, indexed by lane
    const float4* down_row; // row y = 8
    const float4* lptr;     // pixel to the left of (lane, row 0); row stride TW
    const float4* rptr;     // pixel to the right
    float* D;               // &D[0][0][lane]
    float2* rcs;
    float* stage;           // &stage[0][0]
    float2* pre;            // &pre[0][lane]
    int rem[4];             // remote neighbour strip id per side (0 up, 1 down, 2 left, 3 right) or -1
    uint4* outbox;          // own outbox: [RS_OUTBOX_ENTRIES][3]
    uint4* side_out;        // lane 0 / lane 31: where the left / right column entries of row 0 go (null: nothing to publish)
};

struct Cta {
    const ResProb* P;
    unsigned long long* bar; // = P->bar
    int* status;             // = P->status
    Ctl* ctl;
    struct ClusterCtl* xc;   // cluster-scope barrier only (null otherwise)
    int cta, G, lane, wid, nw;
    unsigned epoch;
    unsigned long long acc[3]; // optional cycle accounting (thread 0): reduce+arrive, poll, decode+broadcast
    bool prof;
};

// ---- grid barrier carrying an exact sum ----------------------------------------------------------
// Split in two so that independent work (the halo fetch) can sit between arrival and completion.
// grid_arrive: this thread's group terms g0 (and g1 when a lane holds two groups) are converted to limbs
// against the scale 2^S, summed over the CTA and added to the barrier words.
__device__ __forceinline__ void limbs_to_smem(Cta& c, float g0, float g1, int S)
{
    Ctl* ctl = c.ctl;
    // ---- thread -> four signed 24-bit limbs in units 2^(S-18), 2^(S-42), 2^(S-66), 2^(S-90) ----
    // (binary32 only: scaling by powers of two and the remainders are exact)
    const float sc = __int_as_float((127 + 18 - S) << 23);
    int l0, l1, l2, l3;
    bool ovf;
    {
        const float v = g0 * sc;
        ovf = !(fabsf(v) < 16777216.0f); // |g| >= 2^(S+6), Inf or NaN
        const float vv = ovf ? 0.0f : v; // an overflowing term contributes nothing (its limbs would spill into the counts)
        l0 = __float2int_rn(vv);
        const float v1 = (vv - (float)l0) * 16777216.0f;
        l1 = __float2int_rn(v1);
        const float v2 = (v1 - (float)l1) * 16777216.0f;
        l2 = __float2int_rn(v2);
        const float v3 = (v2 - (float)l2) * 16777216.0f;
        l3 = __float2int_rn(v3);
    }
    {
        const float v = g1 * sc;
        const bool o1 = !(fabsf(v) < 16777216.0f);
        ovf = ovf || o1;
        const float vv = o1 ? 0.0f : v;
        const int m0 = __float2int_rn(vv);
        const float v1 = (vv - (float)m0) * 16777216.0f;
        const int m1 = __float2int_rn(v1);
        const float v2 = (v1 - (float)m1) * 16777216.0f;
        const int m2 = __float2int_rn(v2);
        const float v3 = (v2 - (float)m2) * 16777216.0f;
        l0 += m0; l1 += m1; l2 += m2; l3 += __float2int_rn(v3);
    }
    const int s0 = __reduce_add_sync(0xffffffffu, l0);
    const int s1 = __reduce_add_sync(0xffffffffu, l1);
    const int s2 = __reduce_add_sync(0xffffffffu, l2);
    const int s3 = __reduce_add_sync(0xffffffffu, l3);
    const bool wovf = __any_sync(0xffffffffu, ovf);
    if (c.lane == 0) {
        ctl->limb[c.wid][0] = s0;
        ctl->limb[c.wid][1] = s1;
        ctl->limb[c.wid][2] = s2;
        ctl->limb[c.wid][3] = s3;
        ctl->ovf[c.wid] = wovf ? 1 : 0;
    }
    __syncthreads();
}
__device__ __forceinline__ void grid_arrive(Cta& c, float g0, float g1, int S, long long& t0, long long& t1)
{
    Ctl* ctl = c.ctl;
    if (c.prof) t0 = clock64();
    limbs_to_smem(c, g0, g1, S);
    if (c.wid == 0 && c.lane < 4) {
        unsigned long long* buf = c.bar + (size_t)(c.epoch & 1u) * 4 * BAR_STRIDE;
        long long sum = 0;
        int any = 0;
        // four warps per trip: their shared-memory loads overlap
#pragma unroll 4
        for (int w = 0; w < c.nw; ++w) {
            sum += (long long)ctl->limb[w][c.lane];
            any |= ctl->ovf[w];
        }
        unsigned long long contrib = (1ull << 48) + (unsigned long long)(sum + LIMB_BIAS);
        if (c.lane == 0 && any) contrib += (1ull << 56);
        red_add_u64(buf + (size_t)c.lane * BAR_STRIDE, contrib);
    }
    if (c.prof) t1 = clock64();
}

// grid_wait: poll the barrier words until all G CTAs have arrived, decode, verify the scale, broadcast.
// Returns 0 = accepted (result in res, S updated for the next reduction of this kind), 1 = redo with the new S.
__device__ __forceinline__ int grid_wait(Cta& c, int& S, bool& grown, float& res, bool& ok, long long t0, long long t1)
{
    Ctl* ctl = c.ctl;
    long long t2 = 0;
    if (c.wid == 0 && c.lane == 0) {
        unsigned long long* buf = c.bar + (size_t)(c.epoch & 1u) * 4 * BAR_STRIDE;
        unsigned long long* prev = ctl->prev[c.epoch & 1u];
        unsigned long long d[4];
        unsigned spins = 0;
        for (;;) {
            bool done = true;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                d[j] = ld_u64_volatile(buf + (size_t)j * BAR_STRIDE) - prev[j];
                if ((int)((d[j] >> 48) & 0xFF) != c.G) done = false;
            }
            if (done) break;
            if ((++spins & 0xffu) == 0) {
                // watchdog: a peer's abort or ~seconds of polling => leave instead of hanging the GPU
                if (*(volatile int*)c.status || spins > (1u << 23)) {
                    atomicExch(c.status, 1);
                    atomicCAS(c.status + 1, 0, 100 + (int)(c.epoch & 0xffff));
                    ctl->abort = 1;
                    break;
                }
            }
        }
        if (c.prof) t2 = clock64();
        long long L[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            prev[j] += d[j];
            L[j] = (long long)(d[j] & ((1ull << 48) - 1)) - (long long)c.G * LIMB_BIAS;
        }
        const int novf = (int)((d[0] >> 56) & 0xFF);
        bool T_is_zero;
        const float r = limbs_to_float_rn(L, S - 90, T_is_zero);
        int code = 0, newS = S;
        if (novf) {
            code = 1; newS = min(S + 24, S_MAX);
            if (S >= S_MAX) code = 0; // Inf/NaN terms: give up, the result is garbage anyway
        } else if (T_is_zero) {
            if (!grown && S > S_MIN) { code = 1; newS = max(S - 64, S_MIN); }
        } else {
            const int e = ilogb_f32(fabsf(r));
            if (!grown && e < S - 24 && S > S_MIN) { code = 1; newS = max(e + 4, S_MIN); }
            else newS = max(min(e + 4, S_MAX), S_MIN);
        }
        ctl->bc = r;
        ctl->bc_code = code;
        ctl->bc_S = newS;
    }
    __syncthreads();
    if (c.prof && threadIdx.x == 0) {
        const long long t3 = clock64();
        c.acc[0] += (unsigned long long)(t1 - t0);
        c.acc[1] += (unsigned long long)(t2 - t1);
        c.acc[2] += (unsigned long long)(t3 - t2);
    }
    ++c.epoch;
    if (ctl->abort) { ok = false; res = 0.f; return 0; }
    const int code = ctl->bc_code;
    const int newS = ctl->bc_S;
    res = ctl->bc;
    if (newS > S) grown = true;
    S = newS;
    return code;
}

// ---- cluster-scope barrier (problems of at most 16 CTAs) ---------------------------------------------------------
// A problem that fits one thread-block cluster never touches L2 for its reductions: every CTA PUSHES its four limb sums
// into the shared memory of every CTA of the cluster (st.async through distributed shared memory, completion counted in
// bytes on the receiver's mbarrier), then waits on its OWN mbarrier and decodes locally.  One DSMEM hop (~200 cycles)
// replaces red -> L2 -> poll (~1 700 cycles per barrier for a lone problem, profiles/r2_resident_cycle_accounting.txt).
// Two buffers / two mbarriers alternate with the barrier's parity; a buffer is re-armed for its next use (two barriers
// later) right after its wait completes, which is before this CTA arrives at the barrier in between -- and no peer can
// send for the next use before it has passed that barrier.  Values are fresh per use (no running totals).
constexpr int CL_MAX = 16; // CTAs per cluster (non-portable size, cudaFuncAttributeNonPortableClusterSizeAllowed)
constexpr long long CL_BIAS = 1ll << 40;
struct __align__(16) ClusterCtl {
    unsigned long long x[2][CL_MAX][4]; // [buffer][sender rank][limb]: limb sum + CL_BIAS (bit 62 of limb 0: overflow)
    unsigned long long mbar[2];
};
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* b, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(b)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arm(unsigned long long* b, unsigned tx_bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(b)), "r"(tx_bytes) : "memory");
}
// (default .acquire.cta, the convention of CUTLASS's ClusterBarrier::wait for data that other CTAs of the cluster deliver
// with complete_tx: the payload lands in THIS SM's shared memory and its arrival is what flips the phase.  The explicit
// .acquire.cluster form compiles to an extra CCTL.IVALL + MEMBAR per wait.)
__device__ __forceinline__ bool mbar_try_wait(unsigned long long* b, unsigned parity)
{
    unsigned ok;
    asm volatile("{\n\t.reg .pred p;\n\t"
                 "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                 "selp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(smem_u32(b)), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void cluster_sync_all()
{
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// remote (float data word, mbarrier) store: data lands in CTA `rank`'s copy of *dst and 8 bytes complete on its *mbar
__device__ __forceinline__ void dsmem_push(unsigned long long* dst, unsigned long long* mbar, unsigned rank, unsigned long long v)
{
    unsigned rd, rm;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(rd) : "r"(smem_u32(dst)), "r"(rank));
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(rm) : "r"(smem_u32(mbar)), "r"(rank));
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b64 [%0], %1, [%2];" ::"r"(rd), "l"(v), "r"(rm) : "memory");
}
__device__ __forceinline__ void cl_setup(Cta& c, ClusterCtl* xc)
{
    c.xc = xc;
    if (threadIdx.x == 0) {
        mbar_init(&xc->mbar[0], 1);
        mbar_init(&xc->mbar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        mbar_arm(&xc->mbar[0], (unsigned)c.G * 32u);
        mbar_arm(&xc->mbar[1], (unsigned)c.G * 32u);
    }
    cluster_sync_all(); // nobody pushes before every peer's mbarriers exist
}
__device__ __forceinline__ void cl_arrive(Cta& c, float g0, float g1, int S, long long& t0, long long& t1)
{
    Ctl* ctl = c.ctl;
    ClusterCtl* xc = c.xc;
    if (c.prof) t0 = clock64();
    limbs_to_smem(c, g0, g1, S);
    if (c.wid == 0) {
        // lanes 0..3 hold the CTA's limb sums, every lane then takes (peer = lane / 4 [+ 8], limb = lane % 4)
        long long sum = 0;
        int any = 0;
        if (c.lane < 4)
            for (int w = 0; w < c.nw; ++w) {
                sum += (long long)ctl->limb[w][c.lane];
                any |= ctl->ovf[w];
            }
        unsigned long long v = (unsigned long long)(sum + CL_BIAS);
        if (c.lane == 0 && any) v |= 1ull << 62;
        v = __shfl_sync(0xffffffffu, v, c.lane & 3);
        const unsigned b = c.epoch & 1u;
#pragma unroll
        for (int half = 0; half < CL_MAX / 8; ++half) {
            const int peer = (c.lane >> 2) + 8 * half;
            if (peer < c.G) dsmem_push(&xc->x[b][c.cta][c.lane & 3], &xc->mbar[b], (unsigned)peer, v);
        }
    }
    if (c.prof) t1 = clock64();
}
__device__ __forceinline__ int cl_wait(Cta& c, int& S, bool& grown, float& res, bool& ok, long long t0, long long t1)
{
    Ctl* ctl = c.ctl;
    ClusterCtl* xc = c.xc;
    long long t2 = 0;
    if (c.wid == 0) {
        const unsigned b = c.epoch & 1u, parity = (c.epoch >> 1) & 1u;
        unsigned spins = 0;
        bool aborted = false;
        while (!mbar_try_wait(&xc->mbar[b], parity)) { // (a hardware-assisted sleep, not a busy poll)
            if (++spins > (1u << 18) || ((spins & 0x3fu) == 0 && *(volatile int*)c.status)) { aborted = true; break; }
        }
        if (c.prof) t2 = clock64();
        // sum the G senders' limbs: lane = 4 * sender + limb (senders 0..7), second half for senders 8..15
        long long part = 0;
        int fl = 0;
#pragma unroll
        for (int half = 0; half < CL_MAX / 8; ++half) {
            const int sender = (c.lane >> 2) + 8 * half;
            if (sender < c.G) {
                const unsigned long long w = xc->x[b][sender][c.lane & 3];
                fl |= (int)((w >> 62) & 1ull);
                part += (long long)(w & ((1ull << 62) - 1ull)) - CL_BIAS;
            }
        }
#pragma unroll
        for (int o = 4; o < 32; o <<= 1) {
            part += __shfl_xor_sync(0xffffffffu, part, o);
            fl |= __shfl_xor_sync(0xffffffffu, fl, o);
        }
        long long L[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) L[k] = __shfl_sync(0xffffffffu, part, k);
        const int novf = __shfl_sync(0xffffffffu, fl, 0);
        if (c.lane == 0) {
            if (!aborted) mbar_arm(&xc->mbar[b], (unsigned)c.G * 32u); // for the use after next
            bool T_is_zero;
            const float r = limbs_to_float_rn(L, S - 90, T_is_zero);
            int code = 0, newS = S;
            if (novf) {
                code = 1; newS = min(S + 24, S_MAX);
                if (S >= S_MAX) code = 0;
            } else if (T_is_zero) {
                if (!grown && S > S_MIN) { code = 1; newS = max(S - 64, S_MIN); }
            } else {
                const int e = ilogb_f32(fabsf(r));
                if (!grown && e < S - 24 && S > S_MIN) { code = 1; newS = max(e + 4, S_MIN); }
                else newS = max(min(e + 4, S_MAX), S_MIN);
            }
            if (aborted) {
                atomicExch(c.status, 1);
                atomicCAS(c.status + 1, 0, 300 + (int)(c.epoch & 0xffff));
                ctl->abort = 1;
            }
            ctl->bc = r;
            ctl->bc_code = code;
            ctl->bc_S = newS;
        }
    }
    __syncthreads();
    if (c.prof && threadIdx.x == 0) {
        const long long t3 = clock64();
        c.acc[0] += (unsigned long long)(t1 - t0);
        c.acc[1] += (unsigned long long)(t2 - t1);
        c.acc[2] += (unsigned long long)(t3 - t2);
    }
    ++c.epoch;
    if (ctl->abort) { ok = false; res = 0.f; return 0; }
    const int code = ctl->bc_code;
    const int newS = ctl->bc_S;
    res = ctl->bc;
    if (newS > S) grown = true;
    S = newS;
    return code;
}

// arrive + wait (+ the rare redo with a corrected scale).  Returns the exact sum rounded once to binary32.
// CL selects the cluster-scope barrier (a separate kernel instantiation: the L2 form compiles exactly as before).
template <bool CL>
__device__ __forceinline__ void arrive_t(Cta& c, float g0, float g1, int S, long long& t0, long long& t1)
{
    if constexpr (CL) cl_arrive(c, g0, g1, S, t0, t1);
    else grid_arrive(c, g0, g1, S, t0, t1);
}
template <bool CL>
__device__ __forceinline__ float grid_finish(Cta& c, float g0, float g1, int& S, bool& ok, long long t0, long long t1)
{
    bool grown = false;
    float res;
    for (;;) {
        int redo;
        if constexpr (CL) redo = cl_wait(c, S, grown, res, ok, t0, t1);
        else redo = grid_wait(c, S, grown, res, ok, t0, t1);
        if (!redo) break;
        __syncthreads(); // everybody has read the broadcast before the redo overwrites it
        arrive_t<CL>(c, g0, g1, S, t0, t1);
    }
    return res;
}
template <bool CL>
__device__ __forceinline__ float grid_sum(Cta& c, float g0, float g1, int& S, bool& ok)
{
    long long t0 = 0, t1 = 0;
    arrive_t<CL>(c, g0, g1, S, t0, t1);
    return grid_finish<CL>(c, g0, g1, S, ok, t0, t1);
}

// ---- halo publication / reception ----------------------------------------------------------------
// An outbox entry is 2 x uint4 = four (float, tag) words: (z0, z1 | z2, -) or (X0, X1 | c, s).  Only z travels during the
// PCG iterations: the receiver already holds the neighbour's previous direction (it computed it one iteration ago).
__device__ __forceinline__ void put_entry(uint4* e, unsigned tag, float a, float b, float c2, float d)
{
    st_entry_relaxed(e, tag, a, b);
    st_entry_relaxed(e + 1, tag, c2, d);
}

// called once per row k (fully unrolled) with the entry of pixel (lane, k)
__device__ __forceinline__ void publish_rowcol(const StripCtx& s, int lane, int k, unsigned tag, float a, float b, float c2,
                                               float d)
{
    if (s.rem[0] >= 0 && k == 0) put_entry(s.outbox + 2 * lane, tag, a, b, c2, d);
    if (s.rem[1] >= 0 && k == RS_STRIP_H - 1) put_entry(s.outbox + 2 * (32 + lane), tag, a, b, c2, d);
    if (s.side_out) put_entry(s.side_out + 2 * k, tag, a, b, c2, d); // both columns in one predicated store
}

// What a lane receives: the pixel above / below its column (all lanes) and, for lanes 0..H-1 (left column)
// or 8..8+H-1 (right column), one pixel beside the strip.  Fetched values are parked in shared memory
// (stage[ring slot][6]) so that they do not occupy registers across the barrier.
__device__ __forceinline__ bool entry_ok(const uint4 w0, const uint4 w1, unsigned tag)
{
    return w0.y == tag && w0.w == tag && w1.y == tag && w1.w == tag;
}
// four = false: only [0..2] are written -- [3] keeps the ring pixel's p_a between iterations
__device__ __forceinline__ void entry_park(float* st, const uint4 w0, const uint4 w1, bool four)
{
    *reinterpret_cast<float2*>(st) = make_float2(__uint_as_float(w0.x), __uint_as_float(w0.z));
    st[2] = __uint_as_float(w1.x);
    if (four) st[3] = __uint_as_float(w1.z);
}

// Spin until every remote entry this lane needs carries `tag`.  All loads of a round are in flight together;
// normally the first round succeeds because the neighbours published before they went into the barrier that
// this warp has just arrived at (the call sits between arrival and completion, so its latency hides there).
__device__ __forceinline__ void fetch_halo(const ResProb& P, Ctl* ctl, const StripCtx& s, int lane, unsigned tag, bool four)
{
    const bool left = s.rem[2] >= 0 && lane < RS_STRIP_H;
    const bool right = s.rem[3] >= 0 && lane >= 8 && lane < 8 + RS_STRIP_H;
    const uint4* pu = (s.rem[0] >= 0) ? P.outbox + ((size_t)s.rem[0] * RS_OUTBOX_ENTRIES + 32 + lane) * 2 : nullptr;
    const uint4* pd = (s.rem[1] >= 0) ? P.outbox + ((size_t)s.rem[1] * RS_OUTBOX_ENTRIES + lane) * 2 : nullptr;
    const uint4* ps = left ? P.outbox + ((size_t)s.rem[2] * RS_OUTBOX_ENTRIES + OB_RIGHT + lane) * 2
                           : (right ? P.outbox + ((size_t)s.rem[3] * RS_OUTBOX_ENTRIES + OB_LEFT + lane - 8) * 2 : nullptr);
    const int side_slot = left ? OB_LEFT + lane : OB_RIGHT + lane - 8;
    const uint4 fake = make_uint4(0u, tag, 0u, tag);
    unsigned spins = 0;
    for (;;) {
        uint4 u0 = fake, u1 = fake, d0 = fake, d1 = fake, s0 = fake, s1 = fake;
        if (pu) { u0 = ld_entry_relaxed(pu); u1 = ld_entry_relaxed(pu + 1); }
        if (pd) { d0 = ld_entry_relaxed(pd); d1 = ld_entry_relaxed(pd + 1); }
        if (ps) { s0 = ld_entry_relaxed(ps); s1 = ld_entry_relaxed(ps + 1); }
        if (entry_ok(u0, u1, tag) && entry_ok(d0, d1, tag) && entry_ok(s0, s1, tag)) {
            if (pu) entry_park(s.stage + 4 * lane, u0, u1, four);
            if (pd) entry_park(s.stage + 4 * (32 + lane), d0, d1, four);
            if (ps) entry_park(s.stage + 4 * side_slot, s0, s1, four);
            return;
        }
        if ((++spins & 0xffu) == 0 && (*(volatile int*)P.status || spins > (1u << 22))) {
            atomicExch(P.status, 1);
            atomicCAS(P.status + 1, 0, 200);
            ctl->abort = 1;
            return;
        }
    }
}

// ring <- neighbours' (X_x, X_y, cos, sin)
__device__ __forceinline__ void apply_x(const StripCtx& s, int lane)
{
    if (s.rem[0] >= 0) {
        const float* v = s.stage + 4 * lane;
        s.own[0 * TW + lane + 1] = make_float4(v[0], v[1], v[2], v[3]);
        s.rcs[lane] = make_float2(v[2], v[3]);
    }
    if (s.rem[1] >= 0) {
        const float* v = s.stage + 4 * (32 + lane);
        s.own[(TH - 1) * TW + lane + 1] = make_float4(v[0], v[1], v[2], v[3]);
        s.rcs[32 + lane] = make_float2(v[2], v[3]);
    }
    if (s.rem[2] >= 0 && lane < RS_STRIP_H) {
        const float* v = s.stage + 4 * (OB_LEFT + lane);
        s.own[(lane + 1) * TW + 0] = make_float4(v[0], v[1], v[2], v[3]);
        s.rcs[OB_LEFT + lane] = make_float2(v[2], v[3]);
    }
    if (s.rem[3] >= 0 && lane >= 8 && lane < 8 + RS_STRIP_H) {
        const float* v = s.stage + 4 * (OB_RIGHT + lane - 8);
        s.own[(lane - 8 + 1) * TW + TW - 1] = make_float4(v[0], v[1], v[2], v[3]);
        s.rcs[OB_RIGHT + lane - 8] = make_float2(v[2], v[3]);
    }
}

// One ring pixel's new direction p = z + beta * p_old from the neighbour's published z; p_old is what this warp computed
// for that pixel one iteration ago (p_x, p_y in the ring cell, p_a in st[3]).  FIRST: p_0 = z_0 (PCGInit1).
template <bool FIRST>
__device__ __forceinline__ void ring_update(float4* cell, float* st, float beta, float2 cs)
{
    float p0 = st[0], p1 = st[1], pa = st[2];
    if (!FIRST) {
        const float4 old = *cell;
        p0 = fmaf(beta, old.x, p0);
        p1 = fmaf(beta, old.y, p1);
        pa = fmaf(beta, st[3], pa);
    }
    st[3] = pa;
    *cell = make_float4(p0, p1, cs.y * pa, cs.x * pa);
}

// ring <- neighbours' new direction
template <bool FIRST>
__device__ __forceinline__ void apply_p(const StripCtx& s, int lane, float beta)
{
    const bool lft = lane < RS_STRIP_H;
    const int row = lft ? lane : lane - 8;
    const bool side = (lft && s.rem[2] >= 0) || (!lft && lane >= 8 && lane < 8 + RS_STRIP_H && s.rem[3] >= 0);
    const int slot = (lft ? OB_LEFT : OB_RIGHT) + row;
    if (s.rem[0] >= 0) ring_update<FIRST>(&s.own[0 * TW + lane + 1], s.stage + 4 * lane, beta, s.rcs[lane]);
    if (s.rem[1] >= 0) ring_update<FIRST>(&s.own[(TH - 1) * TW + lane + 1], s.stage + 4 * (32 + lane), beta, s.rcs[32 + lane]);
    // left column (lanes 0..H-1) and right column (lanes 8..8+H-1) in one predicated block
    if (side) ring_update<FIRST>(&s.own[(row + 1) * TW + (lft ? 0 : TW - 1)], s.stage + 4 * slot, beta, s.rcs[slot]);
}

// constraint of a pixel for the current continuation weight (CombinedSolver.h:236-239)
__device__ __forceinline__ float2 constraint_of(const ResProb& P, size_t i, int x, int y, float alpha)
{
    float2 c = P.C[i];
    if (P.lerp_mode) {
        const float om = 1.0f - alpha;
        c.x = om * (float)x + alpha * c.x;
        c.y = om * (float)y + alpha * c.y;
    }
    return c;
}

// flags of pixel k out of the two packed words
__device__ __forceinline__ unsigned flag_of(unsigned flo, unsigned fhi, int k)
{
    return ((k < 4 ? flo : fhi) >> (8 * (k & 3))) & 0xffu;
}

// =====================================================================================================
template <int MAXT, int MINB, bool PROF, bool CL = false>
__global__ void __launch_bounds__(MAXT, MINB) k_resident_t(const ResProb* __restrict__ probs)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ Ctl ctl;
    // Two grid shapes (host: enqueue_group).  Equal-sized problems: (G, count), blockIdx.y = problem.  Otherwise a
    // compact 1-D grid of exactly sum G CTAs, the CTAs of problem k following those of problem k-1.
    const ResProb* Pp = probs + blockIdx.y;
    int cta_in_problem = (int)blockIdx.x;
    if (gridDim.y == 1)
        while (cta_in_problem >= Pp->G) { cta_in_problem -= Pp->G; ++Pp; }
    // the problem descriptor is read all through the kernel: keep a copy in shared memory
    __shared__ ResProb sP;
    static_assert(sizeof(ResProb) % 4 == 0, "ResProb is copied word by word");
    for (int w = threadIdx.x; w < (int)(sizeof(ResProb) / 4); w += blockDim.x)
        reinterpret_cast<int*>(&sP)[w] = reinterpret_cast<const int*>(Pp)[w];
    __syncthreads();
    const ResProb& P = sP;
    StripSmem* S = reinterpret_cast<StripSmem*>(smem_raw);

    constexpr bool LEAN = (MINB >= 3);               // the 128-register variants
    // Rows of phases 2 and 3 whose shared-memory loads are issued together: all eight in the 168-register variants.  All
    // eight spill in the 128-register variants (C1s 28.4 -> 26.6, C2 6.04 -> 5.76, C3 6.00 -> 5.79 pairs/s); groups of
    // four gain C1s / C2 / C3 1.3 ... 1.9 % over not hoisting there, groups of two the same within noise.
    constexpr int HG = LEAN ? 4 : RS_STRIP_H;
    // delta += alpha p after the arrival at the second barrier, under its latency, in the 128-register variants only:
    // fewer live values in phase 2 there (C1s +1.4 %, C3 +1.3 %); at 168 registers it delays the poller (lone problem -1.4 %)
    constexpr bool DEFER = LEAN;
    Cta c;
    c.P = &P; c.bar = P.bar; c.status = P.status; c.ctl = &ctl; c.xc = nullptr; c.cta = cta_in_problem; c.G = P.G;
    c.lane = threadIdx.x & 31; c.wid = threadIdx.x >> 5; c.nw = blockDim.x >> 5; c.epoch = 0;
    c.acc[0] = c.acc[1] = c.acc[2] = 0; c.prof = PROF && (P.prof != nullptr);
    unsigned long long ph[4] = {0, 0, 0, 0}; // cycles in PCG phase 1, 2, 3 and everything else (thread 0)
    long long tk = c.prof ? clock64() : 0;
#define RS_TICK(slot) do { if (c.prof && threadIdx.x == 0) { const long long tn = clock64(); ph[slot] += (unsigned long long)(tn - tk); tk = tn; } } while (0)
#define RS_TOCK() do { if (c.prof && threadIdx.x == 0) tk = clock64(); } while (0)
    const int lane = c.lane, wid = c.wid;
    const int W = P.W, H = P.H;
    const float wr = P.wr, wf = P.wf, wr2 = P.wr2, wf2 = P.wf2;

    if (threadIdx.x == 0) ctl.abort = 0;
    if (threadIdx.x < 8) ctl.prev[threadIdx.x >> 2][threadIdx.x & 3] = 0ull; // the host zeroes P.bar before the launch
    if constexpr (CL) {
        // cluster launch: the problem IS the cluster (host: enqueue_cluster), rank in the cluster = CTA in the problem
        __shared__ ClusterCtl xc;
        cl_setup(c, &xc);
    }

    // ---- which strip is mine, who are my neighbours ----
    const int n = P.n_strips;
    const int s_begin = (int)(((long long)c.cta * n) / c.G), s_end = (int)(((long long)(c.cta + 1) * n) / c.G);
    StripCtx s;
    const int slot = s_begin + wid;
    s.has = slot < s_end;
    s.own = &S[wid].T[0][0];
    s.D = &S[wid].D[0][0][lane];
    s.rcs = S[wid].rcs;
    s.stage = &S[wid].stage[0][0];
    s.pre = &S[wid].pre[0][lane];
    s.up_row = s.own + 0 * TW + 1;
    s.down_row = s.own + (TH - 1) * TW + 1;
    s.lptr = s.own + 1 * TW + lane;
    s.rptr = s.own + 1 * TW + lane + 2;
    s.rem[0] = s.rem[1] = s.rem[2] = s.rem[3] = -1;
    s.outbox = nullptr;
    int sx = 0, sy = 0;
    if (s.has) {
        const int2 xy = P.strip_xy[slot];
        sx = xy.x; sy = xy.y;
        s.outbox = P.outbox + (size_t)slot * RS_OUTBOX_ENTRIES * 2;
        const int nu = (sy > 0) ? P.slot_of_strip[(sy - 1) * P.SX + sx] : -1;
        const int nd = (sy + 1 < P.SY) ? P.slot_of_strip[(sy + 1) * P.SX + sx] : -1;
        const int nl = (sx > 0) ? P.slot_of_strip[sy * P.SX + sx - 1] : -1;
        const int nr = (sx + 1 < P.SX) ? P.slot_of_strip[sy * P.SX + sx + 1] : -1;
        if (nu >= 0) { if (nu >= s_begin && nu < s_end) s.up_row = &S[nu - s_begin].T[TH - 2][1]; else s.rem[0] = nu; }
        if (nd >= 0) { if (nd >= s_begin && nd < s_end) s.down_row = &S[nd - s_begin].T[1][1]; else s.rem[1] = nd; }
        if (nl >= 0) { if (nl >= s_begin && nl < s_end) { if (lane == 0) s.lptr = &S[nl - s_begin].T[1][TW - 2]; } else s.rem[2] = nl; }
        if (nr >= 0) { if (nr >= s_begin && nr < s_end) { if (lane == 31) s.rptr = &S[nr - s_begin].T[1][1]; } else s.rem[3] = nr; }
    }
    s.side_out = nullptr;
    if (s.has && lane == 0 && s.rem[2] >= 0) s.side_out = s.outbox + 2 * OB_LEFT;
    if (s.has && lane == 31 && s.rem[3] >= 0) s.side_out = s.outbox + 2 * OB_RIGHT;
    s.x = sx * RS_STRIP_W + lane;
    s.y0 = sy * RS_STRIP_H;
    const bool any_rem = s.has && (s.rem[0] >= 0 || s.rem[1] >= 0 || s.rem[2] >= 0 || s.rem[3] >= 0); // warp-uniform

    // ---- flags from the mask (constant for the whole launch except the fit bit) ----
    unsigned flo = 0, fhi = 0;
#pragma unroll
    for (int k = 0; k < RS_STRIP_H; ++k) {
        unsigned f = 0;
        const int x = s.x, y = s.y0 + k;
        if (s.has && x < W && y < H) {
            const size_t i = (size_t)y * W + x;
            if (P.M[i] == 0.0f) {
                f = FLAG_ACTIVE;
                if (x + 1 < W && P.M[i + 1] == 0.0f) f |= 1u;
                if (x > 0 && P.M[i - 1] == 0.0f) f |= 2u;
                if (y + 1 < H && P.M[i + W] == 0.0f) f |= 4u;
                if (y > 0 && P.M[i - W] == 0.0f) f |= 8u;
            }
        }
        if (k < 4) flo |= f << (8 * k); else fhi |= f << (8 * (k - 4));
    }

    // registers that live across the PCG loop
    float r0[RS_STRIP_H], r1[RS_STRIP_H], r2[RS_STRIP_H];
    float pa[RS_STRIP_H], cc[RS_STRIP_H], ss[RS_STRIP_H];
    float q0[RS_STRIP_H], q1[RS_STRIP_H], qa[RS_STRIP_H];
#pragma unroll
    for (int k = 0; k < RS_STRIP_H; ++k) { r0[k] = r1[k] = r2[k] = pa[k] = 0.f; cc[k] = 1.f; ss[k] = 0.f; q0[k] = q1[k] = qa[k] = 0.f; }
    // preconditioner entries (position, angle) of own pixel k.  Read through this lambda rather than as s.pre[k * 32] at
    // each use: the plain reads compile to another register assignment of the kernel's set-up code.
    auto pre_of = [&](int k) -> float2 { return s.pre[k * 32]; };
    // every tile cell must hold finite data (the masked stencil multiplies invalid neighbours by 0)
    for (int e = lane; e < TH * TW; e += 32) s.own[e] = make_float4(0.f, 0.f, 0.f, 0.f);
    int S_cost = 0, S_num = 0, S_den = 0, S_bnum = 0, S_sep = 8;
    unsigned seq = 0; // publication sequence number == halo tag
    bool ok = true;
    __syncthreads();

    for (int t = 0; t < P.nCont && ok; ++t) {
        const float alpha_c = (float)(t + 1) / (float)P.nCont; // CombinedSolver.h:199-201
        for (int g = 0; g <= P.nGN && ok; ++g) {
            // ======== prologue: tile <- (X, cos, sin), ring exchange, cost of the current state ========
            ++seq;
#pragma unroll
            for (int k = 0; k < RS_STRIP_H; ++k) {
                float4 e = make_float4(0.f, 0.f, 1.f, 0.f);
                if (flag_of(flo, fhi, k) & FLAG_ACTIVE) {
                    const size_t i = (size_t)(s.y0 + k) * W + s.x;
                    const float2 X = P.X[i];
                    float sn, cs;
                    contract_sincos(P.A[i], sn, cs);
                    cc[k] = cs; ss[k] = sn;
                    e = make_float4(X.x, X.y, cs, sn);
                }
                s.own[(k + 1) * TW + lane + 1] = e;
                if (any_rem) publish_rowcol(s, lane, k, seq, e.x, e.y, e.z, e.w);
            }
            if (any_rem) {
                fetch_halo(P, &ctl, s, lane, seq, true);
                apply_x(s, lane);
            }
            __syncthreads();
            {
                float gs0 = 0.f, gs1 = 0.f;
                float4 up = s.up_row[lane], cur = s.own[1 * TW + lane + 1];
#pragma unroll
                for (int k = 0; k < RS_STRIP_H; ++k) {
                    const float4 dn = (k < RS_STRIP_H - 1) ? s.own[(k + 2) * TW + lane + 1] : s.down_row[lane];
                    const unsigned f = flag_of(flo, fhi, k);
                    if (f & FLAG_ACTIVE) {
                        const float4 lf = s.lptr[k * TW], rt = s.rptr[k * TW];
                        float acc = 0.f;
                        if (f & 1u) acc = cost_nb<0>(acc, cur.x, cur.y, cur.z, cur.w, rt, wr);
                        if (f & 2u) acc = cost_nb<1>(acc, cur.x, cur.y, cur.z, cur.w, lf, wr);
                        if (f & 4u) acc = cost_nb<2>(acc, cur.x, cur.y, cur.z, cur.w, dn, wr);
                        if (f & 8u) acc = cost_nb<3>(acc, cur.x, cur.y, cur.z, cur.w, up, wr);
                        const size_t i = (size_t)(s.y0 + k) * W + s.x;
                        const float2 ct = constraint_of(P, i, s.x, s.y0 + k, alpha_c);
                        if (ct.x >= 0.f && ct.y >= 0.f) acc = cost_fit(acc, cur.x, cur.y, ct.x, ct.y, wf);
                        if (k < 4) gs0 = gs0 + acc; else gs1 = gs1 + acc;
                    }
                    up = cur;
                    cur = dn;
                }
                const float tot = grid_sum<CL>(c, gs0, gs1, S_cost, ok);
                if (!ok) break;
                if (c.cta == 0 && threadIdx.x == 0) P.costs[(size_t)t * (P.nGN + 1) + g] = 0.5f * tot;
                if (P.gn_rtol > 0.0f) {
                    // N4 (opt-in, never on the parity path): stop the Gauss-Newton steps of this continuation step once
                    // a step improves the cost by less than gn_rtol (relative); every CTA holds the same `tot`
                    const float prevc = ctl.prev_cost;
                    __syncthreads();
                    if (threadIdx.x == 0) ctl.prev_cost = tot;
                    if (g > 0 && g < P.nGN && !((prevc - tot) > P.gn_rtol * prevc)) {
                        if (c.cta == 0 && threadIdx.x == 0)
                            for (int gg = g + 1; gg <= P.nGN; ++gg) P.costs[(size_t)t * (P.nGN + 1) + gg] = 0.5f * tot;
                        break;
                    }
                }
            }
            if (g == P.nGN) break; // the trailing prologue only produced the final cost

            // ======== PCGInit1: r = -J^T F, z = pre * r ========
            float num;
            {
                float gs0 = 0.f, gs1 = 0.f;
                float4 up = s.up_row[lane], cur = s.own[1 * TW + lane + 1];
                unsigned nflo = 0, nfhi = 0;
#pragma unroll
                for (int k = 0; k < RS_STRIP_H; ++k) {
                    const float4 dn = (k < RS_STRIP_H - 1) ? s.own[(k + 2) * TW + lane + 1] : s.down_row[lane];
                    unsigned f = flag_of(flo, fhi, k) & ~FLAG_FIT;
                    r0[k] = r1[k] = r2[k] = 0.f;
                    pa[k] = 0.f;
                    s.pre[k * 32] = make_float2(1.0f, 1.0f); // inactive pixels: r stays 0, any finite value works
                    s.D[(0 * RS_STRIP_H + k) * 32] = 0.f;
                    s.D[(1 * RS_STRIP_H + k) * 32] = 0.f;
                    s.D[(2 * RS_STRIP_H + k) * 32] = 0.f;
                    if (f & FLAG_ACTIVE) {
                        const float4 lf = s.lptr[k * TW], rt = s.rptr[k * TW];
                        JtfAcc a;
                        jtf_zero(a);
                        if (f & 1u) jtf_nb<0>(a, cur.x, cur.y, cur.z, cur.w, rt);
                        if (f & 2u) jtf_nb<1>(a, cur.x, cur.y, cur.z, cur.w, lf);
                        if (f & 4u) jtf_nb<2>(a, cur.x, cur.y, cur.z, cur.w, dn);
                        if (f & 8u) jtf_nb<3>(a, cur.x, cur.y, cur.z, cur.w, up);
                        const size_t i = (size_t)(s.y0 + k) * W + s.x;
                        const float2 ct = constraint_of(P, i, s.x, s.y0 + k, alpha_c);
                        const bool fit = (ct.x >= 0.f && ct.y >= 0.f); // arap_plan.t:22
                        if (fit) f |= FLAG_FIT;
                        float g0, g1, ga, DX, DA;
                        jtf_finish(a, cur.x, cur.y, fit, ct.x, ct.y, wr2, wf2, g0, g1, ga, DX, DA);
                        const float pX = guarded_invert(DX), pA = guarded_invert(DA);
                        s.pre[k * 32] = make_float2(pX, pA);
                        r0[k] = -g0; r1[k] = -g1; r2[k] = -ga;
                        const float z0 = pX * r0[k], z1 = pX * r1[k], z2 = pA * r2[k];
                        const float term = dot3(r0[k], r1[k], r2[k], z0, z1, z2);
                        if (k < 4) gs0 = gs0 + term; else gs1 = gs1 + term;
                    }
                    if (k < 4) nflo |= f << (8 * k); else nfhi |= f << (8 * (k - 4));
                    up = cur;
                    cur = dn;
                }
                flo = nflo; fhi = nfhi;
                // publish (z = p_0, p_old = 0) of the boundary so that neighbours rebuild p_0 with beta = 0
                ++seq;
#pragma unroll
                for (int k = 0; k < RS_STRIP_H; ++k) {
                    if (any_rem) {
                        const float2 pre = pre_of(k);
                        publish_rowcol(s, lane, k, seq, pre.x * r0[k], pre.x * r1[k], pre.y * r2[k], 0.f);
                    }
                }
                long long ta0 = 0, ta1 = 0;
                arrive_t<CL>(c, gs0, gs1, S_num, ta0, ta1);
                if (any_rem) fetch_halo(P, &ctl, s, lane, seq, false); // overlaps the barrier latency
                num = grid_finish<CL>(c, gs0, gs1, S_num, ok, ta0, ta1); // solverGPUGaussNewton.t:395 scanAlphaNumerator
                if (!ok) break;
                // p_0 = z_0 into the tile (all warps are past their J^T F reads: grid_sum synchronised)
#pragma unroll
                for (int k = 0; k < RS_STRIP_H; ++k) {
                    const float2 pre = pre_of(k);
                    const float pX = pre.x, pA = pre.y;
                    const float p0 = pX * r0[k], p1 = pX * r1[k];
                    pa[k] = pA * r2[k];
                    s.own[(k + 1) * TW + lane + 1] = make_float4(p0, p1, ss[k] * pa[k], cc[k] * pa[k]);
                }
                if (any_rem) apply_p<true>(s, lane, 0.0f);
                // N4 (opt-in, never on the parity path): relative tolerance on the preconditioned residual norm
                if (threadIdx.x == 0) ctl.stop = (P.pcg_rtol2 > 0.0f) ? P.pcg_rtol2 * num : -1.0f;
                __syncthreads();
            }

            // ======== PCG iterations ========
            RS_TICK(3);
            // Outbox reuse is safe only when a full grid barrier separates two publications to the same entry (a
            // neighbour fetches publication k between its arrival at and the completion of the barrier that follows
            // k).  The fixed-budget loop guarantees that (the last iteration does not publish and the den barrier
            // precedes it); an early exit, or no PCG iteration at all, leaves a publication without its separating
            // barrier before the next prologue publishes again -- those two paths run one extra barrier.
            bool need_sep = (P.nPCG == 0);
            for (int it = 0; it < P.nPCG; ++it) {
                // ---- PCGStep1: q = J^T J p, den = sum p.q.  Inactive pixels hold zeros throughout.
                float gs0 = 0.f, gs1 = 0.f;
                // One code path for every strip: 0/1-masked FMAs (bit-identical to skipping invalid neighbours).  A
                // second, mask-free path for all-interior strips made the kernel SLOWER (7.51 vs 7.88 pairs/s on C1):
                // warps of one CTA then finish phase 1 at different times and the loop body doubles in size.
                float4 up = s.up_row[lane], cur = s.own[1 * TW + lane + 1];
#pragma unroll
                for (int k = 0; k < RS_STRIP_H; ++k) {
                    const float4 dn = (k < RS_STRIP_H - 1) ? s.own[(k + 2) * TW + lane + 1] : s.down_row[lane];
                    const float4 lf = s.lptr[k * TW], rt = s.rptr[k * TW];
                    const unsigned f = flag_of(flo, fhi, k);
                    // validity as 0/1 multipliers (every tile cell holds finite data: tiles are zeroed at start)
                    const float m0 = (f & 1u) ? 1.0f : 0.0f, m1 = (f & 2u) ? 1.0f : 0.0f;
                    const float m2 = (f & 4u) ? 1.0f : 0.0f, m3 = (f & 8u) ? 1.0f : 0.0f;
                    JtjAcc a;
                    jtj_zero(a);
                    jtj_nb_masked<0>(a, cur.x, cur.y, rt, m0);
                    jtj_nb_masked<1>(a, cur.x, cur.y, lf, m1);
                    jtj_nb_masked<2>(a, cur.x, cur.y, dn, m2);
                    jtj_nb_masked<3>(a, cur.x, cur.y, up, m3);
                    jtj_finish(a, cc[k], ss[k], cur.x, cur.y, pa[k], (f & FLAG_FIT) != 0, wr2, wf2, q0[k], q1[k], qa[k]);
                    const float term = dot3(cur.x, cur.y, pa[k], q0[k], q1[k], qa[k]);
                    if (k < 4) gs0 = gs0 + term; else gs1 = gs1 + term;
                    up = cur;
                    cur = dn;
                }
                RS_TICK(0);
                const float den = grid_sum<CL>(c, gs0, gs1, S_den, ok);
                RS_TOCK();
                if (!ok) break;
                const float alpha = (den > 0.0f) ? num / den : 0.0f; // :456-459

                // ---- PCGStep2: delta += alpha p, r -= alpha q, z = pre r, bnum = sum z.r ----
                gs0 = 0.f; gs1 = 0.f;
                const bool pub = any_rem && (it + 1 < P.nPCG);
                ++seq;
                // every shared-memory load of the phase first: the compiler cannot move a later row's loads above an earlier
                // row's delta stores (it cannot prove that D, the tile and pre do not alias), so written row by row the phase
                // pays the shared-memory latency eight times over
#pragma unroll
                for (int kb = 0; kb < RS_STRIP_H; kb += HG) {
                    float hx[HG], hy[HG], hd0[HG], hd1[HG], hd2[HG];
                    float2 hpre[HG];
#pragma unroll
                    for (int j = 0; j < HG; ++j) {
                        const int k = kb + j;
                        if constexpr (!DEFER) {
                            const float4 e = s.own[(k + 1) * TW + lane + 1];
                            const float* Dk = s.D + k * 32;
                            hx[j] = e.x; hy[j] = e.y;
                            hd0[j] = Dk[0 * RS_STRIP_H * 32]; hd1[j] = Dk[1 * RS_STRIP_H * 32]; hd2[j] = Dk[2 * RS_STRIP_H * 32];
                        }
                        hpre[j] = pre_of(k);
                    }
#pragma unroll
                    for (int j = 0; j < HG; ++j) {
                        const int k = kb + j;
                        if constexpr (!DEFER) {
                            float* Dk = s.D + k * 32;
                            Dk[0 * RS_STRIP_H * 32] = fmaf(alpha, hx[j], hd0[j]);
                            Dk[1 * RS_STRIP_H * 32] = fmaf(alpha, hy[j], hd1[j]);
                            Dk[2 * RS_STRIP_H * 32] = fmaf(alpha, pa[k], hd2[j]);
                        }
                        r0[k] = fmaf(-alpha, q0[k], r0[k]);
                        r1[k] = fmaf(-alpha, q1[k], r1[k]);
                        r2[k] = fmaf(-alpha, qa[k], r2[k]);
                        const float pX = hpre[j].x, pA = hpre[j].y;
                        const float z0 = pX * r0[k], z1 = pX * r1[k], z2 = pA * r2[k];
                        const float term = dot3(z0, z1, z2, r0[k], r1[k], r2[k]);
                        if (k < 4) gs0 = gs0 + term; else gs1 = gs1 + term;
                        if (pub) publish_rowcol(s, lane, k, seq, z0, z1, z2, 0.f);
                    }
                }
                RS_TICK(1);
                long long tb0 = 0, tb1 = 0;
                arrive_t<CL>(c, gs0, gs1, S_bnum, tb0, tb1);
                if constexpr (DEFER) {
                    // delta += alpha p feeds no reduction: it runs here, under the latency of the barrier just arrived at
                    // (p -- the tile entries and pa -- does not change before phase 3)
#pragma unroll
                    for (int kb = 0; kb < RS_STRIP_H; kb += HG) {
                        float hx[HG], hy[HG], hd0[HG], hd1[HG], hd2[HG];
#pragma unroll
                        for (int j = 0; j < HG; ++j) {
                            const int k = kb + j;
                            const float4 e = s.own[(k + 1) * TW + lane + 1];
                            const float* Dk = s.D + k * 32;
                            hx[j] = e.x; hy[j] = e.y;
                            hd0[j] = Dk[0 * RS_STRIP_H * 32]; hd1[j] = Dk[1 * RS_STRIP_H * 32]; hd2[j] = Dk[2 * RS_STRIP_H * 32];
                        }
#pragma unroll
                        for (int j = 0; j < HG; ++j) {
                            const int k = kb + j;
                            float* Dk = s.D + k * 32;
                            Dk[0 * RS_STRIP_H * 32] = fmaf(alpha, hx[j], hd0[j]);
                            Dk[1 * RS_STRIP_H * 32] = fmaf(alpha, hy[j], hd1[j]);
                            Dk[2 * RS_STRIP_H * 32] = fmaf(alpha, pa[k], hd2[j]);
                        }
                    }
                }
                if (pub) fetch_halo(P, &ctl, s, lane, seq, false); // overlaps the barrier latency
                const float bnum = grid_finish<CL>(c, gs0, gs1, S_bnum, ok, tb0, tb1);
                RS_TOCK();
                if (!ok) break;
                if (P.trace && c.cta == 0 && threadIdx.x == 0) {
                    float* tr = P.trace + ((size_t)(t * P.nGN + g) * P.nPCG + it) * 3;
                    tr[0] = den; tr[1] = num; tr[2] = bnum;
                }
                const float beta = (num > 0.0f) ? bnum / num : 0.0f; // :544-547
                num = bnum;                                          // :1091
                if (it + 1 == P.nPCG) break; // the direction is not needed after the last iteration
                if (bnum <= ctl.stop) { need_sep = true; break; } // early exit (every CTA decodes the same bnum: a uniform decision)

                // ---- PCGStep3: p = z + beta p (own pixels, then the remote ring) ----
#pragma unroll
                for (int kb = 0; kb < RS_STRIP_H; kb += HG) {
                    float hx[HG], hy[HG];
                    float2 hpre[HG];
#pragma unroll
                    for (int j = 0; j < HG; ++j) {
                        const float4 e = s.own[(kb + j + 1) * TW + lane + 1];
                        hx[j] = e.x; hy[j] = e.y;
                        hpre[j] = pre_of(kb + j);
                    }
#pragma unroll
                    for (int j = 0; j < HG; ++j) {
                        const int k = kb + j;
                        const float pX = hpre[j].x, pA = hpre[j].y;
                        const float p0 = fmaf(beta, hx[j], pX * r0[k]);
                        const float p1 = fmaf(beta, hy[j], pX * r1[k]);
                        pa[k] = fmaf(beta, pa[k], pA * r2[k]);
                        s.own[(k + 1) * TW + lane + 1] = make_float4(p0, p1, ss[k] * pa[k], cc[k] * pa[k]);
                    }
                }
                if (any_rem) apply_p<false>(s, lane, beta);
                __syncthreads();
                RS_TICK(2);
            }
            if (!ok) break;
            if (need_sep) {
                (void)grid_sum<CL>(c, threadIdx.x == 0 ? 1.0f : 0.0f, 0.0f, S_sep, ok); // sum = G: never zero, scale settles at once
                if (!ok) break;
            }

            // ======== PCGLinearUpdate ========
#pragma unroll
            for (int k = 0; k < RS_STRIP_H; ++k) {
                if (flag_of(flo, fhi, k) & FLAG_ACTIVE) {
                    const size_t i = (size_t)(s.y0 + k) * W + s.x;
                    float2 X = P.X[i];
                    X.x = X.x + s.D[(0 * RS_STRIP_H + k) * 32];
                    X.y = X.y + s.D[(1 * RS_STRIP_H + k) * 32];
                    P.X[i] = X;
                    P.A[i] = P.A[i] + s.D[(2 * RS_STRIP_H + k) * 32];
                }
            }
            __syncthreads(); // tile entries (p) are overwritten by the next prologue
        }
    }
    if (c.prof && threadIdx.x == 0) {
        unsigned long long* o = P.prof + (size_t)c.cta * RS_PROF_SLOTS;
        o[0] = ph[0]; o[1] = ph[1]; o[2] = ph[2]; o[3] = ph[3];
        o[4] = c.acc[0]; o[5] = c.acc[1]; o[6] = c.acc[2]; o[7] = c.epoch;
    }
    if constexpr (CL) cluster_sync_all(); // no CTA leaves while a peer may still push into its shared memory
#undef RS_TICK
#undef RS_TOCK
}

// Instantiations: (max threads, min CTAs per SM).  More CTAs per SM = more problems interleaved on an SM,
// which is what hides the barrier latency; the price is a tighter register budget.
using KernelFn = void (*)(const ResProb*);
struct KernelVariant {
    int max_threads, min_blocks;
    KernelFn fn, fn_prof;
};
const KernelVariant g_variants[] = {
    {128, 4, k_resident_t<128, 4, false>, k_resident_t<128, 4, true>},
    {160, 3, k_resident_t<160, 3, false>, k_resident_t<160, 3, true>},
    {192, 2, k_resident_t<192, 2, false>, k_resident_t<192, 2, true>},
    {384, 1, k_resident_t<384, 1, false>, k_resident_t<384, 1, true>},
};
constexpr int g_nvariants = sizeof(g_variants) / sizeof(g_variants[0]);
// the cluster-scope instantiation: up to RS_THREADS_MAX / 32 strips per CTA, one CTA per SM
const KernelFn g_cluster_fn = k_resident_t<RS_THREADS_MAX, 1, false, true>;

// ---- strip table construction -------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_strip_active(int W, int H, int SX, int SY, const float* __restrict__ M,
                                                       unsigned char* __restrict__ active)
{
    const int strip = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (strip >= SX * SY) return;
    const int sx = strip % SX, sy = strip / SX; // row-major id here; ordering happens in k_strip_compact
    const int x = sx * RS_STRIP_W + lane;
    bool any = false;
    if (x < W)
        for (int k = 0; k < RS_STRIP_H; ++k) {
            const int y = sy * RS_STRIP_H + k;
            if (y < H && M[(size_t)y * W + x] == 0.0f) any = true;
        }
    const unsigned b = __ballot_sync(0xffffffffu, any);
    if (lane == 0) active[strip] = b ? 1 : 0;
}

// single block: column-major ordered compaction
__global__ void __launch_bounds__(1024) k_strip_compact(int SX, int SY, const unsigned char* __restrict__ active,
                                                         int2* __restrict__ strip_xy, int* __restrict__ slot_of_strip,
                                                         int* __restrict__ count)
{
    __shared__ int wsum[32];
    __shared__ int base;
    if (threadIdx.x == 0) base = 0;
    __syncthreads();
    const int total = SX * SY, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int start = 0; start < total; start += 1024) {
        const int j = start + threadIdx.x; // column-major: j = sx * SY + sy
        int sx = 0, sy = 0, a = 0;
        if (j < total) {
            sx = j / SY; sy = j - sx * SY;
            a = active[sy * SX + sx];
        }
        const unsigned b = __ballot_sync(0xffffffffu, a != 0);
        const int prefix = __popc(b & ((1u << lane) - 1u));
        if (lane == 0) wsum[wid] = __popc(b);
        __syncthreads();
        int woff = 0;
        for (int w = 0; w < wid; ++w) woff += wsum[w];
        int tot = 0;
        for (int w = 0; w < 32; ++w) tot += wsum[w];
        const int b0 = base;
        if (j < total) {
            if (a) {
                const int slot = b0 + woff + prefix;
                strip_xy[slot] = make_int2(sx, sy);
                slot_of_strip[sy * SX + sx] = slot;
            } else {
                slot_of_strip[sy * SX + sx] = -1;
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) base = b0 + tot;
        __syncthreads();
    }
    if (threadIdx.x == 0) *count = base;
}

} // namespace

// ------------------------------------------------------------------------------------------------ host
// The kernel variant with the most registers per thread that can keep `total_ctas` CTAs of nw warps resident;
// -1 if none can.
static int pick_variant(int nw, long long total_ctas, int sm_count)
{
    for (int v = g_nvariants - 1; v >= 0; --v) {
        if (g_variants[v].max_threads < nw * 32) continue;
        int per_sm = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, (const void*)g_variants[v].fn, nw * 32,
                                                          (size_t)nw * sizeof(StripSmem)) != cudaSuccess)
            continue;
        if ((long long)per_sm * sm_count >= total_ctas) return v;
    }
    return -1;
}

ResidentSolver::ResidentSolver(int maxW, int maxH, int max_slots) : maxW_(maxW), maxH_(maxH)
{
    int dev = 0;
    ARAP_CUDA_CHECK(cudaGetDevice(&dev));
    ARAP_CUDA_CHECK(cudaDeviceGetAttribute(&sm_count_, cudaDevAttrMultiProcessorCount, dev));
    const int SX = (maxW + RS_STRIP_W - 1) / RS_STRIP_W, SY = (maxH + RS_STRIP_H - 1) / RS_STRIP_H;
    strip_cap_ = (size_t)SX * SY;
    slots_.resize(max_slots > 0 ? max_slots : 1);
    for (Slot& sl : slots_) {
        ARAP_CUDA_CHECK(cudaMalloc(&sl.d_strip_xy, strip_cap_ * sizeof(int2)));
        ARAP_CUDA_CHECK(cudaMalloc(&sl.d_slot_of_strip, strip_cap_ * sizeof(int) + strip_cap_)); // + the active bytes
        ARAP_CUDA_CHECK(cudaMalloc(&sl.d_count, sizeof(int)));
        // the outbox only has to hold what can be resident: at most sm_count * max warps strips
        const size_t ob = std::min(strip_cap_, (size_t)sm_count_ * (RS_THREADS_MAX / 32));
        ARAP_CUDA_CHECK(cudaMalloc(&sl.d_outbox, ob * RS_OUTBOX_ENTRIES * 2 * sizeof(uint4)));
        ARAP_CUDA_CHECK(cudaMalloc(&sl.d_bar, 8 * BAR_STRIDE * sizeof(unsigned long long)));
    }
    ARAP_CUDA_CHECK(cudaMallocHost(&h_counts_, slots_.size() * sizeof(int)));
    ARAP_CUDA_CHECK(cudaMalloc(&d_status_, 2 * sizeof(int)));
    ARAP_CUDA_CHECK(cudaMemset(d_status_, 0, 2 * sizeof(int)));
    // the memset ran on the legacy stream, all later work runs on non-blocking streams: finish it here
    ARAP_CUDA_CHECK(cudaDeviceSynchronize());
    ARAP_CUDA_CHECK(cudaMalloc(&d_probs_, slots_.size() * sizeof(ResProb)));
    {
        const int smem = (int)((RS_THREADS_MAX / 32) * sizeof(StripSmem));
        ARAP_CUDA_CHECK(cudaFuncSetAttribute((const void*)g_cluster_fn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        ARAP_CUDA_CHECK(cudaFuncSetAttribute((const void*)g_cluster_fn, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    }
    for (int v = 0; v < g_nvariants; ++v) {
        const int smem = (int)((g_variants[v].max_threads / 32) * sizeof(StripSmem));
        ARAP_CUDA_CHECK(cudaFuncSetAttribute((const void*)g_variants[v].fn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        ARAP_CUDA_CHECK(cudaFuncSetAttribute((const void*)g_variants[v].fn_prof, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    }
}

ResidentSolver::~ResidentSolver()
{
    for (Slot& sl : slots_) {
        cudaFree(sl.d_strip_xy); cudaFree(sl.d_slot_of_strip); cudaFree(sl.d_count); cudaFree(sl.d_outbox); cudaFree(sl.d_bar);
    }
    cudaFreeHost(h_counts_);
    cudaFree(d_status_); cudaFree(d_probs_);
}

void ResidentSolver::prepare_enqueue(int slot, int W, int H, const float* d_M, cudaStream_t stream)
{
    Slot& sl = slots_[slot];
    sl.W = W; sl.H = H;
    sl.SX = (W + RS_STRIP_W - 1) / RS_STRIP_W;
    sl.SY = (H + RS_STRIP_H - 1) / RS_STRIP_H;
    sl.d_M = d_M;
    sl.fits = false;
    sl.n_strips = 0;
    if ((size_t)W * H > (size_t)maxW_ * maxH_ || (size_t)sl.SX * sl.SY > strip_cap_) { h_counts_[slot] = -1; return; }
    unsigned char* d_active = reinterpret_cast<unsigned char*>(sl.d_slot_of_strip + (size_t)sl.SX * sl.SY);
    k_strip_active<<<(sl.SX * sl.SY + 7) / 8, 256, 0, stream>>>(W, H, sl.SX, sl.SY, d_M, d_active);
    k_strip_compact<<<1, 1024, 0, stream>>>(sl.SX, sl.SY, d_active, sl.d_strip_xy, sl.d_slot_of_strip, sl.d_count);
    launches_ += 2;
    ARAP_CUDA_CHECK(cudaMemcpyAsync(&h_counts_[slot], sl.d_count, sizeof(int), cudaMemcpyDeviceToHost, stream));
}

bool ResidentSolver::prepare_finish(int slot)
{
    Slot& sl = slots_[slot];
    sl.fits = false;
    if (h_counts_[slot] < 0) return false;
    sl.n_strips = h_counts_[slot];
    const int max_warps = RS_THREADS_MAX / 32;
    sl.cluster_ctas = 0;
    if (sl.n_strips == 0) { sl.G = 1; sl.NW = 1; sl.fits = true; return true; }
    // small problem: fits one thread-block cluster of at most CL_MAX CTAs x max_warps strips (cluster-scope barrier)
    if (sl.n_strips <= CL_MAX * max_warps) {
        const int cs = (sl.n_strips + max_warps - 1) / max_warps;
        if (cluster_schedulable(cs)) sl.cluster_ctas = cs;
    }
    sl.NW = (sl.n_strips + sm_count_ - 1) / sm_count_;
    if (sl.NW < 4) sl.NW = 4;
    if (sl.NW > max_warps) return false; // does not fit on chip
    sl.G = (sl.n_strips + sl.NW - 1) / sl.NW;
    if (sl.G > sm_count_) sl.G = sm_count_;
    if (sl.G > RS_MAX_CTAS) return false;
    if ((sl.n_strips + sl.G - 1) / sl.G > sl.NW) return false; // balanced split: ceil(n/G) strips per CTA
    if (pick_variant(sl.NW, sl.G, sm_count_) < 0) return false;
    sl.fits = true;
    return true;
}

bool ResidentSolver::prepare(int W, int H, const float* d_M, cudaStream_t stream)
{
    prepare_enqueue(0, W, H, d_M, stream);
    ARAP_CUDA_CHECK(cudaStreamSynchronize(stream));
    return prepare_finish(0);
}

void ResidentSolver::set_problem(int slot, float2* X, float* A, const float2* C, int lerp_mode, float wf, float wr,
                                 float* d_costs, float* d_trace)
{
    Slot& sl = slots_[slot];
    ResProb& p = sl.prob;
    p = ResProb{};
    p.W = sl.W; p.H = sl.H; p.SX = sl.SX; p.SY = sl.SY; p.n_strips = sl.n_strips; p.G = sl.G;
    p.X = X; p.A = A; p.C = C; p.M = sl.d_M; p.lerp_mode = lerp_mode;
    p.wf = wf; p.wr = wr; p.wf2 = wf * wf; p.wr2 = wr * wr;
    p.strip_xy = sl.d_strip_xy; p.slot_of_strip = sl.d_slot_of_strip;
    p.outbox = sl.d_outbox; p.bar = sl.d_bar; p.costs = d_costs; p.trace = d_trace; p.status = d_status_;
}

int ResidentSolver::group_size(int first, int limit) const
{
    int best = 0;
    int nwmax = 0;
    long long ctas = 0;
    for (int cnt = 1; cnt <= limit && first + cnt <= (int)slots_.size(); ++cnt) {
        const Slot& sl = slots_[first + cnt - 1];
        if (!sl.fits) break;
        ctas += sl.G;
        nwmax = std::max(nwmax, sl.NW);
        if (pick_variant(nwmax, ctas, sm_count_) < 0) break;
        best = cnt;
    }
    return best;
}

void ResidentSolver::enqueue_group(int first, int count, int nCont, int nGN, int nPCG, cudaStream_t stream)
{
    int nwmax = 0;
    long long ctas = 0;
    std::vector<ResProb> host(count);
    for (int i = 0; i < count; ++i) {
        Slot& sl = slots_[first + i];
        sl.prob.nCont = nCont; sl.prob.nGN = nGN; sl.prob.nPCG = nPCG;
        sl.prob.pcg_rtol2 = pcg_rtol_ * pcg_rtol_;
        sl.prob.gn_rtol = gn_rtol_;
        sl.prob.prof = (i == 0) ? d_prof_ : nullptr;
        host[i] = sl.prob;
        ctas += sl.G;
        nwmax = std::max(nwmax, sl.NW);
        // barrier words start at zero; halo tags start at 1, so a zeroed outbox is "nothing published yet"
        ARAP_CUDA_CHECK(cudaMemsetAsync(sl.d_bar, 0, 8 * BAR_STRIDE * sizeof(unsigned long long), stream));
        ARAP_CUDA_CHECK(cudaMemsetAsync(sl.d_outbox, 0,
                                          (size_t)(sl.n_strips > 0 ? sl.n_strips : 1) * RS_OUTBOX_ENTRIES * 2 * sizeof(uint4), stream));
    }
    ARAP_CUDA_CHECK(cudaMemcpyAsync(d_probs_ + first, host.data(), count * sizeof(ResProb), cudaMemcpyHostToDevice, stream));
    // the live CTAs of all problems form one 1-D grid; the variant with the most registers that keeps them co-resident
    const int v = pick_variant(nwmax, ctas, sm_count_);
    if (v < 0) arap_fail(1, "resident kernel cannot be co-resident (%lld CTAs of %d warps)", ctas, nwmax);
    last_variant_ = v;
    const int threads = nwmax * 32;
    const size_t smem = (size_t)nwmax * sizeof(StripSmem);
    const ResProb* dp = d_probs_ + first;
    void* args[] = {(void*)&dp};
    const void* fn = d_prof_ ? (const void*)g_variants[v].fn_prof : (const void*)g_variants[v].fn;
    // equal-sized problems keep the 2-D shape (measured 4 % faster on C1: the hardware's placement of a 2-D grid mixes the
    // problems better over the SMs); ragged groups (multi-segment pairs) get the compact grid and its better balance
    const int g0 = slots_[first].G;
    bool equal = true;
    for (int i = 1; i < count; ++i) equal = equal && slots_[first + i].G == g0;
    const dim3 grid = equal ? dim3((unsigned)g0, (unsigned)count, 1) : dim3((unsigned)ctas, 1, 1);
    last_shape_[0] = g_variants[v].max_threads; last_shape_[1] = g_variants[v].min_blocks;
    last_shape_[2] = (int)grid.x; last_shape_[3] = (int)grid.y; last_shape_[4] = threads;
    ARAP_CUDA_CHECK(cudaLaunchCooperativeKernel(fn, grid, dim3(threads, 1, 1), args, smem, stream));
    launches_ += 1;
}

// can the device schedule a cluster of cs CTAs of the cluster kernel at full size?  (asked once per size)
bool ResidentSolver::cluster_schedulable(int cs)
{
    if (cs < 1 || cs > CL_MAX) return false;
    if (cluster_ok_[cs] == 0) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)cs, 1, 1);
        cfg.blockDim = dim3(RS_THREADS_MAX, 1, 1);
        cfg.dynamicSmemBytes = (size_t)(RS_THREADS_MAX / 32) * sizeof(StripSmem);
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = (unsigned)cs; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        int n = 0;
        const cudaError_t e = cudaOccupancyMaxActiveClusters(&n, (const void*)g_cluster_fn, &cfg);
        if (e != cudaSuccess) (void)cudaGetLastError();
        cluster_ok_[cs] = (e == cudaSuccess && n > 0) ? 1 : -1;
    }
    return cluster_ok_[cs] > 0;
}

// how many of the prepared slots first, first+1, ... (at most limit) can go into ONE cluster launch: 0 if the first
// cannot.  Different problems of such a launch need not be co-resident (a cluster is scheduled as a unit, the problems do
// not talk to each other), so the only limit is that a cluster must be schedulable at all.
int ResidentSolver::cluster_run(int first, int limit) const
{
    if (!cluster_barrier_) return 0;
    int n = 0;
    while (n < limit && first + n < (int)slots_.size() && slots_[first + n].fits && slots_[first + n].cluster_ctas > 0) ++n;
    return n;
}

void ResidentSolver::enqueue_cluster(int first, int count, int nCont, int nGN, int nPCG, cudaStream_t stream)
{
    const int max_warps = RS_THREADS_MAX / 32;
    int cs = 1, nmax = 0;
    for (int i = 0; i < count; ++i) {
        cs = std::max(cs, slots_[first + i].cluster_ctas);
        nmax = std::max(nmax, slots_[first + i].n_strips);
    }
    int nw = std::max(4, (nmax + cs - 1) / cs); // strips of the largest problem per CTA (balanced split)
    if (nw > max_warps) arap_fail(1, "cluster launch: %d strips do not fit %d CTAs", nmax, cs);
    std::vector<ResProb> host(count);
    for (int i = 0; i < count; ++i) {
        Slot& sl = slots_[first + i];
        sl.prob.G = cs; // every problem of the launch spreads over the whole cluster
        sl.prob.nCont = nCont; sl.prob.nGN = nGN; sl.prob.nPCG = nPCG;
        sl.prob.pcg_rtol2 = pcg_rtol_ * pcg_rtol_;
        sl.prob.gn_rtol = gn_rtol_;
        sl.prob.prof = nullptr;
        host[i] = sl.prob;
        // halo tags start at 1, so a zeroed outbox is "nothing published yet" (the L2 barrier words are not used)
        ARAP_CUDA_CHECK(cudaMemsetAsync(sl.d_outbox, 0,
                                        (size_t)(sl.n_strips > 0 ? sl.n_strips : 1) * RS_OUTBOX_ENTRIES * 2 * sizeof(uint4), stream));
    }
    ARAP_CUDA_CHECK(cudaMemcpyAsync(d_probs_ + first, host.data(), count * sizeof(ResProb), cudaMemcpyHostToDevice, stream));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(cs * count), 1, 1);
    cfg.blockDim = dim3((unsigned)(nw * 32), 1, 1);
    cfg.dynamicSmemBytes = (size_t)nw * sizeof(StripSmem);
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)cs;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const ResProb* dp = d_probs_ + first;
    last_variant_ = -1;
    last_shape_[0] = RS_THREADS_MAX; last_shape_[1] = 0; // min CTAs/SM "0" marks the cluster kernel
    last_shape_[2] = cs * count; last_shape_[3] = 1; last_shape_[4] = nw * 32;
    ARAP_CUDA_CHECK(cudaLaunchKernelEx(&cfg, g_cluster_fn, dp));
    launches_ += 1;
}

void ResidentSolver::enqueue(float2* X, float* A, const float2* C, int lerp_mode, float wf, float wr, int nCont, int nGN,
                             int nPCG, float* d_costs, float* d_trace, cudaStream_t stream)
{
    set_problem(0, X, A, C, lerp_mode, wf, wr, d_costs, d_trace);
    if (cluster_run(0, 1) == 1 && !d_prof_) enqueue_cluster(0, 1, nCont, nGN, nPCG, stream);
    else enqueue_group(0, 1, nCont, nGN, nPCG, stream);
}

int ResidentSolver::status(cudaStream_t stream)
{
    int st[2] = {0, 0};
    ARAP_CUDA_CHECK(cudaMemcpyAsync(st, d_status_, sizeof(st), cudaMemcpyDeviceToHost, stream));
    ARAP_CUDA_CHECK(cudaStreamSynchronize(stream));
    if (st[0]) {
        ARAP_CUDA_CHECK(cudaMemsetAsync(d_status_, 0, sizeof(st), stream));
        return st[1] ? st[1] : 1;
    }
    return 0;
}

} // namespace arapb200
