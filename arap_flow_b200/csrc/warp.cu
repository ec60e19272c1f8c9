// warp.cu -- forward warp: rasterise the deformed pixel grid into warped RGB, warped mask and the
// per-pixel splat index.
//
// Replaces the single-threaded CPU rasteriser of ARAP/deformation/src/CombinedSolver.h:248-342
// (in-app) == ARAP/warping/src/main.cpp:110-225 (stand-alone tool); edge function PointInTriangleLK
// CombinedSolver.h:61-97 / main.cpp:68-104.  The reference walks the pixel quads in row-major order,
// two triangles per quad, and lets the LAST writer win.  Here the same result is produced without any
// ordering between threads: pass 1 does an integer atomicMax of (triangle sequence number + 1) into a
// uint32 z-buffer for every covered output pixel, pass 2 re-evaluates the winning triangle's
// barycentrics and resolves colour + mask.  The outcome is therefore deterministic and bit-identical
// to the sequential reference.  All float arithmetic uses explicit round-to-nearest intrinsics (no
// FMA contraction), because the reference's colour bytes change under contraction (SURVEY.md section 4).
#include "warp.cuh"

namespace arapb200 {
namespace {

// pass 1: one thread per pixel quad (x, y), x + 1 < W, y + 1 < H, all four corners on the object
__global__ void __launch_bounds__(256) k_splat(int W, int H, const float2* __restrict__ pos,
                                                const unsigned char* __restrict__ mask_red,
                                                unsigned* __restrict__ z)
{
    const int x = blockIdx.x * 32 + (threadIdx.x & 31);
    const int y = blockIdx.y * 8 + (threadIdx.x >> 5);
    if (x + 1 >= W || y + 1 >= H) return;
    const size_t i00 = (size_t)y * W + x, i01 = i00 + 1, i10 = i00 + W, i11 = i10 + 1;
    if (mask_red[i00] | mask_red[i01] | mask_red[i10] | mask_red[i11]) return; // main.cpp:178, 191-196
    const float2 p00 = pos[i00], p01 = pos[i01], p10 = pos[i10], p11 = pos[i11];
    const unsigned id = (unsigned)(2 * i00 + 1);
    splat_tri(W, H, p00, p01, p10, id, z);     // (pos00, pos01, pos10)  main.cpp:197-199
    splat_tri(W, H, p10, p01, p11, id + 1, z); // (pos10, pos01, pos11)  main.cpp:200-202
}

// The weights w applied to the triangle's vertices as vert(i) gives them: (Va*b0 + Vb*b1) + Vc*b2, the colour's operation
// order, minus the pixel (qx, qy).  vert is the pixel grid for the backward flow of k_resolve<true>, a position array
// for the frame-to-frame flows of k_interp (DESIGN.md 4.3, 4.4).
template <class Vert>
__device__ __forceinline__ float2 interp_minus_q(const Bary& w, const Tri& tr, Vert vert, int qx, int qy)
{
    const float2 a = vert(tr.ia), b = vert(tr.ib), c = vert(tr.ic);
    const float sx = __fadd_rn(__fadd_rn(__fmul_rn(a.x, w.b0), __fmul_rn(b.x, w.b1)), __fmul_rn(c.x, w.b2));
    const float sy = __fadd_rn(__fadd_rn(__fmul_rn(a.y, w.b0), __fmul_rn(b.y, w.b1)), __fmul_rn(c.y, w.b2));
    return make_float2(__fsub_rn(sx, (float)qx), __fsub_rn(sy, (float)qy));
}

// The pixel grid as a vertex source: vertex i at its undeformed position.  The backward flow of frame 1 (k_resolve<true>)
// and the backward flow of frame k to frame 0 (k_interp_grid, DESIGN.md 4.9) both use it, so the two agree bit for bit.
struct GridVert {
    int W;
    __device__ __forceinline__ float2 operator()(size_t i) const
    {
        return make_float2((float)(int)(i % W), (float)(int)(i / W));
    }
};

// pass 2: one thread per output pixel.  BFLOW: also the backward flow -- the winning triangle's barycentrics applied to
// its undeformed vertex coordinates give the exact frame-1 source point of the pixel (DESIGN.md 4.3).
template <bool BFLOW>
__global__ void __launch_bounds__(256) k_resolve(int W, int H, const float2* __restrict__ pos,
                                                  const unsigned char* __restrict__ rgb,
                                                  const unsigned* __restrict__ z, unsigned char* __restrict__ out_rgb,
                                                  unsigned char* __restrict__ out_mask, float2* __restrict__ out_bflow)
{
    const size_t N = (size_t)W * H;
    const size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= N) return;
    const unsigned id = z[o];
    unsigned char c0 = 0, c1 = 0, c2 = 0, m = 0;
    float2 bf = make_float2(0.f, 0.f); // nothing landed: the background is static
    if (id) {
        const unsigned t = (id - 1) & 1u;
        const size_t i00 = (id - 1) >> 1, i01 = i00 + 1, i10 = i00 + W, i11 = i10 + 1;
        const size_t ia = t ? i10 : i00, ib = i01, ic = t ? i11 : i10;
        const float2 a = pos[ia], b = pos[ib], c = pos[ic];
        const int x = (int)(o % W), y = (int)(o / W);
        const Bary w = lk(a.x, a.y, b.x, b.y, c.x, c.y, (float)x, (float)y);
        // vec3f val = c0*b0 + c1*b1 + c2*b2, then the truncating vec3f -> vec3uc cast (vec3.h:32-37)
        float v[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const float ca = (float)rgb[3 * ia + k], cb = (float)rgb[3 * ib + k], cc = (float)rgb[3 * ic + k];
            v[k] = __fadd_rn(__fadd_rn(__fmul_rn(ca, w.b0), __fmul_rn(cb, w.b1)), __fmul_rn(cc, w.b2));
        }
        c0 = (unsigned char)__float2int_rz(v[0]);
        c1 = (unsigned char)__float2int_rz(v[1]);
        c2 = (unsigned char)__float2int_rz(v[2]);
        m = 255;
        if (BFLOW)
            bf = interp_minus_q(w, Tri{ia, ib, ic}, GridVert{W}, x, y);
    }
    out_rgb[3 * o] = c0;
    out_rgb[3 * o + 1] = c1;
    out_rgb[3 * o + 2] = c2;
    out_mask[o] = m;
    if (BFLOW) out_bflow[o] = bf;
}

// occlusion of frame 1: one thread per frame-1 pixel, gathering z, bflow and the forward flow (DESIGN.md 4.3)
__global__ void __launch_bounds__(256) k_occlusion(int W, int H, const unsigned char* __restrict__ mask_red,
                                                    const float2* __restrict__ flow, const unsigned* __restrict__ z,
                                                    const float2* __restrict__ bflow, unsigned char* __restrict__ occ)
{
    const size_t N = (size_t)W * H;
    const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= N) return;
    const int seg = mask_red[p] == 0 ? 0 : -1;
    const float2 f = seg == 0 ? flow[p] : make_float2(0.f, 0.f);
    occ[p] = occlusion_of(W, H, (int)(p % W), (int)(p / W), seg, f, bflow,
                          [z](size_t q) { return z[q] != 0 ? 0 : -1; });
}

// interp(z_a, P_a, V)[q] = the weights of q's winning triangle in frame a (lk against P_a) applied to that triangle's
// vertices in V, minus q; (0, 0) where nothing landed (z_a[q] == 0).  (z_{k-1}, P_{k-1}, P_k) is the flow from frame
// k - 1 to frame k, (z_k, P_k, P_{k-1}) the backward flow from frame k to frame k - 1 (DESIGN.md 4.4).
template <class Vert>
__device__ __forceinline__ float2 interp_at(int W, const unsigned* __restrict__ z_a, const float2* __restrict__ P_a,
                                            Vert vert, size_t q)
{
    const unsigned id = z_a[q];
    float2 r = make_float2(0.f, 0.f);
    if (id) {
        const Tri tr = tri_of(W, id);
        const float2 a = P_a[tr.ia], b = P_a[tr.ib], c = P_a[tr.ic];
        const int x = (int)(q % W), y = (int)(q / W);
        const Bary w = lk(a.x, a.y, b.x, b.y, c.x, c.y, (float)x, (float)y);
        r = interp_minus_q(w, tr, vert, x, y);
    }
    return r;
}

__global__ void __launch_bounds__(256) k_interp(int W, int H, const unsigned* __restrict__ z_a,
                                                 const float2* __restrict__ P_a, const float2* __restrict__ V,
                                                 float2* __restrict__ out)
{
    const size_t N = (size_t)W * H;
    const size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= N) return;
    out[q] = interp_at(W, z_a, P_a, [V](size_t i) { return V[i]; }, q);
}

// interp(z_k, P_k, grid): the backward flow of frame k to frame 0 (DESIGN.md 4.9), k_resolve<true>'s for k = 1
__global__ void __launch_bounds__(256) k_interp_grid(int W, int H, const unsigned* __restrict__ z_a,
                                                      const float2* __restrict__ P_a, float2* __restrict__ out)
{
    const size_t N = (size_t)W * H;
    const size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= N) return;
    out[q] = interp_at(W, z_a, P_a, GridVert{W}, q);
}

// query i of frame k: its frame-0 pixel p plus flow0[k][p], and occ0[k][p] (DESIGN.md 4.9); one thread per (k, i)
__global__ void __launch_bounds__(256) k_track_queries(int W, int H, int K, int n, const int2* __restrict__ queries,
                                                        const float2* __restrict__ flow0,
                                                        const unsigned char* __restrict__ occ0,
                                                        float2* __restrict__ pos, unsigned char* __restrict__ qocc)
{
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (size_t)K * n) return;
    const int2 c = queries[t % n];
    const size_t p = (t / n) * ((size_t)W * H) + (size_t)c.y * W + c.x;
    const float2 f = flow0[p];
    pos[t] = make_float2(__fadd_rn((float)c.x, f.x), __fadd_rn((float)c.y, f.y));
    qocc[t] = occ0[p];
}

// occlusion of frame k - 1 >= 1 in frame k: k_occlusion with p's surface taken from frame k - 1's z-buffer instead of
// the input mask (DESIGN.md 4.4)
__global__ void __launch_bounds__(256) k_occlusion_z(int W, int H, const unsigned* __restrict__ z_prev,
                                                      const float2* __restrict__ flow, const unsigned* __restrict__ z,
                                                      const float2* __restrict__ bflow, unsigned char* __restrict__ occ)
{
    const size_t N = (size_t)W * H;
    const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= N) return;
    const int seg = z_prev[p] != 0 ? 0 : -1;
    const float2 f = seg == 0 ? flow[p] : make_float2(0.f, 0.f);
    occ[p] = occlusion_of(W, H, (int)(p % W), (int)(p / W), seg, f, bflow,
                          [z](size_t q) { return z[q] != 0 ? 0 : -1; });
}

// positions from a flow field (main.cpp:160-166); also used for flow extraction X - grid
// (CombinedSolver.h:352-366) with sign = -1
__global__ void __launch_bounds__(256) k_grid_add(int W, int H, const float2* __restrict__ in, float2* __restrict__ out,
                                                   float sign)
{
    const size_t N = (size_t)W * H;
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const float gx = (float)(int)(i % W), gy = (float)(int)(i / W);
    const float2 v = in[i];
    float2 r;
    if (sign > 0.f) {
        r.x = __fadd_rn(gx, v.x);
        r.y = __fadd_rn(gy, v.y);
    } else {
        r.x = __fsub_rn(v.x, gx);
        r.y = __fsub_rn(v.y, gy);
    }
    out[i] = r;
}

} // namespace

int warp_launches_per_call() { return 2; }

void enqueue_warp(int W, int H, const float2* d_pos, const unsigned char* d_rgb, const unsigned char* d_mask_red,
                  unsigned* d_z, unsigned char* d_out_rgb, unsigned char* d_out_mask, cudaStream_t stream,
                  float2* d_out_bflow)
{
    const size_t N = (size_t)W * H;
    ARAP_CUDA_CHECK(cudaMemsetAsync(d_z, 0, N * sizeof(unsigned), stream));
    dim3 g1((W + 31) / 32, (H + 7) / 8);
    k_splat<<<g1, 256, 0, stream>>>(W, H, d_pos, d_mask_red, d_z);
    const unsigned g2 = (unsigned)((N + 255) / 256);
    if (d_out_bflow)
        k_resolve<true><<<g2, 256, 0, stream>>>(W, H, d_pos, d_rgb, d_z, d_out_rgb, d_out_mask, d_out_bflow);
    else
        k_resolve<false><<<g2, 256, 0, stream>>>(W, H, d_pos, d_rgb, d_z, d_out_rgb, d_out_mask, nullptr);
    ARAP_CUDA_CHECK(cudaGetLastError());
}

void enqueue_occlusion(int W, int H, const unsigned char* d_mask_red, const float2* d_flow, const unsigned* d_z,
                       const float2* d_bflow, unsigned char* d_occ, cudaStream_t stream)
{
    const size_t N = (size_t)W * H;
    k_occlusion<<<(unsigned)((N + 255) / 256), 256, 0, stream>>>(W, H, d_mask_red, d_flow, d_z, d_bflow, d_occ);
    ARAP_CUDA_CHECK(cudaGetLastError());
}

int enqueue_warp_seq(int W, int H, int K, const float2* d_pos, const unsigned char* d_rgb,
                     const unsigned char* d_mask_red, unsigned* d_z2, const SeqOut& o, cudaStream_t stream)
{
    const size_t N = (size_t)W * H;
    const unsigned g = (unsigned)((N + 255) / 256);
    int launches = 0;
    for (int k = 0; k < K; ++k) { // frame k + 1
        const float2* P = d_pos + (size_t)k * N;
        unsigned* z = d_z2 + (size_t)(k & 1) * N;
        const unsigned* zp = d_z2 + (size_t)((k + 1) & 1) * N; // frame k's z-buffer (k >= 1)
        float2 *flow = o.flow + (size_t)k * N, *bflow = o.bflow + (size_t)k * N;
        // frame 1 is the single warp of DESIGN.md 4.3: its backward flow comes from k_resolve<true>, against the grid
        enqueue_warp(W, H, P, d_rgb, d_mask_red, z, o.rgb + 3 * N * k, o.mask + N * k, stream, k == 0 ? bflow : nullptr);
        enqueue_pos_to_flow(W, H, P, o.flow0 + (size_t)k * N, stream);
        if (k == 0) {
            enqueue_pos_to_flow(W, H, P, flow, stream);
            enqueue_occlusion(W, H, d_mask_red, flow, z, bflow, o.occ, stream);
        } else {
            k_interp<<<g, 256, 0, stream>>>(W, H, zp, P - N, P, flow);
            k_interp<<<g, 256, 0, stream>>>(W, H, z, P, P - N, bflow);
            k_occlusion_z<<<g, 256, 0, stream>>>(W, H, zp, flow, z, bflow, o.occ + N * k);
        }
        launches += warp_launches_per_call() + (k == 0 ? 3 : 4);
        // tracks (DESIGN.md 4.9) while z_k is live; frame 1 is the consecutive pair, whose outputs are already there
        if (o.bflow0) {
            float2* bflow0 = o.bflow0 + (size_t)k * N;
            unsigned char* occ0 = o.occ0 ? o.occ0 + (size_t)k * N : nullptr;
            if (k == 0) {
                ARAP_CUDA_CHECK(cudaMemcpyAsync(bflow0, bflow, N * sizeof(float2), cudaMemcpyDeviceToDevice, stream));
                if (occ0) ARAP_CUDA_CHECK(cudaMemcpyAsync(occ0, o.occ, N, cudaMemcpyDeviceToDevice, stream));
            } else {
                k_interp_grid<<<g, 256, 0, stream>>>(W, H, z, P, bflow0);
                if (occ0) k_occlusion<<<g, 256, 0, stream>>>(W, H, d_mask_red, o.flow0 + (size_t)k * N, z, bflow0, occ0);
                launches += occ0 ? 2 : 1;
            }
        }
        ARAP_CUDA_CHECK(cudaGetLastError());
    }
    return launches;
}

void enqueue_track_queries(int W, int H, int K, int n, const int2* d_queries, const float2* d_flow0,
                           const unsigned char* d_occ0, float2* d_pos, unsigned char* d_occ, cudaStream_t stream)
{
    const size_t T = (size_t)K * n;
    k_track_queries<<<(unsigned)((T + 255) / 256), 256, 0, stream>>>(W, H, K, n, d_queries, d_flow0, d_occ0, d_pos, d_occ);
    ARAP_CUDA_CHECK(cudaGetLastError());
}

void enqueue_flow_to_pos(int W, int H, const float2* d_flow, float2* d_pos, cudaStream_t stream)
{
    const size_t N = (size_t)W * H;
    k_grid_add<<<(unsigned)((N + 255) / 256), 256, 0, stream>>>(W, H, d_flow, d_pos, 1.f);
    ARAP_CUDA_CHECK(cudaGetLastError());
}

void enqueue_pos_to_flow(int W, int H, const float2* d_pos, float2* d_flow, cudaStream_t stream)
{
    const size_t N = (size_t)W * H;
    k_grid_add<<<(unsigned)((N + 255) / 256), 256, 0, stream>>>(W, H, d_pos, d_flow, -1.f);
    ARAP_CUDA_CHECK(cudaGetLastError());
}

} // namespace arapb200
