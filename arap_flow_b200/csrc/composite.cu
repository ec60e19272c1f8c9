// composite.cu -- "next" row N1 (SURVEY.md 8f): the step right after the warp in the reference's driver.
//   flatten (para_gen.py:136-175): the per-segment outputs of a --multseg pair are layered in segment order; where a
//     later segment's warped mask is non-zero its flow / colour / mask replace what is below (segment 0 is the base).
//   add_bg  (para_gen.py:50-61, 206-212): where the final mask is 0 the colour comes from the background image.
//   match filter + segment masks (para_gen.py:216-223, 468-482, 513-537): "next" row N3, the step right before the solve.
// One thread per pixel; the winning layer is the LAST segment whose mask is non-zero (else segment 0), so the result
// does not depend on any ordering between threads.  Pure select arithmetic: bit-identical to the numpy original.
// Opt-in (arapb200_flatten_ex): the flattened backward flow and the occlusion of frame 1 across the layers, with the
// same occlusion rule as the per-problem warp (warp.cuh occlusion_of, DESIGN.md 4.3).
// arapb200_composite: the same layers over a background that moves by its own affine map, with the forward flow,
// backward flow and occlusion of both (DESIGN.md 4.5).
// The batch's scenes (DESIGN.md 4.6) launch the same composite on layers that stay on the device (composite.cuh).
#include "../../include/arapb200.h"
#include "common.cuh"
#include "composite.cuh"
#include "devmem.cuh"
#include "warp.cuh"

#include <algorithm>
#include <cmath>
#include <mutex>

namespace arapb200 {
namespace {

// the layer in front at pixel i: the last one whose warped mask is non-zero, -1 = none
__device__ __forceinline__ int front_layer(const Layers& L, size_t i)
{
    for (int s = L.n - 1; s >= 0; --s)
        if (L.mask[s][i] != 0) return s;
    return -1;
}

// out_bflow / out_occ may be null (arapb200_flatten passes null for both)
__global__ void __launch_bounds__(256) k_flatten(int W, int H, Layers L, const unsigned char* __restrict__ bg,
                                                  float2* __restrict__ out_flow, unsigned char* __restrict__ out_rgb,
                                                  unsigned char* __restrict__ out_mask, float2* __restrict__ out_bflow,
                                                  unsigned char* __restrict__ out_occ)
{
    const size_t N = (size_t)W * H;
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const int front = front_layer(L, i);
    const int win = front < 0 ? 0 : front; // segment 0 is the base of the flow / colour / mask layering
    const unsigned char m = L.mask[win][i];
    out_flow[i] = L.flow[win][i];
    out_mask[i] = m;
    const unsigned char* src = (bg != nullptr && m == 0) ? bg : L.rgb[win];
    out_rgb[3 * i] = src[3 * i];
    out_rgb[3 * i + 1] = src[3 * i + 1];
    out_rgb[3 * i + 2] = src[3 * i + 2];
    if (out_bflow) out_bflow[i] = front < 0 ? make_float2(0.f, 0.f) : L.bflow[front][i];
    if (out_occ) {
        int seg = -1; // p's surface: the (last) layer whose input mask has p on the object
        for (int s = L.n - 1; s >= 0; --s)
            if (L.src[s][i] == 0) { seg = s; break; }
        const float2 f = seg >= 0 ? L.flow[seg][i] : make_float2(0.f, 0.f);
        out_occ[i] = occlusion_of(W, H, (int)(i % W), (int)(i / W), seg, f, seg >= 0 ? L.bflow[seg] : nullptr,
                                  [&L](size_t q) { return front_layer(L, q); });
    }
}

// ---- background motion (DESIGN.md 4.5): the composite of the layers over an affinely moving background ----
// frame-b pass: colour, mask and backward flow of the composite.  S: frame-b pixel -> background plane, B: frame-b
// pixel -> frame a.  out_bflow may be null (no extras).
__global__ void __launch_bounds__(256) k_composite_b(int W, int H, Layers L, const unsigned char* __restrict__ bg,
                                                      int bgW, int bgH, int bg_x, int bg_y, Affine S, Affine B,
                                                      unsigned char* __restrict__ out_rgb,
                                                      unsigned char* __restrict__ out_mask, float2* __restrict__ out_bflow)
{
    const size_t N = (size_t)W * H;
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const int qx = (int)(i % W), qy = (int)(i / W);
    const int front = front_layer(L, i);
    if (front >= 0) {
        out_mask[i] = L.mask[front][i];
        out_rgb[3 * i] = L.rgb[front][3 * i];
        out_rgb[3 * i + 1] = L.rgb[front][3 * i + 1];
        out_rgb[3 * i + 2] = L.rgb[front][3 * i + 2];
        if (out_bflow) out_bflow[i] = L.bflow[front][i];
        return;
    }
    out_mask[i] = 0;
    const float2 s = affine_at(S, qx, qy);
    sample_bg(bg, bgW, bgH, make_float2(__fadd_rn(s.x, (float)bg_x), __fadd_rn(s.y, (float)bg_y)), out_rgb + 3 * i);
    if (out_bflow) {
        const float2 b = affine_at(B, qx, qy);
        out_bflow[i] = make_float2(__fsub_rn(b.x, (float)qx), __fsub_rn(b.y, (float)qy));
    }
}

// frame-a pass: forward flow and (out_occ non-null) occlusion, the background being surface L.n.  F: frame-a pixel ->
// frame b; bflow_b: the frame-b backward flow k_composite_b wrote (read only for out_occ).  kSrcPrev: L.src are the
// warped masks of frame k-1 of a sequence, p being on layer s where one is 255 -- the "255 - mask" of the flatten recipe
// (DESIGN.md 4.4) read in place.
template <bool kSrcPrev>
__global__ void __launch_bounds__(256) k_composite_a(int W, int H, Layers L, Affine F,
                                                      const float2* __restrict__ bflow_b, float2* __restrict__ out_flow,
                                                      unsigned char* __restrict__ out_occ)
{
    const size_t N = (size_t)W * H;
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const int px = (int)(i % W), py = (int)(i / W);
    int seg = L.n; // p's surface: the (last) layer whose input mask has p on the object, else the background
    for (int s = L.n - 1; s >= 0; --s)
        if (kSrcPrev ? L.src[s][i] == 255 : L.src[s][i] == 0) { seg = s; break; }
    float2 f;
    if (seg < L.n) {
        const int front = front_layer(L, i);
        out_flow[i] = L.flow[front < 0 ? 0 : front][i]; // the flatten's own selection
        f = L.flow[seg][i];
    } else {
        const float2 a = affine_at(F, px, py);
        f = make_float2(__fsub_rn(a.x, (float)px), __fsub_rn(a.y, (float)py));
        out_flow[i] = f;
    }
    if (out_occ)
        out_occ[i] = occlusion_of(W, H, px, py, seg, f, bflow_b, [&L](size_t q) {
            const int s = front_layer(L, q);
            return s < 0 ? L.n : s;
        });
}

// frame 0 of a scene: the input image where any layer's input mask is 0 (the object), the background crop elsewhere
__global__ void __launch_bounds__(256) k_scene_input(int W, int H, Layers L, const unsigned char* __restrict__ rgb,
                                                      const unsigned char* __restrict__ bg, int bgW, int bgH, int bg_x,
                                                      int bg_y, unsigned char* __restrict__ out)
{
    const size_t N = (size_t)W * H;
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    bool object = false;
    for (int s = 0; s < L.n; ++s) object = object || L.src[s][i] == 0;
    const unsigned char* c = rgb + 3 * i;
    if (!object) {
        const int x = min(max((int)(i % W) + bg_x, 0), bgW - 1), y = min(max((int)(i / W) + bg_y, 0), bgH - 1);
        c = bg + 3 * ((size_t)y * bgW + x);
    }
    out[3 * i] = c[0];
    out[3 * i + 1] = c[1];
    out[3 * i + 2] = c[2];
}

// ---- N3: match filter (para_gen.py:216-223) and per-segment masks (:513-537) ----
__global__ void __launch_bounds__(256) k_match_valid(int n, const int4* __restrict__ m, int W1, int H1,
                                                     const unsigned char* __restrict__ l1, int W2, int H2,
                                                     const unsigned char* __restrict__ l2, unsigned char* __restrict__ label)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int4 v = m[i];
    unsigned char keep = 0;
    if (v.x >= 0 && v.y >= 0 && v.z >= 0 && v.w >= 0 && v.x < W1 && v.z < W2 && v.y < H1 && v.w < H2) {
        const long long dx = (long long)v.z - v.x, dy = (long long)v.w - v.y;
        const long long d2 = dx * dx + dy * dy; // sqrt(d2) < 60 and > 0  <=>  0 < d2 < 3600 for integers
        const unsigned char a = l1[(size_t)v.y * W1 + v.x];
        if (d2 > 0 && d2 < 3600 && a > 0 && a == l2[(size_t)v.w * W2 + v.z]) keep = a;
    }
    label[i] = keep; // 0 = dropped (a kept match always has a non-zero label)
}

// order-preserving compaction by one block (n is a few thousand)
__global__ void __launch_bounds__(1024) k_match_compact(int n, const int4* __restrict__ m,
                                                        const unsigned char* __restrict__ label, int4* __restrict__ out_m,
                                                        unsigned char* __restrict__ out_l, int* __restrict__ count)
{
    __shared__ int wsum[32];
    __shared__ int base;
    if (threadIdx.x == 0) base = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int start = 0; start < n; start += 1024) {
        const int i = start + threadIdx.x;
        const unsigned char l = (i < n) ? label[i] : 0;
        const unsigned b = __ballot_sync(0xffffffffu, l != 0);
        if (lane == 0) wsum[wid] = __popc(b);
        __syncthreads();
        int woff = 0, tot = 0;
        for (int w = 0; w < 32; ++w) {
            if (w < wid) woff += wsum[w];
            tot += wsum[w];
        }
        const int b0 = base;
        if (l != 0) {
            const int o = b0 + woff + __popc(b & ((1u << lane) - 1u));
            out_m[o] = m[i];
            out_l[o] = l;
        }
        __syncthreads();
        if (threadIdx.x == 0) base = b0 + tot;
        __syncthreads();
    }
    if (threadIdx.x == 0) *count = base;
}

__global__ void __launch_bounds__(256) k_segment_mask(size_t N, const unsigned char* __restrict__ labels, int segment,
                                                      unsigned char* __restrict__ out)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const unsigned char l = labels[i];
    const bool object = segment > 0 ? (l == (unsigned char)segment) : (l != 0);
    out[i] = object ? 0 : 255; // ARAP_BG = 255 (para_gen.py:30)
}

} // namespace
} // namespace arapb200

using namespace arapb200;

extern "C" int arapb200_filter_matches(int W1, int H1, const uint8_t* labels1, int W2, int H2, const uint8_t* labels2,
                                       const int32_t* matches, int n, int32_t* out_matches, uint8_t* out_labels,
                                       int* n_out)
{
    if (W1 <= 0 || H1 <= 0 || W2 <= 0 || H2 <= 0 || !labels1 || !labels2 || n < 0 || (n > 0 && (!matches || !out_matches)) || !n_out)
        return 1;
    *n_out = 0;
    if (n == 0) return 0;
    return guarded([&]() -> int {
        const size_t N1 = (size_t)W1 * H1, N2 = (size_t)W2 * H2;
        DevBuf<unsigned char> d_l1(N1), d_l2(N2), d_lab(n), d_ol(n);
        DevBuf<int4> d_m(n), d_o(n);
        DevBuf<int> d_cnt(1);
        d_l1.up(labels1);
        d_l2.up(labels2);
        d_m.up((const int4*)matches);
        k_match_valid<<<(n + 255) / 256, 256>>>(n, d_m.p, W1, H1, d_l1.p, W2, H2, d_l2.p, d_lab.p);
        k_match_compact<<<1, 1024>>>(n, d_m.p, d_lab.p, d_o.p, d_ol.p, d_cnt.p);
        int cnt = 0;
        ARAP_CUDA_CHECK(cudaMemcpy(&cnt, d_cnt.p, sizeof(int), cudaMemcpyDeviceToHost));
        if (cnt > 0) {
            ARAP_CUDA_CHECK(cudaMemcpy(out_matches, d_o.p, (size_t)cnt * sizeof(int4), cudaMemcpyDeviceToHost));
            if (out_labels) ARAP_CUDA_CHECK(cudaMemcpy(out_labels, d_ol.p, (size_t)cnt, cudaMemcpyDeviceToHost));
        }
        *n_out = cnt;
        return 0;
    });
}

extern "C" int arapb200_segment_mask(int W, int H, const uint8_t* labels, int segment, uint8_t* out_mask)
{
    if (W <= 0 || H <= 0 || !labels || !out_mask || segment < 0 || segment > 255) return 1;
    return guarded([&]() -> int {
        const size_t N = (size_t)W * H;
        DevBuf<unsigned char> d_l(N), d_o(N);
        d_l.up(labels);
        k_segment_mask<<<(unsigned)((N + 255) / 256), 256>>>(N, d_l.p, segment, d_o.p);
        ARAP_CUDA_CHECK(cudaMemcpy(out_mask, d_o.p, N, cudaMemcpyDeviceToHost));
        return 0;
    });
}

namespace {
// the flatten's and the composite's device workspace, used on the legacy default stream with synchronous copies out
WorkspaceTable composite_workspaces;

int flatten_common(int W, int H, int n_layers, const float* const* flows, const uint8_t* const* rgbs,
                   const uint8_t* const* masks, const uint8_t* background, const uint8_t* const* src_masks,
                   const float* const* bflows, float* out_flow, uint8_t* out_rgb, uint8_t* out_mask, float* out_bflow,
                   uint8_t* out_occ)
{
    if (W <= 0 || H <= 0 || n_layers < 1 || n_layers > MAX_LAYERS || !flows || !rgbs || !masks) return 1;
    if ((out_bflow || out_occ) && !bflows) return 1;
    if (out_occ && !src_masks) return 1;
    const bool ex = out_bflow || out_occ;
    const size_t N = (size_t)W * H;
    // workspace: [layers: flow, rgb, mask (, bflow)(, src mask)][background][outputs: flow, rgb, mask (, bflow)(, occ)]
    struct { size_t flow, rgb, mask, bflow, src; } in[MAX_LAYERS];
    Layout l;
    for (int s = 0; s < n_layers; ++s) {
        in[s].flow = l.take(8 * N);
        in[s].rgb = l.take(3 * N);
        in[s].mask = l.take(N);
        in[s].bflow = l.take(ex ? 8 * N : 0);
        in[s].src = l.take(out_occ ? N : 0);
    }
    const size_t o_bg = l.take(background ? 3 * N : 0), o_flow = l.take(8 * N), o_rgb = l.take(3 * N),
                 o_mask = l.take(N), o_bflow = l.take(out_bflow ? 8 * N : 0), o_occ = l.take(out_occ ? N : 0);
    return guarded([&]() -> int {
        Workspace& ws = composite_workspaces.current();
        std::lock_guard<std::mutex> lock(ws.mu);
        unsigned char* b = ws.buf.reserve(l.bytes());
        auto up = [&](size_t at, const void* h, size_t bytes) {
            ARAP_CUDA_CHECK(cudaMemcpyAsync(b + at, h, bytes, cudaMemcpyHostToDevice, nullptr));
            return b + at;
        };
        Layers L{};
        L.n = n_layers;
        for (int s = 0; s < n_layers; ++s) {
            L.flow[s] = (const float2*)up(in[s].flow, flows[s], 8 * N);
            L.rgb[s] = up(in[s].rgb, rgbs[s], 3 * N);
            L.mask[s] = up(in[s].mask, masks[s], N);
            if (ex) L.bflow[s] = (const float2*)up(in[s].bflow, bflows[s], 8 * N);
            if (out_occ) L.src[s] = up(in[s].src, src_masks[s], N);
        }
        const unsigned char* d_bg = background ? up(o_bg, background, 3 * N) : nullptr;
        k_flatten<<<(unsigned)((N + 255) / 256), 256>>>(W, H, L, d_bg, (float2*)(b + o_flow), b + o_rgb, b + o_mask,
                                                         out_bflow ? (float2*)(b + o_bflow) : nullptr,
                                                         out_occ ? b + o_occ : nullptr);
        ARAP_CUDA_CHECK(cudaMemcpy(out_flow, b + o_flow, 8 * N, cudaMemcpyDeviceToHost));
        ARAP_CUDA_CHECK(cudaMemcpy(out_rgb, b + o_rgb, 3 * N, cudaMemcpyDeviceToHost));
        ARAP_CUDA_CHECK(cudaMemcpy(out_mask, b + o_mask, N, cudaMemcpyDeviceToHost));
        if (out_bflow) ARAP_CUDA_CHECK(cudaMemcpy(out_bflow, b + o_bflow, 8 * N, cudaMemcpyDeviceToHost));
        if (out_occ) ARAP_CUDA_CHECK(cudaMemcpy(out_occ, b + o_occ, N, cudaMemcpyDeviceToHost));
        return 0;
    });
}
} // namespace

extern "C" int arapb200_flatten(int W, int H, int n_layers, const float* const* flows, const uint8_t* const* rgbs,
                                const uint8_t* const* masks, const uint8_t* background, float* out_flow,
                                uint8_t* out_rgb, uint8_t* out_mask)
{
    return flatten_common(W, H, n_layers, flows, rgbs, masks, background, nullptr, nullptr, out_flow, out_rgb, out_mask,
                          nullptr, nullptr);
}

extern "C" int arapb200_flatten_ex(int W, int H, int n_layers, const float* const* flows, const uint8_t* const* rgbs,
                                   const uint8_t* const* masks, const uint8_t* background, const uint8_t* const* src_masks,
                                   const float* const* bflows, float* out_flow, uint8_t* out_rgb, uint8_t* out_mask,
                                   float* out_bflow, uint8_t* out_occ)
{
    return flatten_common(W, H, n_layers, flows, rgbs, masks, background, src_masks, bflows, out_flow, out_rgb, out_mask,
                          out_bflow, out_occ);
}

namespace arapb200 {
namespace {
// 2x3 affine maps in binary64, row-major: (a00 a01 a02; a10 a11 a12).  The derivation of DESIGN.md 4.5, in its order
// (ARAP_NO_CONTRACT, composite.cuh).
struct Aff64 {
    double a[6];
};

ARAP_NO_CONTRACT Aff64 aff_inverse(const Aff64& A, double* det)
{
    const double* a = A.a;
    *det = a[0] * a[4] - a[1] * a[3];
    Aff64 r;
    r.a[0] = a[4] / *det;
    r.a[1] = -a[1] / *det;
    r.a[3] = -a[3] / *det;
    r.a[4] = a[0] / *det;
    r.a[2] = -(r.a[0] * a[2] + r.a[1] * a[5]);
    r.a[5] = -(r.a[3] * a[2] + r.a[4] * a[5]);
    return r;
}

ARAP_NO_CONTRACT Aff64 aff_compose(const Aff64& P, const Aff64& Q) // P o Q
{
    const double* p = P.a;
    const double* q = Q.a;
    Aff64 r;
    for (int row = 0; row < 2; ++row) {
        const double* pr = p + 3 * row;
        r.a[3 * row] = pr[0] * q[0] + pr[1] * q[3];
        r.a[3 * row + 1] = pr[0] * q[1] + pr[1] * q[4];
        r.a[3 * row + 2] = (pr[0] * q[2] + pr[1] * q[5]) + pr[2];
    }
    return r;
}

bool aff_finite(const double* a)
{
    for (int k = 0; k < 6; ++k)
        if (!std::isfinite(a[k])) return false;
    return true;
}

Affine affine_of(const float* c) { return Affine{c[0], c[1], c[2], c[3], c[4], c[5]}; }
} // namespace

bool composite_coeffs(const double* motion_from, const double* motion_to, float c[18])
{
    Aff64 Af{{1.0, 0.0, 0.0, 0.0, 1.0, 0.0}}, At;
    if (motion_from) std::copy(motion_from, motion_from + 6, Af.a);
    std::copy(motion_to, motion_to + 6, At.a);
    if (!aff_finite(Af.a) || !aff_finite(At.a)) return false;
    double det_f = 0.0, det_t = 0.0;
    const Aff64 If = aff_inverse(Af, &det_f), It = aff_inverse(At, &det_t);
    if (det_f == 0.0 || det_t == 0.0) return false;
    const Aff64 m[3] = {aff_compose(At, If), aff_compose(Af, It), It}; // F, B, S
    for (int k = 0; k < 18; ++k) {
        c[k] = (float)m[k / 6].a[k % 6];
        if (!std::isfinite(c[k])) return false;
    }
    return true;
}

void enqueue_composite(int W, int H, const Layers& L, bool src_prev, const unsigned char* d_bg, int bgW, int bgH,
                       int bg_x, int bg_y, const float c[18], float2* d_flow, unsigned char* d_rgb,
                       unsigned char* d_mask, float2* d_bflow, unsigned char* d_occ, cudaStream_t stream)
{
    const unsigned blocks = (unsigned)(((size_t)W * H + 255) / 256);
    k_composite_b<<<blocks, 256, 0, stream>>>(W, H, L, d_bg, bgW, bgH, bg_x, bg_y, affine_of(c + 12), affine_of(c + 6),
                                              d_rgb, d_mask, d_bflow);
    if (src_prev) k_composite_a<true><<<blocks, 256, 0, stream>>>(W, H, L, affine_of(c), d_bflow, d_flow, d_occ);
    else k_composite_a<false><<<blocks, 256, 0, stream>>>(W, H, L, affine_of(c), d_bflow, d_flow, d_occ);
}

void enqueue_scene_input(int W, int H, const Layers& L, const unsigned char* d_rgb, const unsigned char* d_bg, int bgW,
                         int bgH, int bg_x, int bg_y, unsigned char* d_out, cudaStream_t stream)
{
    const unsigned blocks = (unsigned)(((size_t)W * H + 255) / 256);
    k_scene_input<<<blocks, 256, 0, stream>>>(W, H, L, d_rgb, d_bg, bgW, bgH, bg_x, bg_y, d_out);
}
} // namespace arapb200

namespace {
template <class T> bool all_set(const T* const* p, int n)
{
    if (!p) return false;
    for (int s = 0; s < n; ++s)
        if (!p[s]) return false;
    return true;
}
} // namespace

extern "C" int arapb200_composite(int W, int H, int n_layers, const float* const* flows, const uint8_t* const* rgbs,
                                  const uint8_t* const* masks, const uint8_t* const* src_masks,
                                  const float* const* bflows, int bgW, int bgH, const uint8_t* background, int bg_x,
                                  int bg_y, const double* motion_from, const double* motion_to, float* out_flow,
                                  uint8_t* out_rgb, uint8_t* out_mask, float* out_bflow, uint8_t* out_occ,
                                  float* out_coeffs)
{
    // every rejection comes before any CUDA call and any write
    if (W <= 0 || H <= 0 || n_layers < 0 || n_layers > MAX_LAYERS) return 1;
    const bool ex = out_bflow || out_occ;
    if (n_layers > 0 && (!all_set(flows, n_layers) || !all_set(rgbs, n_layers) || !all_set(masks, n_layers) ||
                         !all_set(src_masks, n_layers) || (ex && !all_set(bflows, n_layers))))
        return 1;
    if (!background || bgW <= 0 || bgH <= 0 || !motion_to || !out_flow || !out_rgb || !out_mask) return 1;
    float cf[18];
    if (!composite_coeffs(motion_from, motion_to, cf)) return 1;
    if (out_coeffs) std::copy(cf, cf + 18, out_coeffs);

    const size_t N = (size_t)W * H, NB = (size_t)bgW * bgH;
    // workspace: [layers: flow, rgb, mask, src mask (, bflow)][background][outputs: flow, rgb, mask (, bflow)(, occ)];
    // out_occ reads the whole frame-b bflow, so it has a block whenever either extra is asked for
    struct { size_t flow, rgb, mask, src, bflow; } in[MAX_LAYERS];
    Layout l;
    for (int s = 0; s < n_layers; ++s) {
        in[s].flow = l.take(8 * N);
        in[s].rgb = l.take(3 * N);
        in[s].mask = l.take(N);
        in[s].src = l.take(N);
        in[s].bflow = l.take(ex ? 8 * N : 0);
    }
    const size_t o_bg = l.take(3 * NB), o_flow = l.take(8 * N), o_rgb = l.take(3 * N), o_mask = l.take(N),
                 o_bflow = l.take(ex ? 8 * N : 0), o_occ = l.take(out_occ ? N : 0);
    return guarded([&]() -> int {
        Workspace& ws = composite_workspaces.current();
        std::lock_guard<std::mutex> lock(ws.mu);
        unsigned char* b = ws.buf.reserve(l.bytes());
        auto up = [&](size_t at, const void* h, size_t bytes) {
            ARAP_CUDA_CHECK(cudaMemcpyAsync(b + at, h, bytes, cudaMemcpyHostToDevice, nullptr));
            return b + at;
        };
        Layers L{};
        L.n = n_layers;
        for (int s = 0; s < n_layers; ++s) {
            L.flow[s] = (const float2*)up(in[s].flow, flows[s], 8 * N);
            L.rgb[s] = up(in[s].rgb, rgbs[s], 3 * N);
            L.mask[s] = up(in[s].mask, masks[s], N);
            L.src[s] = up(in[s].src, src_masks[s], N);
            if (ex) L.bflow[s] = (const float2*)up(in[s].bflow, bflows[s], 8 * N);
        }
        const unsigned char* d_bg = up(o_bg, background, 3 * NB);
        enqueue_composite(W, H, L, false, d_bg, bgW, bgH, bg_x, bg_y, cf, (float2*)(b + o_flow), b + o_rgb, b + o_mask,
                          ex ? (float2*)(b + o_bflow) : nullptr, out_occ ? b + o_occ : nullptr, nullptr);
        ARAP_CUDA_CHECK(cudaMemcpy(out_flow, b + o_flow, 8 * N, cudaMemcpyDeviceToHost));
        ARAP_CUDA_CHECK(cudaMemcpy(out_rgb, b + o_rgb, 3 * N, cudaMemcpyDeviceToHost));
        ARAP_CUDA_CHECK(cudaMemcpy(out_mask, b + o_mask, N, cudaMemcpyDeviceToHost));
        if (out_bflow) ARAP_CUDA_CHECK(cudaMemcpy(out_bflow, b + o_bflow, 8 * N, cudaMemcpyDeviceToHost));
        if (out_occ) ARAP_CUDA_CHECK(cudaMemcpy(out_occ, b + o_occ, N, cudaMemcpyDeviceToHost));
        return 0;
    });
}
