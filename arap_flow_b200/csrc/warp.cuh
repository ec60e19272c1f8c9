// warp.cuh -- forward-warp kernels (see warp.cu).  Device pointers, enqueue-only.
#pragma once
#include "common.cuh"

namespace arapb200 {

// z: uint32[W*H] scratch that ends up holding the splat index (1 + 2*(y*W+x) + t, 0 = empty).
// d_out_bflow (may be null): float2[W*H] backward flow, source point of every frame-2 pixel minus the pixel (DESIGN.md 4.3)
void enqueue_warp(int W, int H, const float2* d_pos, const unsigned char* d_rgb, const unsigned char* d_mask_red,
                  unsigned* d_z, unsigned char* d_out_rgb, unsigned char* d_out_mask, cudaStream_t stream,
                  float2* d_out_bflow = nullptr);
// occlusion of frame 1 (0 = visible in frame 2, 255 = not), from the z-buffer and backward flow enqueue_warp left and the
// forward flow d_flow = X - grid
void enqueue_occlusion(int W, int H, const unsigned char* d_mask_red, const float2* d_flow, const unsigned* d_z,
                       const float2* d_bflow, unsigned char* d_occ, cudaStream_t stream);
// Frame sequences (DESIGN.md 4.4).  Every buffer is [K][W*H][...] on the device; frame k (1-based) sits at index k - 1.
struct SeqOut {
    unsigned char *rgb, *mask; // warp of P_k (uint8x3, uint8)
    float2 *flow, *bflow;      // frame k - 1 -> k on the frame k - 1 grid; frame k -> k - 1 on the frame k grid
    unsigned char* occ;        // occlusion of frame k - 1 in frame k (0 visible, 255 not)
    float2* flow0;             // P_k - grid
};
// d_pos: the K position fields P_1 .. P_K (frame 0 is the grid); d_z2: uint32[2][W*H] scratch (the z-buffers of two
// consecutive frames).  Frames are rendered in order.  Returns the number of kernels launched.
int enqueue_warp_seq(int W, int H, int K, const float2* d_pos, const unsigned char* d_rgb,
                     const unsigned char* d_mask_red, unsigned* d_z2, const SeqOut& out, cudaStream_t stream);
void enqueue_flow_to_pos(int W, int H, const float2* d_flow, float2* d_pos, cudaStream_t stream);
void enqueue_pos_to_flow(int W, int H, const float2* d_pos, float2* d_flow, cudaStream_t stream);
int warp_launches_per_call();

#ifdef __CUDACC__
struct Bary {
    float b0, b1, b2;
    bool in;
};

// PointInTriangleLK with w0 = w1 = w2 = 1 (main.cpp:68-104), operation for operation.
__device__ __forceinline__ Bary lk(float x0, float y0, float x1, float y1, float x2, float y2, float sx, float sy)
{
    const float X0 = __fsub_rn(x0, sx), X1 = __fsub_rn(x1, sx), X2 = __fsub_rn(x2, sx);
    const float Y0 = __fsub_rn(y0, sy), Y1 = __fsub_rn(y1, sy), Y2 = __fsub_rn(y2, sy);
    float d01 = __fsub_rn(__fmul_rn(X0, Y1), __fmul_rn(Y0, X1));
    float d12 = __fsub_rn(__fmul_rn(X1, Y2), __fmul_rn(Y1, X2));
    float d20 = __fsub_rn(__fmul_rn(X2, Y0), __fmul_rn(Y2, X0));
    Bary r;
    r.in = false;
    r.b0 = r.b1 = r.b2 = 0.f;
    if ((d01 < 0.f) & (d12 < 0.f) & (d20 < 0.f)) return r; // backfacing
    const float inv = __fdiv_rn(1.f, __fadd_rn(__fadd_rn(d01, d12), d20));
    d01 = __fmul_rn(d01, inv);
    d12 = __fmul_rn(d12, inv);
    d20 = __fmul_rn(d20, inv);
    r.b0 = d12;
    r.b1 = d20;
    r.b2 = d01;
    r.in = (d01 >= 0.f && d12 >= 0.f && d20 >= 0.f); // NaN => not covered
    return r;
}

// atomicMax of id into z over every pixel of the image the triangle (a, b, c) covers
__device__ __forceinline__ void splat_tri(int W, int H, float2 a, float2 b, float2 c, unsigned id, unsigned* z)
{
    // bbox floor(min) .. ceil(max) inclusive, clipped to the image (main.cpp:123-127)
    float minx = floorf(fminf(a.x, fminf(b.x, c.x))), miny = floorf(fminf(a.y, fminf(b.y, c.y)));
    float maxx = ceilf(fmaxf(a.x, fmaxf(b.x, c.x))), maxy = ceilf(fmaxf(a.y, fmaxf(b.y, c.y)));
    if (!(minx > -1e9f)) minx = -1e9f;
    if (!(miny > -1e9f)) miny = -1e9f;
    if (!(maxx < 1e9f)) maxx = 1e9f;
    if (!(maxy < 1e9f)) maxy = 1e9f;
    const int xs = max(0, (int)minx), ys = max(0, (int)miny);
    const int xe = min(W - 1, (int)maxx), ye = min(H - 1, (int)maxy);
    for (int y = ys; y <= ye; ++y)
        for (int x = xs; x <= xe; ++x)
            if (lk(a.x, a.y, b.x, b.y, c.x, c.y, (float)x, (float)y).in) atomicMax(&z[(size_t)y * W + x], id);
}

// vertices of the triangle a splat index names: (x0, y0 + t), (x0 + 1, y0), (x0 + t, y0 + 1) as pixel indices
struct Tri {
    size_t ia, ib, ic;
};
__device__ __forceinline__ Tri tri_of(int W, unsigned id)
{
    const unsigned t = (id - 1) & 1u;
    const size_t i00 = (id - 1) >> 1, i01 = i00 + 1, i10 = i00 + W, i11 = i10 + 1;
    return Tri{t ? i10 : i00, i01, t ? i11 : i10};
}

// The occlusion rule of DESIGN.md 4.3 for frame-1 pixel p = (px, py), shared by the per-problem kernel and the layer
// flatten.  seg: p's surface (-1 = background); f: p's forward flow; bflow: backward flow of p's surface;
// owner(q): the surface that is in front at frame-2 pixel q (-1 = nothing landed).  Returns 0 (visible) or 255.
template <class Owner>
__device__ __forceinline__ unsigned char occlusion_of(int W, int H, int px, int py, int seg, float2 f,
                                                      const float2* __restrict__ bflow, Owner owner)
{
    if (seg < 0) return owner((size_t)py * W + px) < 0 ? 0 : 255; // static background: visible unless covered
    const float tx = __fadd_rn(__fadd_rn((float)px, f.x), 0.5f), ty = __fadd_rn(__fadd_rn((float)py, f.y), 0.5f);
    if (!(tx >= 0.f && tx < (float)W && ty >= 0.f && ty < (float)H)) return 255; // left the frame (or NaN)
    const int qx = (int)floorf(tx), qy = (int)floorf(ty);
    const size_t q = (size_t)qy * W + qx;
    if (owner(q) != seg) return 255;
    const float2 b = bflow[q];
    const float ex = __fadd_rn(b.x, (float)(qx - px)), ey = __fadd_rn(b.y, (float)(qy - py));
    return (fabsf(ex) < 1.f && fabsf(ey) < 1.f) ? 0 : 255;
}
#endif

} // namespace arapb200
