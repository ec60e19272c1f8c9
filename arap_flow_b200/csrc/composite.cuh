// composite.cuh -- the layer composite over a moving background (composite.cu, DESIGN.md 4.5), enqueue-only, for the
// callers that hold the layers on the device: arapb200_composite (its workspace) and the batch's scenes (DESIGN.md 4.6).
#pragma once
#include "common.cuh"

// fp-contract=off keeps a host compiler from fusing a product and a sum where the target has FMA: the host derivations
// of the maps (DESIGN.md 4.5) and of the blur schedule (4.8) are binary64 in a documented order
#if defined(__GNUC__) && !defined(__clang__)
#define ARAP_NO_CONTRACT __attribute__((optimize("fp-contract=off")))
#else
#define ARAP_NO_CONTRACT
#endif

namespace arapb200 {

constexpr int MAX_LAYERS = 32;
struct Layers {
    const float2* flow[MAX_LAYERS];
    const unsigned char* rgb[MAX_LAYERS];
    const unsigned char* mask[MAX_LAYERS];
    const float2* bflow[MAX_LAYERS];      // backward flow of each layer (only read for out_bflow / out_occ)
    const unsigned char* src[MAX_LAYERS]; // frame-a input mask of each layer, 0 = object (flatten: only read for out_occ)
    int n;
};

// F, B, S of DESIGN.md 4.5 rounded to binary32 (c[3][2][3]); motion_from NULL = identity.  false for a non-finite or
// singular motion or a non-finite coefficient.  Host only, no CUDA call.
bool composite_coeffs(const double* motion_from, const double* motion_to, float c[18]);

// k_composite_b then k_composite_a on `stream` with the maps c of composite_coeffs.  d_bflow is required when d_occ is
// given (the occlusion reads the whole frame-b backward flow).  src_prev: L.src holds frame k-1's warped masks and p is
// on layer s where it is 255 (frames k >= 2 of a sequence, DESIGN.md 4.6) instead of the input masks' 0.
void enqueue_composite(int W, int H, const Layers& L, bool src_prev, const unsigned char* d_bg, int bgW, int bgH,
                       int bg_x, int bg_y, const float c[18], float2* d_flow, unsigned char* d_rgb,
                       unsigned char* d_mask, float2* d_bflow, unsigned char* d_occ, cudaStream_t stream);

// frame 0 of a scene (k_scene_input): d_rgb where any layer's input mask L.src is 0, else the background at
// q + (bg_x, bg_y), coordinates clamped to the image as the composite clamps them
void enqueue_scene_input(int W, int H, const Layers& L, const unsigned char* d_rgb, const unsigned char* d_bg, int bgW,
                         int bgH, int bg_x, int bg_y, unsigned char* d_out, cudaStream_t stream);

#ifdef __CUDACC__
// a 2x3 map rounded to binary32, shared by the composite and the motion blur (DESIGN.md 4.5, 4.8)
struct Affine {
    float m00, m01, m02, m10, m11, m12;
};

__device__ __forceinline__ float2 affine_at(const Affine& M, int x, int y)
{
    const float fx = (float)x, fy = (float)y;
    return make_float2(__fadd_rn(__fadd_rn(__fmul_rn(M.m00, fx), __fmul_rn(M.m01, fy)), M.m02),
                       __fadd_rn(__fadd_rn(__fmul_rn(M.m10, fx), __fmul_rn(M.m11, fy)), M.m12));
}

// bilinear sample of the uint8x3 background at s, coordinates clamped to the image (NaN -> 0)
__device__ __forceinline__ void sample_bg(const unsigned char* __restrict__ bg, int bgW, int bgH, float2 s,
                                          unsigned char* __restrict__ out)
{
    const float sx = fminf(fmaxf(s.x, 0.f), (float)(bgW - 1)), sy = fminf(fmaxf(s.y, 0.f), (float)(bgH - 1));
    const int x0 = (int)floorf(sx), y0 = (int)floorf(sy);
    const int x1 = min(x0 + 1, bgW - 1), y1 = min(y0 + 1, bgH - 1);
    const float fx = __fsub_rn(sx, (float)x0), fy = __fsub_rn(sy, (float)y0);
    const float gx = __fsub_rn(1.f, fx), gy = __fsub_rn(1.f, fy);
    const unsigned char* r0 = bg + 3 * (size_t)y0 * bgW;
    const unsigned char* r1 = bg + 3 * (size_t)y1 * bgW;
    for (int c = 0; c < 3; ++c) {
        const float top = __fadd_rn(__fmul_rn((float)r0[3 * x0 + c], gx), __fmul_rn((float)r0[3 * x1 + c], fx));
        const float bot = __fadd_rn(__fmul_rn((float)r1[3 * x0 + c], gx), __fmul_rn((float)r1[3 * x1 + c], fx));
        out[c] = (unsigned char)min(255, __float2int_rn(__fadd_rn(__fmul_rn(top, gy), __fmul_rn(bot, fy))));
    }
}
#endif

} // namespace arapb200
