// composite.cuh -- the layer composite over a moving background (composite.cu, DESIGN.md 4.5), enqueue-only, for the
// callers that hold the layers on the device: arapb200_composite (its workspace) and the batch's scenes (DESIGN.md 4.6).
#pragma once
#include "common.cuh"

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

} // namespace arapb200
