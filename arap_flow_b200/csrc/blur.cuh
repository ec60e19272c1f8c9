// blur.cuh -- motion blur of a scene's images from the continuation states (blur.cu, DESIGN.md 4.8), enqueue-only.
#pragma once
#include "composite.cuh"

namespace arapb200 {

constexpr int BLUR_MAX_SAMPLES = 64;

// One sub-frame of a blurred image: the layers at the lerp of continuation states j0 and j0 + 1 (-1 = the pixel grid)
// with weight w, over the background sampled through smap = inv(A(i)) rounded to binary32 (row-major 2x3).
struct BlurSub {
    int j0;
    float w;
    float smap[6];
};

// The n_samples sub-frames of one image of a scene (DESIGN.md 4.8): image -1 = frame 0, 0 = the pair, k = frame k of
// the n_frames frames at steps (motion A; frame_motions A_1 .. A_K).  false, with nothing written, for arguments outside
// the definition's ranges and for a sub-frame motion that is non-finite or singular or whose maps are non-finite.
// Host only, no CUDA call.
bool blur_schedule(int nCont, int n_frames, const int* steps, const double* motion, const double* frame_motions,
                   int n_samples, double shutter, int image, BlurSub* out);

// the layers of a scene in one sub-frame: positions lerped between qa and qb (null = the pixel grid), input masks
struct BlurLayers {
    const float2* qa[MAX_LAYERS];
    const float2* qb[MAX_LAYERS];
    const unsigned char* mask_red[MAX_LAYERS];
    int n;
};

#ifdef __CUDACC__
// Sub-frame j of S: clears the L.n z-buffers d_z[L.n][W*H], splats every layer into its own (k_blur_splat) and adds the
// sub-frame's colour into d_acc (k_blur_accum; sub-frame 0 stores, sub-frame S - 1 writes the rounded mean to d_out).
// Returns the kernels launched (2).
int enqueue_blur_subframe(int W, int H, const BlurLayers& L, float w, const float smap[6], const unsigned char* d_rgb,
                          const unsigned char* d_bg, int bgW, int bgH, int bg_x, int bg_y, unsigned* d_z,
                          ushort4* d_acc, int j, int S, unsigned char* d_out, cudaStream_t stream);
#endif

} // namespace arapb200
