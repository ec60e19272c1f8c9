// blur.cu -- motion blur of a scene's images (DESIGN.md 4.8): the mean of S sub-frame renders over the trailing shutter.
// A sub-frame is the scene's composite colour at intermediate geometry: every layer splatted at positions lerped between
// two continuation states (k_splat's rule, one z-buffer per layer), the front layer's colour resolved as k_resolve does,
// the background sampled through the sub-frame's inverse motion as k_composite_b does.  The helpers are the warp's and
// the composite's own (warp.cuh, composite.cuh), so each rule has one copy.  The mean is integer arithmetic on bytes,
// independent of any summation order.
#include "blur.cuh"
#include "warp.cuh"

#include <algorithm>
#include <cmath>

namespace arapb200 {
namespace {

// one component of the lerp: w == 0 and w == 1 select a state exactly (the other may hold anything)
__device__ __forceinline__ float lerp_rn(float a, float b, float w)
{
    return w == 0.f ? a : (w == 1.f ? b : __fadd_rn(a, __fmul_rn(w, __fsub_rn(b, a))));
}

__device__ __forceinline__ float2 blur_pos(const float2* qa, const float2* qb, float w, int W, size_t i)
{
    const float2 g = make_float2((float)(int)(i % W), (float)(int)(i / W));
    const float2 a = qa ? qa[i] : g, b = qb ? qb[i] : g;
    return make_float2(lerp_rn(a.x, b.x, w), lerp_rn(a.y, b.y, w));
}

// k_splat for layer blockIdx.z at the lerped positions, into its own z-buffer z[blockIdx.z]
__global__ void __launch_bounds__(256) k_blur_splat(int W, int H, BlurLayers L, float w, unsigned* __restrict__ z)
{
    const int s = blockIdx.z;
    const int x = blockIdx.x * 32 + (threadIdx.x & 31);
    const int y = blockIdx.y * 8 + (threadIdx.x >> 5);
    if (x + 1 >= W || y + 1 >= H) return;
    const size_t i00 = (size_t)y * W + x, i01 = i00 + 1, i10 = i00 + W, i11 = i10 + 1;
    const unsigned char* m = L.mask_red[s];
    if (m[i00] | m[i01] | m[i10] | m[i11]) return;
    const float2 *qa = L.qa[s], *qb = L.qb[s];
    const float2 p00 = blur_pos(qa, qb, w, W, i00), p01 = blur_pos(qa, qb, w, W, i01);
    const float2 p10 = blur_pos(qa, qb, w, W, i10), p11 = blur_pos(qa, qb, w, W, i11);
    const unsigned id = (unsigned)(2 * i00 + 1);
    unsigned* zs = z + (size_t)s * W * H;
    splat_tri(W, H, p00, p01, p10, id, zs);
    splat_tri(W, H, p10, p01, p11, id + 1, zs);
}

// one thread per pixel: the sub-frame's colour (front layer resolved at the lerped positions, else the background), added
// into acc; first: store instead of add; FINAL: write (sum + S/2) / S as bytes instead of storing the sum
template <bool FINAL>
__global__ void __launch_bounds__(256) k_blur_accum(int W, int H, BlurLayers L, float w, Affine S,
                                                     const unsigned* __restrict__ z, const unsigned char* __restrict__ rgb,
                                                     const unsigned char* __restrict__ bg, int bgW, int bgH, int bg_x,
                                                     int bg_y, bool first, int n_samples, ushort4* __restrict__ acc,
                                                     unsigned char* __restrict__ out)
{
    const size_t N = (size_t)W * H;
    const size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= N) return;
    const int qx = (int)(o % W), qy = (int)(o / W);
    int front = -1;
    unsigned id = 0;
    for (int s = L.n - 1; s >= 0; --s) {
        id = z[(size_t)s * N + o];
        if (id) {
            front = s;
            break;
        }
    }
    unsigned char c[3];
    if (front >= 0) {
        const Tri tr = tri_of(W, id);
        const float2 *qa = L.qa[front], *qb = L.qb[front];
        const float2 a = blur_pos(qa, qb, w, W, tr.ia), b = blur_pos(qa, qb, w, W, tr.ib),
                     cc = blur_pos(qa, qb, w, W, tr.ic);
        const Bary bw = lk(a.x, a.y, b.x, b.y, cc.x, cc.y, (float)qx, (float)qy);
#pragma unroll
        for (int k = 0; k < 3; ++k) { // k_resolve's colour and truncating cast
            const float ca = (float)rgb[3 * tr.ia + k], cb = (float)rgb[3 * tr.ib + k], cx = (float)rgb[3 * tr.ic + k];
            c[k] = (unsigned char)__float2int_rz(
                __fadd_rn(__fadd_rn(__fmul_rn(ca, bw.b0), __fmul_rn(cb, bw.b1)), __fmul_rn(cx, bw.b2)));
        }
    } else {
        const float2 s = affine_at(S, qx, qy);
        sample_bg(bg, bgW, bgH, make_float2(__fadd_rn(s.x, (float)bg_x), __fadd_rn(s.y, (float)bg_y)), c);
    }
    ushort4 a = first ? make_ushort4(0, 0, 0, 0) : acc[o];
    a.x += c[0];
    a.y += c[1];
    a.z += c[2];
    if (FINAL) {
        const unsigned h = (unsigned)n_samples / 2u;
        out[3 * o] = (unsigned char)((a.x + h) / (unsigned)n_samples);
        out[3 * o + 1] = (unsigned char)((a.y + h) / (unsigned)n_samples);
        out[3 * o + 2] = (unsigned char)((a.z + h) / (unsigned)n_samples);
    } else {
        acc[o] = a;
    }
}

} // namespace

ARAP_NO_CONTRACT bool blur_schedule(int nCont, int n_frames, const int* steps, const double* motion,
                                    const double* frame_motions, int n_samples, double shutter, int image, BlurSub* out)
{
    if (nCont < 1 || n_frames < 0 || !motion || (n_frames > 0 && (!steps || !frame_motions)) || n_samples < 1 ||
        n_samples > BLUR_MAX_SAMPLES || !(shutter >= 0.0 && shutter <= 1.0) || image < -1 || image > n_frames || !out)
        return false;
    for (int k = 0; k < n_frames; ++k)
        if (steps[k] < 0 || steps[k] >= nCont || (k > 0 && steps[k] <= steps[k - 1])) return false;
    static const double I[6] = {1.0, 0.0, 0.0, 0.0, 1.0, 0.0};
    // the image's knot i_hi, interval, motion at the knot and the previous knot's motion (DESIGN.md 4.8 table)
    int i_hi, delta;
    const double *A_hi, *A_prev;
    double D[6];
    if (image == 0) {
        i_hi = nCont - 1;
        delta = nCont;
        A_hi = motion;
        A_prev = I;
    } else if (image > 0) {
        i_hi = steps[image - 1];
        delta = i_hi - (image > 1 ? steps[image - 2] : -1);
        A_hi = frame_motions + 6 * (image - 1);
        A_prev = image > 1 ? frame_motions + 6 * (image - 2) : I;
    } else { // frame 0: extrapolated backwards at the first interval's velocity; no previous knot
        i_hi = -1;
        delta = n_frames > 0 ? steps[0] + 1 : nCont;
        A_hi = I;
        A_prev = nullptr;
    }
    const double* A_first = n_frames > 0 ? frame_motions : motion;
    for (int e = 0; e < 6; ++e) D[e] = A_prev ? A_prev[e] - A_hi[e] : I[e] - A_first[e];
    BlurSub tab[BLUR_MAX_SAMPLES];
    for (int j = 0; j < n_samples; ++j) {
        const double u = n_samples == 1 ? 0.0 : (shutter * j) / (n_samples - 1);
        const double i = i_hi - u * delta;
        double A[6];
        for (int e = 0; e < 6; ++e) A[e] = (A_prev && u == 1.0) ? A_prev[e] : A_hi[e] + u * D[e];
        float c[18];
        if (!composite_coeffs(nullptr, A, c)) return false;
        const int j0 = std::min(std::max((int)std::floor(i), -1), nCont - 2);
        tab[j].j0 = j0;
        tab[j].w = (float)(i - j0);
        std::copy(c + 12, c + 18, tab[j].smap);
    }
    std::copy(tab, tab + n_samples, out);
    return true;
}

int enqueue_blur_subframe(int W, int H, const BlurLayers& L, float w, const float smap[6], const unsigned char* d_rgb,
                          const unsigned char* d_bg, int bgW, int bgH, int bg_x, int bg_y, unsigned* d_z,
                          ushort4* d_acc, int j, int S, unsigned char* d_out, cudaStream_t stream)
{
    const size_t N = (size_t)W * H;
    ARAP_CUDA_CHECK(cudaMemsetAsync(d_z, 0, (size_t)L.n * N * sizeof(unsigned), stream));
    const dim3 g1((W + 31) / 32, (H + 7) / 8, L.n);
    k_blur_splat<<<g1, 256, 0, stream>>>(W, H, L, w, d_z);
    const unsigned g2 = (unsigned)((N + 255) / 256);
    const Affine M{smap[0], smap[1], smap[2], smap[3], smap[4], smap[5]};
    if (j == S - 1)
        k_blur_accum<true><<<g2, 256, 0, stream>>>(W, H, L, w, M, d_z, d_rgb, d_bg, bgW, bgH, bg_x, bg_y, j == 0, S,
                                                   d_acc, d_out);
    else
        k_blur_accum<false><<<g2, 256, 0, stream>>>(W, H, L, w, M, d_z, d_rgb, d_bg, bgW, bgH, bg_x, bg_y, j == 0, S,
                                                    d_acc, d_out);
    ARAP_CUDA_CHECK(cudaGetLastError());
    return 2;
}

} // namespace arapb200
