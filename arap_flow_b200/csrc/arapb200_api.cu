// arapb200_api.cu -- the flat C ABI of include/arapb200.h (host buffers in, host buffers out).
#include "../../include/arapb200.h"
#include "composite.cuh"
#include "devmem.cuh"
#include "pipeline.cuh"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <memory>
#include <mutex>
#include <vector>

using namespace arapb200;

namespace {

// the stand-alone warp calls (warp_image, the Opt.h mirror's copyResultToCPU), each on its device's non-blocking stream
WorkspaceTable warp_workspaces;

int warp_common(int W, int H, const float* pos_or_flow, bool is_flow, const uint8_t* rgb, const uint8_t* mask_red,
                uint8_t* out_rgb, uint8_t* out_mask, uint32_t* out_splat, float* out_bflow = nullptr,
                uint8_t* out_occ = nullptr)
{
    if (W <= 0 || H <= 0 || !pos_or_flow || !rgb || !mask_red || !out_rgb || !out_mask) return 1;
    const size_t N = (size_t)W * H;
    const bool ex = out_bflow || out_occ; // the occlusion needs the backward flow
    Layout l;
    const size_t o_in = l.take(8 * N), o_pos = l.take(8 * N), o_z = l.take(4 * N), o_rgb = l.take(3 * N),
                 o_orgb = l.take(3 * N), o_m = l.take(N), o_om = l.take(N), o_bf = l.take(ex ? 8 * N : 0),
                 o_fl = l.take(out_occ ? 8 * N : 0), o_occ = l.take(out_occ ? N : 0);
    Workspace& ws = warp_workspaces.current();
    std::lock_guard<std::mutex> g(ws.mu);
    unsigned char* b = ws.buf.reserve(l.bytes());
    cudaStream_t s = ws.stream();
    float2* d_in = (float2*)(b + o_in);
    float2* d_pos = (float2*)(b + o_pos);
    unsigned* d_z = (unsigned*)(b + o_z);
    float2* d_bf = ex ? (float2*)(b + o_bf) : nullptr;
    ARAP_CUDA_CHECK(cudaMemcpyAsync(d_in, pos_or_flow, 8 * N, cudaMemcpyHostToDevice, s));
    ARAP_CUDA_CHECK(cudaMemcpyAsync(b + o_rgb, rgb, 3 * N, cudaMemcpyHostToDevice, s));
    ARAP_CUDA_CHECK(cudaMemcpyAsync(b + o_m, mask_red, N, cudaMemcpyHostToDevice, s));
    const float2* pos = d_in;
    if (is_flow) {
        enqueue_flow_to_pos(W, H, d_in, d_pos, s);
        pos = d_pos;
    }
    enqueue_warp(W, H, pos, b + o_rgb, b + o_m, d_z, b + o_orgb, b + o_om, s, d_bf);
    if (out_occ) {
        const float2* flow = d_in; // forward flow: given, or X - grid exactly as the batch path extracts it
        if (!is_flow) {
            enqueue_pos_to_flow(W, H, d_in, (float2*)(b + o_fl), s);
            flow = (const float2*)(b + o_fl);
        }
        enqueue_occlusion(W, H, b + o_m, flow, d_z, d_bf, b + o_occ, s);
        ARAP_CUDA_CHECK(cudaMemcpyAsync(out_occ, b + o_occ, N, cudaMemcpyDeviceToHost, s));
    }
    ARAP_CUDA_CHECK(cudaMemcpyAsync(out_rgb, b + o_orgb, 3 * N, cudaMemcpyDeviceToHost, s));
    ARAP_CUDA_CHECK(cudaMemcpyAsync(out_mask, b + o_om, N, cudaMemcpyDeviceToHost, s));
    if (out_splat) ARAP_CUDA_CHECK(cudaMemcpyAsync(out_splat, d_z, 4 * N, cudaMemcpyDeviceToHost, s));
    if (out_bflow) ARAP_CUDA_CHECK(cudaMemcpyAsync(out_bflow, d_bf, 8 * N, cudaMemcpyDeviceToHost, s));
    ARAP_CUDA_OR_RETURN(cudaStreamSynchronize(s));
    return 0;
}

// forget a slot's tracks request (DESIGN.md 4.9)
void drop_tracks(HostProblem& hp)
{
    hp.tracks = false;
    hp.trk_flow0 = hp.trk_bflow0 = nullptr;
    hp.trk_occ0 = nullptr;
    hp.queries.clear();
    hp.query_pos = nullptr;
    hp.query_occ = nullptr;
}

} // namespace

struct arapb200_batch {
    int maxW, maxH, max_problems, nCont, nGN, nPCG, backend;
    std::unique_ptr<BatchPipeline> pipe;
    std::vector<HostProblem> slots;
    std::vector<char> pending;
    std::vector<HostProblem> todo;
    // scenes queued for the next run (HostScene::first holds the first slot until run() maps it into todo) and, per
    // slot, the queued scene that owns it (-1 = none)
    std::vector<HostScene> scenes;
    std::vector<int> scene_of;
    float ms[3] = {0, 0, 0};
    long long launches = 0;
};

extern "C" {

const char* arapb200_version(void) { return "arapb200 0.1.0 (sm_100a)"; }

int arapb200_device_info(int* sm_count, size_t* l2_bytes, int* cc_major, int* cc_minor)
{
    return guarded([&]() -> int {
        int dev = 0;
        ARAP_CUDA_OR_RETURN(cudaGetDevice(&dev));
        cudaDeviceProp p;
        ARAP_CUDA_OR_RETURN(cudaGetDeviceProperties(&p, dev));
        if (sm_count) *sm_count = p.multiProcessorCount;
        if (l2_bytes) *l2_bytes = (size_t)p.l2CacheSize;
        if (cc_major) *cc_major = p.major;
        if (cc_minor) *cc_minor = p.minor;
        return 0;
    });
}

int arapb200_warp(int W, int H, const float* pos, const uint8_t* rgb, const uint8_t* mask_red, uint8_t* out_rgb,
                  uint8_t* out_mask, uint32_t* out_splat)
{
    return guarded([&]() -> int {
        return warp_common(W, H, pos, false, rgb, mask_red, out_rgb, out_mask, out_splat);
    });
}

int arapb200_warp_flow(int W, int H, const float* flow, const uint8_t* rgb, const uint8_t* mask_red,
                       uint8_t* out_rgb, uint8_t* out_mask, uint32_t* out_splat)
{
    return guarded([&]() -> int {
        return warp_common(W, H, flow, true, rgb, mask_red, out_rgb, out_mask, out_splat);
    });
}

int arapb200_warp_ex(int W, int H, const float* pos_or_flow, int is_flow, const uint8_t* rgb, const uint8_t* mask_red,
                     uint8_t* out_rgb, uint8_t* out_mask, uint32_t* out_splat, float* out_bflow, uint8_t* out_occ)
{
    return guarded([&]() -> int {
        return warp_common(W, H, pos_or_flow, is_flow != 0, rgb, mask_red, out_rgb, out_mask, out_splat, out_bflow,
                           out_occ);
    });
}

int arapb200_warp_seq(int W, int H, int K, const float* pos, const uint8_t* rgb, const uint8_t* mask_red,
                      uint8_t* out_rgb, uint8_t* out_mask, float* out_flow, float* out_bflow, uint8_t* out_occ,
                      float* out_flow0)
{
    return guarded([&]() -> int {
        if (W <= 0 || H <= 0 || K <= 0 || !pos || !rgb || !mask_red || !out_rgb || !out_mask) return 1;
        const size_t N = (size_t)W * H, F = N * K;
        DevBuf<float2> d_pos(F), d_flow(F), d_bflow(F), d_flow0(F);
        DevBuf<unsigned char> d_rgb(3 * N), d_mask(N), d_orgb(3 * F), d_omask(F), d_occ(F);
        DevBuf<unsigned> d_z(2 * N);
        d_pos.up((const float2*)pos);
        d_rgb.up(rgb);
        d_mask.up(mask_red);
        const SeqOut o{d_orgb.p, d_omask.p, d_flow.p, d_bflow.p, d_occ.p, d_flow0.p};
        enqueue_warp_seq(W, H, K, d_pos.p, d_rgb.p, d_mask.p, d_z.p, o, nullptr);
        d_orgb.down(out_rgb);
        d_omask.down(out_mask);
        if (out_flow) d_flow.down((float2*)out_flow);
        if (out_bflow) d_bflow.down((float2*)out_bflow);
        if (out_occ) d_occ.down(out_occ);
        if (out_flow0) d_flow0.down((float2*)out_flow0);
        ARAP_CUDA_OR_RETURN(cudaDeviceSynchronize());
        return 0;
    });
}

int arapb200_warp_tracks(int W, int H, int K, const float* pos, const uint8_t* mask_red, float* out_bflow0,
                         uint8_t* out_occ0)
{
    return guarded([&]() -> int {
        if (W <= 0 || H <= 0 || K <= 0 || !pos || !mask_red) return 1;
        // the batch's kernels: enqueue_warp_seq with the tracks of DESIGN.md 4.9 (colours are not asked for: black rgb)
        const size_t N = (size_t)W * H, F = N * K;
        DevBuf<float2> d_pos(F), d_flow(F), d_bflow(F), d_flow0(F), d_bflow0(F);
        DevBuf<unsigned char> d_rgb(3 * N), d_mask(N), d_orgb(3 * F), d_omask(F), d_occ(F), d_occ0(F);
        DevBuf<unsigned> d_z(2 * N);
        d_pos.up((const float2*)pos);
        d_mask.up(mask_red);
        ARAP_CUDA_OR_RETURN(cudaMemsetAsync(d_rgb.p, 0, 3 * N, nullptr));
        const SeqOut o{d_orgb.p, d_omask.p, d_flow.p, d_bflow.p, d_occ.p, d_flow0.p, d_bflow0.p, d_occ0.p};
        enqueue_warp_seq(W, H, K, d_pos.p, d_rgb.p, d_mask.p, d_z.p, o, nullptr);
        if (out_bflow0) d_bflow0.down((float2*)out_bflow0);
        if (out_occ0) d_occ0.down(out_occ0);
        ARAP_CUDA_OR_RETURN(cudaDeviceSynchronize());
        return 0;
    });
}

int arapb200_deform(int W, int H, const uint8_t* rgb, const uint8_t* mask_red, const int32_t* matches, int n_matches,
                    int nCont, int nGN, int nPCG, int backend, float* out_flow, uint8_t* out_rgb, uint8_t* out_mask,
                    float* out_costs)
{
    return guarded([&]() -> int {
        if (W <= 0 || H <= 0 || !rgb || !mask_red || (n_matches > 0 && !matches)) return 1;
        BatchPipeline pipe(W, H, 1, nCont, nGN, nPCG, backend);
        HostProblem hp;
        hp.W = W; hp.H = H; hp.rgb = rgb; hp.mask_red = mask_red; hp.matches = matches; hp.n_matches = n_matches;
        hp.out_flow = out_flow; hp.out_rgb = out_rgb; hp.out_mask = out_mask; hp.out_costs = out_costs;
        return pipe.run(&hp, 1);
    });
}

arapb200_batch* arapb200_batch_create(int maxW, int maxH, int max_problems, int nCont, int nGN, int nPCG, int backend)
{
    if (maxW <= 0 || maxH <= 0 || max_problems <= 0) return nullptr;
    if (nCont < 0 || nGN < 0 || nPCG < 0 || backend < ARAPB200_BACKEND_AUTO || backend > ARAPB200_BACKEND_RESIDENT) return nullptr;
    arapb200_batch* b = nullptr;
    const int rc = guarded([&]() -> int {
        b = new arapb200_batch;
        b->maxW = maxW; b->maxH = maxH; b->max_problems = max_problems;
        b->nCont = nCont; b->nGN = nGN; b->nPCG = nPCG; b->backend = backend;
        b->pipe.reset(new BatchPipeline(maxW, maxH, max_problems, nCont, nGN, nPCG, backend));
        b->slots.resize(max_problems);
        b->pending.assign(max_problems, 0);
        b->scene_of.assign(max_problems, -1);
        return 0;
    });
    if (rc) { delete b; return nullptr; }
    return b;
}

void arapb200_batch_destroy(arapb200_batch* b) { delete b; }

int arapb200_batch_submit(arapb200_batch* b, int slot, int W, int H, const uint8_t* rgb, const uint8_t* mask_red,
                          const int32_t* matches, int n_matches, float* out_flow, uint8_t* out_rgb,
                          uint8_t* out_mask, float* out_costs)
{
    return arapb200_batch_submit_ex(b, slot, W, H, rgb, mask_red, matches, n_matches, out_flow, out_rgb, out_mask,
                                    out_costs, nullptr, nullptr);
}

int arapb200_batch_submit_ex(arapb200_batch* b, int slot, int W, int H, const uint8_t* rgb, const uint8_t* mask_red,
                             const int32_t* matches, int n_matches, float* out_flow, uint8_t* out_rgb,
                             uint8_t* out_mask, float* out_costs, float* out_bflow, uint8_t* out_occ)
{
    return arapb200_batch_submit_seq(b, slot, W, H, rgb, mask_red, matches, n_matches, out_flow, out_rgb, out_mask,
                                     out_costs, out_bflow, out_occ, 0, nullptr, nullptr, nullptr, nullptr, nullptr,
                                     nullptr, nullptr);
}

int arapb200_batch_submit_seq(arapb200_batch* b, int slot, int W, int H, const uint8_t* rgb, const uint8_t* mask_red,
                              const int32_t* matches, int n_matches, float* out_flow, uint8_t* out_rgb,
                              uint8_t* out_mask, float* out_costs, float* out_bflow, uint8_t* out_occ, int n_frames,
                              const int* steps, uint8_t* seq_rgb, uint8_t* seq_mask, float* seq_flow,
                              float* seq_bflow, uint8_t* seq_occ, float* seq_flow0)
{
    return guarded([&]() -> int {
        if (!b || slot < 0 || slot >= b->max_problems) return 1;
        if (b->scene_of[slot] >= 0) {
            fprintf(stderr, "arapb200: batch_submit: slot %d belongs to a scene queued for the next run\n", slot);
            return 1;
        }
        // everything run() will dereference is checked here, while the caller can still be told
        if (W <= 0 || H <= 0 || (size_t)W * H > (size_t)b->maxW * b->maxH || !rgb || !mask_red || n_matches < 0 ||
            (n_matches > 0 && !matches)) {
            fprintf(stderr, "arapb200: batch_submit: bad problem (%dx%d in a %dx%d batch, %d matches, null input?)\n", W, H,
                    b->maxW, b->maxH, n_matches);
            return 1;
        }
        const bool any_out = seq_rgb || seq_mask || seq_flow || seq_bflow || seq_occ || seq_flow0;
        if (n_frames < 0 || (n_frames == 0 && any_out) || (n_frames > 0 && (!steps || !seq_rgb || !seq_mask))) {
            fprintf(stderr, "arapb200: batch_submit_seq: %d frames with%s step list and%s outputs (rgb and mask required)\n",
                    n_frames, steps ? "" : " no", any_out ? "" : " no");
            return 1;
        }
        for (int k = 0; k < n_frames; ++k)
            if (steps[k] < 0 || steps[k] >= b->nCont || (k > 0 && steps[k] <= steps[k - 1])) {
                fprintf(stderr, "arapb200: batch_submit_seq: steps must increase strictly within [0, %d]; step %d is %d\n",
                        b->nCont - 1, k, steps[k]);
                return 1;
            }
        HostProblem& hp = b->slots[slot];
        hp.W = W; hp.H = H; hp.rgb = rgb; hp.mask_red = mask_red; hp.matches = matches; hp.n_matches = n_matches;
        hp.out_flow = out_flow; hp.out_rgb = out_rgb; hp.out_mask = out_mask; hp.out_costs = out_costs;
        hp.out_bflow = out_bflow; hp.out_occ = out_occ;
        hp.steps.assign(steps, steps + n_frames);
        hp.seq_rgb = seq_rgb; hp.seq_mask = seq_mask; hp.seq_flow = seq_flow; hp.seq_bflow = seq_bflow;
        hp.seq_occ = seq_occ; hp.seq_flow0 = seq_flow0;
        hp.scene = false; // the slot may have been a scene layer in an earlier run
        drop_tracks(hp); // a new problem drops an earlier tracks request
        b->pending[slot] = 1;
        return 0;
    });
}

int arapb200_batch_submit_scene(arapb200_batch* b, int slot, int n_layers, int W, int H, const uint8_t* rgb,
                                const uint8_t* const* masks_red, const int32_t* const* matches, const int* n_matches,
                                int bgW, int bgH, const uint8_t* background, int bg_x, int bg_y, const double* motion,
                                int n_frames, const int* steps, const double* frame_motions, float* out_flow,
                                uint8_t* out_rgb, uint8_t* out_mask, float* out_bflow, uint8_t* out_occ, uint8_t* out_rgb0,
                                float* out_costs, uint8_t* seq_rgb, uint8_t* seq_mask, float* seq_flow, float* seq_bflow,
                                uint8_t* seq_occ)
{
    return guarded([&]() -> int {
        // every rejection comes before anything is queued
        if (!b || n_layers < 1 || n_layers > MAX_LAYERS || slot < 0 || slot > b->max_problems - n_layers) return 1;
        for (int s = slot; s < slot + n_layers; ++s)
            if (b->scene_of[s] >= 0) {
                fprintf(stderr, "arapb200: batch_submit_scene: slot %d belongs to another queued scene\n", s);
                return 1;
            }
        if (W <= 0 || H <= 0 || (size_t)W * H > (size_t)b->maxW * b->maxH || !rgb || !masks_red || !matches ||
            !n_matches) {
            fprintf(stderr, "arapb200: batch_submit_scene: bad scene (%dx%d in a %dx%d batch, null input?)\n", W, H,
                    b->maxW, b->maxH);
            return 1;
        }
        for (int s = 0; s < n_layers; ++s)
            if (!masks_red[s] || n_matches[s] < 0 || (n_matches[s] > 0 && !matches[s])) {
                fprintf(stderr, "arapb200: batch_submit_scene: layer %d: null mask or bad match list\n", s);
                return 1;
            }
        if (!background || bgW <= 0 || bgH <= 0 || !motion || !out_flow || !out_rgb || !out_mask) {
            fprintf(stderr, "arapb200: batch_submit_scene: null background, motion or pair output, or bad background size\n");
            return 1;
        }
        const bool any_out = seq_rgb || seq_mask || seq_flow || seq_bflow || seq_occ;
        if (n_frames < 0 || (n_frames == 0 && any_out) ||
            (n_frames > 0 && (!steps || !frame_motions || !seq_rgb || !seq_mask))) {
            fprintf(stderr, "arapb200: batch_submit_scene: %d frames with%s step list,%s motions and%s outputs (rgb and "
                    "mask required)\n", n_frames, steps ? "" : " no", frame_motions ? "" : " no", any_out ? "" : " no");
            return 1;
        }
        for (int k = 0; k < n_frames; ++k)
            if (steps[k] < 0 || steps[k] >= b->nCont || (k > 0 && steps[k] <= steps[k - 1])) {
                fprintf(stderr, "arapb200: batch_submit_scene: steps must increase strictly within [0, %d]; step %d is %d\n",
                        b->nCont - 1, k, steps[k]);
                return 1;
            }
        HostScene sc;
        sc.maps.resize(18 * (size_t)(1 + n_frames));
        bool ok = composite_coeffs(nullptr, motion, sc.maps.data());
        for (int k = 0; k < n_frames && ok; ++k) // frame k + 1: A_k -> A_{k+1}, A_0 = identity
            ok = composite_coeffs(k == 0 ? nullptr : frame_motions + 6 * (k - 1), frame_motions + 6 * k,
                                  sc.maps.data() + 18 * (k + 1));
        if (!ok) {
            fprintf(stderr, "arapb200: batch_submit_scene: non-finite or singular motion\n");
            return 1;
        }
        sc.first = slot;
        sc.n = n_layers;
        sc.W = W; sc.H = H;
        sc.background = background; sc.bgW = bgW; sc.bgH = bgH; sc.bg_x = bg_x; sc.bg_y = bg_y;
        sc.out_flow = out_flow; sc.out_rgb = out_rgb; sc.out_mask = out_mask; sc.out_bflow = out_bflow;
        sc.out_occ = out_occ; sc.out_rgb0 = out_rgb0;
        sc.seq_rgb = seq_rgb; sc.seq_mask = seq_mask; sc.seq_flow = seq_flow; sc.seq_bflow = seq_bflow;
        sc.seq_occ = seq_occ;
        sc.motions.assign(motion, motion + 6);
        if (n_frames > 0) sc.motions.insert(sc.motions.end(), frame_motions, frame_motions + 6 * (size_t)n_frames);
        const size_t cn = (size_t)b->nCont * (b->nGN + 1);
        for (int s = 0; s < n_layers; ++s) {
            HostProblem& hp = b->slots[slot + s];
            hp = HostProblem{};
            hp.W = W; hp.H = H; hp.rgb = rgb; hp.mask_red = masks_red[s]; hp.matches = matches[s];
            hp.n_matches = n_matches[s];
            hp.out_costs = out_costs ? out_costs + cn * s : nullptr;
            hp.steps.assign(steps, steps + n_frames);
            hp.scene = true;
            b->pending[slot + s] = 1;
            b->scene_of[slot + s] = (int)b->scenes.size();
        }
        b->scenes.push_back(std::move(sc));
        return 0;
    });
}

int arapb200_batch_scene_blur(arapb200_batch* b, int slot, int n_samples, double shutter, uint8_t* blur_rgb,
                              uint8_t* blur_rgb0, uint8_t* seq_blur_rgb)
{
    return guarded([&]() -> int {
        // every rejection comes before the scene is changed
        if (!b || slot < 0 || slot >= b->max_problems) return 1;
        const int q = b->scene_of[slot];
        if (q < 0 || b->scenes[q].first != slot) {
            fprintf(stderr, "arapb200: batch_scene_blur: slot %d is not the first slot of a queued scene\n", slot);
            return 1;
        }
        HostScene& sc = b->scenes[q];
        const int K = (int)(sc.maps.size() / 18) - 1;
        if (n_samples < 1 || n_samples > BLUR_MAX_SAMPLES || !(shutter >= 0.0 && shutter <= 1.0) || !blur_rgb ||
            (blur_rgb0 && !sc.out_rgb0) || (seq_blur_rgb && K == 0)) {
            fprintf(stderr, "arapb200: batch_scene_blur: bad request (%d samples, shutter %g, null blur_rgb, or a frame-0 "
                    "or frame output the scene does not have)\n", n_samples, shutter);
            return 1;
        }
        const std::vector<int>& steps = b->slots[slot].steps;
        std::vector<BlurSub> tab((size_t)(K + 2) * n_samples);
        for (int image = -1; image <= K; ++image) {
            if ((image < 0 && !blur_rgb0) || (image > 0 && !seq_blur_rgb)) continue;
            if (!blur_schedule(b->nCont, K, steps.data(), sc.motions.data(), sc.motions.data() + 6, n_samples, shutter,
                               image, tab.data() + (size_t)(image + 1) * n_samples)) {
                fprintf(stderr, "arapb200: batch_scene_blur: image %d has a non-finite or singular sub-frame motion\n",
                        image);
                return 1;
            }
        }
        std::vector<int> states; // what the sub-frames read: j0 unless w == 1, j0 + 1 unless w == 0; never the grid
        for (int image = -1; image <= K; ++image) {
            if ((image < 0 && !blur_rgb0) || (image > 0 && !seq_blur_rgb)) continue;
            for (int j = 0; j < n_samples; ++j) {
                const BlurSub& e = tab[(size_t)(image + 1) * n_samples + j];
                if (e.w != 1.f && e.j0 >= 0) states.push_back(e.j0);
                if (e.w != 0.f) states.push_back(e.j0 + 1);
            }
        }
        std::sort(states.begin(), states.end());
        states.erase(std::unique(states.begin(), states.end()), states.end());
        sc.blur_S = n_samples;
        sc.blur.swap(tab);
        sc.blur_states.swap(states);
        sc.blur_rgb = blur_rgb;
        sc.blur_rgb0 = blur_rgb0;
        sc.seq_blur_rgb = seq_blur_rgb;
        return 0;
    });
}

int arapb200_batch_tracks(arapb200_batch* b, int slot, float* flow0, float* bflow0, uint8_t* occ0, int n_queries,
                          const int32_t* queries, float* query_pos, uint8_t* query_occ)
{
    return guarded([&]() -> int {
        // every rejection comes before anything is changed
        if (!b || slot < 0 || slot >= b->max_problems) return 1;
        const int q = b->scene_of[slot];
        HostScene* sc = q >= 0 && b->scenes[q].first == slot ? &b->scenes[q] : nullptr;
        HostProblem& hp = b->slots[slot];
        const bool plain = q < 0 && b->pending[slot] && !hp.scene;
        const int K = sc ? (int)(sc->maps.size() / 18) - 1 : plain ? (int)hp.steps.size() : 0;
        if (K == 0) {
            fprintf(stderr, "arapb200: batch_tracks: slot %d holds no problem or scene queued with frames\n", slot);
            return 1;
        }
        const int W = sc ? sc->W : hp.W, H = sc ? sc->H : hp.H;
        bool ok = n_queries >= 0 && (flow0 || bflow0 || occ0 || n_queries > 0) &&
                  (n_queries == 0 ? !query_pos && !query_occ : queries && query_pos);
        for (int i = 0; ok && i < n_queries; ++i)
            ok = queries[2 * i] >= 0 && queries[2 * i] < W && queries[2 * i + 1] >= 0 && queries[2 * i + 1] < H;
        if (!ok) {
            fprintf(stderr, "arapb200: batch_tracks: bad request (nothing asked for, %d queries, null queries or "
                    "query_pos, query outputs without queries, or a query outside the %dx%d frame)\n", n_queries, W, H);
            return 1;
        }
        std::vector<float> maps(sc ? 18 * (size_t)K : 0);
        for (int k = 1; sc && k <= K; ++k) // frame 0 -> frame k of the background: composite_coeffs(NULL, A_k)
            if (!composite_coeffs(nullptr, sc->motions.data() + 6 * k, maps.data() + 18 * (k - 1))) {
                fprintf(stderr, "arapb200: batch_tracks: frame %d's motion gives non-finite maps\n", k);
                return 1;
            }
        auto attach = [&](auto& t) {
            t.tracks = true;
            t.trk_flow0 = flow0; t.trk_bflow0 = bflow0; t.trk_occ0 = occ0;
            t.queries.assign(queries, queries + 2 * (size_t)n_queries);
            t.query_pos = query_pos; t.query_occ = query_occ;
        };
        if (sc) {
            attach(*sc);
            sc->track_maps.swap(maps);
        } else {
            attach(hp);
        }
        return 0;
    });
}

int arapb200_blur_schedule(int nCont, int n_frames, const int* steps, const double* motion,
                           const double* frame_motions, int n_samples, double shutter, int image, int* out_state,
                           float* out_w, float* out_smap)
{
    if (!out_state || !out_w || !out_smap || n_samples < 1 || n_samples > BLUR_MAX_SAMPLES) return 1;
    BlurSub tab[BLUR_MAX_SAMPLES];
    if (!blur_schedule(nCont, n_frames, steps, motion, frame_motions, n_samples, shutter, image, tab)) return 1;
    for (int j = 0; j < n_samples; ++j) {
        out_state[j] = tab[j].j0;
        out_w[j] = tab[j].w;
        std::copy(tab[j].smap, tab[j].smap + 6, out_smap + 6 * j);
    }
    return 0;
}

int arapb200_batch_run(arapb200_batch* b)
{
    return guarded([&]() -> int {
        if (!b) return 1;
        b->ms[0] = b->ms[1] = b->ms[2] = 0.f;
        const long long l0 = b->pipe->launches();
        b->todo.clear();
        std::vector<int> at(b->max_problems, -1); // slot -> index in todo
        for (int s = 0; s < b->max_problems; ++s)
            if (b->pending[s]) {
                at[s] = (int)b->todo.size();
                b->todo.push_back(b->slots[s]);
                b->pending[s] = 0;
            }
        std::vector<HostScene> scenes;
        scenes.swap(b->scenes);
        b->scene_of.assign(b->max_problems, -1);
        for (HostScene& sc : scenes) {
            sc.first = at[sc.first]; // a scene's slots are consecutive and all pending
            for (int s = 0; s < sc.n; ++s) {
                b->todo[sc.first + s].blur_states = sc.blur_states;
                b->todo[sc.first + s].tracks = sc.tracks; // a tracked scene's layers keep their frame k -> 0 flows
            }
        }
        for (HostProblem& hp : b->slots) drop_tracks(hp); // the run drops the tracks requests, as it drops the scenes
        const int rc = b->pipe->run(b->todo.data(), (int)b->todo.size(), scenes.data(), (int)scenes.size());
        if (rc) return rc;
        b->ms[0] = b->pipe->last_ms_total();
        b->ms[1] = b->pipe->last_ms_solve();
        b->ms[2] = b->pipe->last_ms_warp();
        b->launches = b->pipe->launches() - l0;
        return 0;
    });
}

int arapb200_batch_timing(arapb200_batch* b, float* ms3)
{
    return guarded([&]() -> int {
        if (!b || !ms3) return 1;
        ms3[0] = b->ms[0]; ms3[1] = b->ms[1]; ms3[2] = b->ms[2];
        return 0;
    });
}

long long arapb200_batch_launches(arapb200_batch* b) { return b ? b->launches : 0; }

int arapb200_batch_resident_count(arapb200_batch* b) { return b ? b->pipe->last_resident_count() : 0; }

int arapb200_batch_launch_info(arapb200_batch* b, int* info6)
{
    if (!b || !info6) return 1;
    b->pipe->last_launch_info(info6);
    return 0;
}

int arapb200_batch_set_option(arapb200_batch* b, const char* name, double value)
{
    return guarded([&]() -> int {
        if (!b || !name) return 1;
        if (strcmp(name, "pcg_rtol") == 0) {
            if (!(value >= 0.0) || value >= 1.0) return 1;
            b->pipe->set_pcg_rtol((float)value);
            return 0;
        }
        if (strcmp(name, "cluster_barrier") == 0) return 0; // no effect, accepted for compatibility (include/arapb200.h)
        if (strcmp(name, "gn_rtol") == 0) {
            if (!(value >= 0.0) || value >= 1.0) return 1;
            b->pipe->set_gn_rtol((float)value);
            return 0;
        }
        if (strcmp(name, "lm") == 0) { // 1: solver kind "LMGPU" for every Opt_ProblemSolve of the schedule; 0 (default): gaussNewtonGPU
            b->pipe->set_lm(value != 0.0);
            return 0;
        }
        return 1;
    });
}

// ------------------------------------------------------------------------------------ debug / parity
int arapb200_debug_gn_solve(int W, int H, float* X, float* A, const float* U, const float* C, const float* M,
                            float wf, float wr, int nGN, int nPCG, int backend, float* costs, float* scal)
{
    return guarded([&]() -> int {
        const size_t N = (size_t)W * H;
        DevBuf<float2> dX(N), dU(N), dC(N);
        DevBuf<float> dA(N), dM(N);
        DevBuf<float> dtr(scal ? (size_t)3 * nGN * nPCG : 0);
        dX.up((const float2*)X); dU.up((const float2*)U); dC.up((const float2*)C); dA.up(A); dM.up(M);
        ARAP_CUDA_OR_RETURN(cudaDeviceSynchronize());
        GnPlan plan(W, H, 0, backend);
        plan.set_parameter("nIterations", &nGN);
        plan.set_parameter("lIterations", &nPCG);
        if (scal) plan.set_trace(dtr.p);
        void* pp[7] = {dX.p, dA.p, dU.p, dC.p, dM.p, &wf, &wr};
        plan.init(pp);
        if (costs) costs[0] = (float)plan.current_cost();
        int g = 0;
        while (plan.step(pp)) {
            ++g;
            if (costs) costs[g] = (float)plan.current_cost();
        }
        dX.down((float2*)X);
        dA.down(A);
        if (scal) dtr.down(scal);
        ARAP_CUDA_OR_RETURN(cudaDeviceSynchronize());
        return 0;
    });
}

// UrShape == pixel grid on every active pixel?  (what GnPlan::choose_backend checks on the device)
static bool host_urshape_is_grid(int W, int H, const float* U, const float* M)
{
    for (int y = 0; y < H; ++y)
        for (int x = 0; x < W; ++x) {
            const size_t i = (size_t)y * W + x;
            if (M[i] == 0.0f && (U[2 * i] != (float)x || U[2 * i + 1] != (float)y)) return false;
        }
    return true;
}

static int debug_setup(int W, int H, const float* X, const float* A, const float* U, const float* C, const float* M,
                       float wf, float wr, StreamSolver& s, DevBuf<float2>& dX, DevBuf<float2>& dU, DevBuf<float2>& dC,
                       DevBuf<float>& dA, DevBuf<float>& dM)
{
    const size_t N = (size_t)W * H;
    std::vector<float> zeros(2 * N, 0.f);
    dX.up((const float2*)(X ? X : zeros.data()));
    dU.up((const float2*)U);
    dC.up((const float2*)C);
    dA.up(A);
    dM.up(M);
    ARAP_CUDA_OR_RETURN(cudaDeviceSynchronize());
    s.bind(dX.p, dA.p, dU.p, dC.p, dM.p, wf, wr, nullptr);
    s.set_general(!host_urshape_is_grid(W, H, U, M));
    s.enqueue_prep(nullptr);
    return 0;
}

// three planes (PL_* indices) -> interleaved [N][3], zero outside the object
static void gather3(const StreamSolver& s, const int planes[3], size_t N, float* out3, const std::vector<unsigned char>& flags)
{
    std::vector<float> tmp(N);
    for (int k = 0; k < 3; ++k) {
        s.download_plane(planes[k], tmp.data());
        for (size_t i = 0; i < N; ++i) out3[3 * i + k] = (flags[i] & FLAG_ACTIVE) ? tmp[i] : 0.f;
    }
}

int arapb200_debug_eval_jtf(int W, int H, const float* X, const float* A, const float* U, const float* C,
                            const float* M, float wf, float wr, float* r3, float* pre3)
{
    return guarded([&]() -> int {
        const size_t N = (size_t)W * H;
        DevBuf<float2> dX(N), dU(N), dC(N);
        DevBuf<float> dA(N), dM(N);
        StreamSolver s(W, H);
        if (int rc = debug_setup(W, H, X, A, U, C, M, wf, wr, s, dX, dU, dC, dA, dM)) return rc;
        s.enqueue_pcg_init(nullptr);
        ARAP_CUDA_OR_RETURN(cudaDeviceSynchronize());
        std::vector<unsigned char> flags(N);
        s.download_flags(flags.data());
        const int r_planes[3] = {PL_R, PL_R + 1, PL_R + 2};
        gather3(s, r_planes, N, r3, flags);
        const int pre_planes[3] = {PL_PRE, PL_PRE, PL_PRE + 1};
        gather3(s, pre_planes, N, pre3, flags);
        return 0;
    });
}

int arapb200_debug_apply_jtj(int W, int H, const float* A, const float* U, const float* C, const float* M, float wf,
                             float wr, const float* p3, float* q3, float* dot)
{
    return guarded([&]() -> int {
        const size_t N = (size_t)W * H;
        DevBuf<float2> dX(N), dU(N), dC(N);
        DevBuf<float> dA(N), dM(N);
        StreamSolver s(W, H);
        if (int rc = debug_setup(W, H, nullptr, A, U, C, M, wf, wr, s, dX, dU, dC, dA, dM)) return rc;
        const StreamDev& v = s.host_view();
        ARAP_CUDA_OR_RETURN(cudaDeviceSynchronize());
        std::vector<float> tmp(N);
        for (int k = 0; k < 3; ++k) {
            for (size_t i = 0; i < N; ++i) tmp[i] = p3[3 * i + k];
            s.upload_plane(PL_P + k, tmp.data());
        }
        s.enqueue_step_a(true, 0, nullptr);
        ARAP_CUDA_OR_RETURN(cudaDeviceSynchronize());
        std::vector<unsigned char> flags(N);
        s.download_flags(flags.data());
        const int q_planes[3] = {PL_Q, PL_Q + 1, PL_Q + 2};
        gather3(s, q_planes, N, q3, flags);
        StreamScalars sc;
        ARAP_CUDA_OR_RETURN(cudaMemcpy(&sc, v.sc, sizeof(sc), cudaMemcpyDeviceToHost));
        if (dot) *dot = sc.den;
        return 0;
    });
}

int arapb200_debug_cost(int W, int H, const float* X, const float* A, const float* U, const float* C, const float* M,
                        float wf, float wr, float* cost)
{
    return guarded([&]() -> int {
        const size_t N = (size_t)W * H;
        DevBuf<float2> dX(N), dU(N), dC(N);
        DevBuf<float> dA(N), dM(N);
        dX.up((const float2*)X); dU.up((const float2*)U); dC.up((const float2*)C); dA.up(A); dM.up(M);
        ARAP_CUDA_OR_RETURN(cudaDeviceSynchronize());
        StreamSolver s(W, H);
        s.bind(dX.p, dA.p, dU.p, dC.p, dM.p, wf, wr, nullptr);
        s.set_general(!host_urshape_is_grid(W, H, U, M));
        s.enqueue_init(nullptr);
        s.read_back(nullptr, cost, nullptr);
        return 0;
    });
}

// Cycle accounting of the resident kernel on one problem (see solver_resident.cu, RS_TICK):
// prof[cta][8] = cycles in {phase1, phase2, phase3, other, barrier skew, barrier poll, barrier fold}, epochs.
// info = {n_strips, ctas, warps per cta}; *ms = device time of the launch.
int arapb200_debug_resident_profile(int W, int H, const uint8_t* mask_red, const int32_t* matches, int n_matches,
                                    int nCont, int nGN, int nPCG, unsigned long long* prof, int* info, float* ms)
{
    return guarded([&]() -> int {
        const size_t N = (size_t)W * H;
        std::vector<MatchRec> recs;
        build_match_records(W, H, mask_red, matches, n_matches, recs);
        DevBuf<unsigned char> dmask(N);
        DevBuf<float2> dX(N), dU(N), dC(N);
        DevBuf<float> dA(N), dM(N), dcost((size_t)nCont * (nGN + 1));
        DevBuf<MatchRec> dm(recs.size());
        DevBuf<unsigned long long> dprof(RS_MAX_CTAS * RS_PROF_SLOTS);
        dmask.up(mask_red);
        if (!recs.empty()) dm.up(recs.data());
        ARAP_CUDA_OR_RETURN(cudaMemset(dprof.p, 0, RS_MAX_CTAS * RS_PROF_SLOTS * sizeof(unsigned long long)));
        enqueue_reset_state(W, H, dmask.p, dX.p, dU.p, dA.p, dM.p, nullptr);
        enqueue_target_image(W, H, dm.p, (int)recs.size(), dC.p, nullptr);
        ARAP_CUDA_OR_RETURN(cudaDeviceSynchronize());
        ResidentSolver rs(W, H);
        if (!rs.prepare(W, H, dM.p, nullptr)) return 3;
        rs.set_profile(dprof.p);
        const EventHandle e0 = make_event(), e1 = make_event();
        cudaEventRecord(e0.get(), nullptr);
        rs.enqueue(dX.p, dA.p, dC.p, 1, sqrtf(100.f), sqrtf(0.01f), nCont, nGN, nPCG, dcost.p, nullptr, nullptr);
        cudaEventRecord(e1.get(), nullptr);
        ARAP_CUDA_OR_RETURN(cudaDeviceSynchronize());
        if (ms) cudaEventElapsedTime(ms, e0.get(), e1.get());
        if (int st = rs.status(nullptr)) return 100 + st;
        dprof.down(prof);
        ARAP_CUDA_OR_RETURN(cudaDeviceSynchronize());
        if (info) { info[0] = rs.n_strips(); info[1] = rs.ctas(); info[2] = rs.warps(); }
        return 0;
    });
}

// The same accounting for the first of `copies` identical problems sharing one cooperative launch: what the phases and
// the barriers of one problem cost while its co-resident neighbours compete for the SM and for L2.
int arapb200_debug_resident_profile_group(int W, int H, const uint8_t* mask_red, const int32_t* matches, int n_matches,
                                          int copies, int nCont, int nGN, int nPCG, unsigned long long* prof, int* info,
                                          float* ms)
{
    return guarded([&]() -> int {
        if (copies < 1 || copies > 16) return 1;
        const size_t N = (size_t)W * H;
        std::vector<MatchRec> recs;
        build_match_records(W, H, mask_red, matches, n_matches, recs);
        DevBuf<unsigned char> dmask(N);
        DevBuf<float2> dU(N);
        DevBuf<float> dM(N);
        DevBuf<MatchRec> dm(recs.size());
        DevBuf<unsigned long long> dprof(RS_MAX_CTAS * RS_PROF_SLOTS);
        std::vector<DevBuf<float2>> dX, dC;
        std::vector<DevBuf<float>> dA, dcost;
        dmask.up(mask_red);
        if (!recs.empty()) dm.up(recs.data());
        ARAP_CUDA_OR_RETURN(cudaMemset(dprof.p, 0, RS_MAX_CTAS * RS_PROF_SLOTS * sizeof(unsigned long long)));
        ResidentSolver rs(W, H, copies);
        for (int i = 0; i < copies; ++i) {
            dX.emplace_back(N);
            dC.emplace_back(N);
            dA.emplace_back(N);
            dcost.emplace_back((size_t)nCont * (nGN + 1));
            enqueue_reset_state(W, H, dmask.p, dX[i].p, dU.p, dA[i].p, dM.p, nullptr);
            enqueue_target_image(W, H, dm.p, (int)recs.size(), dC[i].p, nullptr);
            rs.prepare_enqueue(i, W, H, dM.p, nullptr);
        }
        ARAP_CUDA_OR_RETURN(cudaDeviceSynchronize());
        for (int i = 0; i < copies; ++i) {
            if (!rs.prepare_finish(i)) return 3;
            rs.set_problem(i, dX[i].p, dA[i].p, dC[i].p, 1, sqrtf(100.f), sqrtf(0.01f), dcost[i].p, nullptr);
        }
        if (rs.group_size(0, copies) < copies) return 4; // they must share ONE launch
        rs.set_profile(dprof.p);
        const EventHandle e0 = make_event(), e1 = make_event();
        cudaEventRecord(e0.get(), nullptr);
        rs.enqueue_group(0, copies, nCont, nGN, nPCG, nullptr);
        cudaEventRecord(e1.get(), nullptr);
        ARAP_CUDA_OR_RETURN(cudaDeviceSynchronize());
        if (ms) cudaEventElapsedTime(ms, e0.get(), e1.get());
        if (int st = rs.status(nullptr)) return 100 + st;
        dprof.down(prof);
        ARAP_CUDA_OR_RETURN(cudaDeviceSynchronize());
        if (info) { info[0] = rs.n_strips(); info[1] = rs.ctas(); info[2] = rs.warps(); }
        return 0;
    });
}

} // extern "C"

// device-side sincos / exact-sum probes
namespace {
__global__ void k_dbg_sincos(int n, const float* a, float* s, float* c)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) contract_sincos(a[i], s[i], c[i]);
}
// one block; thread t sums terms t, t+B, ... sequentially in binary32?  No: each term is its own
// "group term": the block folds them exactly in chunks of blockDim.x.
__global__ void k_dbg_exact_sum(size_t n, const float* t, float* out)
{
    __shared__ double red[64];
    // level 1: per-chunk block sums; level 2: chunk results are folded with a second exact pass below
    extern __shared__ double chunks[]; // 2 * nchunks
    const size_t nchunks = (n + blockDim.x - 1) / blockDim.x;
    for (size_t c = 0; c < nchunks; ++c) {
        size_t i = c * blockDim.x + threadIdx.x;
        float g = (i < n) ? t[i] : 0.f;
        HL b = block_exact_sum(g, red);
        if (threadIdx.x == 0) {
            chunks[2 * c] = b.h;
            chunks[2 * c + 1] = b.l;
        }
        __syncthreads();
    }
    if (threadIdx.x < 32) {
        // fold the chunk partials 32 at a time, carrying the running (h, l) in lane 0's slot
        HL run = {0.0, 0.0};
        for (size_t base = 0; base < nchunks; base += 31) {
            HL v = {0.0, 0.0};
            const size_t idx = base + threadIdx.x;
            if (threadIdx.x < 31 && idx < nchunks) { v.h = chunks[2 * idx]; v.l = chunks[2 * idx + 1]; }
            if (threadIdx.x == 31) v = run;
            run = warp_combine(v);
        }
        if (threadIdx.x == 0) *out = hl_to_float(run);
    }
}
// the streaming back-end's reduction path on its own: every block publishes its exact partial into one wide
// fixed-point accumulator (common.cuh), a second kernel decodes it
__global__ void __launch_bounds__(256) k_dbg_wide_publish(size_t n, const float* t, unsigned long long* acc)
{
    __shared__ double red[64];
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const HL b = block_exact_sum((i < n) ? t[i] : 0.f, red);
    if (threadIdx.x == 0) wide_add(acc, blockIdx.x, b.h);
    if (threadIdx.x == 1) wide_add(acc, blockIdx.x, b.l);
}
__global__ void __launch_bounds__(32) k_dbg_wide_decode(const unsigned long long* acc, float* out)
{
    const float v = wide_round(wide_fetch(acc, threadIdx.x & 15));
    if (threadIdx.x == 0) *out = v;
}
} // namespace

extern "C" {

int arapb200_debug_wide_sum(size_t n, const float* t, float* sum)
{
    return guarded([&]() -> int {
        if (n == 0 || n > ((size_t)1 << 26)) return 1;
        DevBuf<float> dt(n), dsum(1);
        DevBuf<unsigned long long> acc(WA_WORDS);
        dt.up(t);
        ARAP_CUDA_OR_RETURN(cudaMemset(acc.p, 0, WA_WORDS * sizeof(unsigned long long)));
        k_dbg_wide_publish<<<(unsigned)((n + 255) / 256), 256>>>(n, dt.p, acc.p);
        k_dbg_wide_decode<<<1, 32>>>(acc.p, dsum.p);
        dsum.down(sum);
        ARAP_CUDA_OR_RETURN(cudaDeviceSynchronize());
        return 0;
    });
}

int arapb200_debug_sincos(int n, const float* a, float* s, float* c)
{
    return guarded([&]() -> int {
        DevBuf<float> da(n), ds(n), dc(n);
        da.up(a);
        k_dbg_sincos<<<(n + 255) / 256, 256>>>(n, da.p, ds.p, dc.p);
        ds.down(s);
        dc.down(c);
        ARAP_CUDA_OR_RETURN(cudaDeviceSynchronize());
        return 0;
    });
}

int arapb200_debug_exact_sum(size_t n, const float* t, float* sum)
{
    return guarded([&]() -> int {
        if (n > (size_t)256 * 2048) return 1;
        DevBuf<float> dt(n), dsum(1);
        dt.up(t);
        const size_t nchunks = (n + 255) / 256;
        k_dbg_exact_sum<<<1, 256, 2 * nchunks * sizeof(double)>>>(n, dt.p, dsum.p);
        dsum.down(sum);
        ARAP_CUDA_OR_RETURN(cudaDeviceSynchronize());
        return 0;
    });
}

} // extern "C"
