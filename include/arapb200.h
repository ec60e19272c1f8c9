/*
 * arapb200.h -- flat C ABI above the Opt.h level: what the reference's L3/L4 code does around the
 * solver (ARAP/deformation/src/CombinedSolver.h, ARAP/deformation/src/main.cpp,
 * ARAP/warping/src/main.cpp), as whole-image calls with plain pointers and sizes.  This is the
 * surface a Terra host reaches with terralib.includec (INTEGRATION.md) and the one bench.py / the
 * Python mirror bind with ctypes.  All functions return 0 on success, non-zero on failure (message on
 * stderr); nothing in the library calls exit(): failures inside the Opt_* entry points are recorded on the
 * plan (arapb200_plan_error).
 */
#ifndef ARAPB200_H
#define ARAPB200_H

#include <stddef.h>
#include <stdint.h>

#ifndef ARAPB200_API
#define ARAPB200_API __attribute__((visibility("default")))
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define ARAPB200_BACKEND_AUTO 0     /* resident when the problem fits on chip, else streaming */
#define ARAPB200_BACKEND_STREAM 1   /* graph-captured 2-kernel PCG iteration, state in L2/HBM */
#define ARAPB200_BACKEND_RESIDENT 2 /* persistent cooperative kernel, state in registers/smem */

/* library / device info: fills sm_count, l2_bytes, cc_major, cc_minor (any may be NULL) */
ARAPB200_API int arapb200_device_info(int* sm_count, size_t* l2_bytes, int* cc_major, int* cc_minor);
ARAPB200_API const char* arapb200_version(void);

/* ---- forward warp (replaces ARAP/warping/src/main.cpp:145-225 == CombinedSolver.h:280-342) ----
 * Host buffers.  pos float2[W*H] absolute positions, rgb uint8x3[W*H], mask_red uint8[W*H]
 * (0 = object).  Outputs: out_rgb uint8x3[W*H], out_mask uint8[W*H] (255 where something landed),
 * out_splat uint32[W*H] = 1 + 2*(y*W+x) + t of the winning triangle (0 = empty); out_splat may be NULL. */
ARAPB200_API int arapb200_warp(int W, int H, const float* pos, const uint8_t* rgb, const uint8_t* mask_red,
                  uint8_t* out_rgb, uint8_t* out_mask, uint32_t* out_splat);
/* warp tool front half (warping/src/main.cpp:160-166): positions = grid + flow, then warp */
ARAPB200_API int arapb200_warp_flow(int W, int H, const float* flow, const uint8_t* rgb, const uint8_t* mask_red,
                       uint8_t* out_rgb, uint8_t* out_mask, uint32_t* out_splat);
/* The warp with its opt-in extra outputs (DESIGN.md 4.3).  pos_or_flow: absolute positions (is_flow = 0, as
 * arapb200_warp; forward flow = pos - grid) or a forward flow (is_flow = 1, as arapb200_warp_flow; positions = grid + flow).
 * out_rgb, out_mask, out_splat as arapb200_warp; out_rgb and out_mask are required, every other output may be NULL.
 * out_bflow float2[W*H]: backward flow on the frame-2 grid, the exact frame-1 source point of every pixel something
 * landed on minus the pixel, (0, 0) elsewhere.  out_occ uint8[W*H]: occlusion of frame 1, 0 = the pixel is visible in
 * frame 2, 255 = it is not (covered, folded, never rasterised or out of the frame). */
ARAPB200_API int arapb200_warp_ex(int W, int H, const float* pos_or_flow, int is_flow, const uint8_t* rgb,
                                  const uint8_t* mask_red, uint8_t* out_rgb, uint8_t* out_mask, uint32_t* out_splat,
                                  float* out_bflow, uint8_t* out_occ);
/* A frame sequence from position fields the caller holds (DESIGN.md 4.4), e.g. X after each of several Opt_ProblemSolve
 * calls.  pos float2[K][W*H]: P_1 .. P_K, absolute positions; frame 0 is the input image on the pixel grid.  Every output
 * is [K][W*H][...] contiguous, index k - 1 holding frame k.  out_rgb uint8x3 / out_mask uint8: arapb200_warp of P_k
 * (required).  out_flow float2: frame k - 1 -> k on the frame k - 1 grid (k = 1: P_1 - grid; k >= 2: at every pixel
 * something landed on in frame k - 1, the weights of its winning triangle applied to that triangle's vertices in P_k,
 * minus the pixel; (0, 0) elsewhere).  out_bflow float2: frame k -> k - 1 on the frame k grid, the same with the roles
 * of the frames swapped (k = 1: arapb200_warp_ex's out_bflow).  out_occ uint8: occlusion of frame k - 1 in frame k
 * (0 visible, 255 not; k = 1: arapb200_warp_ex's out_occ).  out_flow0 float2: P_k - grid.  Every output but out_rgb and
 * out_mask may be NULL.  Colours are always sampled from the frame-0 image. */
ARAPB200_API int arapb200_warp_seq(int W, int H, int K, const float* pos, const uint8_t* rgb, const uint8_t* mask_red,
                                   uint8_t* out_rgb, uint8_t* out_mask, float* out_flow, float* out_bflow,
                                   uint8_t* out_occ, float* out_flow0);
/* Tracks from frame 0 (DESIGN.md 4.9) of the frame sequence arapb200_warp_seq renders from the same pos and mask_red:
 * out_bflow0 float2[K][W*H], frame k -> frame 0 on the frame k grid (at every pixel something landed on in frame k, the
 * weights of its winning triangle applied to that triangle's vertices on the pixel grid, minus the pixel; (0, 0)
 * elsewhere); out_occ0 uint8[K][W*H], the occlusion of frame 0 in frame k (0 visible, 255 not: arapb200_warp_ex's rule
 * with the forward flow P_k - grid, frame k's z-buffer and out_bflow0).  Index k - 1 holds frame k; frame 1 is
 * arapb200_warp_seq's out_bflow and out_occ.  The same bits as arapb200_batch_tracks.  Either output may be NULL.
 * Returns non-zero for W, H or K <= 0 and a NULL pos or mask_red. */
ARAPB200_API int arapb200_warp_tracks(int W, int H, int K, const float* pos, const uint8_t* mask_red, float* out_bflow0,
                                      uint8_t* out_occ0);

/* ---- one image / segment, end to end (replaces deformSingle, deformation/src/main.cpp:140-160:
 * border pins :130-136, resetGPU + continuation CombinedSolver.h:172-242, solve, warp, flow :352-366).
 * Host buffers in, host buffers out.  matches int32[4*n] (x1 y1 x2 y2) WITHOUT the border pins.
 * out_flow float2[W*H]; out_rgb/out_mask as arapb200_warp; out_costs float[nCont*(nGN+1)] (may be
 * NULL): cost at init and after every Gauss-Newton step of every continuation step. */
ARAPB200_API int arapb200_deform(int W, int H, const uint8_t* rgb, const uint8_t* mask_red, const int32_t* matches,
                    int n_matches, int nCont, int nGN, int nPCG, int backend, float* out_flow,
                    uint8_t* out_rgb, uint8_t* out_mask, float* out_costs);

/* ---- "next" row N1: layer flatten + background composite (replaces para_gen.py:136-175 flatten and :50-61 add_bg).
 * n_layers per-segment results of one --multseg pair, in segment order: flows[s] float2[W*H], rgbs[s] uint8x3[W*H],
 * masks[s] uint8[W*H] (warped masks, non-zero = object).  Later segments overwrite earlier ones where their mask is
 * non-zero; where the final mask is 0 the colour is taken from `background` (uint8x3[W*H], may be NULL). */
ARAPB200_API int arapb200_flatten(int W, int H, int n_layers, const float* const* flows, const uint8_t* const* rgbs,
                                  const uint8_t* const* masks, const uint8_t* background, float* out_flow,
                                  uint8_t* out_rgb, uint8_t* out_mask);
/* arapb200_flatten with the extra outputs of the layers (DESIGN.md 4.3).  src_masks[s] uint8[W*H]: segment s's frame-1
 * input mask (0 = object); bflows[s] float2[W*H]: its backward flow (arapb200_warp_ex / arapb200_batch_submit_ex).
 * out_bflow float2[W*H]: the backward flow of the front layer (the last one whose warped mask is non-zero), (0, 0) where
 * there is none.  out_occ uint8[W*H]: occlusion of frame 1 across the layers (0 visible, 255 not).  out_bflow and out_occ
 * may be NULL; out_bflow needs bflows, out_occ needs bflows and src_masks.  With both NULL this is arapb200_flatten. */
ARAPB200_API int arapb200_flatten_ex(int W, int H, int n_layers, const float* const* flows, const uint8_t* const* rgbs,
                                     const uint8_t* const* masks, const uint8_t* background,
                                     const uint8_t* const* src_masks, const float* const* bflows, float* out_flow,
                                     uint8_t* out_rgb, uint8_t* out_mask, float* out_bflow, uint8_t* out_occ);
/* The layers of arapb200_flatten_ex over a background that moves by its own affine map (DESIGN.md 4.5): renders frame b
 * from frame a.  A motion is a row-major 2x3 binary64 matrix mapping background-plane points to frame pixels; the plane
 * has frame 0's coordinates.  motion_from is frame a's motion (NULL = identity, the pair case), motion_to frame b's.
 * n_layers (0 .. 32) layers as arapb200_flatten_ex: flows, rgbs, masks (warped), src_masks (frame-a input masks, 0 =
 * object; required, they decide which frame-a pixels are background) and bflows (required for out_bflow / out_occ).
 * n_layers == 0 is a pure background-motion pair.  background uint8x3[bgW*bgH], sampled bilinearly at
 * inv(motion_to)(q) + (bg_x, bg_y) where no layer is in front, coordinates clamped to the image.
 * out_flow float2[W*H] (frame a: the flatten's flow on object pixels, the background's motion elsewhere), out_rgb,
 * out_mask (objects only, as the flatten) and out_bflow float2[W*H] (frame b), out_occ uint8[W*H] (frame a, 0 visible
 * in frame b, 255 not).  out_bflow, out_occ and out_coeffs may be NULL; out_coeffs float[3][2][3] receives the binary32
 * maps the kernels use: F (frame a -> b), B (frame b -> a), S (frame b -> background plane).  Returns non-zero before
 * any CUDA call and without writing anything for: W or H <= 0, n_layers outside [0, 32], a missing layer array or
 * entry (src_masks included) when n_layers > 0, out_bflow / out_occ without bflows when n_layers > 0, a NULL
 * background or bgW / bgH <= 0, a NULL motion_to, a non-finite or singular motion or non-finite derived maps, and a
 * NULL out_flow, out_rgb or out_mask.  With both motions the identity and a W x H background at (0, 0), rgb, mask,
 * bflow and occ are arapb200_flatten_ex's with that background bit for bit. */
ARAPB200_API int arapb200_composite(int W, int H, int n_layers, const float* const* flows, const uint8_t* const* rgbs,
                                    const uint8_t* const* masks, const uint8_t* const* src_masks,
                                    const float* const* bflows, int bgW, int bgH, const uint8_t* background, int bg_x,
                                    int bg_y, const double* motion_from, const double* motion_to, float* out_flow,
                                    uint8_t* out_rgb, uint8_t* out_mask, float* out_bflow, uint8_t* out_occ,
                                    float* out_coeffs);

/* ---- "next" row N3: match ingestion on the device (replaces the Python loops of para_gen.py:216-223 valid_cnstr,
 * :468-482 filter, :513-537 per-segment masks).
 * labels1 uint8[W1*H1], labels2 uint8[W2*H2]: the segment-label images of frame 1 and 2 (0 = background).
 * A raw match (x1 y1 x2 y2) is kept iff both points are inside their images, 0 < |p2 - p1| < 60 px, the label under
 * p1 is non-zero and equals the label under p2.  Order is preserved (later constraints overwrite earlier ones
 * downstream, CombinedSolver.h:223-242).  out_matches int32[4*n], out_labels uint8[n] (label under p1 of every kept
 * match; may be NULL), *n_out = number kept.  Negative coordinates are rejected (the reference would wrap them). */
ARAPB200_API int arapb200_filter_matches(int W1, int H1, const uint8_t* labels1, int W2, int H2, const uint8_t* labels2,
                                         const int32_t* matches, int n, int32_t* out_matches, uint8_t* out_labels,
                                         int* n_out);
/* The mask image arap_deform expects (red channel 0 = solve here, 255 = ARAP_BG, para_gen.py:30): segment > 0 selects
 * one label (--multseg, :526-527), segment == 0 selects every non-zero label (:515-516).  out_mask uint8[W*H]. */
ARAPB200_API int arapb200_segment_mask(int W, int H, const uint8_t* labels, int segment, uint8_t* out_mask);

/* ---- batched, pipelined variant: many independent (image, segment) problems per GPU --------- */
typedef struct arapb200_batch arapb200_batch;
/* max_problems problems of at most maxW x maxH in flight on the current device */
ARAPB200_API arapb200_batch* arapb200_batch_create(int maxW, int maxH, int max_problems, int nCont, int nGN, int nPCG,
                                      int backend);
ARAPB200_API void arapb200_batch_destroy(arapb200_batch* b);
/* enqueue problem `slot` (0 <= slot < max_problems); host pointers must stay valid until _wait */
ARAPB200_API int arapb200_batch_submit(arapb200_batch* b, int slot, int W, int H, const uint8_t* rgb,
                          const uint8_t* mask_red, const int32_t* matches, int n_matches, float* out_flow,
                          uint8_t* out_rgb, uint8_t* out_mask, float* out_costs);
/* arapb200_batch_submit plus the extra outputs of arapb200_warp_ex for this problem: out_bflow float2[W*H], out_occ
 * uint8[W*H] (either may be NULL).  Buffers for them are allocated for a slot the first time it asks; with both NULL
 * this is exactly arapb200_batch_submit. */
ARAPB200_API int arapb200_batch_submit_ex(arapb200_batch* b, int slot, int W, int H, const uint8_t* rgb,
                                          const uint8_t* mask_red, const int32_t* matches, int n_matches,
                                          float* out_flow, uint8_t* out_rgb, uint8_t* out_mask, float* out_costs,
                                          float* out_bflow, uint8_t* out_occ);
/* arapb200_batch_submit_ex plus a frame sequence taken from the continuation schedule (DESIGN.md 4.4): steps int[n_frames]
 * lists continuation steps, strictly increasing, each in [0, nCont - 1]; frame k is the solver's state after step
 * steps[k - 1], rendered as arapb200_warp_seq renders P_k, with seq_rgb .. seq_flow0 its outputs ([n_frames][W*H][...]).
 * seq_rgb and seq_mask are required, the others may be NULL.  The step list is copied: it need not outlive the call.
 * Returns non-zero, and queues nothing, for n_frames < 0, outputs without frames, a missing seq_rgb / seq_mask or a
 * step list that is not strictly increasing within [0, nCont - 1].  With n_frames == 0 and NULL sequence outputs this is
 * exactly arapb200_batch_submit_ex.  A slot allocates its sequence buffers (37 B/px per frame on the device) the first
 * time it asks and grows them for a longer list.  Frames are copied straight into the caller's buffers; pinned
 * buffers make that copy faster.  A resident group in which any problem asks for frames runs one launch per
 * continuation step (same results bit for bit). */
ARAPB200_API int arapb200_batch_submit_seq(arapb200_batch* b, int slot, int W, int H, const uint8_t* rgb,
                                           const uint8_t* mask_red, const int32_t* matches, int n_matches,
                                           float* out_flow, uint8_t* out_rgb, uint8_t* out_mask, float* out_costs,
                                           float* out_bflow, uint8_t* out_occ, int n_frames, const int* steps,
                                           uint8_t* seq_rgb, uint8_t* seq_mask, float* seq_flow, float* seq_bflow,
                                           uint8_t* seq_occ, float* seq_flow0);
/* A scene (DESIGN.md 4.6): one image, its n_layers segments and a background with its own motion, solved, warped and
 * composited in the batch without the layers leaving the device.  Slots slot .. slot + n_layers - 1 take one layer each,
 * in segment order (later layers are in front, as in arapb200_flatten); layer s is an ordinary problem with the shared
 * W x H and rgb, its own masks_red[s] (0 = object) and its own matches[s] / n_matches[s], grouped and launched as run()
 * groups any problems.  The solve and the warp read rgb only on the object, so rgb may be the raw image.
 * The pair: out_flow, out_rgb, out_mask, out_bflow, out_occ are exactly arapb200_composite of the layers' ordinary
 * outputs (flow, rgb, mask, backward flow, input mask) with motion_from = NULL and motion_to = motion (row-major 2x3
 * binary64, required; the identity gives a still background), over background uint8x3[bgW*bgH] at origin (bg_x, bg_y).
 * out_flow, out_rgb and out_mask are required; out_bflow, out_occ, out_rgb0 and out_costs may be NULL.
 * out_costs float[n_layers][nCont][nGN+1]: the layers' cost logs.
 * out_rgb0 uint8x3[W*H], frame 0: rgb where any masks_red[s] is 0, else background[q + (bg_x, bg_y)] (coordinates clamped
 * to the image, as the composite clamps them).
 * Frames: n_frames > 0 asks every layer for the frames of steps (as arapb200_batch_submit_seq) and frame_motions
 * double[n_frames][2][3] gives A_1 .. A_K.  Frame k is arapb200_composite of the layers' frame k with motion_from =
 * A_{k-1} (A_0 = identity) and motion_to = A_k, and as source masks the input masks for k = 1 and 255 - (the layers'
 * warped masks of frame k - 1) for k >= 2 (lib.composite_seq).  seq_rgb uint8x3, seq_mask uint8, seq_flow float2,
 * seq_bflow float2, seq_occ uint8, each [n_frames][W*H][...]; seq_rgb and seq_mask are required with frames, the others
 * may be NULL.  Steps and motions are copied: they need not outlive the call; every other buffer must stay valid until
 * the run.
 * Only the composited outputs (and out_costs) are copied to the host; the scene keeps a device buffer of its own for the
 * background, frame 0 and 21 B/px per composited frame (the pair and each frame), allocated the first time and grown for
 * a larger scene.  Its kernels count in arapb200_batch_launches and in the total and warp spans of arapb200_batch_timing.
 * Returns non-zero, and queues nothing, for: a NULL batch; n_layers outside [1, 32]; slots outside the batch; slots that
 * belong to another scene queued for the same run; W or H <= 0, or W * H above the batch's maxW * maxH; a NULL rgb,
 * masks_red, matches or n_matches array, a NULL mask, a negative n_matches[s], or a NULL matches[s] with
 * n_matches[s] > 0; a NULL background, bgW or bgH <= 0, a NULL motion, a NULL out_flow, out_rgb or out_mask; n_frames
 * < 0, frame outputs without frames, frames without steps, frame_motions, seq_rgb or seq_mask, a step list that is not
 * strictly increasing within [0, nCont - 1]; and a non-finite or singular motion (or non-finite derived maps) among
 * motion and frame_motions.  Until the next arapb200_batch_run, an ordinary submit into a slot of a queued scene is
 * refused too. */
ARAPB200_API int arapb200_batch_submit_scene(arapb200_batch* b, int slot, int n_layers, int W, int H, const uint8_t* rgb,
                                             const uint8_t* const* masks_red, const int32_t* const* matches,
                                             const int* n_matches, int bgW, int bgH, const uint8_t* background,
                                             int bg_x, int bg_y, const double* motion, int n_frames, const int* steps,
                                             const double* frame_motions, float* out_flow, uint8_t* out_rgb,
                                             uint8_t* out_mask, float* out_bflow, uint8_t* out_occ, uint8_t* out_rgb0,
                                             float* out_costs, uint8_t* seq_rgb, uint8_t* seq_mask, float* seq_flow,
                                             float* seq_bflow, uint8_t* seq_occ);
/* Motion blur of a queued scene (DESIGN.md 4.8): the "final pass" next to the scene's sharp images.  Each blurred image
 * is the mean, per pixel and channel (sum + S/2) / S in integers, of n_samples = S sub-frame renders over a trailing
 * shutter that is open for the fraction `shutter` of the interval before the image's time: the layers splatted at
 * positions lerped between the continuation states, over the background at the lerped motion.  Masks, flows, backward
 * flows and occlusion stay as they are (defined at the frame times).  slot is the scene's first slot.
 * blur_rgb uint8x3[W*H], required: the blurred pair.  blur_rgb0 uint8x3[W*H], may be NULL: the blurred frame 0, which
 * extrapolates backwards at the first interval's velocity; it needs a scene that asked for out_rgb0.  seq_blur_rgb
 * uint8x3[n_frames][W*H], may be NULL: the blurred frames; it needs a scene with frames.  With n_samples = 1 or shutter
 * = 0 the blurred images are the sharp ones (frame 0: where the layers' warp at the grid covers the pixel or no layer has
 * it on its object).  Applies to the next run only; a second call replaces the first.  The sub-frames need the layers'
 * states after individual continuation steps, so a resident group holding a blurred layer runs one launch per step
 * (same results bit for bit).  Per blurred image the run launches 2 * n_samples more kernels, counted in
 * arapb200_batch_launches and in the warp span of arapb200_batch_timing; the scene keeps a second device buffer of
 * 4 B/px per layer + 8 B/px + 3 B/px per blurred image, and each layer 8 B/px per continuation state its sub-frames read.
 * Returns non-zero, and changes nothing, for: a NULL batch; a slot that is not the first slot of a scene queued for the
 * next run; n_samples outside [1, 64]; a shutter that is NaN or outside [0, 1]; a NULL blur_rgb; a blur_rgb0 for a
 * scene without out_rgb0; a seq_blur_rgb for a scene without frames; and a sub-frame motion of an image asked for that
 * is non-finite or singular or whose maps are non-finite (arapb200_blur_schedule; frame 0's extrapolation can produce
 * one). */
ARAPB200_API int arapb200_batch_scene_blur(arapb200_batch* b, int slot, int n_samples, double shutter, uint8_t* blur_rgb,
                                           uint8_t* blur_rgb0, uint8_t* seq_blur_rgb);
/* Tracks from frame 0 to every frame (DESIGN.md 4.9) for the next run: slot holds a problem queued with frames
 * (arapb200_batch_submit_seq, n_frames > 0) or is the first slot of a scene queued with frames.  Every output is
 * frame-major, index k - 1 holding frame k; each dense one may be NULL.
 * flow0 float2[K][W*H], frame 0 -> k on the frame 0 grid: P_k - grid for a problem (the bits of its seq_flow0), and for a
 * scene the flow of the layer whose input mask has the pixel on its object (the last one), else the background's A_k(p)
 * - p.  bflow0 float2[K][W*H], frame k -> 0 on the frame k grid: arapb200_warp_tracks's out_bflow0 for a problem; for a
 * scene the front layer's (the last one whose frame-k warped mask is non-zero), else inv(A_k)(q) - q.  occ0 uint8[K][W*H]:
 * the occlusion of frame 0 in frame k (0 visible, 255 not), the rule of arapb200_warp_ex for a problem and of
 * arapb200_composite (motion_from = NULL, motion_to = A_k) for a scene.  Frame 1's bflow0 and occ0 are the sequence's
 * frame-1 bflow and occ.
 * queries int32[n_queries][2]: (x, y) pixels of frame 0, copied; query_pos float2[K][n_queries] = (x, y) + flow0[k] at
 * the query, query_occ uint8[K][n_queries] = occ0[k] there (may be NULL), gathered on the device.
 * The run computes the dense outputs on the device whichever are asked for: a problem's slot keeps 9 B/px per frame more,
 * a scene's layers 8 B/px per frame each and the scene's buffer 17 B/px per frame and 9 B per query and frame; outputs
 * are copied straight into the caller's buffers.  The kernels count in arapb200_batch_launches and in the warp span of
 * arapb200_batch_timing: per frame k >= 2, two for a problem and one per scene layer; per frame two for a scene; one
 * gather with queries.  Applies to the next run only; a second call replaces the first, and a new submit into the
 * problem's slot drops it.
 * Returns non-zero, and changes nothing, for: a NULL batch; a slot that holds no problem queued with frames and is not
 * the first slot of a scene queued with frames; nothing asked for (every dense output NULL and n_queries == 0);
 * n_queries < 0; queries without a queries array or without query_pos (query_occ may be NULL); query_pos or query_occ
 * without queries; a query outside the W x H frame; and, for a scene, a frame motion A_k whose maps are non-finite. */
ARAPB200_API int arapb200_batch_tracks(arapb200_batch* b, int slot, float* flow0, float* bflow0, uint8_t* occ0,
                                       int n_queries, const int32_t* queries, float* query_pos, uint8_t* query_occ);
/* The sub-frame table a blurred scene uses for one image (DESIGN.md 4.8); host only, no CUDA call.  nCont, the frames'
 * steps and motions as arapb200_batch_submit_scene takes them (n_frames 0: steps and frame_motions may be NULL);
 * image -1 = frame 0, 0 = the pair, k = frame k.  Per sub-frame j < n_samples: out_state[j] = j0, the lower continuation
 * state of the lerp (-1 = the pixel grid), out_w[j] = its weight w (the positions are state j0 + w * (state j0+1 - state
 * j0)), out_smap[6 j .. 6 j + 5] = the binary32 map from the frame to the background plane (row-major 2x3).  Returns
 * non-zero, and writes nothing, for: NULL outputs; nCont < 1; n_frames < 0; a NULL motion; frames without steps or
 * frame_motions; a step list that is not strictly increasing within [0, nCont - 1]; n_samples outside [1, 64]; a
 * shutter that is NaN or outside [0, 1]; image outside [-1, n_frames]; and a sub-frame motion that is non-finite or
 * singular or whose maps are non-finite. */
ARAPB200_API int arapb200_blur_schedule(int nCont, int n_frames, const int* steps, const double* motion,
                                        const double* frame_motions, int n_samples, double shutter, int image,
                                        int* out_state, float* out_w, float* out_smap);
/* run everything submitted since the last run; returns after all outputs are in host memory */
ARAPB200_API int arapb200_batch_run(arapb200_batch* b);
/* device milliseconds of the last run: [0] total, [1] solve kernels only, [2] warp kernels only (with the scenes'
 * composite kernels) */
ARAPB200_API int arapb200_batch_timing(arapb200_batch* b, float* ms3);
/* number of kernel launches issued by the last run (the scenes' composite kernels and the tracks' kernels included) */
ARAPB200_API long long arapb200_batch_launches(arapb200_batch* b);

/* how many problems of the last run were solved by the resident (on-chip) back-end; the rest took the streaming one */
ARAPB200_API int arapb200_batch_resident_count(arapb200_batch* b);

/* shape of the last cooperative launch of the last run: info6 = {problems sharing the launch, kernel variant's max
 * threads, variant's min CTAs per SM, grid.x, grid.y, threads per CTA}; zeros when every problem streamed.  Lets a test
 * assert that it exercised the launch shape a benchmark times. */
ARAPB200_API int arapb200_batch_launch_info(arapb200_batch* b, int* info6);

/* Options beyond the reference's behaviour; every one defaults to "off" and none is on the parity path.
 *   "pcg_rtol" (SURVEY.md 8f N4): 0 <= value < 1.  > 0: a PCG loop ends as soon as r.z <= value^2 * (r.z at its start)
 *   instead of always running lIterations iterations.  Changes results (by design).  Both back-ends honour it (the
 *   streaming one turns the remaining kernels of its captured graph into no-ops).
 *   "gn_rtol": 0 <= value < 1.  > 0: the Gauss-Newton steps of a continuation step end as soon as one of them lowers
 *   the cost by less than value (relative) instead of always running nIterations steps; the skipped entries of
 *   out_costs repeat the last cost.  Same scope and caveats as "pcg_rtol" (both back-ends).
 *   "cluster_barrier": accepted for compatibility, any value, no effect: every resident problem uses the L2 barrier.  The
 *   cluster-scope barrier it once selected gave the same bits and was slower on every workload (DESIGN.md 4.1).
 *   "lm": 1 = every Opt_ProblemSolve of the schedule is run by the reference's other solver kind, "LMGPU"
 *   (Levenberg-Marquardt trust region, Q-based exit of the linear loops, step acceptance / revert;
 *   ARAP/API/src/solverGPUGaussNewton.t with UsesLambda()) with its default solver parameters (:26-39), one problem at a
 *   time; nIterations / lIterations stay upper bounds.  Changes results (a different algorithm); out_costs holds the
 *   accepted cost after init and after every step, entries of steps not taken repeat the last one.  0 (default) =
 *   gaussNewtonGPU, what the ARAP app requests (CombinedSolverBase.h:76).
 * Returns non-zero for unknown names / bad values. */
ARAPB200_API int arapb200_batch_set_option(arapb200_batch* b, const char* name, double value);

/* Error state of a plan made by Opt_ProblemPlan (include/Opt.h).  Opt_ProblemInit / Step / Solve have no error return
 * in the reference's ABI (ARAP/API/release/include/Opt.h:60-68) and the reference exits the process on a CUDA failure
 * (ARAP/API/src/solverGPUGaussNewton.t:59-73); this library records the failure instead: 0 = fine, otherwise the code of
 * the first failure (Opt_ProblemCurrentCost then returns NaN and Opt_ProblemStep reports "finished"). */
struct Opt_Plan;
ARAPB200_API int arapb200_plan_error(struct Opt_Plan* plan);

/* Opt_InitializationParameters.collectPerKernelTimingInfo (ARAP/API/release/include/Opt.h:22-24, util.t:404-510): every
 * kernel launch of a solve is bracketed by a CUDA event pair under the reference's kernel name and aggregated at the end of
 * the solve (when Opt_ProblemStep returns 0 / Opt_ProblemSolve returns).  Such a plan runs on the streaming back-end with
 * eager launches (a persistent kernel has nothing to time per kernel; results are the same bits).  With verbosityLevel > 0
 * the table is printed like the reference's Timer:evaluate does; this call returns it in any case: copies at most
 * cap - 1 characters into buf (may be NULL), returns the full length (0 = no finished solve / no timing). */
ARAPB200_API size_t arapb200_plan_timing_report(struct Opt_Plan* plan, char* buf, size_t cap);

/* Opt_ProblemDefine(state, file, "LMGPU") selects the reference's other solver kind (ARAP/API/src/o.t:121-124,
 * ARAP/API/src/solverGPUGaussNewton.t with UsesLambda(): Levenberg-Marquardt trust region around the same PCG, Q-based
 * early exit of the linear loop, step acceptance / revert; never requested by the ARAP app).  Its solver parameters
 * (Opt_SetSolverParameter, :26-39, :140-157) are floats -- min_relative_decrease, min_trust_region_radius,
 * max_trust_region_radius, q_tolerance, function_tolerance, trust_region_radius, radius_decrease_factor,
 * min_lm_diagonal, max_lm_diagonal -- and the int residual_reset_period.  This call reports what the last
 * Opt_ProblemStep of such a plan did: info6 = trust-region radius after the step, linear iterations run, verdict
 * (1 accepted, 0 reverted, 2 function tolerance reached, 3 radius below the minimum), model cost, cost at the trial
 * point, last Q.  Returns 0, or 1 when the plan is not an LM plan. */
ARAPB200_API int arapb200_plan_lm_info(struct Opt_Plan* plan, float info6[6]);

/* ---- debug / parity entry points (unit-level comparison against the oracle) ----------------- */
/* one Opt_ProblemSolve on host buffers: X float2[N] and A float[N] in/out; U, C float2[N]; M float[N];
 * costs float[nGN+1] (may be NULL); scal float[nGN*nPCG*3] (den, num, bnum per PCG iteration; may be NULL) */
ARAPB200_API int arapb200_debug_gn_solve(int W, int H, float* X, float* A, const float* U, const float* C, const float* M,
                            float wf, float wr, int nGN, int nPCG, int backend, float* costs, float* scal);
/* r = -J^T F and pre (float3[N] each, zero on inactive pixels) */
ARAPB200_API int arapb200_debug_eval_jtf(int W, int H, const float* X, const float* A, const float* U, const float* C,
                            const float* M, float wf, float wr, float* r3, float* pre3);
/* q = J^T J p (float3[N]); *dot = p.q per the summation contract */
ARAPB200_API int arapb200_debug_apply_jtj(int W, int H, const float* A, const float* U, const float* C, const float* M,
                             float wf, float wr, const float* p3, float* q3, float* dot);
/* cost per the contract */
ARAPB200_API int arapb200_debug_cost(int W, int H, const float* X, const float* A, const float* U, const float* C,
                        const float* M, float wf, float wr, float* cost);
/* cycle accounting of the resident kernel: prof uint64[160*16] (per CTA: cycles in PCG phase 1/2/3, other,
 * barrier skew / poll / fold, barrier count), info int[3] = {strips, CTAs, warps per CTA}, *ms = launch time */
ARAPB200_API int arapb200_debug_resident_profile(int W, int H, const uint8_t* mask_red, const int32_t* matches,
                                                 int n_matches, int nCont, int nGN, int nPCG,
                                                 unsigned long long* prof, int* info, float* ms);
/* the same for the first of `copies` (1..16) identical problems that share ONE cooperative launch: what one problem's
 * phases and barriers cost next to co-resident neighbours; returns 4 when they do not fit one launch */
ARAPB200_API int arapb200_debug_resident_profile_group(int W, int H, const uint8_t* mask_red, const int32_t* matches,
                                                       int n_matches, int copies, int nCont, int nGN, int nPCG,
                                                       unsigned long long* prof, int* info, float* ms);
/* contract sincos and exact sum on the device */
ARAPB200_API int arapb200_debug_sincos(int n, const float* a, float* s, float* c);
ARAPB200_API int arapb200_debug_exact_sum(size_t n, const float* t, float* sum);
/* the same sum through the streaming back-end's fence-free wide fixed-point accumulators (one block per 256 terms) */
ARAPB200_API int arapb200_debug_wide_sum(size_t n, const float* t, float* sum);

#ifdef __cplusplus
}
#endif
#endif
