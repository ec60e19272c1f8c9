"""ctypes binding of libarapb200.so (include/Opt.h + include/arapb200.h).

The shared library is the product; this module only marshals numpy buffers into its C ABI.  There is no
fallback of any kind: if the library is missing or no CUDA device is present, calls raise.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# ARAPB200_LIB selects another build of the same library (A/B measurements, tools/build_variant.sh)
LIB_PATH = os.environ.get("ARAPB200_LIB") or os.path.join(_HERE, "libarapb200.so")

BACKEND_AUTO, BACKEND_STREAM, BACKEND_RESIDENT = 0, 1, 2

# every symbol include/Opt.h and include/arapb200.h declare
OPT_SYMBOLS = [
    "Opt_NewState", "Opt_ProblemDefine", "Opt_ProblemDelete", "Opt_ProblemPlan", "Opt_PlanFree",
    "Opt_SetSolverParameter", "Opt_ProblemSolve", "Opt_ProblemInit", "Opt_ProblemStep", "Opt_ProblemCurrentCost",
]
ARAP_SYMBOLS = [
    "arapb200_device_info", "arapb200_version", "arapb200_warp", "arapb200_warp_flow", "arapb200_deform",
    "arapb200_batch_create", "arapb200_batch_destroy", "arapb200_batch_submit", "arapb200_batch_run",
    "arapb200_batch_timing", "arapb200_batch_launches", "arapb200_debug_gn_solve", "arapb200_debug_eval_jtf",
    "arapb200_debug_apply_jtj", "arapb200_debug_cost", "arapb200_debug_sincos", "arapb200_debug_exact_sum",
    "arapb200_debug_resident_profile", "arapb200_debug_resident_profile_group", "arapb200_flatten", "arapb200_filter_matches", "arapb200_segment_mask",
    "arapb200_batch_set_option", "arapb200_batch_resident_count", "arapb200_debug_wide_sum", "arapb200_plan_error", "arapb200_plan_lm_info", "arapb200_plan_timing_report",
    "arapb200_batch_launch_info", "arapb200_warp_ex", "arapb200_batch_submit_ex", "arapb200_flatten_ex",
    "arapb200_warp_seq", "arapb200_batch_submit_seq", "arapb200_composite", "arapb200_batch_submit_scene",
    "arapb200_batch_scene_blur", "arapb200_blur_schedule",
]


class OptInitializationParameters(C.Structure):
    _fields_ = [("doublePrecision", C.c_int), ("verbosityLevel", C.c_int),
                ("collectPerKernelTimingInfo", C.c_int), ("threadsPerBlock", C.c_int)]


_f32p = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
_u8p = np.ctypeslib.ndpointer(dtype=np.uint8, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")

_lib = None


def load():
    """Load the library (raises if it has not been built: run `python -c 'import __graft_entry__ as g; g.build()'`)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: build it with arap_flow_b200/csrc/Makefile (no CPU fallback exists)")
    L = C.CDLL(LIB_PATH)
    L.arapb200_version.restype = C.c_char_p
    L.arapb200_device_info.argtypes = [C.POINTER(C.c_int), C.POINTER(C.c_size_t), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.arapb200_warp.argtypes = [C.c_int, C.c_int, _f32p, _u8p, _u8p, _u8p, _u8p, C.c_void_p]
    L.arapb200_warp_flow.argtypes = [C.c_int, C.c_int, _f32p, _u8p, _u8p, _u8p, _u8p, C.c_void_p]
    L.arapb200_deform.argtypes = [C.c_int, C.c_int, _u8p, _u8p, _i32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                  _f32p, _u8p, _u8p, C.c_void_p]
    L.arapb200_batch_create.argtypes = [C.c_int] * 7
    L.arapb200_batch_create.restype = C.c_void_p
    L.arapb200_batch_destroy.argtypes = [C.c_void_p]
    L.arapb200_batch_destroy.restype = None
    L.arapb200_batch_submit.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.arapb200_batch_run.argtypes = [C.c_void_p]
    L.arapb200_batch_timing.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
    L.arapb200_batch_launches.argtypes = [C.c_void_p]
    L.arapb200_batch_launches.restype = C.c_longlong
    L.arapb200_debug_gn_solve.argtypes = [C.c_int, C.c_int, _f32p, _f32p, _f32p, _f32p, _f32p, C.c_float, C.c_float,
                                          C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    L.arapb200_debug_eval_jtf.argtypes = [C.c_int, C.c_int, _f32p, _f32p, _f32p, _f32p, _f32p, C.c_float, C.c_float,
                                          _f32p, _f32p]
    L.arapb200_debug_apply_jtj.argtypes = [C.c_int, C.c_int, _f32p, _f32p, _f32p, _f32p, C.c_float, C.c_float,
                                           _f32p, _f32p, C.POINTER(C.c_float)]
    L.arapb200_debug_cost.argtypes = [C.c_int, C.c_int, _f32p, _f32p, _f32p, _f32p, _f32p, C.c_float, C.c_float,
                                      C.POINTER(C.c_float)]
    L.arapb200_debug_sincos.argtypes = [C.c_int, _f32p, _f32p, _f32p]
    L.arapb200_debug_exact_sum.argtypes = [C.c_size_t, _f32p, C.POINTER(C.c_float)]
    # Opt.h
    L.Opt_NewState.argtypes = [OptInitializationParameters]
    L.Opt_NewState.restype = C.c_void_p
    L.Opt_ProblemDefine.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p]
    L.Opt_ProblemDefine.restype = C.c_void_p
    L.Opt_ProblemDelete.argtypes = [C.c_void_p, C.c_void_p]
    L.Opt_ProblemDelete.restype = None
    L.Opt_ProblemPlan.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_uint)]
    L.Opt_ProblemPlan.restype = C.c_void_p
    L.Opt_PlanFree.argtypes = [C.c_void_p, C.c_void_p]
    L.Opt_PlanFree.restype = None
    L.Opt_SetSolverParameter.argtypes = [C.c_void_p, C.c_void_p, C.c_char_p, C.c_void_p]
    L.Opt_SetSolverParameter.restype = None
    for n in ("Opt_ProblemSolve", "Opt_ProblemInit"):
        getattr(L, n).argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]
        getattr(L, n).restype = None
    L.Opt_ProblemStep.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]
    L.Opt_ProblemStep.restype = C.c_int
    L.Opt_ProblemCurrentCost.argtypes = [C.c_void_p, C.c_void_p]
    L.Opt_ProblemCurrentCost.restype = C.c_double
    _lib = L
    return L


def _c(a, dt):
    return np.ascontiguousarray(a, dtype=dt)


def _check(rc, what):
    if rc != 0:
        raise RuntimeError(f"{what} failed with code {rc}")


def device_info():
    sm, l2, ma, mi = C.c_int(), C.c_size_t(), C.c_int(), C.c_int()
    _check(load().arapb200_device_info(C.byref(sm), C.byref(l2), C.byref(ma), C.byref(mi)), "arapb200_device_info")
    return dict(sm_count=sm.value, l2_bytes=l2.value, cc=(ma.value, mi.value))


def warp(pos, rgb, mask_red, want_splat=True):
    """Forward warp from absolute positions (== CombinedSolver::copyResultToCPU).  Returns (rgb, mask, splat)."""
    H, W = mask_red.shape
    o_rgb = np.zeros((H, W, 3), np.uint8)
    o_m = np.zeros((H, W), np.uint8)
    sp = np.zeros((H, W), np.uint32) if want_splat else None
    _check(load().arapb200_warp(W, H, _c(pos, np.float32), _c(rgb, np.uint8), _c(mask_red, np.uint8), o_rgb, o_m,
                                sp.ctypes.data if want_splat else None), "arapb200_warp")
    return o_rgb, o_m, sp


def warp_flow(flow, rgb, mask_red, want_splat=True):
    """warp_image: forward warp from a flow field (ARAP/warping/src/main.cpp:145-225)."""
    H, W = mask_red.shape
    o_rgb = np.zeros((H, W, 3), np.uint8)
    o_m = np.zeros((H, W), np.uint8)
    sp = np.zeros((H, W), np.uint32) if want_splat else None
    _check(load().arapb200_warp_flow(W, H, _c(flow, np.float32), _c(rgb, np.uint8), _c(mask_red, np.uint8), o_rgb, o_m,
                                     sp.ctypes.data if want_splat else None), "arapb200_warp_flow")
    return o_rgb, o_m, sp


def warp_ex(pos_or_flow, rgb, mask_red, is_flow=False):
    """The warp with its extra outputs (include/arapb200.h arapb200_warp_ex, DESIGN.md 4.3): absolute positions, or a
    forward flow with is_flow=True.  Returns a dict: rgb, mask, splat as warp(); bflow[H,W,2] f32, the backward flow on
    the frame-2 grid; occ[H,W] u8, the occlusion of frame 1 (0 visible in frame 2, 255 not)."""
    H, W = mask_red.shape
    out = dict(rgb=np.zeros((H, W, 3), np.uint8), mask=np.zeros((H, W), np.uint8), splat=np.zeros((H, W), np.uint32),
               bflow=np.zeros((H, W, 2), np.float32), occ=np.zeros((H, W), np.uint8))
    L = load()
    L.arapb200_warp_ex.argtypes = [C.c_int, C.c_int, _f32p, C.c_int, _u8p, _u8p, _u8p, _u8p, C.c_void_p, C.c_void_p,
                                   C.c_void_p]
    _check(L.arapb200_warp_ex(W, H, _c(pos_or_flow, np.float32), int(bool(is_flow)), _c(rgb, np.uint8),
                              _c(mask_red, np.uint8), out["rgb"], out["mask"], out["splat"].ctypes.data,
                              out["bflow"].ctypes.data, out["occ"].ctypes.data), "arapb200_warp_ex")
    return out


SEQ_KEYS = ("rgb", "mask", "flow", "bflow", "occ", "flow0")


def _seq_arrays(K, H, W):
    return dict(rgb=np.zeros((K, H, W, 3), np.uint8), mask=np.zeros((K, H, W), np.uint8),
                flow=np.zeros((K, H, W, 2), np.float32), bflow=np.zeros((K, H, W, 2), np.float32),
                occ=np.zeros((K, H, W), np.uint8), flow0=np.zeros((K, H, W, 2), np.float32))


def warp_seq(positions, rgb, mask_red):
    """A frame sequence from position fields (include/arapb200.h arapb200_warp_seq, DESIGN.md 4.4): positions[K,H,W,2]
    are P_1 .. P_K, frame 0 is the input image on the pixel grid.  Returns a dict of arrays with a leading K axis, index
    k - 1 holding frame k: rgb, mask (the warp of P_k), flow (frame k-1 -> k on the frame k-1 grid), bflow (frame k ->
    k-1 on the frame k grid), occ (occlusion of frame k-1 in frame k, 0 visible, 255 not), flow0 (P_k - grid)."""
    H, W = mask_red.shape
    pos = _c(positions, np.float32)
    K = pos.shape[0]
    assert pos.shape == (K, H, W, 2), pos.shape
    out = _seq_arrays(K, H, W)
    L = load()
    L.arapb200_warp_seq.argtypes = [C.c_int, C.c_int, C.c_int, _f32p, _u8p, _u8p] + [C.c_void_p] * 6
    _check(L.arapb200_warp_seq(W, H, K, pos, _c(rgb, np.uint8), _c(mask_red, np.uint8),
                               *[out[k].ctypes.data for k in SEQ_KEYS]), "arapb200_warp_seq")
    return out


def deform(rgb, mask_red, matches, nCont=19, nGN=8, nPCG=400, backend=BACKEND_AUTO):
    """arap_deform for one image/segment: returns (flow[H,W,2], warped_rgb, warped_mask, costs[nCont,nGN+1])."""
    H, W = mask_red.shape
    m = _c(matches, np.int32).reshape(-1, 4)
    flow = np.zeros((H, W, 2), np.float32)
    o_rgb = np.zeros((H, W, 3), np.uint8)
    o_m = np.zeros((H, W), np.uint8)
    costs = np.zeros((nCont, nGN + 1), np.float32)
    _check(load().arapb200_deform(W, H, _c(rgb, np.uint8), _c(mask_red, np.uint8), m, len(m), nCont, nGN, nPCG,
                                  backend, flow, o_rgb, o_m, costs.ctypes.data), "arapb200_deform")
    return flow, o_rgb, o_m, costs


def flatten(flows, rgbs, masks, background=None):
    """Layer the per-segment results of a --multseg pair and composite the background (para_gen.py:136-175, 50-61)."""
    n = len(flows)
    H, W = masks[0].shape
    fl = [_c(f, np.float32) for f in flows]
    rg = [_c(r, np.uint8) for r in rgbs]
    mk = [_c(m, np.uint8) for m in masks]
    P = C.c_void_p * n
    bg = _c(background, np.uint8) if background is not None else None
    o_f = np.zeros((H, W, 2), np.float32)
    o_r = np.zeros((H, W, 3), np.uint8)
    o_m = np.zeros((H, W), np.uint8)
    L = load()
    L.arapb200_flatten.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p]
    _check(L.arapb200_flatten(W, H, n, P(*[a.ctypes.data for a in fl]), P(*[a.ctypes.data for a in rg]),
                              P(*[a.ctypes.data for a in mk]), bg.ctypes.data if bg is not None else None,
                              o_f.ctypes.data, o_r.ctypes.data, o_m.ctypes.data), "arapb200_flatten")
    return o_f, o_r, o_m


def flatten_ex(flows, rgbs, masks, src_masks=None, bflows=None, background=None, extras=True):
    """flatten() plus, with extras, the flattened backward flow and the occlusion of frame 1 across the layers
    (arapb200_flatten_ex).  src_masks: each segment's frame-1 input mask (0 = object); bflows: each segment's backward
    flow; both are needed with extras.  Returns a dict flow, rgb, mask (+ bflow[H,W,2] f32, occ[H,W] u8 with extras)."""
    n = len(flows)
    H, W = masks[0].shape
    arrs = [None if group is None else [_c(a, dt) for a in group] for group, dt in
            ((flows, np.float32), (rgbs, np.uint8), (masks, np.uint8), (src_masks, np.uint8), (bflows, np.float32))]
    P = C.c_void_p * n
    ptrs = [None if group is None else P(*[a.ctypes.data for a in group]) for group in arrs]
    bg = _c(background, np.uint8) if background is not None else None
    out = dict(flow=np.zeros((H, W, 2), np.float32), rgb=np.zeros((H, W, 3), np.uint8), mask=np.zeros((H, W), np.uint8))
    if extras:
        out.update(bflow=np.zeros((H, W, 2), np.float32), occ=np.zeros((H, W), np.uint8))
    L = load()
    L.arapb200_flatten_ex.argtypes = [C.c_int] * 3 + [C.c_void_p] * 11
    _check(L.arapb200_flatten_ex(W, H, n, ptrs[0], ptrs[1], ptrs[2], bg.ctypes.data if bg is not None else None, ptrs[3],
                                 ptrs[4], out["flow"].ctypes.data, out["rgb"].ctypes.data, out["mask"].ctypes.data,
                                 out["bflow"].ctypes.data if extras else None, out["occ"].ctypes.data if extras else None),
           "arapb200_flatten_ex")
    return out


COMPOSITE_ARGTYPES = [C.c_int] * 3 + [C.c_void_p] * 5 + [C.c_int] * 2 + [C.c_void_p] + [C.c_int] * 2 + [C.c_void_p] * 8


def _motion(m):
    m = np.ascontiguousarray(m, np.float64)
    if m.shape != (2, 3):
        raise ValueError(f"a motion is a 2x3 affine matrix, got shape {m.shape}")
    return m


def composite(flows, rgbs, masks, src_masks, bflows, background, motion, motion_from=None, origin=(0, 0), extras=True,
              shape=None):
    """The layers of flatten_ex over a background that moves by its own affine map (arapb200_composite, DESIGN.md 4.5):
    frame b rendered from frame a.  motion / motion_from: 2x3 float64 maps from the background plane to frames b / a
    (motion_from None = identity, the pair case).  background uint8[bgH,bgW,3]; frame pixel q of a still background shows
    background[q + origin].  src_masks: each layer's frame-a input mask (0 = object); bflows: each layer's backward flow,
    needed with extras.  shape=(H, W) is needed only with no layers.  Returns a dict flow (frame a), rgb, mask (frame b),
    coeffs[3,2,3] f32 (the maps F: a -> b, B: b -> a, S: b -> background plane, as the kernels used them), and with
    extras bflow[H,W,2] (frame b) and occ[H,W] (frame a, 0 visible in frame b, 255 not)."""
    n = len(masks)
    H, W = masks[0].shape if n else shape
    groups = [None if g is None else [_c(a, dt) for a in g] for g, dt in
              ((flows, np.float32), (rgbs, np.uint8), (masks, np.uint8), (src_masks, np.uint8), (bflows, np.float32))]
    P = C.c_void_p * n
    ptrs = [None if g is None or n == 0 else P(*[a.ctypes.data for a in g]) for g in groups]
    bg = _c(background, np.uint8)
    mt = _motion(motion)
    mf = None if motion_from is None else _motion(motion_from)
    out = dict(flow=np.zeros((H, W, 2), np.float32), rgb=np.zeros((H, W, 3), np.uint8), mask=np.zeros((H, W), np.uint8),
               coeffs=np.zeros((3, 2, 3), np.float32))
    if extras:
        out.update(bflow=np.zeros((H, W, 2), np.float32), occ=np.zeros((H, W), np.uint8))
    L = load()
    L.arapb200_composite.argtypes = COMPOSITE_ARGTYPES
    _check(L.arapb200_composite(W, H, n, *ptrs, bg.shape[1], bg.shape[0], bg.ctypes.data, int(origin[0]), int(origin[1]),
                                None if mf is None else mf.ctypes.data, mt.ctypes.data, out["flow"].ctypes.data,
                                out["rgb"].ctypes.data, out["mask"].ctypes.data,
                                out["bflow"].ctypes.data if extras else None, out["occ"].ctypes.data if extras else None,
                                out["coeffs"].ctypes.data), "arapb200_composite")
    return out


def composite_seq(seqs, src_masks, background, motions, origin=(0, 0)):
    """A layered frame sequence over a moving background (DESIGN.md 4.5).  seqs: per layer, the out["seq"] dict of
    Batch.submit(..., frames=...) (K frames each); src_masks: the layers' input masks; motions[K] the background's
    motions A_1 .. A_K (frame 0 has the identity; synth.motion_path gives the chord path).  Frame k is composite() of the
    layers' frame k with motion_from = A_{k-1}, motion = A_k and as source masks the input masks for k = 1 and
    255 - mask[k-1] for k >= 2.  Frame 0 is the caller's: it must show the background crop
    background[oy:oy+H, ox:ox+W] where no layer is.  Returns composite()'s keys (with extras) stacked on a leading K axis."""
    K = len(motions)
    assert seqs and all(len(q["mask"]) == K for q in seqs), "one seq per layer, K frames each, K = len(motions)"
    frames = []
    for k in range(K):
        src = list(src_masks) if k == 0 else [255 - q["mask"][k - 1] for q in seqs]
        frames.append(composite([q["flow"][k] for q in seqs], [q["rgb"][k] for q in seqs], [q["mask"][k] for q in seqs],
                                src, [q["bflow"][k] for q in seqs], background, motions[k],
                                motion_from=None if k == 0 else motions[k - 1], origin=origin))
    return {key: np.stack([f[key] for f in frames]) for key in frames[0]}


BLUR_SCHEDULE_ARGTYPES = [C.c_int] * 2 + [C.c_void_p] * 3 + [C.c_int, C.c_double, C.c_int] + [C.c_void_p] * 3


def blur_schedule(nCont, steps, motion, frame_motions, n_samples, shutter, image):
    """The sub-frame table of one blurred image of a scene (arapb200_blur_schedule, DESIGN.md 4.8): image -1 = frame 0,
    0 = the pair, k = frame k of the frames at `steps` (None or empty: no frames) with motions frame_motions (A_1 ..
    A_K); motion is the pair's A.  Returns (state int32[S], the lower continuation state of each sub-frame's lerp, -1 =
    the pixel grid; w float32[S], its weight; smap float32[S,2,3], the map from the frame to the background plane)."""
    st = np.ascontiguousarray([] if steps is None else steps, np.int32).reshape(-1)
    K = len(st)
    fm = np.ascontiguousarray(np.asarray(frame_motions, np.float64).reshape(-1, 2, 3)) if K else None
    if K and len(fm) != K:
        raise ValueError(f"{len(fm)} frame motions for {K} frames")
    A = _motion(motion)
    S = int(n_samples)
    state, w, smap = np.zeros(max(S, 1), np.int32), np.zeros(max(S, 1), np.float32), np.zeros((max(S, 1), 2, 3), np.float32)
    L = load()
    L.arapb200_blur_schedule.argtypes = BLUR_SCHEDULE_ARGTYPES
    _check(L.arapb200_blur_schedule(int(nCont), K, st.ctypes.data if K else None, A.ctypes.data,
                                    fm.ctypes.data if K else None, S, float(shutter), int(image), state.ctypes.data,
                                    w.ctypes.data, smap.ctypes.data), "arapb200_blur_schedule")
    return state, w, smap


def filter_matches(matches, labels1, labels2):
    """N3: keep the matches para_gen.valid_cnstr keeps (para_gen.py:216-223, 468-482), in order.
    Returns (matches int32[k,4], labels uint8[k])."""
    m = _c(np.asarray(matches, np.int32).reshape(-1, 4), np.int32)
    l1, l2 = _c(labels1, np.uint8), _c(labels2, np.uint8)
    n = m.shape[0]
    out = np.zeros((max(n, 1), 4), np.int32)
    lab = np.zeros(max(n, 1), np.uint8)
    cnt = C.c_int(0)
    L = load()
    L.arapb200_filter_matches.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                          C.c_void_p, C.c_void_p, C.POINTER(C.c_int)]
    _check(L.arapb200_filter_matches(l1.shape[1], l1.shape[0], l1.ctypes.data, l2.shape[1], l2.shape[0], l2.ctypes.data,
                                     m.ctypes.data, n, out.ctypes.data, lab.ctypes.data, C.byref(cnt)),
           "arapb200_filter_matches")
    return out[:cnt.value].copy(), lab[:cnt.value].copy()


def segment_mask(labels, segment=0):
    """N3: the mask image arap_deform expects (0 = solve, 255 = ARAP_BG): one label (--multseg) or all (segment=0)."""
    l = _c(labels, np.uint8)
    out = np.zeros(l.shape, np.uint8)
    L = load()
    L.arapb200_segment_mask.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
    _check(L.arapb200_segment_mask(l.shape[1], l.shape[0], l.ctypes.data, int(segment), out.ctypes.data),
           "arapb200_segment_mask")
    return out


class Batch:
    """Many independent (image, segment) problems on the current device (arapb200_batch_*)."""

    def __init__(self, maxW, maxH, max_problems, nCont=19, nGN=8, nPCG=400, backend=BACKEND_AUTO):
        self.L = load()
        self.nCont, self.nGN = nCont, nGN
        self.h = self.L.arapb200_batch_create(maxW, maxH, max_problems, nCont, nGN, nPCG, backend)
        if not self.h:
            raise RuntimeError("arapb200_batch_create failed")
        self._keep = {}

    def set_option(self, name: str, value: float):
        """Opt-in behaviour beyond the reference (include/arapb200.h): e.g. set_option("pcg_rtol", 1e-3)."""
        self.L.arapb200_batch_set_option.argtypes = [C.c_void_p, C.c_char_p, C.c_double]
        _check(self.L.arapb200_batch_set_option(self.h, name.encode(), float(value)), "arapb200_batch_set_option")

    def submit(self, slot, rgb, mask_red, matches, out=None, extras=False, frames=None):
        """Queue one problem.  `out` may be the dict a previous submit() of the same image size returned: its arrays are
        then written in place instead of allocating fresh ones (what a caller looping over many pairs does).
        extras=True: the dict also gets bflow[H,W,2] f32 (backward flow) and occ[H,W] u8 (occlusion of frame 1, 0 visible,
        255 not), as lib.warp_ex computes them on the solved positions (arapb200_batch_submit_ex).
        frames: a strictly increasing list of continuation steps in [0, nCont-1]; the dict then also gets "seq", the
        dict lib.warp_seq returns for the solver's states after those steps (arapb200_batch_submit_seq)."""
        H, W = mask_red.shape
        rgb = _c(rgb, np.uint8)
        mask_red = _c(mask_red, np.uint8)
        m = _c(matches, np.int32).reshape(-1, 4)
        if out is None or out["flow"].shape != (H, W, 2):
            out = dict(flow=np.zeros((H, W, 2), np.float32), rgb=np.zeros((H, W, 3), np.uint8),
                       mask=np.zeros((H, W), np.uint8), costs=np.zeros((self.nCont, self.nGN + 1), np.float32))
        if extras and "bflow" not in out:
            out.update(bflow=np.zeros((H, W, 2), np.float32), occ=np.zeros((H, W), np.uint8))
        steps = None
        if frames is not None:
            steps = np.ascontiguousarray(frames, np.int32).reshape(-1)
            if "seq" not in out or out["seq"]["mask"].shape[0] != len(steps):
                out["seq"] = _seq_arrays(len(steps), H, W)
        self._keep[slot] = (rgb, mask_red, m, out)
        args = (self.h, slot, W, H, rgb.ctypes.data, mask_red.ctypes.data, m.ctypes.data, len(m), out["flow"].ctypes.data,
                out["rgb"].ctypes.data, out["mask"].ctypes.data, out["costs"].ctypes.data)
        if steps is not None:
            self.L.arapb200_batch_submit_seq.argtypes = (self.L.arapb200_batch_submit.argtypes +
                                                         [C.c_void_p, C.c_void_p, C.c_int] + [C.c_void_p] * 7)
            seq = out["seq"]
            _check(self.L.arapb200_batch_submit_seq(
                *args, out["bflow"].ctypes.data if extras else None, out["occ"].ctypes.data if extras else None,
                len(steps), steps.ctypes.data, *[seq[k].ctypes.data for k in SEQ_KEYS]), "arapb200_batch_submit_seq")
        elif extras:
            self.L.arapb200_batch_submit_ex.argtypes = self.L.arapb200_batch_submit.argtypes + [C.c_void_p, C.c_void_p]
            _check(self.L.arapb200_batch_submit_ex(*args, out["bflow"].ctypes.data, out["occ"].ctypes.data),
                   "arapb200_batch_submit_ex")
        else:
            _check(self.L.arapb200_batch_submit(*args), "arapb200_batch_submit")
        return out

    SCENE_KEYS = ("flow", "rgb", "mask", "bflow", "occ")

    def submit_scene(self, slot, rgb, masks, matches, background, motion, origin=(0, 0), frames=None, frame_motions=None,
                     input_frame=False, out=None, blur=None):
        """Queue a scene (arapb200_batch_submit_scene, DESIGN.md 4.6): one image rgb, its segments' masks (0 = object, in
        segment order) with one match list each, and a background uint8[bgH,bgW,3] that moves by the 2x3 float64 map
        `motion` (frame pixel q of a still background shows background[q + origin]).  The layers take slots
        slot .. slot + len(masks) - 1, are solved and warped like submit(..., extras=True) problems and composited on the
        device; only the composite is copied out.  Returns a dict with composite()'s image keys (flow, rgb, mask, bflow,
        occ: what composite() gives for those layers with motion_from=None), costs[n_layers, nCont, nGN+1], with
        input_frame=True rgb0[H,W,3] (frame 0: rgb on the objects, the background crop elsewhere), and with frames (a
        strictly increasing list of continuation steps) and frame_motions (A_1 .. A_K, e.g. synth.motion_path) "seq",
        stacked like composite_seq()'s result.  `out` may be the dict a previous submit_scene() of the same shape returned:
        its arrays are then written in place.
        blur=(n_samples, shutter): motion blur (arapb200_batch_scene_blur, DESIGN.md 4.8) adds blur_rgb[H,W,3], with
        input_frame blur_rgb0[H,W,3], and with frames seq["blur_rgb"][K,H,W,3]: each image averaged over n_samples
        sub-frames of a trailing shutter open for the fraction `shutter` of the interval before it.  The sub-frame table
        of every image to blur is checked (lib.blur_schedule) before anything is queued, so a request the library would
        refuse raises with no scene queued."""
        n = len(masks)
        H, W = masks[0].shape
        rgb = _c(rgb, np.uint8)
        mk = [_c(m, np.uint8) for m in masks]
        mt = [_c(m, np.int32).reshape(-1, 4) for m in matches]
        if len(mt) != n:
            raise ValueError(f"{n} masks but {len(mt)} match lists")
        bg = _c(background, np.uint8)
        A = _motion(motion)
        steps = fm = None
        K = 0
        if frames is not None:
            steps = np.ascontiguousarray(frames, np.int32).reshape(-1)
            K = len(steps)
        if frame_motions is not None:
            fm = np.ascontiguousarray(np.asarray(frame_motions, np.float64).reshape(-1, 2, 3))
            if len(fm) != K:   # the library reads one motion per frame
                raise ValueError(f"{len(fm)} frame motions for {K} frames")
        if blur is not None:
            for image in ([-1] if input_frame else []) + list(range(K + 1)):
                blur_schedule(self.nCont, steps, A, fm, blur[0], blur[1], image)
        if out is None or out["flow"].shape != (H, W, 2) or out["costs"].shape[0] != n:
            out = dict(flow=np.zeros((H, W, 2), np.float32), rgb=np.zeros((H, W, 3), np.uint8),
                       mask=np.zeros((H, W), np.uint8), bflow=np.zeros((H, W, 2), np.float32),
                       occ=np.zeros((H, W), np.uint8), costs=np.zeros((n, self.nCont, self.nGN + 1), np.float32))
        if input_frame and "rgb0" not in out:
            out["rgb0"] = np.zeros((H, W, 3), np.uint8)
        elif not input_frame:
            out.pop("rgb0", None)
        if K and ("seq" not in out or out["seq"]["mask"].shape[0] != K):
            out["seq"] = dict(flow=np.zeros((K, H, W, 2), np.float32), rgb=np.zeros((K, H, W, 3), np.uint8),
                              mask=np.zeros((K, H, W), np.uint8), bflow=np.zeros((K, H, W, 2), np.float32),
                              occ=np.zeros((K, H, W), np.uint8))
        elif not K:
            out.pop("seq", None)
        P = C.c_void_p * n
        ptrs = (P(*[m.ctypes.data for m in mk]), P(*[m.ctypes.data for m in mt]), (C.c_int * n)(*[len(m) for m in mt]))
        self._keep[slot] = (rgb, mk, mt, bg, A, steps, fm, ptrs, out)
        seq = out.get("seq")
        if blur is not None:
            out.setdefault("blur_rgb", np.zeros((H, W, 3), np.uint8))
            if input_frame:
                out.setdefault("blur_rgb0", np.zeros((H, W, 3), np.uint8))
            else:
                out.pop("blur_rgb0", None)
            if K:
                seq.setdefault("blur_rgb", np.zeros((K, H, W, 3), np.uint8))
        else:
            out.pop("blur_rgb", None)
            out.pop("blur_rgb0", None)
            if seq is not None:
                seq.pop("blur_rgb", None)
        self.L.arapb200_batch_submit_scene.argtypes = ([C.c_void_p] + [C.c_int] * 4 + [C.c_void_p] * 4 + [C.c_int] * 2 +
                                                       [C.c_void_p] + [C.c_int] * 2 + [C.c_void_p, C.c_int] +
                                                       [C.c_void_p] * 14)
        _check(self.L.arapb200_batch_submit_scene(
            self.h, slot, n, W, H, rgb.ctypes.data, *ptrs, bg.shape[1], bg.shape[0], bg.ctypes.data, int(origin[0]),
            int(origin[1]), A.ctypes.data, K, None if steps is None else steps.ctypes.data,
            None if fm is None else fm.ctypes.data, *[out[k].ctypes.data for k in self.SCENE_KEYS],
            out["rgb0"].ctypes.data if input_frame else None, out["costs"].ctypes.data,
            *[None if seq is None else seq[k].ctypes.data for k in ("rgb", "mask", "flow", "bflow", "occ")]),
            "arapb200_batch_submit_scene")
        if blur is not None:
            n_samples, shutter = blur
            self.L.arapb200_batch_scene_blur.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double] + [C.c_void_p] * 3
            _check(self.L.arapb200_batch_scene_blur(
                self.h, slot, int(n_samples), float(shutter), out["blur_rgb"].ctypes.data,
                out["blur_rgb0"].ctypes.data if input_frame else None, seq["blur_rgb"].ctypes.data if K else None),
                "arapb200_batch_scene_blur")
        return out

    def run(self):
        _check(self.L.arapb200_batch_run(self.h), "arapb200_batch_run")

    def timing_ms(self):
        ms = (C.c_float * 3)()
        self.L.arapb200_batch_timing(self.h, ms)
        return dict(total=ms[0], solve=ms[1], warp=ms[2])

    def launches(self):
        return int(self.L.arapb200_batch_launches(self.h))

    def resident_count(self):
        """Problems of the last run() that the resident back-end solved (the others streamed)."""
        self.L.arapb200_batch_resident_count.argtypes = [C.c_void_p]
        return int(self.L.arapb200_batch_resident_count(self.h))

    def launch_info(self):
        """Shape of the last cooperative launch of the last run() (zeros if every problem streamed)."""
        info = (C.c_int * 6)()
        self.L.arapb200_batch_launch_info.argtypes = [C.c_void_p, C.POINTER(C.c_int)]
        _check(self.L.arapb200_batch_launch_info(self.h, info), "arapb200_batch_launch_info")
        return dict(problems_per_launch=info[0], variant=(info[1], info[2]), grid=(info[3], info[4]), threads=info[5])

    def close(self):
        if self.h:
            self.L.arapb200_batch_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---- unit-level parity entry points -----------------------------------------------------------------
def debug_gn_solve(X, A, U, Cn, M, nGN, nPCG, wf, wr, backend=BACKEND_AUTO, trace=False):
    H, W = M.shape
    X = _c(X, np.float32).copy()
    A = _c(A, np.float32).copy()
    costs = np.zeros(nGN + 1, np.float32)
    scal = np.zeros((nGN, nPCG, 3), np.float32) if trace else None
    _check(load().arapb200_debug_gn_solve(W, H, X, A, _c(U, np.float32), _c(Cn, np.float32), _c(M, np.float32),
                                          wf, wr, nGN, nPCG, backend, costs.ctypes.data,
                                          scal.ctypes.data if trace else None), "arapb200_debug_gn_solve")
    return X, A, costs, scal


def debug_eval_jtf(X, A, U, Cn, M, wf, wr):
    H, W = M.shape
    r = np.zeros((H, W, 3), np.float32)
    pre = np.zeros((H, W, 3), np.float32)
    _check(load().arapb200_debug_eval_jtf(W, H, _c(X, np.float32), _c(A, np.float32), _c(U, np.float32),
                                          _c(Cn, np.float32), _c(M, np.float32), wf, wr, r, pre), "debug_eval_jtf")
    return r, pre


def debug_apply_jtj(A, U, Cn, M, p, wf, wr):
    H, W = M.shape
    q = np.zeros((H, W, 3), np.float32)
    d = C.c_float()
    _check(load().arapb200_debug_apply_jtj(W, H, _c(A, np.float32), _c(U, np.float32), _c(Cn, np.float32),
                                           _c(M, np.float32), wf, wr, _c(p, np.float32), q, C.byref(d)), "debug_apply_jtj")
    return q, np.float32(d.value)


def debug_cost(X, A, U, Cn, M, wf, wr):
    H, W = M.shape
    c = C.c_float()
    _check(load().arapb200_debug_cost(W, H, _c(X, np.float32), _c(A, np.float32), _c(U, np.float32),
                                      _c(Cn, np.float32), _c(M, np.float32), wf, wr, C.byref(c)), "debug_cost")
    return np.float32(c.value)


def debug_resident_profile(mask_red, matches, nCont, nGN, nPCG, copies=1):
    """Cycle accounting of the resident kernel (thread 0 of every CTA) for one problem, or for the first of `copies`
    identical problems sharing one cooperative launch.  Returns (prof[G, 16], info, ms)."""
    H, W = mask_red.shape
    m = _c(matches, np.int32).reshape(-1, 4)
    prof = np.zeros((160, 16), np.uint64)
    info = (C.c_int * 3)()
    ms = C.c_float()
    L = load()
    L.arapb200_debug_resident_profile.argtypes = [C.c_int, C.c_int, _u8p, _i32p, C.c_int, C.c_int, C.c_int, C.c_int,
                                                  C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_float)]
    L.arapb200_debug_resident_profile_group.argtypes = [C.c_int, C.c_int, _u8p, _i32p, C.c_int, C.c_int, C.c_int, C.c_int,
                                                        C.c_int, C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_float)]
    if copies > 1:
        _check(L.arapb200_debug_resident_profile_group(W, H, _c(mask_red, np.uint8), m, len(m), copies, nCont, nGN, nPCG,
                                                       prof.ctypes.data, info, C.byref(ms)), "debug_resident_profile_group")
    else:
        _check(L.arapb200_debug_resident_profile(W, H, _c(mask_red, np.uint8), m, len(m), nCont, nGN, nPCG,
                                                 prof.ctypes.data, info, C.byref(ms)), "debug_resident_profile")
    G = info[1]
    return prof[:G], dict(strips=info[0], ctas=info[1], warps=info[2]), ms.value


def debug_sincos(a):
    a = _c(a, np.float32).ravel()
    s = np.zeros_like(a)
    c = np.zeros_like(a)
    _check(load().arapb200_debug_sincos(a.size, a, s, c), "debug_sincos")
    return s, c


def debug_wide_sum(t):
    t = _c(t, np.float32).ravel()
    out = C.c_float()
    L = load()
    L.arapb200_debug_wide_sum.argtypes = [C.c_size_t, _f32p, C.POINTER(C.c_float)]
    _check(L.arapb200_debug_wide_sum(t.size, t, C.byref(out)), "debug_wide_sum")
    return np.float32(out.value)


def debug_exact_sum(t):
    t = _c(t, np.float32).ravel()
    out = C.c_float()
    _check(load().arapb200_debug_exact_sum(t.size, t, C.byref(out)), "debug_exact_sum")
    return np.float32(out.value)
