"""CUDA path vs the CPU oracle, through the C ABI (libarapb200.so).  Bit-exact unless stated otherwise."""
import os

import numpy as np
import pytest

from arap_flow_b200 import flowio, lib, synth
from tests.helpers import cat512_flo, epe, random_problem, synth_gn_problem

pytestmark = pytest.mark.gpu


def _eq(a, b):
    """value equality (treats -0 == +0), NaN-free"""
    return np.array_equal(np.asarray(a), np.asarray(b))


# ------------------------------------------------------------------------------------- scalar contract
def test_contract_sincos_bit_exact(oracle):
    rng = np.random.default_rng(1)
    a = np.concatenate([rng.uniform(-10, 10, 20000), rng.uniform(-1e-3, 1e-3, 2000), [0.0, 1e4, -3e4]]).astype(np.float32)
    s, c = lib.debug_sincos(a)
    ref = np.array([oracle.sincos(float(x)) for x in a])
    assert _eq(s, ref[:, 0]) and _eq(c, ref[:, 1])


def test_exact_sum_bit_exact(oracle):
    rng = np.random.default_rng(2)
    for n in (1, 33, 256, 5000, 200000):
        t = (rng.standard_normal(n) * 10.0 ** rng.uniform(-6, 6, n)).astype(np.float32)
        assert lib.debug_exact_sum(t) == oracle.exact_sum(t)


def _exact_f32_sum(t):
    """Sum of binary32 values, exact in integer arithmetic (units of 2^-149), rounded ONCE to nearest-even binary32."""
    import math
    from fractions import Fraction
    T = sum(int(Fraction(float(x)) * (1 << 149)) for x in t)
    if T == 0:
        return np.float32(0.0)
    a, nb = abs(T), abs(T).bit_length()
    sh = max(nb - 24, 0)
    q, rem = a >> sh, a & ((1 << sh) - 1)
    if sh and (rem > (1 << (sh - 1)) or (rem == (1 << (sh - 1)) and (q & 1))):
        q += 1
    return np.float32(math.copysign(math.ldexp(q, sh - 149), T))


def test_wide_accumulator_sums_exactly(oracle):
    """The streaming back-end's fence-free 320-bit accumulators: exact whatever the arrival order, rounded once --
    wide dynamic range, massive cancellation, negative totals, round-to-even ties, subnormal totals, zeros."""
    rng = np.random.default_rng(11)
    cases = []
    for n in (1, 257, 5000, 100000):
        cases.append((rng.standard_normal(n) * 10.0 ** rng.uniform(-30, 30, n)).astype(np.float32))
    x = (rng.standard_normal(20000) * 10.0 ** rng.uniform(-10, 10, 20000)).astype(np.float32)
    # cancellation ACROSS blocks over 200 binades (inside one 256-term block the (h, l) partial is the contract's
    # binned sum, exact only up to ~2^-98 of the block's largest term: keep every block on one exponent so that the
    # partials are exact and the accumulator alone is under test)
    blocks = [np.ldexp(rng.integers(-255, 256, 256).astype(np.float32), int(e)) for e in rng.integers(-100, 100, 150)]
    blocks = blocks + [-b for b in blocks] + [np.ldexp(np.float32([3.0] + [0.0] * 255), -120)]
    order = rng.permutation(len(blocks))
    cases.append(np.concatenate([blocks[i] for i in order]).astype(np.float32))                        # total = 3 * 2^-120
    cases.append(-np.abs(x))                                                                           # negative total
    cases.append(np.float32([16777216.0, 1.0]))                                                        # tie -> even (down)
    cases.append(np.float32([16777218.0, 1.0]))                                                        # tie -> even (up)
    cases.append(np.float32([16777216.0, 1.0, 1e-30]))                                                 # sticky breaks the tie
    cases.append(np.float32([1e-45] * 700 + [-3e-45] * 100))                                           # subnormal total
    cases.append(np.float32([3e38, 3e38, -3e38, -2.9e38]))                                             # partials beyond FLT_MAX
    cases.append(np.zeros(1000, np.float32))
    for t in cases:
        want = _exact_f32_sum(t)
        got = lib.debug_wide_sum(t)
        assert got == want and np.signbit(got) == np.signbit(want), (len(t), got, want)
    # and it agrees with the oracle's and the resident path's summation on PCG-like data
    t = (rng.standard_normal(200000) ** 2 * 10.0 ** rng.uniform(-8, 2, 200000)).astype(np.float32)
    assert lib.debug_wide_sum(t) == oracle.exact_sum(t) == lib.debug_exact_sum(t)


# ------------------------------------------------------------------------------------- single kernels
@pytest.mark.parametrize("W,H,seed", [(37, 29, 0), (64, 64, 1), (100, 70, 2), (33, 5, 3), (1, 9, 4)])
def test_kernels_bit_exact(oracle, W, H, seed):
    pr = random_problem(W, H, seed)
    wf, wr = oracle.WF, oracle.WR
    r_o, pre_o = oracle.eval_jtf(pr["X"], pr["A"], pr["U"], pr["C"], pr["M"])
    r_g, pre_g = lib.debug_eval_jtf(pr["X"], pr["A"], pr["U"], pr["C"], pr["M"], wf, wr)
    assert _eq(r_g, r_o) and _eq(pre_g, pre_o)
    q_o, d_o = oracle.apply_jtj(pr["A"], pr["U"], pr["C"], pr["M"], pr["p"])
    q_g, d_g = lib.debug_apply_jtj(pr["A"], pr["U"], pr["C"], pr["M"], pr["p"], wf, wr)
    assert _eq(q_g, q_o) and d_g == d_o
    assert lib.debug_cost(pr["X"], pr["A"], pr["U"], pr["C"], pr["M"], wf, wr) == \
        oracle.cost(pr["X"], pr["A"], pr["U"], pr["C"], pr["M"])


def test_kernels_empty_and_full_masks(oracle):
    for p_in in (0.0, 1.0):
        pr = random_problem(40, 33, 7, p_inactive=p_in)
        q_o, d_o = oracle.apply_jtj(pr["A"], pr["U"], pr["C"], pr["M"], pr["p"])
        q_g, d_g = lib.debug_apply_jtj(pr["A"], pr["U"], pr["C"], pr["M"], pr["p"], oracle.WF, oracle.WR)
        assert _eq(q_g, q_o) and d_g == d_o


# ------------------------------------------------------------------------------------- Opt_ProblemSolve level
@pytest.mark.parametrize("backend", [lib.BACKEND_STREAM, lib.BACKEND_RESIDENT])
@pytest.mark.parametrize("W,H,seed,nGN,nPCG", [(64, 64, 0, 3, 40), (150, 97, 1, 2, 60), (96, 128, 2, 2, 25)])
def test_gn_solve_bit_exact(oracle, backend, W, H, seed, nGN, nPCG):
    pr = synth_gn_problem(oracle, W, H, seed, fd=2)
    Xo, Ao, co, so = oracle.gn_solve(pr["X"], pr["A"], pr["U"], pr["C"], pr["M"], nGN, nPCG, trace=True)
    Xg, Ag, cg, sg = lib.debug_gn_solve(pr["X"], pr["A"], pr["U"], pr["C"], pr["M"], nGN, nPCG, oracle.WF, oracle.WR,
                                        backend=backend, trace=True)
    assert _eq(sg, so), "per-iteration PCG scalars (den, num, bnum) differ"
    assert _eq(cg, co) and _eq(Xg, Xo) and _eq(Ag, Ao)


def test_gn_solve_random_state_bit_exact(oracle):
    """start from a perturbed state with non-zero angles (exercises every sin/cos path)"""
    pr = random_problem(80, 60, 11, p_inactive=0.2, n_cstr=40)
    Xo, Ao, co, so = oracle.gn_solve(pr["X"], pr["A"], pr["U"], pr["C"], pr["M"], 2, 30, trace=True)
    Xg, Ag, cg, sg = lib.debug_gn_solve(pr["X"], pr["A"], pr["U"], pr["C"], pr["M"], 2, 30, oracle.WF, oracle.WR,
                                        backend=lib.BACKEND_STREAM, trace=True)
    assert _eq(sg, so) and _eq(cg, co) and _eq(Xg, Xo) and _eq(Ag, Ao)


# ------------------------------------------------------------------------------------- whole arap_deform path
@pytest.mark.parametrize("backend", [lib.BACKEND_STREAM, lib.BACKEND_RESIDENT])
def test_deform_c0_full_schedule(oracle, backend):
    """BASELINE config C0 (64x64, fd=1), the full 19 x 8 x 400 schedule."""
    sp = synth.config("C0")
    mask = sp.masks[0]
    Xo, Ao, co = oracle.solve(mask, sp.matches)
    flo_o = oracle.flow(Xo)
    rgb_o, m_o, sp_o = oracle.warp(Xo, sp.rgb, mask)
    flo_g, rgb_g, m_g, cg = lib.deform(sp.rgb, mask, sp.matches, backend=backend)
    act = mask == 0
    # north_star tolerances, stated: flow within 1e-3 px mean EPE, final energy within 1e-4 relative
    assert epe(flo_g, flo_o, act).mean() < 1e-3
    assert abs(float(cg[-1, -1]) - float(co[-1, -1])) <= 1e-4 * abs(float(co[-1, -1]))
    # ... and in fact the contract makes it exact
    assert _eq(flo_g, flo_o) and _eq(cg, co)
    assert _eq(rgb_g, rgb_o) and _eq(m_g, m_o)
    assert (flo_g[~act] == 0).all()


def test_deform_multiseg_shared_constraints(oracle):
    """--multseg quirk (para_gen.py:523-536): every segment run gets the SAME constraint file; foreign matches
    are dropped by the mask test.  Reduced schedule."""
    sp = synth.synth(128, 96, 4, 3, 2000)
    for mask in sp.masks:
        Xo, Ao, co = oracle.solve(mask, sp.matches, nCont=3, nGN=2, nPCG=40)
        flo_g, rgb_g, m_g, cg = lib.deform(sp.rgb, mask, sp.matches, nCont=3, nGN=2, nPCG=40)
        assert _eq(flo_g, oracle.flow(Xo)) and _eq(cg, co)
        rgb_o, m_o, _ = oracle.warp(Xo, sp.rgb, mask)
        assert _eq(rgb_g, rgb_o) and _eq(m_g, m_o)


def test_deform_edge_cases(oracle):
    sp = synth.synth(40, 36, 1, 1, 3)
    # empty object: nothing moves, nothing lands
    none = np.full((36, 40), 255, np.uint8)
    flo, rgb, m, c = lib.deform(sp.rgb, none, sp.matches, nCont=2, nGN=1, nPCG=5)
    assert not flo.any() and not rgb.any() and not m.any() and not c.any()
    # no matches at all; object touching the border gets pinned there
    mask = sp.masks[0].copy()
    mask[:, :6] = 0
    Xo, Ao, co = oracle.solve(mask, np.zeros((0, 4), np.int32), nCont=2, nGN=2, nPCG=10)
    flo, rgb, m, c = lib.deform(sp.rgb, mask, np.zeros((0, 4), np.int32), nCont=2, nGN=2, nPCG=10)
    assert _eq(flo, oracle.flow(Xo)) and _eq(c, co)
    # duplicate sources (later wins) and off-object / out-of-image sources are ignored
    mm = np.array([[20, 18, 23, 18], [20, 18, 21, 20], [0, 0, 5, 5], [39, 35, 30, 30], [-3, 2, 1, 1]], np.int32)
    Xo, Ao, co = oracle.solve(sp.masks[0], mm, nCont=2, nGN=2, nPCG=30)
    flo, rgb, m, c = lib.deform(sp.rgb, sp.masks[0], mm, nCont=2, nGN=2, nPCG=30)
    assert _eq(flo, oracle.flow(Xo)) and _eq(c, co)


# ------------------------------------------------------------------------------------- forward warp
def test_warp_golden_cat512(oracle, gold, tmp_path):
    rgb = flowio.read_png_rgb(os.path.join(gold, "cat512_iRGB.png"))
    msk = flowio.read_png_mask_red(os.path.join(gold, "cat512_iMsk.png"))
    flo = flowio.read_flo(cat512_flo(tmp_path))
    r, m, sp = lib.warp_flow(flo, rgb, msk)
    assert _eq(m, flowio.read_png_rgb(os.path.join(gold, "cat512_wMsk.png"))[..., 0])          # shipped golden
    assert _eq(r, flowio.read_png_rgb(os.path.join(gold, "cat512_reftool_wRGB.png")))          # reference tool
    ro, mo, spo = oracle.warp(oracle.flow_to_pos(flo), rgb, msk)
    assert _eq(sp, spo) and _eq(r, ro) and _eq(m, mo)                                          # splat indices


def test_warp_reference_tool_cases(oracle, gold):
    z = np.load(os.path.join(gold, "warp_reftool_cases.npz"))
    for name in ("warp_a", "warp_b", "warp_c"):
        r, m, sp = lib.warp_flow(z[f"{name}__flow"], z[f"{name}__rgb"], z[f"{name}__mask"])
        assert _eq(r, z[f"{name}__ref_rgb"]) and _eq(m, z[f"{name}__ref_mask"]), name
        _, _, spo = oracle.warp(oracle.flow_to_pos(z[f"{name}__flow"]), z[f"{name}__rgb"], z[f"{name}__mask"])
        assert _eq(sp, spo), name


@pytest.mark.parametrize("W,H,amp,seed", [(97, 61, 4.0, 0), (200, 120, 40.0, 1), (64, 64, 0.0, 2), (3, 2, 1.0, 3)])
def test_warp_random_vs_oracle(oracle, W, H, amp, seed):
    rng = np.random.default_rng(seed)
    rgb = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    mask = np.where(rng.random((H, W)) < 0.2, 255, 0).astype(np.uint8)
    pos = (oracle.grid(W, H) + rng.standard_normal((H, W, 2)) * amp).astype(np.float32)
    if amp > 10:  # degenerate + non-finite corners
        pos[5, 5] = pos[5, 6]
        pos[10, 10] = np.nan
        pos[12, 12] = np.inf
    r, m, sp = lib.warp(pos, rgb, mask)
    ro, mo, spo = oracle.warp(pos, rgb, mask)
    assert _eq(sp, spo) and _eq(r, ro) and _eq(m, mo)


def test_warp_full_size_properties():
    """1920x1080 (C4 shape): identity flow reproduces the interior of the object exactly; deterministic."""
    sp = synth.config("C4")
    mask = sp.masks[0]
    zero = np.zeros((1080, 1920, 2), np.float32)
    r1, m1, s1 = lib.warp_flow(zero, sp.rgb, mask)
    r2, m2, s2 = lib.warp_flow(zero, sp.rgb, mask)
    assert _eq(r1, r2) and _eq(m1, m2) and _eq(s1, s2)
    act = mask == 0
    quad = act[:-1, :-1] & act[1:, :-1] & act[:-1, 1:] & act[1:, 1:]
    cov = np.zeros_like(act)
    for dy in (0, 1):
        for dx in (0, 1):
            cov[dy:1080 - 1 + dy, dx:1920 - 1 + dx] |= quad
    assert _eq(m1 == 255, cov)
    assert _eq(r1[cov], sp.rgb[cov])


# ------------------------------------------------------------------------------------- Opt.h boundary
def test_opt_h_boundary_through_ctypes(oracle):
    """Drive the library exactly as OptSolver does (ARAP/shared/OptSolver.h:43-91) with torch-owned device images."""
    import ctypes as C
    import torch
    L = lib.load()
    pr = synth_gn_problem(oracle, 72, 56, seed=4, fd=2)
    dev = torch.device("cuda:0")
    t = {k: torch.from_numpy(np.ascontiguousarray(pr[k])).to(dev) for k in ("X", "A", "U", "C", "M")}
    torch.cuda.synchronize()
    st = L.Opt_NewState(lib.OptInitializationParameters(0, 0, 0, 0))
    plan_file = os.path.join(os.path.dirname(lib.LIB_PATH), "arap_plan.t").encode()
    prob = L.Opt_ProblemDefine(st, plan_file, b"gaussNewtonGPU")
    dims = (C.c_uint * 2)(72, 56)
    plan = L.Opt_ProblemPlan(st, prob, dims)
    assert st and prob and plan
    nGN, nPCG = C.c_uint(3), C.c_uint(35)
    L.Opt_SetSolverParameter(st, plan, b"nIterations", C.byref(nGN))
    L.Opt_SetSolverParameter(st, plan, b"lIterations", C.byref(nPCG))
    L.Opt_SetSolverParameter(st, plan, b"no_such_parameter", C.byref(nGN))  # warns at most
    wf, wr = C.c_float(float(oracle.WF)), C.c_float(float(oracle.WR))
    pp = (C.c_void_p * 7)(t["X"].data_ptr(), t["A"].data_ptr(), t["U"].data_ptr(), t["C"].data_ptr(),
                          t["M"].data_ptr(), C.cast(C.byref(wf), C.c_void_p), C.cast(C.byref(wr), C.c_void_p))
    L.Opt_ProblemSolve(st, plan, pp)
    cost = L.Opt_ProblemCurrentCost(st, plan)
    Xo, Ao, co, _ = oracle.gn_solve(pr["X"], pr["A"], pr["U"], pr["C"], pr["M"], 3, 35)
    assert _eq(t["X"].cpu().numpy(), Xo) and _eq(t["A"].cpu().numpy(), Ao) and np.float32(cost) == co[-1]
    # stepwise API (launchProfiledSolve, OptUtils.h:47-64) on a fresh state gives the same trajectory
    t2 = {k: torch.from_numpy(np.ascontiguousarray(pr[k])).to(dev) for k in ("X", "A")}
    torch.cuda.synchronize()
    pp[0], pp[1] = t2["X"].data_ptr(), t2["A"].data_ptr()
    L.Opt_ProblemInit(st, plan, pp)
    costs = [L.Opt_ProblemCurrentCost(st, plan)]
    while L.Opt_ProblemStep(st, plan, pp):
        costs.append(L.Opt_ProblemCurrentCost(st, plan))
    assert _eq(np.float32(costs), co) and L.Opt_ProblemStep(st, plan, pp) == 0
    assert _eq(t2["X"].cpu().numpy(), Xo)
    L.Opt_PlanFree(st, plan)
    L.Opt_ProblemDelete(st, prob)


# ------------------------------------------------------------------------------------- full-size configs
@pytest.mark.parametrize("cfg,kw", [("C1", dict(nCont=2, nGN=2, nPCG=60)), ("C3", dict(nCont=1, nGN=2, nPCG=40))])
def test_full_size_backends_and_oracle_agree(oracle, cfg, kw):
    """854x480 (C1) and 1024x436 (C3) at a reduced schedule: oracle == streaming == resident, bit for bit."""
    sp = synth.config(cfg)
    mask = sp.masks[0]
    Xo, Ao, co = oracle.solve(mask, sp.matches, **kw)
    for backend in (lib.BACKEND_STREAM, lib.BACKEND_RESIDENT):
        flo, rgb, m, c = lib.deform(sp.rgb, mask, sp.matches, backend=backend, **kw)
        assert _eq(c, co), (cfg, backend)
        assert _eq(flo, oracle.flow(Xo)), (cfg, backend)
    rgb_o, m_o, _ = oracle.warp(Xo, sp.rgb, mask)
    assert _eq(rgb, rgb_o) and _eq(m, m_o)


def test_c4_streams_and_matches_oracle(oracle):
    """1920x1080 (C4): too large for the on-chip state, AUTO falls back to streaming; still exact."""
    sp = synth.config("C4")
    mask = sp.masks[0]
    kw = dict(nCont=1, nGN=1, nPCG=12)
    Xo, Ao, co = oracle.solve(mask, sp.matches, **kw)
    flo, rgb, m, c = lib.deform(sp.rgb, mask, sp.matches, backend=lib.BACKEND_AUTO, **kw)
    assert _eq(c, co) and _eq(flo, oracle.flow(Xo))


def test_full_schedule_size_independent_properties():
    """C1 at the full 19x8x400 schedule through the default (resident) path: deterministic run to run,
    zero flow off the object, matches met, cost trajectory finite and decreasing within each continuation step."""
    sp = synth.config("C1")
    mask = sp.masks[0]
    f1, r1, m1, c1 = lib.deform(sp.rgb, mask, sp.matches)
    f2, r2, m2, c2 = lib.deform(sp.rgb, mask, sp.matches)
    assert _eq(f1, f2) and _eq(c1, c2) and _eq(r1, r2) and _eq(m1, m2)
    act = mask == 0
    assert (f1[~act] == 0).all() and np.isfinite(f1).all() and np.isfinite(c1).all()
    err = np.array([np.hypot(*(f1[y1, x1] - (x2 - x1, y2 - y1))) for x1, y1, x2, y2 in sp.matches])
    assert err.max() < 0.05, err.max()
    assert (c1[:, -1] <= c1[:, 0]).all()


def test_batch_api_matches_single_problem_calls():
    """arapb200_batch_*: problems that share one cooperative launch give exactly the single-problem results."""
    sps = [synth.synth(160, 120, 1, 2, 300 + i) for i in range(4)] + [synth.synth(160, 120, 2, 3, 400)]
    jobs = [(s, s.masks[0]) for s in sps] + [(sps[-1], sps[-1].masks[1])]
    kw = dict(nCont=2, nGN=2, nPCG=40)
    b = lib.Batch(160, 120, len(jobs), **kw)
    outs = [b.submit(i, s.rgb, m, s.matches) for i, (s, m) in enumerate(jobs)]
    b.run()
    assert b.launches() > 0
    for o, (s, m) in zip(outs, jobs):
        flow, rgb, wm, costs = lib.deform(s.rgb, m, s.matches, **kw)
        assert _eq(o["flow"], flow) and _eq(o["costs"], costs) and _eq(o["rgb"], rgb) and _eq(o["mask"], wm)
    b.close()


def test_flatten_and_background_composite_vs_numpy_restatement():
    """N1: para_gen.flatten + add_bg on the GPU vs oracle/pycomposite.py (line-by-line numpy restatement)."""
    from oracle import pycomposite as PC
    rng = np.random.default_rng(3)
    H, W, n = 75, 131, 4
    flows = [rng.standard_normal((H, W, 2)).astype(np.float32) for _ in range(n)]
    rgbs = [rng.integers(0, 256, (H, W, 3), dtype=np.uint8) for _ in range(n)]
    masks = [np.where(rng.random((H, W)) < 0.3, 255, 0).astype(np.uint8) for _ in range(n)]
    bg = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    f_o, r_o, m_o = PC.flatten(flows, rgbs, masks)
    f_g, r_g, m_g = lib.flatten(flows, rgbs, masks)
    assert _eq(f_g, f_o) and _eq(r_g, r_o) and _eq(m_g, m_o)
    f_g, r_g, m_g = lib.flatten(flows, rgbs, masks, background=bg)
    assert _eq(r_g, PC.add_bg(r_o, m_o, bg)) and _eq(f_g, f_o) and _eq(m_g, m_o)
    # single layer: flatten is the identity, background fills where nothing landed
    f1, r1, m1 = lib.flatten(flows[:1], rgbs[:1], masks[:1], background=bg)
    assert _eq(f1, flows[0]) and _eq(m1, masks[0]) and _eq(r1, PC.add_bg(rgbs[0], masks[0], bg))


def test_opt_h_multiple_live_states_and_plans(oracle):
    """Opt_NewState has no matching free and is called again on every re-plan (CombinedSolver.h:155-159): several
    states / plans of different sizes must coexist and interleave."""
    import ctypes as C
    import torch
    L = lib.load()
    plan_file = os.path.join(os.path.dirname(lib.LIB_PATH), "arap_plan.t").encode()
    dev = torch.device("cuda:0")
    jobs = []
    for (W, H, seed) in ((64, 48, 21), (96, 40, 22)):
        pr = synth_gn_problem(oracle, W, H, seed=seed, fd=2)
        st = L.Opt_NewState(lib.OptInitializationParameters(0, 0, 0, 0))
        prob = L.Opt_ProblemDefine(st, plan_file, b"gaussNewtonGPU")
        plan = L.Opt_ProblemPlan(st, prob, (C.c_uint * 2)(W, H))
        t = {k: torch.from_numpy(np.ascontiguousarray(pr[k])).to(dev) for k in ("X", "A", "U", "C", "M")}
        jobs.append(dict(pr=pr, st=st, prob=prob, plan=plan, t=t))
    torch.cuda.synchronize()
    nGN, nPCG = C.c_uint(2), C.c_uint(25)
    wf, wr = C.c_float(float(oracle.WF)), C.c_float(float(oracle.WR))
    for rep in range(2):          # two Opt_ProblemSolve calls per plan, interleaved (= two continuation steps)
        for j in jobs:
            t = j["t"]
            L.Opt_SetSolverParameter(j["st"], j["plan"], b"nIterations", C.byref(nGN))
            L.Opt_SetSolverParameter(j["st"], j["plan"], b"lIterations", C.byref(nPCG))
            pp = (C.c_void_p * 7)(t["X"].data_ptr(), t["A"].data_ptr(), t["U"].data_ptr(), t["C"].data_ptr(),
                                  t["M"].data_ptr(), C.cast(C.byref(wf), C.c_void_p), C.cast(C.byref(wr), C.c_void_p))
            L.Opt_ProblemSolve(j["st"], j["plan"], pp)
            j.setdefault("costs", []).append(L.Opt_ProblemCurrentCost(j["st"], j["plan"]))
    for j in jobs:
        pr = j["pr"]
        X, A, c1, _ = oracle.gn_solve(pr["X"], pr["A"], pr["U"], pr["C"], pr["M"], 2, 25)
        X, A, c2, _ = oracle.gn_solve(X, A, pr["U"], pr["C"], pr["M"], 2, 25)
        assert _eq(j["t"]["X"].cpu().numpy(), X) and _eq(j["t"]["A"].cpu().numpy(), A)
        assert _eq(np.float32(j["costs"]), np.float32([c1[-1], c2[-1]]))
        L.Opt_PlanFree(j["st"], j["plan"])
        L.Opt_ProblemDelete(j["st"], j["prob"])


def test_multiseg_pair_end_to_end_c2_shape(oracle):
    """BASELINE config C2 (854x480, 4 segments, fd=3) at a reduced schedule: four independent per-segment solves share
    one cooperative launch, every segment receives the SAME constraint file, then the layers are flattened."""
    from oracle import pycomposite as PC
    sp = synth.config("C2")
    kw = dict(nCont=1, nGN=2, nPCG=30)
    b = lib.Batch(sp.W, sp.H, 4, **kw)
    outs = [b.submit(s, sp.rgb, sp.masks[s], sp.matches) for s in range(4)]
    b.run()
    flows, rgbs, masks = [], [], []
    for s, o in enumerate(outs):
        Xo, Ao, co = oracle.solve(sp.masks[s], sp.matches, **kw)
        assert _eq(o["flow"], oracle.flow(Xo)) and _eq(o["costs"], co), s
        r_o, m_o, _ = oracle.warp(Xo, sp.rgb, sp.masks[s])
        assert _eq(o["rgb"], r_o) and _eq(o["mask"], m_o), s
        flows.append(o["flow"]); rgbs.append(o["rgb"]); masks.append(o["mask"])
    f_g, r_g, m_g = lib.flatten(flows, rgbs, masks)
    f_o, r_o, m_o = PC.flatten(flows, rgbs, masks)
    assert _eq(f_g, f_o) and _eq(r_g, r_o) and _eq(m_g, m_o)
    b.close()


def test_match_filter_and_segment_masks_n3():
    """N3: device-side valid_cnstr filter + per-segment masks vs para_gen.py's own results (fixture) and the numpy
    restatement, including order, out-of-range points, zero-length matches and empty inputs."""
    from oracle import pycomposite as PC
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "para_gen_cases.npz"))
    mk1, mk2, m = z["vc_mk1"], z["vc_mk2"], z["vc_matches"]
    km, kl = lib.filter_matches(m, mk1, mk2)
    assert _eq(km, m[z["vc_keep"]]) and _eq(kl, mk1[km[:, 1], km[:, 0]])
    # a larger random case against the restatement (> 1024 matches: several compaction rounds)
    rng = np.random.default_rng(3)
    H, W = 120, 200
    l1 = rng.integers(0, 4, (H, W)).astype(np.uint8)
    l2 = np.roll(l1, (2, -3), axis=(0, 1))
    n = 5000
    mm = np.stack([rng.integers(0, W + 3, n), rng.integers(0, H + 3, n), rng.integers(0, W + 3, n), rng.integers(0, H + 3, n)], 1)
    mm[:, 2] = np.clip(mm[:, 0] + rng.integers(-4, 5, n), 0, None)
    mm[:, 3] = np.clip(mm[:, 1] + rng.integers(-4, 5, n), 0, None)
    km, kl = lib.filter_matches(mm, l1, l2)
    om, ol = PC.filter_matches(mm, l1, l2)
    assert len(om) > 100 and _eq(km, om) and _eq(kl, ol)
    km, kl = lib.filter_matches(np.zeros((0, 4), np.int32), l1, l2)
    assert km.shape == (0, 4) and kl.shape == (0,)
    for seg in (0, 1, 3):
        assert _eq(lib.segment_mask(l1, seg), PC.segment_mask(l1, seg))
    # and the fixture's flatten case through the GPU path
    f, r, k = lib.flatten(list(z["fl_flows"]), list(z["fl_rgbs"]), list(z["fl_masks"]))
    assert _eq(f, z["fl_out_flow"]) and _eq(r, z["fl_out_rgb"]) and _eq(k, z["fl_out_mask"])
    f, r, k = lib.flatten([z["bg_bg"][..., :2].astype(np.float32)], [z["bg_im"]], [z["bg_mk"]], background=z["bg_bg"])
    assert _eq(r, z["bg_out"])


def test_opt_in_pcg_tolerance_n4(oracle):
    """N4: the convergence-aware schedule is opt-in.  Off (default, or set back to 0) the result is the bit-exact parity
    result; on, the solve ends earlier with a flow close to the full-budget one, and a tolerance nobody reaches
    (1e-30) changes nothing."""
    sp = synth.synth(160, 128, nseg=1, fd=2, seed=5)
    kw = dict(nCont=3, nGN=3, nPCG=200)
    b = lib.Batch(sp.W, sp.H, 1, backend=lib.BACKEND_RESIDENT, **kw)

    def run():
        o = b.submit(0, sp.rgb, sp.masks[0], sp.matches)
        b.run()
        return {k: v.copy() for k, v in o.items()}, b.timing_ms()["solve"]

    full, t_full = run()
    Xo, Ao, co = oracle.solve(sp.masks[0], sp.matches, **kw)
    assert _eq(full["flow"], oracle.flow(Xo)) and _eq(full["costs"], co)
    b.set_option("pcg_rtol", 1e-30)
    same, _ = run()
    assert _eq(same["flow"], full["flow"]) and _eq(same["costs"], full["costs"])
    b.set_option("pcg_rtol", 1e-2)
    fast, t_fast = run()
    # the early-exit path against the ORACLE's implementation of the same rule (not against itself): bit-exact
    try:
        oracle.set_rtol(1e-2, 0.0)
        Xe, Ae, ce = oracle.solve(sp.masks[0], sp.matches, **kw)
        assert _eq(fast["flow"], oracle.flow(Xe)) and _eq(fast["costs"], ce)
        oracle.set_rtol(1e-2, 1e-2)
        Xe2, Ae2, ce2 = oracle.solve(sp.masks[0], sp.matches, **kw)
    finally:
        oracle.set_rtol(0.0, 0.0)
    act = sp.masks[0] == 0
    d = np.linalg.norm(fast["flow"] - full["flow"], axis=-1)[act]
    assert t_fast < 0.8 * t_full, (t_fast, t_full)
    assert d.mean() < 0.5 and abs(fast["costs"][-1, -1] - full["costs"][-1, -1]) < 0.2 * abs(full["costs"][-1, -1]) + 1e-3, (d.mean(), fast["costs"][-1], full["costs"][-1])
    b.set_option("gn_rtol", 1e-2)
    faster, t_faster = run()
    assert _eq(faster["flow"], oracle.flow(Xe2)) and _eq(faster["costs"], ce2)
    d2 = np.linalg.norm(faster["flow"] - full["flow"], axis=-1)[act]
    assert t_faster <= t_fast * 1.05 and d2.mean() < 0.5, (t_faster, t_fast, d2.mean())
    assert np.all(np.diff(faster["costs"], axis=1) <= 1e-6 * np.abs(faster["costs"][:, :-1]) + 1e-9)  # skipped steps repeat the cost
    b.set_option("pcg_rtol", 0.0)
    b.set_option("gn_rtol", 0.0)
    again, _ = run()
    assert _eq(again["flow"], full["flow"])
    with pytest.raises(RuntimeError):
        b.set_option("no_such_option", 1.0)
    b.close()
    # the streaming back-end honours pcg_rtol too (the rest of its captured graph turns into no-ops): same bits as the
    # oracle's early exit, and back to the fixed-budget result when switched off again
    bs = lib.Batch(sp.W, sp.H, 1, backend=lib.BACKEND_STREAM, **kw)
    bs.set_option("pcg_rtol", 1e-2)
    o = bs.submit(0, sp.rgb, sp.masks[0], sp.matches)
    bs.run()
    assert _eq(o["flow"], oracle.flow(Xe)) and _eq(o["costs"], ce)     # (no time bound: at this size the graph is launch-bound)
    bs.set_option("gn_rtol", 1e-2)                                      # ... and gn_rtol, alone or with pcg_rtol
    o = bs.submit(0, sp.rgb, sp.masks[0], sp.matches)
    bs.run()
    assert _eq(o["flow"], oracle.flow(Xe2)) and _eq(o["costs"], ce2)
    bs.set_option("pcg_rtol", 0.0)
    o = bs.submit(0, sp.rgb, sp.masks[0], sp.matches)
    bs.run()
    try:
        oracle.set_rtol(0.0, 1e-2)
        Xe3, Ae3, ce3 = oracle.solve(sp.masks[0], sp.matches, **kw)
    finally:
        oracle.set_rtol(0.0, 0.0)
    assert _eq(o["flow"], oracle.flow(Xe3)) and _eq(o["costs"], ce3)
    assert not _eq(ce3, full["costs"])                                  # the rule did fire
    bs.set_option("gn_rtol", 0.0)
    o = bs.submit(0, sp.rgb, sp.masks[0], sp.matches)
    bs.run()
    assert _eq(o["flow"], full["flow"]) and _eq(o["costs"], full["costs"])
    bs.close()


@pytest.mark.parametrize("W,H,seed", [(70, 45, 0), (128, 96, 1)])
def test_general_urshape_bit_exact(oracle, W, H, seed):
    """An Opt.h caller may bind any UrShape image (arap_plan.t:4); the ARAP app binds the pixel grid.  A non-grid rest
    shape (anisotropic scale + smooth warp) takes the general-d kernels and matches the oracle bit for bit, GN solve,
    costs and per-iteration PCG scalars."""
    pr = random_problem(W, H, seed)
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float32)
    U = np.stack([1.25 * xx + 0.3 * np.sin(yy / 7.0), 0.8 * yy + 0.2 * np.cos(xx / 5.0)], -1).astype(np.float32)
    X0 = (U + pr["X"] - pr["U"]).astype(np.float32)
    Cn = np.where(pr["C"] >= 0, pr["C"] * np.float32(1.1), pr["C"]).astype(np.float32)
    Xo, Ao, co, so = oracle.gn_solve(X0, pr["A"], U, Cn, pr["M"], 2, 30, trace=True)
    Xg, Ag, cg, sg = lib.debug_gn_solve(X0, pr["A"], U, Cn, pr["M"], 2, 30, oracle.WF, oracle.WR, backend=lib.BACKEND_AUTO, trace=True)
    assert _eq(Xg, Xo) and _eq(Ag, Ao) and _eq(cg, co) and _eq(sg, so)
    # single kernels with the general rest shape
    r_o, pre_o = oracle.eval_jtf(X0, pr["A"], U, Cn, pr["M"])
    r_g, pre_g = lib.debug_eval_jtf(X0, pr["A"], U, Cn, pr["M"], oracle.WF, oracle.WR)
    assert _eq(r_g, r_o) and _eq(pre_g, pre_o)
    q_o, d_o = oracle.apply_jtj(pr["A"], U, Cn, pr["M"], pr["p"])
    q_g, d_g = lib.debug_apply_jtj(pr["A"], U, Cn, pr["M"], pr["p"], oracle.WF, oracle.WR)
    assert _eq(q_g, q_o) and d_g == d_o
    assert lib.debug_cost(X0, pr["A"], U, Cn, pr["M"], oracle.WF, oracle.WR) == oracle.cost(X0, pr["A"], U, Cn, pr["M"])
    # and the pixel grid through the same entry point still takes the specialised path with identical results
    Xo, Ao, co, _ = oracle.gn_solve(pr["X"], pr["A"], pr["U"], pr["C"], pr["M"], 1, 20)
    Xg, Ag, cg, _ = lib.debug_gn_solve(pr["X"], pr["A"], pr["U"], pr["C"], pr["M"], 1, 20, oracle.WF, oracle.WR, backend=lib.BACKEND_STREAM)
    assert _eq(Xg, Xo) and _eq(Ag, Ao) and _eq(cg, co)


@pytest.mark.parametrize("backend", [lib.BACKEND_STREAM, lib.BACKEND_RESIDENT])
@pytest.mark.parametrize("kw", [dict(nCont=1, nGN=1, nPCG=0), dict(nCont=1, nGN=0, nPCG=5), dict(nCont=2, nGN=1, nPCG=1),
                                dict(nCont=1, nGN=2, nPCG=1)])
def test_degenerate_schedules(oracle, backend, kw):
    """Zero PCG iterations, zero Gauss-Newton steps, single iterations: the loops' boundary cases (Opt accepts any
    nIterations / lIterations, solverGPUGaussNewton.t:1016-1103)."""
    sp = synth.synth(48, 40, nseg=1, fd=2, seed=3)
    fl, rgb, msk, costs = lib.deform(sp.rgb, sp.masks[0], sp.matches, backend=backend, **kw)
    Xo, Ao, co = oracle.solve(sp.masks[0], sp.matches, **kw)
    assert _eq(fl, oracle.flow(Xo)) and _eq(costs, co)


def test_conditioning_bounds_the_gap_to_any_rounding_order():
    """Parity with the reference's own solver cannot be measured here (DESIGN.md section 2); what can be measured is how
    much ANY rounding-order difference can move the result.  One-ulp perturbations of the two weights through the full
    Opt.h call sequence on a DeepMatching-like problem (C3 geometry, reduced schedule) move the flow by far less than the
    north-star tolerance of 1e-3 px mean EPE and the energy by far less than 1e-4 relative."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("sensitivity", os.path.join(os.path.dirname(os.path.dirname(__file__)), "tools", "sensitivity.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    res = mod.run("C3", 6, 4, 150)
    assert res["worst_mean_epe_px"] < 1e-4 and res["worst_rel_cost_diff"] < 1e-5, res


def test_cluster_scope_barrier_equals_l2_barrier(oracle):
    """Opt-in: small problems (each fits one thread-block cluster) run with a cluster-scope barrier -- limb sums pushed
    through distributed shared memory, mbarrier completion -- instead of the L2 barrier.  Same bits as the L2 path and as the
    oracle; any number of problems per launch; mixed with a large problem in one batch."""
    sps = [synth.synth(160, 120, 1, 2, 500 + i) for i in range(5)] + [synth.synth(320, 200, 2, 3, 600)]
    jobs = [(s, s.masks[0]) for s in sps] + [(sps[-1], sps[-1].masks[1])]
    kw = dict(nCont=2, nGN=2, nPCG=60)
    b = lib.Batch(320, 200, len(jobs), **kw)
    res = {}
    for mode in (1, 0):
        b.set_option("cluster_barrier", mode)
        outs = [b.submit(i, s.rgb, m, s.matches) for i, (s, m) in enumerate(jobs)]
        b.run()
        info = b.launch_info()
        res[mode] = ([{k: v.copy() for k, v in o.items()} for o in outs], info)
    assert res[1][1]["variant"][1] == 0 and res[1][1]["problems_per_launch"] == len(jobs), res[1][1]   # ONE cluster launch
    assert res[0][1]["variant"][1] != 0, res[0][1]
    for a, c in zip(res[1][0], res[0][0]):
        assert _eq(a["flow"], c["flow"]) and _eq(a["costs"], c["costs"]) and _eq(a["rgb"], c["rgb"])
    for o, (s, m) in zip(res[1][0], jobs):
        Xo, Ao, co = oracle.solve(m, s.matches, **kw)
        assert _eq(o["flow"], oracle.flow(Xo)) and _eq(o["costs"], co)
    b.close()
    # a batch that mixes small problems with one that needs the L2 barrier (C1 size)
    big = synth.config("C1")
    small = synth.synth(854, 480, 1, 1, 77, axes=(0.1, 0.1))
    kw = dict(nCont=1, nGN=1, nPCG=30)
    b = lib.Batch(854, 480, 3, **kw)
    b.set_option("cluster_barrier", 1)
    outs = [b.submit(0, small.rgb, small.masks[0], small.matches), b.submit(1, big.rgb, big.masks[0], big.matches),
            b.submit(2, small.rgb, small.masks[0], small.matches)]
    b.run()
    for o, s in zip(outs, (small, big, small)):
        Xo, Ao, co = oracle.solve(s.masks[0], s.matches, **kw)
        assert _eq(o["flow"], oracle.flow(Xo)) and _eq(o["costs"], co)
    b.close()
