"""The resident back-end on the mask geometries real segments produce (objects on the image border, holes, many
components, one-pixel lines, isolated pixels, ragged masks, images smaller than one strip) and on the launch shapes they
select (warps per CTA, co-resident variants, the on-chip limit, mixed batches, tiny problems).  Every comparison is
bit-exact against the CPU oracle, computed here from seeds."""
import numpy as np
import pytest

from arap_flow_b200 import lib, synth
from tests.helpers import (GEOMETRY_CASES, MASKS, ellipse, energy_bound, energy_f64, geometry_gn_problem,
                           geometry_matches, mask_full, strip_count)

pytestmark = pytest.mark.gpu

SCHED = dict(nCont=2, nGN=2, nPCG=40)
SHAPE = dict(nCont=1, nGN=2, nPCG=30)        # launch-shape tests: the shape is the point, keep the oracle cheap


@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _eq(a, b):
    return np.array_equal(np.asarray(a), np.asarray(b))


def _first_diff(a, b):
    d = np.argwhere(np.asarray(a) != np.asarray(b))
    return tuple(int(v) for v in d[0]) if len(d) else None


def _rgb(W, H, seed):
    return np.random.default_rng(seed).integers(0, 256, (H, W, 3), dtype=np.uint8)


def _job(mask, seed):
    H, W = mask.shape
    return dict(rgb=_rgb(W, H, seed), mask=mask, matches=geometry_matches(mask, seed))


def _run(jobs, kw, backend=lib.BACKEND_AUTO, options=(), maxWH=None):
    W = maxWH[0] if maxWH else max(j["mask"].shape[1] for j in jobs)
    H = maxWH[1] if maxWH else max(j["mask"].shape[0] for j in jobs)
    b = lib.Batch(W, H, len(jobs), backend=backend, **kw)
    try:
        for k, v in options:
            b.set_option(k, v)
        outs = [b.submit(i, j["rgb"], j["mask"], j["matches"]) for i, j in enumerate(jobs)]
        b.run()
        return outs, b.launch_info(), b.resident_count()
    finally:
        b.close()


def _check_vs_oracle(oracle, o, job, kw, lm=False):
    mask = job["mask"]
    if lm:
        Xo, _, co, _ = oracle.solve_lm(mask, job["matches"], **kw)
    else:
        Xo, _, co = oracle.solve(mask, job["matches"], **kw)
    assert _eq(o["costs"], co), (o["costs"], co)
    fo = oracle.flow(Xo)
    assert _eq(o["flow"], fo), ("first differing pixel (y, x, c)", _first_diff(o["flow"], fo))
    rgb_o, m_o, _ = oracle.warp(Xo, job["rgb"], mask)
    assert _eq(o["rgb"], rgb_o) and _eq(o["mask"], m_o)


def _expect_launch(info, exp, problems=1, variant=(384, 1), grid=None):
    """A single problem, or several whose CTAs sum to at most SMs, always gets the 168-register variant: it is tried first
    (pick_variant) and keeps at least one CTA of up to 12 warps per SM."""
    assert info["threads"] == 32 * exp["NW"], (info, exp)
    assert info["variant"] == variant, info
    assert info["problems_per_launch"] == problems, info
    assert info["grid"] == (grid if grid is not None else (exp["G"], 1)), (info, exp)


# ------------------------------------------------------------------------------ a. single problem, unit level
@pytest.mark.parametrize("perturbed", [False, True], ids=["rest", "perturbed"])
@pytest.mark.parametrize("name,W,H", GEOMETRY_CASES)
def test_resident_gn_solve_geometry(oracle, name, W, H, perturbed):
    """Opt_ProblemSolve on the resident back-end vs the oracle: X, A, cost per Gauss-Newton step and every PCG iteration's
    (den, num, bnum); then the reported cost against the float64 energy of the returned state."""
    mask = MASKS[name](W, H, 11)
    pr = geometry_gn_problem(oracle, mask, 11, perturbed)
    nGN, nPCG = 2, 40
    Xo, Ao, co, so = oracle.gn_solve(pr["X"], pr["A"], pr["U"], pr["C"], pr["M"], nGN, nPCG, trace=True)
    Xg, Ag, cg, sg = lib.debug_gn_solve(pr["X"], pr["A"], pr["U"], pr["C"], pr["M"], nGN, nPCG, oracle.WF, oracle.WR,
                                        backend=lib.BACKEND_RESIDENT, trace=True)
    assert _eq(sg, so), ("first differing (GN step, PCG iteration, scalar)", _first_diff(sg, so))
    assert _eq(cg, co), (cg, co)
    assert _eq(Xg, Xo), ("first differing X (y, x, c)", _first_diff(Xg, Xo))
    assert _eq(Ag, Ao), ("first differing A (y, x)", _first_diff(Ag, Ao))
    E0, E = energy_f64(oracle, pr["X"], pr["A"], pr), energy_f64(oracle, Xg, Ag, pr)
    assert abs(float(cg[0]) - E0) <= energy_bound(E0, E0), (cg[0], E0)
    assert abs(float(cg[-1]) - E) <= energy_bound(E, E0), (cg[-1], E, E0)


# ------------------------------------------------------------------------------ b. whole arap_deform path
@pytest.mark.parametrize("name,W,H", [(f"border_{s}", 854, 480) for s in ("left", "right", "top", "bottom", "all")] +
                                     [(f"border_{s}", 1024, 436) for s in ("right", "bottom", "all")])
def test_deform_border_objects(oracle, sms, name, W, H):
    """Objects on the image border at C1 / C3 size: the border pins land on object pixels, the last strip column has lanes
    x >= W next to object pixels (and for H = 436 the last strip row rows y >= H)."""
    job = _job(MASKS[name](W, H, 5), 5)
    exp = strip_count(job["mask"], sms)
    (o,), info, nres = _run([job], SCHED)
    assert nres == 1
    _expect_launch(info, exp)
    _check_vs_oracle(oracle, o, job, SCHED)


# ------------------------------------------------------------------------------ c. launch shapes
def _ellipse_nw(W, H, nw, sms):
    """Axes (fraction of the frame) of synth's centred ellipse that gives `nw` warps per CTA on this device."""
    inside = np.zeros((H, W), bool)
    inside[2:H - 2, 2:W - 2] = True
    for a in np.arange(0.20, 0.50, 0.002):
        m = np.where(ellipse(W, H, W / 2.0, H / 2.0, a * W, a * H) & inside, 0, 255).astype(np.uint8)
        if strip_count(m, sms)["NW"] == nw:
            return float(a)
    pytest.fail(f"no ellipse gives NW = {nw} with {sms} SMs")


def _synth_nw(nw, sms, seed=1000):
    a = _ellipse_nw(854, 480, nw, sms)
    sp = synth.synth(854, 480, 1, 1, seed, axes=(a, a))
    return dict(rgb=sp.rgb, mask=sp.masks[0], matches=sp.matches)


@pytest.mark.parametrize("shape", ["nw5", "nw6", "nw8", "full854x480", "full1024x436"])
def test_warps_per_cta(oracle, sms, shape):
    """Enlarged C1 ellipses (NW = 5, 6, 8) and full frames (NW = 11 and 12 with 148 SMs): CTAs of 5..12 warps, their
    shared-memory sizes and local / remote neighbour mixes."""
    if shape.startswith("nw"):
        job = _synth_nw(int(shape[2:]), sms)
    else:
        W, H = (int(v) for v in shape[4:].split("x"))
        job = _job(mask_full(W, H), 7)
    exp = strip_count(job["mask"], sms)
    if shape.startswith("nw"):
        assert exp["NW"] == int(shape[2:])
    (o,), info, nres = _run([job], SHAPE)
    assert nres == 1
    _expect_launch(info, exp)
    _check_vs_oracle(oracle, o, job, SHAPE)


def test_three_coresident_nw5_problems(oracle, sms):
    """Three NW = 5 problems in one launch need three CTAs per SM: only the 128-register variant of up to 160 threads keeps
    that many (3 x 5 warps x 128 registers), so the grouped hoisting and the deferred delta update run with five warps."""
    jobs = [_synth_nw(5, sms, seed=1000 + i) for i in range(3)]
    exps = [strip_count(j["mask"], sms) for j in jobs]
    assert len({e["G"] for e in exps}) == 1 and exps[0]["NW"] == 5 and 3 * exps[0]["G"] > 2 * sms
    outs, info, nres = _run(jobs, SHAPE)
    assert nres == 3
    _expect_launch(info, exps[0], problems=3, variant=(160, 3), grid=(exps[0]["G"], 3))
    for o, j in zip(outs, jobs):
        _check_vs_oracle(oracle, o, j, SHAPE)


def _limit_masks(sms):
    """Full frame of exactly SMs x 12 strips (ragged right and bottom edge), and one of SMs x 12 + 1 strips."""
    fit = mask_full(32 * sms - 5, 93)
    more = np.full((93, 32 * sms + 1), 255, np.uint8)
    more[:, :32 * sms] = 0
    more[0, -1] = 0
    return fit, more


def test_on_chip_limit(oracle, sms):
    """SMs x 12 strips stay resident (12 warps x 12,480 B of shared memory, 384 threads x 168 registers: one CTA per SM);
    one strip more streams under AUTO, and under RESIDENT is refused with an error."""
    fit, more = _limit_masks(sms)
    kw = dict(nCont=1, nGN=1, nPCG=20)
    job = _job(fit, 3)
    exp = strip_count(fit, sms)
    assert exp == dict(strips=12 * sms, NW=12, G=sms, fits=True)
    (o,), info, nres = _run([job], kw)
    assert nres == 1
    _expect_launch(info, exp)
    _check_vs_oracle(oracle, o, job, kw)
    job = _job(more, 4)
    assert not strip_count(more, sms)["fits"]
    (o,), info, nres = _run([job], kw)
    assert nres == 0 and info["threads"] == 0
    _check_vs_oracle(oracle, o, job, kw)
    with pytest.raises(RuntimeError):
        _run([job], kw, backend=lib.BACKEND_RESIDENT)


def test_mixed_batch_nw5_with_small(oracle, sms):
    """A NW = 5 problem with a 64x64 one: the compact 1-D grid, the small problem in CTAs wider than its own NW."""
    jobs = [_synth_nw(5, sms), _job(MASKS["border_all"](64, 64, 2), 2)]
    exps = [strip_count(j["mask"], sms) for j in jobs]
    assert exps[1]["NW"] == 4 and exps[0]["G"] + exps[1]["G"] <= sms
    outs, info, nres = _run(jobs, SHAPE)
    assert nres == 2
    _expect_launch(info, exps[0], problems=2, grid=(exps[0]["G"] + exps[1]["G"], 1))
    for o, j in zip(outs, jobs):
        _check_vs_oracle(oracle, o, j, SHAPE)


@pytest.mark.parametrize("case", ["sizes", "empty_between"])
def test_mixed_batch_geometries(oracle, sms, case):
    """Problems of different W x H in one launch; an empty segment between two real ones."""
    if case == "sizes":
        jobs = [_job(MASKS["border_left"](203, 77, 1), 1), _job(MASKS["holes"](150, 97, 2), 2),
                _job(MASKS["ragged"](320, 200, 3), 3), _job(MASKS["full"](31, 7), 4)]
    else:
        jobs = [_job(MASKS["border_all"](203, 77, 1), 1), _job(MASKS["empty"](203, 77), 2),
                _job(MASKS["components"](203, 77, 3), 3)]
    exps = [strip_count(j["mask"], sms) for j in jobs]
    ctas = sum(e["G"] for e in exps)
    assert max(e["NW"] for e in exps) == 4 and ctas <= sms
    outs, info, nres = _run(jobs, SCHED)
    assert nres == len(jobs)
    _expect_launch(info, dict(NW=4), problems=len(jobs), grid=(ctas, 1))
    for o, j in zip(outs, jobs):
        _check_vs_oracle(oracle, o, j, SCHED)
    if case == "empty_between":
        assert not outs[1]["flow"].any() and not outs[1]["costs"].any() and not outs[1]["mask"].any()


def test_mixed_batch_streaming_between_resident(oracle, sms):
    """[resident, too large (streams), resident]: the streaming problem splits the resident run in two launches."""
    _, more = _limit_masks(sms)
    jobs = [_job(MASKS["border_right"](203, 77, 1), 1), _job(more, 4), _job(MASKS["holes"](203, 77, 2), 2)]
    kw = dict(nCont=1, nGN=1, nPCG=20)
    outs, info, nres = _run(jobs, kw)
    assert nres == 2
    _expect_launch(info, strip_count(jobs[2]["mask"], sms))          # the last launch: the third problem alone
    for o, j in zip(outs, jobs):
        _check_vs_oracle(oracle, o, j, kw)


def test_tiny_and_border_problems_one_launch(oracle, sms):
    """1-strip problems (one of them a 5x3 image) and border-touching ones share one launch: one CTA each for the tiny
    problems, ragged CTA counts on the compact grid."""
    jobs = [_job(MASKS["single"](203, 77, 1), 1), _job(MASKS["full"](5, 3), 2), _job(MASKS["border_all"](203, 77, 3), 3),
            _job(MASKS["lines"](150, 97, 4), 4), _job(MASKS["pixels"](203, 77, 5), 5)]
    exps = [strip_count(j["mask"], sms) for j in jobs]
    assert all(e["fits"] and e["NW"] == 4 for e in exps) and exps[0]["strips"] == exps[1]["strips"] == 1
    Gs = [e["G"] for e in exps]
    grid = (Gs[0], len(jobs)) if len(set(Gs)) == 1 else (sum(Gs), 1)
    outs, info, nres = _run(jobs, SCHED, maxWH=(203, 97))
    assert nres == len(jobs)
    _expect_launch(info, dict(NW=4), problems=len(jobs), grid=grid)
    for o, j in zip(outs, jobs):
        _check_vs_oracle(oracle, o, j, SCHED)


# ------------------------------------------------------------------------------ d. the other solver kinds, same masks
@pytest.mark.parametrize("name", ["border_right", "holes", "ragged"])
@pytest.mark.parametrize("kind", ["stream", "lm"])
def test_other_solvers_on_geometries(oracle, kind, name):
    job = _job(MASKS[name](150, 97, 6), 6)
    kw = dict(nCont=2, nGN=2, nPCG=30)
    if kind == "stream":
        (o,), _, nres = _run([job], kw, backend=lib.BACKEND_STREAM)
        assert nres == 0
    else:
        (o,), _, _ = _run([job], kw, options=[("lm", 1)])
    _check_vs_oracle(oracle, o, job, kw, lm=kind == "lm")
