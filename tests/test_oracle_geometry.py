"""CPU half of the mask-geometry tests: the resident back-end's launch arithmetic mirrored in numpy, and the float64
energy bound that tests/test_gpu_resident_geometry.py applies to the kernel, proven here on the oracle."""
import numpy as np
import pytest

from tests.helpers import GEOMETRY_CASES, MASKS, energy_bound, energy_f64, geometry_gn_problem, mask_full, strip_count

def test_strip_count_hand_made():
    sc = strip_count
    assert sc(mask_full(854, 480), 148) == dict(strips=27 * 60, NW=11, G=148, fits=True)
    assert sc(mask_full(1024, 436), 148) == dict(strips=32 * 55, NW=12, G=147, fits=True)
    # the on-chip limit: SMs x 12 strips fit, one more does not
    for sms in (148, 132):
        full = mask_full(32 * sms - 5, 93)
        assert sc(full, sms) == dict(strips=sms * 12, NW=12, G=sms, fits=True)
        more = np.full((93, 32 * sms + 1), 255, np.uint8)
        more[:, :32 * sms] = 0
        more[0, -1] = 0
        r = sc(more, sms)
        assert r["strips"] == sms * 12 + 1 and not r["fits"]
    assert sc(mask_full(5, 3), 148) == dict(strips=1, NW=4, G=1, fits=True)
    assert sc(mask_full(33, 9), 148)["strips"] == 4
    assert sc(np.full((40, 70), 255, np.uint8), 148) == dict(strips=0, NW=1, G=1, fits=True)
    # the four corners of one strip are one strip; the next pixel to the right / below starts another
    m = np.full((40, 70), 255, np.uint8)
    m[8, 32] = m[8, 63] = m[15, 32] = m[15, 63] = 0
    assert sc(m, 148)["strips"] == 1
    m[8, 64] = 0
    m[16, 32] = 0
    assert sc(m, 148)["strips"] == 3
    # lanes x >= W of the last strip column and rows y >= H of the last strip row hold nothing
    m = np.full((17, 33), 255, np.uint8)
    m[16, 32] = 0
    assert sc(m, 148)["strips"] == 1
    # NW: at least 4, else strips / SMs rounded up; G: strips / NW rounded up, at most SMs
    m = np.full((480, 854), 255, np.uint8)
    m[:8 * 24, :32 * 25] = 0                                          # 600 strips
    assert sc(m, 148) == dict(strips=600, NW=5, G=120, fits=True)
    m = np.full((64, 64), 255, np.uint8)
    m[:, :40] = 0                                                     # 8 x 2 strips
    assert sc(m, 148) == dict(strips=16, NW=4, G=4, fits=True)


@pytest.mark.parametrize("perturbed", [False, True], ids=["rest", "perturbed"])
@pytest.mark.parametrize("name,W,H", GEOMETRY_CASES)
def test_oracle_cost_is_the_float64_energy(oracle, name, W, H, perturbed):
    """The cost the oracle reports equals 0.5 * sum r^2 evaluated in float64 at the state it returns, within the bound
    the GPU tests put on the kernel's returned state (energy_bound)."""
    mask = MASKS[name](W, H, 11)
    pr = geometry_gn_problem(oracle, mask, 11, perturbed)
    E0 = energy_f64(oracle, pr["X"], pr["A"], pr)
    X, A, costs, _ = oracle.gn_solve(pr["X"], pr["A"], pr["U"], pr["C"], pr["M"], 2, 40)
    E = energy_f64(oracle, X, A, pr)
    assert abs(float(costs[0]) - E0) <= energy_bound(E0, E0), (costs[0], E0)
    assert abs(float(costs[-1]) - E) <= energy_bound(E, E0), (costs[-1], E, E0)
    if name == "empty":
        assert E == 0.0 and not costs.any()
    else:
        assert E < E0 or E == E0 == 0.0     # the solve did something on this geometry, or had nothing to do
