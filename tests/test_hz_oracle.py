"""Pins the HagerZhang line-search oracle (linesearch/hager_zhang.h:54-552; SURVEY.md 8(f) rank 2 --
oracle first, the device path is the next round's work; no GPU here):
  1. the reference's four 1-D known-answer tests (src/test/hager_zhang_test.cc:101-141);
  2. bit for bit against oracle/_ref = the reference's own hager_zhang.h compiled on the
     Eigen-API shim (its recorded outputs for the same inputs, reference_outputs.py): random
     1-D searches and Lbfgs / Bfgs / GradientDescent<F, HagerZhang> runs;
  3. the committed fixture that build produced (tests/golden/hz_*.npz).
"""
import glob
import os

import numpy as np
import pytest

from oracle import oracle_binding as ob
import reference_outputs as ro

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
IMPLS = ["oracle", "ref"]
KEYS = ("x", "value", "gradient", "num_iterations", "status", "nfev", "x_delta", "f_delta",
        "gradient_norm")
# (((c4 v + c3) v + c2) v + c1) v + c0
QUADRATIC = lambda a, b, c: [0.0, 0.0, a, b, c]  # noqa: E731  hager_zhang_test.cc:40-58
CUBIC = [0.0, 1.0, 0.0, -3.0, 2.0]               # :60-72  v^3 - 3 v + 2
FLAT_QUARTIC = [1.0, 0.0, 0.0, 1e-8, 0.0]        # :74-85  1e-8 v + v^4


@pytest.mark.parametrize("impl", IMPLS)
def test_case1_convex_quadratic_minimum(impl):  # :101-106
    alpha, f_at, _, _ = ro.hz_search_poly(QUADRATIC(1.0, -2.0, 0.0), 0.0, 1.0, impl)
    assert abs(alpha - 1.0) <= 1e-6 and abs(f_at - (-1.0)) <= 1e-6


@pytest.mark.parametrize("impl", IMPLS)
def test_case2_cubic_local_minimum(impl):  # :107-112
    alpha, f_at, _, _ = ro.hz_search_poly(CUBIC, 0.0, 1.0, impl)
    assert abs(alpha - 1.0) <= 1e-6 and abs(f_at) <= 1e-6


@pytest.mark.parametrize("impl", IMPLS)
def test_case3_ill_scaled_quadratic_stays_bounded(impl):  # :113-120
    alpha, f_at, _, _ = ro.hz_search_poly(QUADRATIC(1e6, -1e6, 2.5e5), 0.0, 1.0, impl)
    assert abs(alpha - 0.5) <= 1e-6 and abs(f_at) <= 1e-3 and 0.0 < alpha < 1.0


@pytest.mark.parametrize("impl", IMPLS)
def test_case4_flat_region_terminates(impl):  # :121-127
    alpha, f_at, _, _ = ro.hz_search_poly(FLAT_QUARTIC, 0.0, 1.0, impl)
    assert alpha > 0.0 and np.isfinite(alpha) and f_at <= 0.0


def test_oracle_equals_reference_on_random_searches():
    rng = np.random.default_rng(0)
    calls = []
    for _ in range(1500):
        c = rng.uniform(-2, 2, 5)
        c[0] = abs(c[0]) + 0.1  # bounded below
        a0, x0 = float(10 ** rng.uniform(-3, 2)), float(rng.uniform(-2, 2))
        calls.append(((c, x0, a0), {}))
    o = ro.stacked("hz_search_poly", [ob.hz_search_poly(*args) for args, _ in calls])
    r = ro.sweep("hz_search_poly", calls)
    assert ro.equal(o["step"], r["step"]) and ro.equal(o["nfev"], r["nfev"])
    assert o["nfev"].sum() > 2000 and o["nfev"].max() >= 5  # bracket expansion, secant and bisection steps all ran


@pytest.mark.parametrize("solver,dtype,d", [
    (ob.LBFGS, np.float64, 2), (ob.LBFGS, np.float64, 37), (ob.LBFGS, np.float32, 37), (ob.LBFGS, np.float64, 128),
    (ob.BFGS, np.float64, 8), (ob.BFGS, np.float32, 37),
    (ob.GRADIENT_DESCENT, np.float64, 8), (ob.GRADIENT_DESCENT, np.float64, 37)])
@pytest.mark.parametrize("policy", [ob.POLICY_WARP_TREE, ob.POLICY_DMMA_TREE])
def test_solvers_with_hager_zhang_equal_reference_headers(solver, dtype, d, policy):
    """Lbfgs<F, 10, HagerZhang>, Bfgs<F, HagerZhang>, GradientDescent<F, HagerZhang>."""
    x0 = ob.fill_uniform((8, d), 0, 77 + d, -2.0, 2.0, dtype)
    stop = ob.default_stop()
    stop.num_iterations = 300
    kw = dict(stop=stop, policy=policy, linesearch=ob.LS_HAGER_ZHANG)
    a = ob.minimize(solver, ob.FN_ROSENBROCK, x0, impl="oracle", **kw)
    b = ro.minimize(solver, ob.FN_ROSENBROCK, x0, impl="ref", **kw)
    assert all(ro.equal(a[k], b[k]) for k in KEYS)


@pytest.mark.parametrize("impl", IMPLS)
def test_lbfgs_with_hager_zhang_solves_the_verify_cc_starts(impl):
    """verify.cc:168-173 Far / Near with the alternative LineSearch policy."""
    r = ro.minimize(ob.LBFGS, ob.FN_ROSENBROCK, np.array([[15.0, 8.0], [-1.0, 2.0]]), impl=impl,
                    linesearch=ob.LS_HAGER_ZHANG)
    for x in r["x"]:
        assert (1 - x[0]) ** 2 + 100 * (x[1] - x[0] ** 2) ** 2 < 1e-4


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "hz_*.npz"))))
def test_oracle_reproduces_committed_reference_fixtures(path):
    """Fixtures were produced by oracle/_ref (tests/golden/make_golden_hz.py)."""
    z = np.load(path)
    r = ob.minimize(int(z["solver"]), int(z["family"]), z["x0"], policy=int(z["policy"]),
                    linesearch=ob.LS_HAGER_ZHANG)
    for k in ("x", "value", "gradient", "num_iterations", "status", "nfev"):
        assert np.array_equal(r[k].view(np.uint8), z[k].view(np.uint8)), k
