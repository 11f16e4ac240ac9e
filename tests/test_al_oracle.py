"""Pins the AugmentedLagrangian CPU oracle (oracle/cno_al_oracle.h; SURVEY.md 8(f) rank 1 --
oracle first, the device path is the next round's work; no GPU here):
  1. against the known answers the reference's own tests hold
     (src/test/augmented_lagrangian_test.cc: the ToAugmentedLagrangian closed forms :397-490,
     the KKT solves :492-625, the outer-loop behaviour :627-692);
  2. bit for bit against oracle/_ref = the reference's own augmented_lagrangian.h,
     function_penalty.h and function_expressions.h compiled on the Eigen-API shim (its recorded
     outputs for the same inputs, reference_outputs.py), and against the fixture that build
     produced (tests/golden/al_*.npz).
"""
import glob
import os

import numpy as np
import pytest

from oracle import oracle_binding as ob
import reference_outputs as ro

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
IMPLS = ["oracle", "ref"]
KEYS = ("x", "equality_multipliers", "inequality_multipliers", "penalty", "max_violation",
        "max_lagrangian_gradient", "num_iterations", "status", "nfev", "x_delta", "f_delta",
        "gradient_norm")
FINISHED = 6

penalty_evaluation_tolerance = 1e-12  # augmented_lagrangian_test.cc:43-46
kkt_primal_tolerance = 1e-3
kkt_dual_tolerance = 1e-2
feasibility_tolerance = 1e-5


def _quadratic(center, scale):
    """scale/2 |x - center|^2 up to a constant, as a DenseQuadratic data row [A col-major | b]."""
    d = len(center)
    return np.array([list((scale * np.eye(d)).T.ravel()) + [scale * c for c in center]])


# ---- ToAugmentedLagrangian closed forms (:397-490) ---------------------------
def test_composite_equality_only_matches_closed_form():
    v, g = ob.al_evaluate(ob.FN_HALF_SQUARED_NORM, np.array([[3.0, 4.0]]), [ob.CON_AFFINE],
                          [[1.0, 0.0, 1.0]], 1, [2.0], [], 3.0)
    assert abs(v[0] - 22.5) <= penalty_evaluation_tolerance
    # grad = x + (lambda + rho c) grad c = (3 + (2 + 3*2), 4)
    assert np.allclose(g[0], [11.0, 4.0], atol=1e-12)


def test_composite_inequality_phr_inactive_side():
    v, g = ob.al_evaluate(ob.FN_HALF_SQUARED_NORM, np.array([[3.0, 0.0]]), [ob.CON_AFFINE],
                          [[1.0, 0.0, 0.5]], 0, [], [7.0], 4.0)
    assert abs(v[0] - (-1.625)) <= penalty_evaluation_tolerance
    assert np.array_equal(g[0], [3.0, 0.0])  # the PHR term is constant there


def test_composite_inequality_phr_active_side():
    v, g = ob.al_evaluate(ob.FN_HALF_SQUARED_NORM, np.array([[0.0, 0.0]]), [ob.CON_AFFINE],
                          [[1.0, 0.0, 0.5]], 0, [], [7.0], 4.0)
    assert abs(v[0] - 4.0) <= penalty_evaluation_tolerance
    # d/dx0 of (1/8) max(0, 7 - 4 (x0 - 0.5))^2 at 0 = -(7 + 2) = -9
    assert np.allclose(g[0], [-9.0, 0.0], atol=1e-12)


def test_composite_gradient_matches_finite_differences():
    rng = np.random.default_rng(0)
    d, B = 8, 5
    x = rng.uniform(-1, 1, (B, d))
    rows = rng.uniform(-1, 1, (B, 4, d + 1))
    kinds = [ob.CON_AFFINE, ob.CON_SQNORM, ob.CON_AFFINE, ob.CON_SQNORM]
    rows[:, 3, d] = 3.0  # t - x.x > 0 somewhere, < mu/rho elsewhere
    lam, mu, rho = rng.uniform(-1, 1, (B, 2)), rng.uniform(0, 2, (B, 2)), rng.uniform(0.5, 3, B)
    v, g = ob.al_evaluate(ob.FN_ROSENBROCK, x, kinds, rows, 2, lam, mu, rho)
    h = 1e-6
    for k in range(d):
        e = np.zeros(d)
        e[k] = h
        vp, _ = ob.al_evaluate(ob.FN_ROSENBROCK, x + e, kinds, rows, 2, lam, mu, rho)
        vm, _ = ob.al_evaluate(ob.FN_ROSENBROCK, x - e, kinds, rows, 2, lam, mu, rho)
        assert np.allclose((vp - vm) / (2 * h), g[:, k], rtol=2e-5, atol=2e-5)


# ---- KKT solves (:492-625) -------------------------------------------------------
@pytest.mark.parametrize("impl", IMPLS)
def test_kkt_equality_only_quadratic(impl):  # :492-539
    r = ro.al_minimize(ob.FN_HALF_SQUARED_NORM, np.array([[5.0, 5.0]]), [ob.CON_AFFINE],
                       [[1.0, 0.0, 1.0]], 1, penalty0=1.0, impl=impl)
    x = r["x"][0]
    assert abs(x[0] - 1.0) <= kkt_primal_tolerance and abs(x[1]) <= kkt_primal_tolerance
    assert abs(x[0] - 1.0) <= feasibility_tolerance
    assert abs(r["equality_multipliers"][0, 0] - (-1.0)) <= kkt_dual_tolerance


@pytest.mark.parametrize("impl", IMPLS)
def test_kkt_inequality_active_recovers_multiplier(impl):  # :541-581
    r = ro.al_minimize(ob.FN_DENSE_QUADRATIC, np.array([[5.0, 5.0]]), [ob.CON_AFFINE],
                       [[-1.0, 0.0, -1.0]], 0, penalty0=1.0, data=_quadratic([2.0, 0.0], 1.0), impl=impl)
    x, mu = r["x"][0], r["inequality_multipliers"][0, 0]
    assert abs(x[0] - 1.0) <= kkt_primal_tolerance and abs(x[1]) <= kkt_primal_tolerance
    assert 1.0 - x[0] >= -feasibility_tolerance
    assert mu >= -kkt_dual_tolerance and abs(mu - 1.0) <= kkt_dual_tolerance


@pytest.mark.parametrize("impl", IMPLS)
def test_kkt_both_equality_and_inequality_active(impl):  # :583-625
    r = ro.al_minimize(ob.FN_DENSE_QUADRATIC, np.array([[1.0, 1.0]]), [ob.CON_AFFINE, ob.CON_AFFINE],
                       [[1.0, 0.0, 0.5], [-1.0, -1.0, -2.0]], 1, penalty0=1.0,
                       data=_quadratic([1.0, 2.0], 2.0), impl=impl)
    x = r["x"][0]
    assert abs(x[0] - 0.5) <= kkt_primal_tolerance and abs(x[1] - 1.5) <= kkt_primal_tolerance
    assert abs(x[0] - 0.5) <= feasibility_tolerance
    assert 2.0 - (x[0] + x[1]) >= -feasibility_tolerance
    assert r["inequality_multipliers"][0, 0] >= -kkt_dual_tolerance


# ---- outer-loop behaviour (:627-692) ----------------------------------------------
@pytest.mark.parametrize("impl", IMPLS)
def test_outer_feasible_start_converges_immediately(impl):  # :627-659
    r = ro.al_minimize(ob.FN_HALF_SQUARED_NORM, np.array([[0.0, 0.0]]), [ob.CON_AFFINE],
                       [[0.0, 0.0, 0.0]], 1, penalty0=1.0, impl=impl)
    assert np.all(np.abs(r["x"][0]) <= kkt_primal_tolerance)
    assert r["status"][0] == FINISHED and r["num_iterations"][0] <= 5


@pytest.mark.parametrize("impl", IMPLS)
def test_outer_no_constraints_is_unconstrained(impl):  # :661-692
    r = ro.al_minimize(ob.FN_HALF_SQUARED_NORM, np.array([[5.0, 5.0]]), [], np.zeros((0, 3)), 0,
                       penalty0=1.0, impl=impl)
    assert np.all(np.abs(r["x"][0]) <= kkt_primal_tolerance) and r["status"][0] == FINISHED


@pytest.mark.parametrize("impl", IMPLS)
def test_outer_penalty_holds_flat_on_feasible_problem_and_growth_can_be_disabled(impl):  # :694-764
    r = ro.al_minimize(ob.FN_HALF_SQUARED_NORM, np.array([[0.0, 0.0]]), [ob.CON_AFFINE],
                       [[0.0, 0.0, 0.0]], 1, penalty0=2.5, impl=impl)
    assert r["penalty"][0] == 2.5  # max_violation = 0 <= 0.25 * 0: never grows
    cfg = ob.al_default_config()
    cfg.penalty_growth_factor = 1.0
    r = ro.al_minimize(ob.FN_HALF_SQUARED_NORM, np.array([[5.0, 5.0]]), [ob.CON_AFFINE],
                       [[1.0, 0.0, 1.0]], 1, penalty0=3.0, config=cfg, impl=impl)
    assert r["penalty"][0] == 3.0 and abs(r["x"][0, 0] - 1.0) <= kkt_primal_tolerance


# ---- oracle == the reference's own headers, bit for bit -------------------------------
def _same(a, b):
    return all(ro.equal(a[k], b[k]) for k in KEYS)


def _random_case(seed, d, B, dtype, per_instance):
    rng = np.random.default_rng(seed)
    x0 = ob.fill_uniform((B, d), 0, seed, -1.5, 1.5, dtype)
    kinds = [ob.CON_AFFINE, ob.CON_SQNORM, ob.CON_AFFINE]
    shape = (B, 3, d + 1) if per_instance else (3, d + 1)
    rows = rng.uniform(-1, 1, shape).astype(dtype)
    rows[..., 1, d] = 2.0 + rng.uniform(0, 1, shape[:-2])  # ball radius^2: |x|^2 <= t
    return x0, kinds, rows


@pytest.mark.parametrize("policy", [ob.POLICY_WARP_TREE, ob.POLICY_EIGEN_SSE2, ob.POLICY_DMMA_TREE])
@pytest.mark.parametrize("dtype,d,n_eq,per_instance", [
    (np.float64, 2, 1, False), (np.float64, 8, 1, True), (np.float64, 37, 0, True),
    (np.float64, 8, 3, False), (np.float32, 8, 1, True)])
def test_al_oracle_equals_reference_headers(policy, dtype, d, n_eq, per_instance):
    x0, kinds, rows = _random_case(31 + d, d, 6, dtype, per_instance)
    stop = ob.al_default_stop()
    stop.num_iterations = 12  # bounded: a hard instance can run to the outer iteration limit
    kw = dict(policy=policy, outer_stop=stop)
    a = ob.al_minimize(ob.FN_ROSENBROCK, x0, kinds, rows, n_eq, impl="oracle", **kw)
    b = ro.al_minimize(ob.FN_ROSENBROCK, x0, kinds, rows, n_eq, impl="ref", **kw)
    assert _same(a, b)
    # user-set initial multipliers / penalty, non-default config and inner preset
    cfg = ob.al_default_config()
    cfg.warmup_max_inner_iterations = 0
    cfg.violation_shrink_ratio = 0.5
    cfg.multiplier_max = 5.0
    kw.update(config=cfg, inner_stop=ob.conservative_stop(), eq0=0.25, ineq0=0.5, penalty0=2.0)
    a = ob.al_minimize(ob.FN_HALF_SQUARED_NORM, x0, kinds, rows, n_eq, impl="oracle", **kw)
    b = ro.al_minimize(ob.FN_HALF_SQUARED_NORM, x0, kinds, rows, n_eq, impl="ref", **kw)
    assert _same(a, b)


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "al_*.npz"))))
def test_al_oracle_reproduces_committed_reference_fixtures(path):
    """Fixtures were produced by oracle/_ref (tests/golden/make_golden_al.py)."""
    z = np.load(path)
    stop = ob.al_default_stop()
    stop.num_iterations = int(z["outer_limit"])
    r = ob.al_minimize(int(z["family"]), z["x0"], z["kinds"], z["rows"], int(z["n_eq"]), outer_stop=stop,
                       policy=int(z["policy"]))
    for k in KEYS:
        assert np.array_equal(r[k].view(np.uint8), z[k].view(np.uint8)), k
    done = z["status"] == FINISHED
    assert np.all(z["max_violation"][done] <= 1e-5)  # Finished = primal feasible (progress.h:240-247)
