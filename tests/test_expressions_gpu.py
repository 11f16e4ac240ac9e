"""Function composition on the device (include/cppoptlib_b200/expressions.h; SURVEY.md 8 row a4) and the
user-functor boundary (device.cuh) against the REFERENCE'S OWN operators and FunctionCRTP functors
(oracle/_ref: function_expressions.h:403-518 compiled on the Eigen-API shim; its recorded outputs for the same inputs,
reference_outputs.py), bit for bit: every output array of Solver::Minimize, for Lbfgs / Bfgs / GradientDescent /
ConjugatedGradientDescent / NewtonDescent and both line searches, plus value/gradient evaluation
(FunctionExpr::operator()).  Fixtures tests/golden/expr_*.npz hold further comparisons with the whole outputs."""
import glob
import os

import numpy as np
import pytest

from oracle import oracle_binding as ob
import reference_outputs as ro
import usertest_binding as ut

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
KEYS = ("num_iterations", "status", "nfev", "x", "value", "gradient", "x_delta", "f_delta", "gradient_norm")
SOLVER_IDS = {"lbfgs": (ob.LBFGS, ob.LS_MORE_THUENTE, 0), "bfgs": (ob.BFGS, ob.LS_MORE_THUENTE, 1),
              "gd": (ob.GRADIENT_DESCENT, ob.LS_MORE_THUENTE, 3), "cg": (ob.CONJUGATED_GRADIENT_DESCENT, ob.LS_MORE_THUENTE, 4),
              "newton": (ob.NEWTON, ob.LS_MORE_THUENTE, 2), "lbfgs_hz": (ob.LBFGS, ob.LS_HAGER_ZHANG, 5),
              "bfgs_hz": (ob.BFGS, ob.LS_HAGER_ZHANG, 6)}


LEAVES = (ob.EXPR_BOWL, ob.EXPR_DOWNGRADE)


def _same(a, b, expr=None, keys=KEYS):
    """Every output array bit for bit.  nfev only for single functors: the reference-side counter ticks once per
    LEAF evaluation (a composite of two functions counts 2 per evaluation), the device counts composite evaluations."""
    for k in keys:
        if k == "nfev" and expr not in LEAVES:
            continue
        assert ro.equal(a[k], b[k]), f"{k} differs"


def _x0(B, d, seed, dtype=np.float64, lo=-2.0, hi=2.0):
    return ob.fill_uniform((B, d), 0, seed, lo, hi, dtype)


CASES = [  # (expr, d, dtype, param, solvers)
    (ob.EXPR_BOWL, 16, np.float64, -2.5, ("lbfgs", "bfgs", "gd", "cg", "lbfgs_hz", "bfgs_hz")),
    (ob.EXPR_BOWL, 64, np.float64, 0.75, ("lbfgs", "cg")),
    (ob.EXPR_BOWL, 37, np.float32, 0.5, ("lbfgs",)),
    (ob.EXPR_ROSEN_PLUS_HALF, 8, np.float64, 0.0, ("lbfgs", "bfgs", "gd", "cg", "lbfgs_hz", "bfgs_hz")),
    (ob.EXPR_ROSEN_PLUS_HALF, 37, np.float64, 0.0, ("lbfgs", "lbfgs_hz")),
    (ob.EXPR_ROSEN_PLUS_HALF, 128, np.float64, 0.0, ("lbfgs",)),
    (ob.EXPR_ROSEN_PLUS_HALF, 37, np.float32, 0.0, ("lbfgs",)),
    (ob.EXPR_PROD, 8, np.float64, 0.0, ("lbfgs", "bfgs")),
    (ob.EXPR_PROD, 37, np.float64, 0.0, ("lbfgs",)),
    (ob.EXPR_SUB, 8, np.float64, 0.0, ("lbfgs", "bfgs")),
    (ob.EXPR_PENALTY, 8, np.float64, 0.0, ("lbfgs", "bfgs")),
    (ob.EXPR_PENALTY, 37, np.float64, 0.0, ("lbfgs",)),
    (ob.EXPR_ZERO_MUL, 8, np.float64, 0.0, ("lbfgs", "bfgs")),
]


@pytest.mark.parametrize("expr,d,dtype,param,solvers", CASES)
def test_first_mode_composites_equal_reference_operators(expr, d, dtype, param, solvers):
    x0 = _x0(24, d, 100 + expr + d, dtype)
    stop = ob.default_stop()
    stop.num_iterations = 300
    for s in solvers:
        sid, ls, dev_id = SOLVER_IDS[s]
        if s in ("gd", "cg"):
            stop.num_iterations = 40
        ref = ro.ref_minimize_expr(expr, sid, x0, param=param, stop=stop, linesearch=ls)
        got = ut.minimize(expr, dev_id, x0, param=param, stop=stop)
        _same(got, ref, expr)
        assert int(got["num_iterations"].max()) > 1


@pytest.mark.parametrize("expr,d", [(ob.EXPR_SECOND_SUM, 8), (ob.EXPR_SECOND_SUM, 37), (ob.EXPR_SECOND_PROD, 2)])
def test_second_mode_composites_newton_and_preconditioned_lbfgs(expr, d):
    """Hessians composed node by node (hess_f + hess_g, c * hess_f, the product rule with its non-symmetric rounding:
    function_expressions.h:133,247,304-305) feed NewtonDescent and Lbfgs's diagonal-preconditioner branch."""
    x0 = _x0(16, d, 7 + d, lo=-1.5, hi=1.5)
    stop = ob.default_stop()
    stop.num_iterations = 60
    ref = ro.ref_minimize_expr(expr, ob.NEWTON, x0, stop=stop)
    got = ut.minimize(expr, 2, x0, mode=2, stop=stop)
    _same(got, ref)
    ref = ro.ref_minimize_expr(expr, ob.LBFGS, x0, stop=stop)   # Second mode: lbfgs.h:116-139
    got = ut.minimize(expr, 0, x0, mode=2, stop=stop)
    _same(got, ref)


@pytest.mark.parametrize("expr,d", [(ob.EXPR_SECOND_SUM, 8), (ob.EXPR_SECOND_SUM, 37), (ob.EXPR_SECOND_PROD, 2)])
def test_condition_hessian_of_second_mode_composites(expr, d):
    """Progress::condition_hessian (progress.h:203-210) of a composite on request (cno_<tag>_condition_hessian): the
    Hessian composed node by node on the device -- for the product not bitwise symmetric -- against the reference's own
    Progress::Update on the reference's own composite (oracle/_ref), bit for bit."""
    x = _x0(24, d, 11 + d, lo=-1.5, hi=1.5)
    got = ut.condition_hessian(expr, x)
    ref = ro.ref_minimize_expr(expr, 100, x)["value"]  # solver id 100: the condition number of the composite at x
    assert ro.equal(got, ref)
    assert np.all(got >= d * 0.99)


def test_function_expr_downgrade_kat_and_first_mode_use():
    """src/test/augmented_lagrangian_test.cc:882-896: a Second-mode source bound through a First-mode FunctionExpr
    evaluates to 20.25 / (12, -3) at (3, -1.5); minimised as a First-mode function (no preconditioner branch)."""
    f, g = ut.evaluate(ob.EXPR_DOWNGRADE, np.array([[3.0, -1.5]]))
    assert f[0] == 20.25 and g[0, 0] == 12.0 and g[0, 1] == -3.0
    rf, rg = ro.ref_evaluate_expr(ob.EXPR_DOWNGRADE, np.array([[3.0, -1.5]]))
    assert ro.equal(f, rf) and ro.equal(g, rg)
    x0 = _x0(8, 2, 5)
    ref = ro.ref_minimize_expr(ob.EXPR_DOWNGRADE, ob.LBFGS, x0)  # FunctionExpr<double, First, 2> wrapped = Second source
    got = ut.minimize(ob.EXPR_DOWNGRADE, 0, x0, mode=1)
    _same(got, ref, ob.EXPR_DOWNGRADE)
    got2 = ut.minimize(ob.EXPR_DOWNGRADE, 0, x0, mode=2)        # used AS Second mode: the other branch of lbfgs.h
    assert not np.array_equal(got2["num_iterations"], got["num_iterations"]) or \
        not np.array_equal(got2["x"].view(np.uint8), got["x"].view(np.uint8))


@pytest.mark.parametrize("expr,d", [(ob.EXPR_ROSEN_PLUS_HALF, 8), (ob.EXPR_PROD, 37), (ob.EXPR_PENALTY, 8),
                                    (ob.EXPR_SUB, 8), (ob.EXPR_ZERO_MUL, 8), (ob.EXPR_BOWL, 64)])
def test_evaluate_equals_reference_operators(expr, d):
    x = _x0(64, d, 11 + d, lo=-3.0, hi=3.0)
    f, g = ut.evaluate(expr, x, param=0.75)
    rf, rg = ro.ref_evaluate_expr(expr, x, param=0.75)
    assert ro.equal(f, rf)
    assert ro.equal(g, rg)


def test_user_functor_stepwise_solve_equals_one_shot():
    """ADVICE r1: SetCallback on a user functor used to be dropped silently.  cno_<tag>_minimize_steps: rounds of K
    iterations with the state parked in between == the fused solve == the reference, bit for bit."""
    x0 = _x0(20, 37, 3)
    ref = ro.ref_minimize_expr(ob.EXPR_ROSEN_PLUS_HALF, ob.LBFGS, x0)
    seen = []
    got = ut.minimize_steps(ob.EXPR_ROSEN_PLUS_HALF, 0, x0, 7, callback=lambda t: seen.append(int((t["status"] == 0).sum())))
    _same(got, ref)
    assert got["rounds"] == -(-int(got["num_iterations"].max()) // 7) and len(seen) == got["rounds"] and seen[-1] == 0


def test_mul_by_zero_never_evaluates_the_source():
    """function_expressions.h:219-227: c == 0 returns 0 / zero gradient without touching f -- also where f is not finite."""
    x = np.full((4, 8), 1e100)  # Rosenbrock overflows to inf there, 0.5 |x|^2 does not
    f, g = ut.evaluate(ob.EXPR_ZERO_MUL, x)
    assert np.all(np.isfinite(f)) and np.all(g == x)  # 0 * Rosenbrock(1e200) would be NaN; the rest is HalfSquaredNorm


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "expr_*.npz"))))
def test_composites_match_reference_fixtures(path):
    """tests/golden/expr_*.npz were produced by oracle/_ref (make_golden_expr.py)."""
    z = np.load(path)
    got = ut.minimize(int(z["expr"]), int(z["device_solver"]), z["x0"], param=float(z["param"]), mode=int(z["mode"]))
    _same(got, {k: z[k] for k in KEYS}, int(z["expr"]))


def test_user_functor_lbfgs_m5_equals_reference():
    """Lbfgs<Bowl, 5> (lbfgs.h:40-41) through CNO_INSTANTIATE_FUNCTION_M; a tag compiled for m = 10 refuses m = 5."""
    x0 = _x0(24, 16, 77)
    ref = ro.ref_minimize_expr(ob.EXPR_BOWL, ob.LBFGS, x0, param=-2.5, lbfgs_m=5)
    got = ut.minimize(ob.EXPR_BOWL, 0, x0, param=-2.5, lbfgs_m=5)
    _same(got, ref, ob.EXPR_BOWL)
    ref10 = ro.ref_minimize_expr(ob.EXPR_BOWL, ob.LBFGS, x0, param=-2.5)
    assert not ro.equal(ref10["x"], ref["x"])
    from cppnumericalsolvers_b200 import _lib
    with pytest.raises(_lib.CnoError):
        ut.minimize(ob.EXPR_BOWL, 0, _x0(4, 64, 1), param=0.75, lbfgs_m=5)  # bowl64 was compiled for m = 10 only
