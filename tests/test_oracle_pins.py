"""Pins the CPU oracle (no GPU):
  1. against every golden vector the reference's own tests hold for this path:
     the 7 cstep KATs (src/test/cstep_test.cc:54-204), verify.cc Far/Near
     (src/test/verify.cc:23,129,168-173,187-188,192), the Dockerfile.test quadratic
     (:35-42) and the AL-test half-norm solve (augmented_lagrangian_test.cc:661-683);
  2. bit for bit against oracle/_ref = the reference's own headers compiled on the
     Eigen-API shim: its recorded outputs for the same inputs (reference_outputs.py),
     and the committed fixtures that build produced.
"""
import glob
import os

import numpy as np
import pytest

from oracle import oracle_binding as ob
import reference_outputs as ro

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
IMPLS = ["oracle", "ref"]


# ---- src/test/cstep_test.cc -------------------------------------------------
@pytest.mark.parametrize("impl", IMPLS)
def test_cstep_case1_quadratic_model(impl):  # :54-72
    io, brackt, info, ret = ro.cstep([0, 0, -1, 0, 0, 0, 3, 1.5, 2, 0, 10], 0, impl=impl)
    assert ret == 0 and info == 1 and brackt == 1
    assert abs(io[6] - 1.0) < 1e-12
    assert io[0] == 0.0 and io[3] == 3.0 and io[4] == 1.5 and io[5] == 2.0


@pytest.mark.parametrize("impl", IMPLS)
def test_cstep_case2_sign_flip(impl):  # :81-100
    io, brackt, info, ret = ro.cstep([0, 2, -2, 0, 0, 0, 3, 0.5, 1, 0, 10], 0, impl=impl)
    assert ret == 0 and info == 2 and brackt == 1
    assert abs(io[6] - 2.0) < 1e-12
    assert (io[0], io[1], io[2]) == (3.0, 0.5, 1.0)
    assert (io[3], io[4], io[5]) == (0.0, 2.0, -2.0)


@pytest.mark.parametrize("impl", IMPLS)
def test_cstep_case3_advance(impl):  # :109-127
    io, brackt, info, ret = ro.cstep([0, 8, -4, 0, 0, 0, 1, 4.5, -3, 0, 20], 0, impl=impl)
    assert ret == 0 and info == 3 and brackt == 0
    assert 1.0 < io[6] <= 20.0
    assert (io[0], io[1], io[2]) == (1.0, 4.5, -3.0)


@pytest.mark.parametrize("impl", IMPLS)
def test_cstep_case4_extrapolate(impl):  # :138-151
    io, brackt, info, ret = ro.cstep([0, 5, -1, 0, 0, 0, 1, 3.99, -1.03, 0, 50], 0, impl=impl)
    assert ret == 0 and info == 4 and brackt == 0 and io[6] == 50.0


@pytest.mark.parametrize("impl", IMPLS)
def test_cstep_clamp(impl):  # :155-168
    io, brackt, info, ret = ro.cstep([0, 0, -1, 0, 0, 0, 3, 1.5, 2, 0.1, 0.75], 0, impl=impl)
    assert ret == 0 and 0.1 <= io[6] <= 0.75


@pytest.mark.parametrize("impl", IMPLS)
def test_cstep_safeguard(impl):  # :175-191
    io, brackt, info, ret = ro.cstep([0, 0, -1, 1, 0.5, 1.5, 0.99, 0.49, 1.4, 0, 2], 1, impl=impl)
    assert ret == 0 and info == 1 and brackt == 1
    assert 0.0 <= io[6] <= 0.66 + 1e-12


@pytest.mark.parametrize("impl", IMPLS)
def test_cstep_rejects_non_descent(impl):  # :196-204
    io, brackt, info, ret = ro.cstep([0, 0, 1, 0, 0, 0, 1, 0.5, 0.5, 0, 10], 0, impl=impl)
    assert ret == -1


def test_cstep_oracle_equals_reference_random():
    rng = np.random.default_rng(7)
    calls = []
    for _ in range(2000):
        stx, stp = sorted(rng.uniform(0, 4, 2))
        if stx == stp:
            continue
        io = [stx, rng.normal(), -abs(rng.normal()) - 1e-3, rng.uniform(0, 6), rng.normal(),
              rng.normal(), stp, rng.normal(), rng.normal(), 0.0, 50.0]
        br = int(rng.integers(0, 2))
        calls.append(((io, br), {}))
    a = ro.stacked("cstep", [ob.cstep(*args) for args, _ in calls])
    b = ro.sweep("cstep", calls)
    assert ro.equal(a["io"], b["io"]) and ro.equal(a["flags"], b["flags"])


# ---- src/test/verify.cc, Dockerfile.test, augmented_lagrangian_test.cc ------
PRECISION = 1e-4  # verify.cc:23


def _rosen2(x):
    return (1 - x[0]) ** 2 + 100 * (x[1] - x[0] ** 2) ** 2


@pytest.mark.parametrize("impl", IMPLS)
@pytest.mark.parametrize("solver", [ob.LBFGS, ob.BFGS, ob.NEWTON])
@pytest.mark.parametrize("x0", [[15.0, 8.0], [-1.0, 2.0]])  # verify.cc:168-173
def test_verify_cc_rosenbrock_far_near(impl, solver, x0):
    r = ro.minimize(solver, ob.FN_ROSENBROCK, np.array([x0]), impl=impl)
    assert abs(_rosen2(r["x"][0])) < PRECISION  # verify.cc:129
    assert r["status"][0] != 1  # not IterationLimit


@pytest.mark.parametrize("impl", IMPLS)
@pytest.mark.parametrize("x0", [[15.0, 8.0], [-1.0, 2.0]])
def test_verify_cc_gradient_descent_far_near(impl, x0):
    """SOLVER_SETUP_CONSERVATIVE(GradientDescent, RosenbrockGradient), verify.cc:185."""
    r = ro.minimize(ob.GRADIENT_DESCENT, ob.FN_ROSENBROCK, np.array([x0]), impl=impl,
                    stop=ob.conservative_stop())
    assert abs(_rosen2(r["x"][0])) < PRECISION


@pytest.mark.parametrize("impl", IMPLS)
@pytest.mark.parametrize("x0", [[15.0, 8.0], [-1.0, 2.0]])
def test_verify_cc_conjugated_gradient_descent_far_near(impl, x0):
    """SOLVER_SETUP(ConjugatedGradientDescent, RosenbrockGradient), verify.cc:186."""
    r = ro.minimize(ob.CONJUGATED_GRADIENT_DESCENT, ob.FN_ROSENBROCK, np.array([x0]), impl=impl)
    assert abs(_rosen2(r["x"][0])) < PRECISION
    assert r["status"][0] != 1


@pytest.mark.parametrize("impl", IMPLS)
def test_dockerfile_quadratic(impl):  # Dockerfile.test:35-42
    r = ro.minimize(ob.LBFGS, ob.FN_DIAG_QUADRATIC, np.array([[-10.0, 2.0]]), impl=impl)
    assert abs(r["x"][0, 0]) < 1e-4 and abs(r["x"][0, 1]) < 1e-4
    assert abs(r["value"][0] - 5.0) < 1e-4


@pytest.mark.parametrize("impl", IMPLS)
def test_al_test_half_norm(impl):  # augmented_lagrangian_test.cc:661-683 (inner solve)
    r = ro.minimize(ob.LBFGS, ob.FN_HALF_SQUARED_NORM, np.array([[5.0, 5.0]]), impl=impl)
    assert np.all(np.abs(r["x"][0]) < 1e-6)


def test_probe_numbers_from_survey():
    """SURVEY.md 6: an independent survey-time restatement saw these counts."""
    r = ob.minimize(ob.LBFGS, ob.FN_ROSENBROCK, np.array([[15.0, 8.0], [-1.0, 2.0]]))
    assert list(r["num_iterations"]) == [45, 42]
    assert list(r["status"]) == [4, 3]
    r = ob.minimize(ob.BFGS, ob.FN_ROSENBROCK, np.array([[15.0, 8.0], [-1.0, 2.0]]))
    assert list(r["num_iterations"]) == [121, 37]
    r = ob.minimize(ob.LBFGS, ob.FN_DIAG_QUADRATIC, np.array([[-10.0, 2.0]]))
    assert list(r["num_iterations"]) == [10] and list(r["nfev"]) == [11]


# ---- oracle == the reference's own code, bit for bit -------------------------
KEYS = ("x", "value", "gradient", "num_iterations", "status", "nfev", "x_delta", "f_delta",
        "gradient_norm")


def _same(a, b, keys=KEYS):
    return all(ro.equal(a[k], b[k]) for k in keys)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("policy", [ob.POLICY_WARP_TREE, ob.POLICY_EIGEN_SSE2, ob.POLICY_DMMA_TREE])
@pytest.mark.parametrize("solver,d", [(ob.LBFGS, 2), (ob.LBFGS, 3), (ob.LBFGS, 37), (ob.LBFGS, 128),
                                      (ob.BFGS, 2), (ob.BFGS, 32), (ob.BFGS, 37),
                                      (ob.NEWTON, 2), (ob.NEWTON, 8)])
def test_oracle_equals_reference_headers(dtype, policy, solver, d):
    B = 6 if d >= 64 else 16
    x0 = ob.fill_uniform((B, d), 1000 * d, 99, -2.0, 2.0, dtype)
    a = ob.minimize(solver, ob.FN_ROSENBROCK, x0, policy=policy, impl="oracle")
    b = ro.minimize(solver, ob.FN_ROSENBROCK, x0, policy=policy, impl="ref")
    assert _same(a, b)


def _random_stop(rng):
    """A random Progress setting that can fire every stopping rule of progress.h:212-300 within a few dozen iterations."""
    s = ob.default_stop()
    s.num_iterations = int(rng.choice([3, 7, 25, 60, 10000]))
    s.x_delta = float(rng.choice([0.0, 1e-9, 1e-4, 1e-2]))
    s.x_delta_violations = int(rng.integers(1, 4))
    s.f_delta = float(rng.choice([0.0, 0.0, 1e-8, 1e-3, 1e-1]))
    s.f_delta_violations = int(rng.integers(1, 4))
    s.f_delta_relative = int(rng.integers(0, 2))
    s.gradient_norm = float(rng.choice([0.0, 1e-5, 1e-2, 1.0]))
    s.gradient_norm_relative = int(rng.integers(0, 2))
    s.past = int(rng.integers(0, 9))
    s.past_delta = float(rng.choice([1e-10, 1e-6, 1e-2]))
    return s


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("solver", [ob.LBFGS, ob.BFGS, ob.NEWTON, ob.GRADIENT_DESCENT, ob.CONJUGATED_GRADIENT_DESCENT])
def test_oracle_equals_reference_headers_under_random_progress_settings(solver, dtype):
    """The ORDER of the tests in Progress::Update decides the reported status (SURVEY.md 3.4): 40 random settings per
    solver -- iteration limits, x / f deltas with 1-3 allowed violations, absolute and relative thresholds, past windows
    0-8 -- through the C oracle and through the reference's own progress.h (oracle/_ref); every output equal bit for
    bit, and every solver's sweep ends in at least three different statuses."""
    if solver == ob.CONJUGATED_GRADIENT_DESCENT and dtype == np.float32:
        pytest.skip("ConjugatedGradientDescent is fp64 only (the reference mixes double into ScalarType vectors)")
    rng = np.random.default_rng(1234 + 10 * solver + (dtype == np.float32))
    d, B = 8, 8
    calls = []
    for k in range(40):
        stop = _random_stop(rng)
        if solver in (ob.GRADIENT_DESCENT, ob.CONJUGATED_GRADIENT_DESCENT):
            stop.num_iterations = min(stop.num_iterations, 60)
        x0 = ob.fill_uniform((B, d), 17 * k, 4321, -2.0, 2.0, dtype)
        calls.append(((solver, ob.FN_ROSENBROCK, x0), {"stop": stop}))
    a = ro.stacked("minimize", [ob.minimize(*args, **kw) for args, kw in calls])
    b = ro.sweep("minimize", calls)
    assert _same(a, b), [k for k in KEYS if not ro.equal(a[k], b[k])]
    seen = set(a["status"].ravel().tolist())
    assert len(seen) >= 3, seen


def test_fused_lu_oracle_equals_reference_headers():
    """CNO_POLICY_DMMA_LU: the oracle's lu_solve(fused = 1) == the reference's newton_descent.h / armijo.h /
    progress.h on the shim whose lu().solve() fuses every multiply-subtract under this policy; d = 64 (the shape
    the tensor-core kernel is built for), 12 and Rosenbrock d = 8; and the committed fixture."""
    rng = np.random.default_rng(11)
    for d, B in ((64, 6), (12, 5)):
        M = rng.uniform(-1, 1, (B, d, d))
        A = np.einsum("bki,bkj->bij", M, M) / d + np.eye(d)
        A = (A + A.transpose(0, 2, 1)) / 2
        if d == 64:
            A[1] = (M[1] + M[1].T) / 2  # indefinite: pivots move
        bvec = rng.uniform(-1, 1, (B, d))
        data = np.concatenate([A.transpose(0, 2, 1).reshape(B, -1), bvec], axis=1)
        x0 = rng.uniform(-2, 2, (B, d))
        stop = ob.default_stop()
        stop.num_iterations = 6
        a = ob.minimize(ob.NEWTON, ob.FN_DENSE_QUADRATIC, x0, data=data, impl="oracle", policy=ob.POLICY_DMMA_LU, stop=stop)
        b = ro.minimize(ob.NEWTON, ob.FN_DENSE_QUADRATIC, x0, data=data, impl="ref", policy=ob.POLICY_DMMA_LU, stop=stop)
        assert _same(a, b)
        c = ob.minimize(ob.NEWTON, ob.FN_DENSE_QUADRATIC, x0, data=data, impl="oracle", stop=stop)
        assert not np.array_equal(a["x"].view(np.uint64), c["x"].view(np.uint64))
    x0 = ob.fill_uniform((16, 8), 8000, 99, -2.0, 2.0)
    assert _same(ob.minimize(ob.NEWTON, ob.FN_ROSENBROCK, x0, policy=ob.POLICY_DMMA_LU, impl="oracle"),
                 ro.minimize(ob.NEWTON, ob.FN_ROSENBROCK, x0, policy=ob.POLICY_DMMA_LU, impl="ref"))


def test_condition_hessian_oracle_equals_reference_progress_update():
    """progress.condition_hessian (progress.h:203-210): the oracle's restatement == the value the reference's own
    Progress::Update leaves (oracle/_ref: H.norm() * H.inverse().norm() on the shim), fp64 (both LU policies), fp32,
    dense quadratics and the Rosenbrock Hessian; and the known answer for H = I."""
    rng = np.random.default_rng(1)
    for d, B, dt in ((64, 4, np.float64), (12, 5, np.float64), (64, 3, np.float32)):
        M = rng.uniform(-1, 1, (B, d, d))
        A = np.einsum("bki,bkj->bij", M, M) / d + np.eye(d)
        A = (A + A.transpose(0, 2, 1)) / 2
        bvec = rng.uniform(-1, 1, (B, d))
        data = np.concatenate([A.transpose(0, 2, 1).reshape(B, -1), bvec], 1).astype(dt)
        x = rng.uniform(-2, 2, (B, d)).astype(dt)
        for pol in ((None, ob.POLICY_DMMA_LU) if dt == np.float64 else (None,)):
            a = ob.condition_hessian(ob.FN_DENSE_QUADRATIC, x, data=data, policy=pol)
            r = ro.condition_hessian(ob.FN_DENSE_QUADRATIC, x, data=data, policy=pol, impl="ref")
            assert ro.equal(a, r)
            truth = np.array([np.linalg.norm(A[i]) * np.linalg.norm(np.linalg.inv(A[i])) for i in range(B)])
            assert np.allclose(a, truth, rtol=1e-4 if dt == np.float32 else 1e-10)
    x = ob.fill_uniform((6, 8), 0, 3, -2.0, 2.0)
    assert ro.equal(ob.condition_hessian(ob.FN_ROSENBROCK, x), ro.condition_hessian(ob.FN_ROSENBROCK, x, impl="ref"))
    assert np.allclose(ob.condition_hessian(ob.FN_HALF_SQUARED_NORM, x), 8.0, rtol=1e-15)  # ||I||_F ||I^-1||_F = d


def test_fused_lu_oracle_reproduces_committed_reference_fixture():
    """tests/golden/newton_dense_quadratic_d64_dmma_lu.npz was produced by oracle/_ref (make_golden.py)."""
    z = np.load(os.path.join(GOLDEN, "newton_dense_quadratic_d64_dmma_lu.npz"))
    r = ob.minimize(ob.NEWTON, ob.FN_DENSE_QUADRATIC, z["x0"], data=z["data"], policy=ob.POLICY_DMMA_LU)
    for k in ("x", "value", "gradient", "num_iterations", "status", "nfev"):
        assert np.array_equal(r[k].view(np.uint8), z[k].view(np.uint8)), k


@pytest.mark.parametrize("policy", [ob.POLICY_WARP_TREE, ob.POLICY_EIGEN_SSE2, ob.POLICY_DMMA_TREE])
@pytest.mark.parametrize("solver,dtype,d", [
    (ob.GRADIENT_DESCENT, np.float64, 2), (ob.GRADIENT_DESCENT, np.float64, 8),
    (ob.GRADIENT_DESCENT, np.float64, 37), (ob.GRADIENT_DESCENT, np.float32, 37),
    (ob.CONJUGATED_GRADIENT_DESCENT, np.float64, 2), (ob.CONJUGATED_GRADIENT_DESCENT, np.float64, 8),
    (ob.CONJUGATED_GRADIENT_DESCENT, np.float64, 37)])
def test_oracle_descent_solvers_equal_reference_headers(policy, solver, dtype, d):
    """gradient_descent.h / conjugated_gradient_descent.h / armijo.h:52-68 compiled from the reference."""
    x0 = ob.fill_uniform((8, d), 77 * d, 5, -2.0, 2.0, dtype)
    stop = ob.default_stop()
    stop.num_iterations = 400  # bounded: these solvers crawl on Rosenbrock
    a = ob.minimize(solver, ob.FN_ROSENBROCK, x0, policy=policy, impl="oracle", stop=stop)
    b = ro.minimize(solver, ob.FN_ROSENBROCK, x0, policy=policy, impl="ref", stop=stop)
    assert _same(a, b)


def test_oracle_equals_reference_dense_quadratic():
    rng = np.random.default_rng(3)
    d, B = 12, 5
    M = rng.uniform(-1, 1, (B, d, d))
    A = np.einsum("bki,bkj->bij", M, M) / d + np.eye(d)
    bvec = rng.uniform(-1, 1, (B, d))
    data = np.concatenate([A.transpose(0, 2, 1).reshape(B, -1), bvec], axis=1)
    x0 = rng.uniform(-2, 2, (B, d))
    for solver in (ob.LBFGS, ob.BFGS, ob.NEWTON):
        a = ob.minimize(solver, ob.FN_DENSE_QUADRATIC, x0, data=data, impl="oracle")
        b = ro.minimize(solver, ob.FN_DENSE_QUADRATIC, x0, data=data, impl="ref")
        assert _same(a, b)
        xs = np.linalg.solve(A, bvec[..., None])[..., 0]
        assert np.allclose(a["x"], xs, atol=1e-4)


@pytest.mark.parametrize("path", sorted(p for p in glob.glob(os.path.join(GOLDEN, "*_rosenbrock_*.npz"))
                                        if not os.path.basename(p).startswith(("al_", "hz_", "lbfgsb_"))))  # incl. gd_*, cg_* (lbfgsb_*: tests/test_lbfgsb.py)
def test_oracle_reproduces_committed_reference_fixtures(path):
    """Fixtures were produced by oracle/_ref (tests/golden/make_golden.py)."""
    z = np.load(path)
    r = ob.minimize(int(z["solver"]), int(z["family"]), z["x0"], policy=int(z["policy"]))
    for k in ("x", "value", "gradient", "num_iterations", "status", "nfev"):
        assert np.array_equal(r[k].view(np.uint8), z[k].view(np.uint8)), k


def test_reference_pins_d2_fixture():
    z = np.load(os.path.join(GOLDEN, "reference_pins_d2.npz"))
    for tag, solver, family, x0 in [
        ("lbfgs_far", ob.LBFGS, ob.FN_ROSENBROCK, [15.0, 8.0]),
        ("bfgs_near", ob.BFGS, ob.FN_ROSENBROCK, [-1.0, 2.0]),
        ("newton_far", ob.NEWTON, ob.FN_ROSENBROCK, [15.0, 8.0]),
        ("lbfgs_quadratic", ob.LBFGS, ob.FN_DIAG_QUADRATIC, [-10.0, 2.0]),
    ]:
        r = ob.minimize(solver, family, np.array([x0]))
        assert np.array_equal(r["x"][0], z[tag + "_x"])
        assert r["num_iterations"][0] == z[tag + "_it"] and r["status"][0] == z[tag + "_status"]


# ---- arithmetic specification -------------------------------------------------
def test_reduction_spec_warp_tree_matches_numpy_model():
    rng = np.random.default_rng(0)
    for d in (1, 2, 31, 32, 33, 64, 100, 128, 200):
        t = rng.normal(size=d)
        E = (d + 31) // 32
        v = np.zeros(32 * E)
        v[:d] = t
        v = v.reshape(32, E).copy()
        w = 1
        while w < E:
            for j in range(0, E - w, 2 * w):
                v[:, j] = v[:, j] + v[:, j + w]
            w *= 2
        p = v[:, 0].copy()
        for off in (16, 8, 4, 2, 1):
            p = p + p[np.arange(32) ^ off]
        import ctypes as C
        got = ob.oracle_lib().cno_oracle_reduce_sum_f64(
            t.ctypes.data_as(C.POINTER(C.c_double)), d, ob.POLICY_WARP_TREE)
        assert got == p[0]


def test_reduction_spec_dmma_tree_matches_numpy_model():
    """CNO_POLICY_DMMA_TREE = what two mma.sync.m8n8k4.f64 (A = ones) compute."""
    import ctypes as C
    rng = np.random.default_rng(1)
    for d in (1, 2, 32, 37, 128, 200):
        t = rng.normal(size=d)
        E = (d + 31) // 32
        v = np.zeros(32 * E)
        v[:d] = t
        v = v.reshape(32, E).copy()
        w = 1
        while w < E:
            for j in range(0, E - w, 2 * w):
                v[:, j] = v[:, j] + v[:, j + w]
            w *= 2
        p = v[:, 0]
        S = [(((0.0 + p[4 * n]) + p[4 * n + 1]) + p[4 * n + 2]) + p[4 * n + 3] for n in range(8)]
        T = [S[2 * j] + S[2 * j + 1] for j in range(4)]
        want = (((0.0 + T[0]) + T[1]) + T[2]) + T[3]
        got = ob.oracle_lib().cno_oracle_reduce_sum_f64(
            t.ctypes.data_as(C.POINTER(C.c_double)), d, ob.POLICY_DMMA_TREE)
        assert got == want


def test_fill_uniform_is_splitmix64():
    a = ob.fill_uniform((4,), 0, 12345, -2.0, 2.0)

    def mix(z):
        z &= (1 << 64) - 1
        z ^= z >> 30
        z = (z * 0xBF58476D1CE4E5B9) & ((1 << 64) - 1)
        z ^= z >> 27
        z = (z * 0x94D049BB133111EB) & ((1 << 64) - 1)
        z ^= z >> 31
        return z
    for k in range(4):
        z = mix(12345 + (k + 1) * 0x9E3779B97F4A7C15)
        u = (z >> 11) * 2.0 ** -53
        assert a[k] == -2.0 + 4.0 * u


def test_oracle_logistic_matches_closed_form():
    """The logistic functor (not in the reference; SURVEY.md 8(d)) against numpy."""
    rng = np.random.default_rng(5)
    B, n, d, lam = 3, 256, 64, 1e-2
    X = rng.uniform(-1, 1, (B, n, d))
    y = np.sign(rng.normal(size=(B, n)))
    w = rng.normal(size=(B, d)) * 0.3
    data = np.concatenate([X.transpose(0, 2, 1).reshape(B, -1), y], axis=1)
    for dtype, tol in ((np.float64, 1e-9), (np.float32, 2e-4)):
        f, g = ob.evaluate(ob.FN_LOGISTIC, w.astype(dtype), data=data.astype(dtype), n=n, param=lam)
        m = y * np.einsum("bnd,bd->bn", X, w)
        f_ref = np.log1p(np.exp(-m)).sum(1) + 0.5 * lam * (w * w).sum(1)
        g_ref = -np.einsum("bn,bnd->bd", y / (1 + np.exp(m)), X) + lam * w
        assert np.allclose(f, f_ref, rtol=tol * 10, atol=tol * 100)
        assert np.allclose(g, g_ref, rtol=0, atol=tol * 500)


@pytest.mark.parametrize("d", [2, 8, 37, 128])
def test_oracle_second_mode_lbfgs_equals_reference_headers(d):
    """Lbfgs<RosenbrockFull> (Second mode -> diagonal preconditioner, lbfgs.h:116-139)."""
    x0 = ob.fill_uniform((8 if d < 100 else 2, d), 0, 5, -2.0, 2.0)  # the reference inverts H every iteration
    a = ob.minimize(ob.LBFGS, ob.FN_ROSENBROCK, x0, mode=2)
    b = ro.minimize(ob.LBFGS, ob.FN_ROSENBROCK, x0, mode=2, impl="ref")
    assert _same(a, b, ("x", "value", "gradient", "num_iterations", "status", "nfev"))
