"""Lbfgsb<F, 5> (solver/lbfgsb.h:44-538; SURVEY.md 8(f) rank 4) -- the device kernel csrc/cno_lbfgsb.cuh against the
REFERENCE'S OWN header compiled on the Eigen-API shim (oracle/_ref: cno_ref_lbfgsb_minimize; its recorded outputs for the
same inputs, reference_outputs.py) and against the fixtures that build produced (tests/golden/lbfgsb_*.npz), bit for bit
on every output array.
CPU: the device source under the warp emulation (tests/emu).  GPU (-m gpu): the kernel through the C ABI
(cno_lbfgsb_minimize) and the Python / C++ mirrors."""
import ctypes as C
import glob
import os
import subprocess

import numpy as np
import pytest
import torch

from oracle import oracle_binding as ob
import reference_outputs as ro

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
KEYS = ("num_iterations", "status", "nfev", "x", "value", "gradient", "x_delta", "f_delta", "gradient_norm")


@pytest.fixture(scope="module")
def emu():
    here = os.path.join(os.path.dirname(__file__), "emu")
    subprocess.run(["make", "-s", "-C", here], check=True)
    return C.CDLL(os.path.join(here, "libcno_emu.so"))


def _emulated(emu, x0, lo, hi, stop=None, m=0):
    B, d = x0.shape
    stop = stop if stop is not None else ob.lbfgsb_stop()
    prob = ob.Problem(ob.FN_ROSENBROCK, 0, d, 0, 0.0, None, 0, ob.device_policy(x0.dtype), 0, m)
    r = dict(x=np.zeros_like(x0), value=np.zeros(B), gradient=np.zeros_like(x0), num_iterations=np.zeros(B, np.uint32),
             status=np.zeros(B, np.int8), nfev=np.zeros(B, np.uint32), x_delta=np.zeros(B), f_delta=np.zeros(B),
             gradient_norm=np.zeros(B))
    out = ob.BatchOut(*[r[n].ctypes.data for n, _ in ob.BatchOut._fields_])
    lo_a = None if lo is None else np.ascontiguousarray(lo, dtype=np.float64)
    hi_a = None if hi is None else np.ascontiguousarray(hi, dtype=np.float64)
    stride = d if (lo_a is not None and lo_a.ndim == 2) else 0
    assert emu.emu_lbfgsb(C.byref(prob), C.c_longlong(B), C.c_void_p(x0.ctypes.data),
                          None if lo_a is None else C.c_void_p(lo_a.ctypes.data),
                          None if hi_a is None else C.c_void_p(hi_a.ctypes.data), C.c_longlong(stride), C.byref(stop),
                          C.byref(out)) == 0
    return r


def _fixture(path):
    z = np.load(path)
    lo = z["lower"] if "lower" in z.files else None
    hi = z["upper"] if "upper" in z.files else None
    return z, lo, hi


# ---- CPU: the device source under emulation ----------------------------------------------------------------
@pytest.mark.parametrize("name", ["rosenbrock_d2_unbounded_verify_starts", "rosenbrock_d8_box",
                                  "rosenbrock_d37_per_instance_boxes"])
def test_emulated_lbfgsb_matches_reference_fixtures(emu, name):
    z, lo, hi = _fixture(os.path.join(GOLDEN, f"lbfgsb_{name}.npz"))
    n = min(4, z["x0"].shape[0])
    r = _emulated(emu, np.ascontiguousarray(z["x0"][:n]), None if lo is None or lo.ndim == 1 else lo[:n],
                  None if hi is None or hi.ndim == 1 else hi[:n]) if (lo is not None and lo.ndim == 2) else \
        _emulated(emu, np.ascontiguousarray(z["x0"][:n]), lo, hi)
    for k in KEYS:
        assert np.array_equal(r[k].view(np.uint8), z[k][:n].view(np.uint8)), k


def test_reference_verify_starts_reach_the_minimum():
    """src/test/verify.cc:187-190 with :168-173,129: Lbfgsb on RosenbrockGradient from (15, 8) and (-1, 2) reaches
    f < 1e-4 (the fixture is the reference's own run)."""
    z = np.load(os.path.join(GOLDEN, "lbfgsb_rosenbrock_d2_unbounded_verify_starts.npz"))
    assert np.all(z["value"] < 1e-4) and np.all(np.abs(z["x"] - 1.0) < 1e-3)


def test_emulated_lbfgsb_active_bounds_and_infeasible_start(emu):
    """A start outside the box is projected first (:145-150); the solution sits on the active faces with a non-zero
    gradient there and a small projected gradient."""
    x0 = ob.fill_uniform((3, 8), 0, 5, -3.0, 3.0)
    lo, hi = np.full(8, -0.5), np.full(8, 0.8)
    r = _emulated(emu, x0, lo, hi)
    o = ro.ref_lbfgsb_minimize(ob.FN_ROSENBROCK, x0, lo, hi)
    for k in KEYS:
        assert ro.equal(r[k], o[k]), k
    assert np.all(r["x"] <= 0.8) and np.all(r["x"] >= -0.5) and np.any(r["x"] == 0.8)


def test_emulated_lbfgsb_m10_equals_reference_header(emu):
    """Lbfgsb<F, 10> (lbfgsb.h:44-45: m is a template parameter): the kernel with ten pairs (2k up to 20 lanes of the
    compact representation) == the reference's own Lbfgsb<F, 10>, bit for bit; it differs from m = 5."""
    x0 = ob.fill_uniform((1, 8), 0, 9, -2.5, 2.5)
    lo, hi = np.full(8, -1.0), np.full(8, 1.5)
    stop = ob.lbfgsb_stop()
    stop.num_iterations = 30  # (past ten iterations the history is full and wraps: both regimes are covered)
    r = _emulated(emu, x0, lo, hi, stop=stop, m=10)
    o = ro.ref_lbfgsb_minimize(ob.FN_ROSENBROCK, x0, lo, hi, stop=stop, m=10)
    for k in KEYS:
        assert ro.equal(r[k], o[k]), k
    o5 = ro.ref_lbfgsb_minimize(ob.FN_ROSENBROCK, x0, lo, hi, stop=stop)
    assert not ro.equal(o5["num_iterations"], o["num_iterations"]) or not ro.equal(o5["x"], o["x"])


# ---- GPU -----------------------------------------------------------------------------------------------------------
def _gpu(x0, lo, hi, stop=None, fn=None, m=5):
    import cppnumericalsolvers_b200 as cn
    dev = "cuda:0"
    d = x0.shape[1]
    solver = cn.Lbfgsb(m=m) if stop is None else cn.Lbfgsb(cn.Progress.from_c(stop), m=m)
    t = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    solver.SetBounds(t(lo), t(hi))
    fn = fn if fn is not None else cn.Rosenbrock(d, torch.float64 if x0.dtype == np.float64 else torch.float32)
    assert solver.supported(fn)
    st, pr = solver.Minimize(fn, cn.BatchedFunctionState(torch.from_numpy(x0).to(dev)))
    torch.cuda.synchronize()
    return dict(x=st.x.cpu().numpy(), value=st.value.cpu().numpy(), gradient=st.gradient.cpu().numpy(),
                num_iterations=pr.num_iterations.cpu().numpy().astype(np.uint32), status=pr.status.cpu().numpy(),
                nfev=pr.nfev.cpu().numpy().astype(np.uint32), x_delta=pr.x_delta.cpu().numpy(),
                f_delta=pr.f_delta.cpu().numpy(), gradient_norm=pr.gradient_norm.cpu().numpy())


@pytest.mark.gpu
@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "lbfgsb_*.npz"))))
def test_gpu_lbfgsb_matches_reference_fixtures(path):
    z, lo, hi = _fixture(path)
    r = _gpu(z["x0"], lo, hi)
    for k in KEYS:
        assert np.array_equal(r[k].view(np.uint8), z[k].view(np.uint8)), k


@pytest.mark.gpu
@pytest.mark.parametrize("d,B", [(8, 256), (37, 128), (64, 96), (128, 64)])
def test_gpu_lbfgsb_bitwise_equals_reference_header(d, B):
    rng = np.random.default_rng(d)
    x0 = ob.fill_uniform((B, d), 0, 31 + d, -2.5, 2.5)
    lo = rng.uniform(-1.5, -0.2, (B, d))
    hi = lo + rng.uniform(0.3, 2.0, (B, d))
    r, o = _gpu(x0, lo, hi), ro.ref_lbfgsb_minimize(ob.FN_ROSENBROCK, x0, lo, hi)
    for k in KEYS:
        assert ro.equal(r[k], o[k]), k
    assert np.all(r["x"] >= lo) and np.all(r["x"] <= hi)
    # one shared box, and no box at all (the unbounded path: every coordinate free, no breakpoint visited)
    r, o = _gpu(x0[:32], np.full(d, -0.5), np.full(d, 0.8)), ro.ref_lbfgsb_minimize(ob.FN_ROSENBROCK, x0[:32], np.full(d, -0.5), np.full(d, 0.8))
    for k in KEYS:
        assert ro.equal(r[k], o[k]), k
    stop = ob.lbfgsb_stop()
    stop.num_iterations = 80
    r, o = _gpu(x0[:32], None, None, stop), ro.ref_lbfgsb_minimize(ob.FN_ROSENBROCK, x0[:32], None, None, stop=stop)
    for k in KEYS:
        assert ro.equal(r[k], o[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("d,B", [(8, 128), (37, 96), (128, 48)])
def test_gpu_lbfgsb_m10_bitwise_equals_reference_header(d, B):
    """Lbfgsb<F, 10>: GPU == the reference's own Lbfgsb<F, 10> (oracle/_ref), per-instance boxes and unbounded."""
    rng = np.random.default_rng(100 + d)
    x0 = ob.fill_uniform((B, d), 0, 77 + d, -2.5, 2.5)
    lo = rng.uniform(-1.5, -0.2, (B, d))
    hi = lo + rng.uniform(0.3, 2.0, (B, d))
    r, o = _gpu(x0, lo, hi, m=10), ro.ref_lbfgsb_minimize(ob.FN_ROSENBROCK, x0, lo, hi, m=10)
    for k in KEYS:
        assert ro.equal(r[k], o[k]), k
    stop = ob.lbfgsb_stop()
    stop.num_iterations = 60
    r, o = _gpu(x0[:24], None, None, stop, m=10), ro.ref_lbfgsb_minimize(ob.FN_ROSENBROCK, x0[:24], None, None, stop=stop, m=10)
    for k in KEYS:
        assert ro.equal(r[k], o[k]), k
