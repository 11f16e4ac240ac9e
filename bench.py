#!/usr/bin/env python
"""bench.py -- batched L-BFGS instances/second, Rosenbrock d=128 fp64, m=10
(BASELINE.json configs[1]), on N B200s of one node.

One "step" = one batched Solver::Minimize over B = 2^20 instances per GPU
(x0 generated on the device by the counter-based generator of SURVEY.md 8(d),
resident in HBM when the timed region starts; 1 GiB of x0 per GPU > 126 MB L2,
so nothing is cache-warm between steps) + the global stop test (convergence
bitmaps, one all-gather) + the D2H read of `status` (SURVEY.md 8(d)).  Timing:
CUDA events on the launching stream bracketed by barrier + synchronize, max
over ranks.

  value     whole-job instances/s, device-resident inputs
  e2e       the same metric through the host-buffer C-ABI call
            cno_minimize_host (pinned host x0 -> H2D -> solve -> D2H of the whole
            returned state/progress), WALL-CLOCK around the call, max over ranks
  roofline  two yardsticks for the dominant kernel, both from THIS run's
            iteration counts and kernel time:
              (hbm)     ALGORITHMIC bytes of the state-streaming model
                        (SURVEY.md 8(d): w*d*(2 k_t + 6) per iteration) against
                        MEASURED_PEAKS.json's copy bandwidth.  The fused kernel
                        keeps the (s, y) history on chip, so this fraction can
                        exceed 1; `traffic` (ncu DRAM bytes per launch) shows
                        what HBM really moved.
              (compute) the resource that binds: the FP64 datapath.  FP64-pipe
                        warp instructions (+ FP64 tensor-core MMAs at their
                        measured issue cost) per solver iteration come from the
                        ncu instruction mix committed under profiles/; achieved
                        = that x the run's iterations / kernel time, peak =
                        SMs x 4 sub-partitions x 0.5 FP64 warp-instr/clk x the
                        SM clock sampled during the run.
  cpu_baseline  the CPU oracle (plain-C port of the reference path, OpenMP over
            instances, every host core the process may use) on a bounded prefix
            of the same batch.
  parity    >= 256 strided instances of the TIMED batch checked against the CPU
            oracle inside this run (iteration counts, status, x* bits).
  strong    (N > 1) the same global B = 2^20 split over the N GPUs.
  other_configs  (N = 1) BASELINE.json configs[2..4]: device timing + binding pipe.

--dump-outputs DIR writes what the last timed step returned as DIR/<name>.npy (float64):
x, value, gradient and the progress arrays of a fixed, seeded sample of the batch
(instance_index.npy names the instances) and the gathered done bitmap, so that two
builds can be compared output for output on the same inputs.

--impl reference times the reference's own CPU implementation of the path on the
host cores: oracle/_ref (the reference's headers compiled against the Eigen-API
shim) or the plain-C oracle port -- whichever is present; it says which.  The
thread count is the number of cores the process may run on (sched_getaffinity),
set explicitly: torchrun's OMP_NUM_THREADS=1 does not apply.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

D = 128
M = 10
SEED = 12345
LOG2_B = 20
HBM_FALLBACK_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback
METRIC = "batched L-BFGS instances/sec (Rosenbrock d=128)"
DUMP_INSTANCES = 16384  # --dump-outputs: instances sampled from the batch
DUMP_SEED = 2024


def host_threads() -> int:
    """Cores this process may run on -- what both CPU legs use, whatever OMP_NUM_THREADS says."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def algorithmic_bytes(iters, w=8, d=D, m=M):
    """SURVEY.md 8(d): sum_t w*d*(2*min(t, m) + 6), t = 0..K-1, summed over instances."""
    import numpy as np
    K = iters.astype(np.int64)
    full = np.maximum(K - m, 0)
    ramp = np.minimum(K, m)
    pairs = full * m + ramp * (ramp - 1) // 2
    return int((w * d * (6 * K + 2 * pairs)).sum())


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self._stop.is_set():
            try:
                out = subprocess.run(
                    ["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                     "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                self.rows.append([c.strip() for c in out.strip().split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 7:
                continue
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
            except ValueError:
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_leg(kind_pref: str, target_seconds: float, log2_b: int, threads: int):
    """Times the CPU implementation on a bounded prefix of the batch (same x0), `threads` OpenMP threads."""
    import numpy as np
    from oracle import oracle_binding as ob
    kind = "port"
    impl = "oracle"
    if kind_pref == "reference" and ob.ref_available():
        kind, impl = "reference", "ref"
    chunk = 64 * threads
    done, t_total, first = 0, 0.0, 0
    iters = []
    while t_total < target_seconds and done < (1 << log2_b):
        x0 = ob.fill_uniform((chunk, D), first, SEED, -2.0, 2.0)
        r = ob.minimize(ob.LBFGS, ob.FN_ROSENBROCK, x0, impl=impl, threads=threads)
        t_total += r["seconds"]
        done += chunk
        first += chunk * D
        iters.append(r["num_iterations"])
    return {"value": done / t_total, "unit": "instances/s", "cores": threads, "kind": kind,
            "sample": f"first {done} instances of the batch (same x0 stream), {t_total:.1f} s, "
                      f"OpenMP schedule(dynamic) on {threads} threads, "
                      f"mean {float(np.concatenate(iters).mean()):.1f} iterations"
            }, done, t_total


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = host_threads()
    vals = []
    for _ in range(args.warmup):
        cpu_leg("reference", 0.5, LOG2_B, threads)
    base = None
    t0 = time.perf_counter()
    for _ in range(args.steps):
        base, done, secs = cpu_leg("reference", args.ref_seconds, LOG2_B, threads)
        vals.append((done, secs))
    total_inst = sum(v[0] for v in vals)
    total_s = sum(v[1] for v in vals)
    value = total_inst / total_s
    base["value"] = value
    # the plain-C port on the same cores, reported beside the reference-headers build
    port, _, _ = cpu_leg("port", min(args.ref_seconds, 4.0), LOG2_B, threads)
    line = {
        "impl": "reference", "metric": METRIC,
        "value": value, "unit": "instances/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total_s / max(args.steps, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": f"Rosenbrock d=128 fp64, L-BFGS m=10, default stopping preset, "
                               f"bounded prefix of the B=2^{LOG2_B} batch per step",
                   "host_threads": threads,
                   "omp_num_threads_env": os.environ.get("OMP_NUM_THREADS")},
        "cpu_baseline": base,
        "cpu_port_same_cores": port,
        "e2e": {"value": value, "unit": "instances/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "wall_s": time.perf_counter() - t0,
    }
    print(json.dumps(line))
    return 0


def load_instr_mix():
    """FP64-pipe / DMMA warp instructions per solver iteration of the headline kernel, from the ncu
    source-level counts committed under profiles/ (tools/ncu_summary.py writes the file)."""
    for name in ("r02_instr_mix.json", "r01_instr_mix.json"):
        p = os.path.join(ROOT, "profiles", name)
        if os.path.exists(p):
            j = json.load(open(p))
            j["source"] = f"profiles/{name}"
            return j
    return None


def parity_sample(x0, state, prog, n_samples: int, threads: int):
    """`n_samples` strided instances of the timed batch against the CPU oracle: iteration counts, status
    and x* bit for bit.  Raises on any difference (a fast wrong answer is not a benchmark)."""
    import numpy as np
    import torch
    from oracle import oracle_binding as ob
    B = x0.shape[0]
    idx = torch.arange(0, B, max(1, B // n_samples), device=x0.device)[:n_samples]
    xs = x0[idx].cpu().numpy()
    ref = ob.minimize(ob.LBFGS, ob.FN_ROSENBROCK, xs, threads=threads)
    it = prog.num_iterations[idx].cpu().numpy().astype(np.uint32)
    st = prog.status[idx].cpu().numpy()
    xg = state.x[idx].cpu().numpy()
    ok_it = bool(np.array_equal(it, ref["num_iterations"]))
    ok_st = bool(np.array_equal(st, ref["status"]))
    ok_x = bool(np.array_equal(xg.view(np.uint64), ref["x"].view(np.uint64)))
    if not (ok_it and ok_st and ok_x):
        raise SystemExit(f"bench.py: parity check failed (iterations {ok_it}, status {ok_st}, x bits {ok_x})")
    return {"instances": int(idx.numel()), "stride": int(max(1, B // n_samples)),
            "iterations_equal": ok_it, "status_equal": ok_st, "x_bits_equal": ok_x,
            "checker": "oracle/libcno_oracle.so (CPU restatement of the reference path)"}


def dump_outputs(out_dir, state, prog, bitmap):
    """Writes one step's returned arrays (see the module docstring) as float64 .npy files: 16 MiB each for the
    sampled x and gradient, well under 64 MiB in all."""
    import numpy as np
    import torch
    B = state.x.shape[0]
    idx = np.sort(np.random.default_rng(DUMP_SEED).choice(B, min(B, DUMP_INSTANCES), replace=False))
    sel = torch.from_numpy(idx).to(state.x.device)
    arrays = {"instance_index": idx, "x": state.x[sel], "value": state.value[sel], "gradient": state.gradient[sel],
              "num_iterations": prog.num_iterations[sel], "status": prog.status[sel], "nfev": prog.nfev[sel],
              "x_delta": prog.x_delta[sel], "f_delta": prog.f_delta[sel], "gradient_norm": prog.gradient_norm[sel],
              "done_bitmap": bitmap}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = a.cpu().numpy() if torch.is_tensor(a) else a
        if name in ("num_iterations", "nfev", "done_bitmap"):
            a = a.view(np.uint32)  # unsigned counters / bit words held in int32 tensors
        np.save(os.path.join(out_dir, f"{name}.npy"), a.astype(np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3, help="timed steps (at least 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--log2-batch", type=int, default=LOG2_B, help="per-GPU batch = 2^this")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--ref-seconds", type=float, default=6.0,
                    help="CPU seconds per step of the reference arm (a bounded prefix of the batch)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the strong-scaling and other-config records")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the arrays the last timed step returned (a seeded sample of the batch) to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the device path's outputs (--impl b200)")

    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist

    import cppnumericalsolvers_b200 as cn
    from cppnumericalsolvers_b200 import distributed as cd

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU: the product has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    threads = host_threads()

    B = 1 << args.log2_batch
    fn = cn.Rosenbrock(D)
    solver = cn.Lbfgs()
    x0 = torch.empty(B, D, dtype=torch.float64, device=dev)
    # shard = contiguous instance range [rank*B, (rank+1)*B) of the global batch
    cn.fill_uniform(x0, rank * B * D, SEED, -2.0, 2.0)
    status_host = torch.empty(B, dtype=torch.int8).pin_memory()
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def make_step(x_in, status_out):
        nwords = (x_in.shape[0] + 31) // 32

        def step():
            state, prog = solver.Minimize(fn, cn.BatchedFunctionState(x_in))
            # global stop test: per-GPU convergence bitmaps, ONE all-gather (NCCL)
            bitmap = cd.gather_done_bitmaps(prog.done_bitmap(), max_words=nwords)
            status_out.copy_(prog.status, non_blocking=True)  # D2H of status (SURVEY.md 8(d))
            return state, prog, bitmap
        return step

    def timed(step, steps, warmup, clocks_index=None):
        for _ in range(warmup):
            step()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sampler = ClockSampler(clocks_index) if clocks_index is not None else None
        if sampler:
            sampler.__enter__()
        barrier()
        e0.record()
        for _ in range(steps):
            out = step()
        e1.record()
        barrier()
        if sampler:
            sampler.__exit__()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), out, sampler

    ms, (state, prog, bitmap), clocks = timed(make_step(x0, status_host), args.steps, args.warmup, local_rank)
    all_done = bool((bitmap == -1).all().item())  # every bit set
    value = world * B * args.steps / (ms * 1e-3)
    clk = clocks.summary()

    # kernel-only timing for the roofline (CUDA events inside cno_minimize, same stream)
    kms = []
    for _ in range(min(args.steps, 3)):
        _, p2 = solver.Minimize(fn, cn.BatchedFunctionState(x0), timed=True)
        kms.append(p2.launch.kernel_ms)
    kernel_ms = sum(kms) / len(kms)
    iters = prog.num_iterations.cpu().numpy()
    nfev = prog.nfev.cpu().numpy()
    status = prog.status.cpu().numpy()
    assert np.array_equal(status, status_host.numpy()), "status D2H of the timed step differs"
    alg_bytes = algorithmic_bytes(iters)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md)"
    achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9
    traffic = None
    for name in ("r02_traffic.json", "r01_traffic.json"):
        tpath = os.path.join(ROOT, "profiles", name)
        if os.path.exists(tpath):
            tj = json.load(open(tpath))
            if tj.get("batch") == B:
                traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
            break

    # the resource that binds: the FP64 datapath (vector FP64 pipe + FP64 tensor-core MMA)
    compute = None
    mix = load_instr_mix()
    if mix is not None:
        props = torch.cuda.get_device_properties(dev)
        sm_clock_hz = (clk["sm_mhz"] or clk["sm_max_mhz"] or 1965.0) * 1e6
        total_iters = float(iters.astype(np.int64).sum())
        # one FP64 warp instruction occupies a sub-partition's 16-lane FP64 pipe for 2 cycles; a DMMA.8x8x4
        # for `dmma_cycles` (measured: tools/fp64_pipe_probe.cu) -- expressed in FP64-instruction equivalents
        dmma_equiv = mix.get("dmma_cycles", 16.0) / 2.0
        per_iter = mix["fp64_per_iteration"] + dmma_equiv * mix["dmma_per_iteration"]
        ach = per_iter * total_iters / (kernel_ms * 1e-3)
        pk = props.multi_processor_count * 4 * 0.5 * sm_clock_hz
        compute = {"bound": "fp64", "achieved": ach / 1e9, "peak": pk / 1e9, "unit": "G FP64 warp-instr/s",
                   "frac": ach / pk, "fp64_per_iteration": mix["fp64_per_iteration"],
                   "dmma_per_iteration": mix["dmma_per_iteration"], "dmma_fp64_equivalents": dmma_equiv,
                   "instr_per_iteration": mix.get("instr_per_iteration"),
                   "sm_clock_mhz": sm_clock_hz / 1e6, "instr_mix_source": mix["source"],
                   "note": "FP64-pipe warp instructions + FP64 tensor-core MMAs (at their measured pipe "
                           "occupancy) per solver iteration x this run's iterations / kernel time, against "
                           "SMs x 4 x 0.5 warp-instr/clk x the SM clock sampled during the run"}

    # ---- parity: strided instances of the timed batch against the CPU oracle ----
    parity = parity_sample(x0, state, prog, 256, threads) if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, state, prog, bitmap)

    # ---- e2e through the host-buffer C ABI call (wall clock around the call) ----
    e2e = None
    if not args.no_e2e:
        hx0 = torch.empty(B, D, dtype=torch.float64).pin_memory()
        hx0.copy_(x0)
        solver.MinimizeHost(fn, hx0)  # warm-up (first touch of the result buffers)
        barrier()
        tt = time.perf_counter()
        ems, h2d, d2h = 0.0, 0, 0
        for _ in range(args.steps):
            hstate, hprog = solver.MinimizeHost(fn, hx0)
            ems += hprog.launch.total_ms
            h2d, d2h = hprog.launch.h2d_bytes, hprog.launch.d2h_bytes
        wall_ms = (time.perf_counter() - tt) * 1e3
        t = torch.tensor([ems, wall_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ems, wall_ms = float(t[0].item()), float(t[1].item())
        assert torch.equal(hstate.x[:1024], state.x[:1024].cpu())
        e2e = {"value": world * B * args.steps / (wall_ms * 1e-3), "unit": "instances/s",
               "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "ms_per_step": wall_ms / args.steps, "device_event_ms_per_step": ems / args.steps,
               "timing": "wall clock around the call, max over ranks",
               "api": "cno_minimize_host (pinned host buffers; H2D, solve, D2H inside the call)"}

    # ---- strong scaling: the same global batch split over the ranks ----
    strong = None
    if world > 1 and not args.no_extra:
        lo, hi = cd.shard_range(B, rank, world)
        xs = torch.empty(hi - lo, D, dtype=torch.float64, device=dev)
        cn.fill_uniform(xs, lo * D, SEED, -2.0, 2.0)
        sh = torch.empty(hi - lo, dtype=torch.int8).pin_memory()
        sms, _, _ = timed(make_step(xs, sh), max(args.steps, 3), 1)
        strong = {"global_batch": B, "batch_per_gpu": hi - lo, "steps": max(args.steps, 3),
                  "ms_per_step": sms / max(args.steps, 3),
                  "value": B * max(args.steps, 3) / (sms * 1e-3), "unit": "instances/s", "scaling": "strong"}
        del xs

    other = None
    if world == 1 and not args.no_extra and args.log2_batch == LOG2_B:
        del x0, state, prog
        torch.cuda.empty_cache()
        import bench_configs
        # c5t = config 5 under CNO_POLICY_DMMA_LU (NewtonDescent's factorisation on the FP64 tensor core)
        other = [bench_configs.run_config(c) for c in ("c3", "c4", "c5", "c5t")]

    if rank == 0:
        cpu = None
        if not args.no_cpu and world == 1:
            cpu, _, _ = cpu_leg("port", args.cpu_seconds, args.log2_batch, threads)
        line = {
            "metric": METRIC,
            "value": value, "unit": "instances/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {
                "workload": "Rosenbrock d=128 fp64, L-BFGS m=10, default stopping preset "
                            "(BASELINE.json configs[1])",
                "batch_per_gpu": B, "global_batch": world * B, "parallelism": f"shard{world}",
                "l2": "x0 is 1 GiB per GPU (> 126 MB L2); no flush needed",
                "start_generator": f"splitmix64 counter stream, seed {SEED}, U(-2,2)",
                "timed_region": "Minimize kernel + done-bitmap kernel + bitmap all-gather + D2H of status",
                "mean_iterations": float(iters.mean()), "mean_nfev": float(nfev.mean()),
                "status_histogram": {str(k): int(v) for k, v in enumerate(np.bincount(status.astype(np.int64) + 1))},
                "all_done_bitmap": all_done,
                "host_threads": threads,
            },
            "e2e": e2e,
            "gpu_launches": args.steps * 2,  # lbfgs_minimize_kernel + done_bitmap_kernel per step
            "roofline": {
                "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic,
                "peak_source": peak_src, "kernel": "lbfgs_minimize_kernel<RosenbrockFn<double,128>,10>",
                "kernel_ms": kernel_ms, "algorithmic_bytes_per_launch": alg_bytes,
                "compute": compute,
                "note": "hbm: algorithmic bytes = state-streaming model w*d*(2k+6)/iteration; the fused "
                        "kernel keeps the (s,y) history on chip (shared memory + Tensor Memory), so this "
                        "frac > 1 means the traffic was removed, not that work was skipped (see `parity`); "
                        "`traffic` = ncu DRAM bytes per launch.  The resource that BINDS the kernel is the "
                        "FP64 datapath: `compute` is the fraction to read.",
            },
            "parity": parity,
            "cpu_baseline": cpu,
            "strong": strong,
            "other_configs": other,
            "clocks": clk,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
