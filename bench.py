#!/usr/bin/env python
"""bench.py — headline benchmark of the GP-inference hot path on B200.

Metric (BASELINE.json): objective evaluations per second.  Default workload = BASELINE config[1]:
`GPR(Matern52).log_marginal_likelihood()` at N=8192, D=8, fp64 (K-build + blocked Cholesky + log-density),
synthetic data of SURVEY.md 8(d).  One "step" = one full evaluation.

  python bench.py --gpus N --steps K --warmup W            our arm (CUDA path through the public API / C ABI)
  python bench.py --impl reference --steps K --warmup W    CPU arm: the oracle port of the reference's
                                                           algorithm on all host cores (TensorFlow is not
                                                           installable here, see DESIGN.md)
Under torchrun (N>1) every rank evaluates its own replica / shard (weak scaling) and the scalar
objectives are summed with ONE asynchronous NCCL all-reduce per step (off the critical path, all complete inside the
timed region); timing = CUDA events, max over ranks.  Every line also carries BASELINE configs[3] (SVGP, 8 latent GPs)
on the same GPUs in each sharding mode of SURVEY 8(e) (`svgp_c4`).
Prints exactly one JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (config index, description)
    "gpr_c2": (2, "GPR Matern52 fp64 N=8192 D=8 log_marginal_likelihood (BASELINE configs[1])"),
    "gpr_c1": (1, "GPR RBF fp64 N=512 D=2 log_marginal_likelihood (BASELINE configs[0])"),
    "sgpr_c3": (3, "SGPR RBF fp32 N=100000 M=1024 D=16 elbo (BASELINE configs[2])"),
    "svgp_c4": (4, "SVGP RBF+White fp32 N=1e6 B=4096 M=2048 P=8 D=16 minibatch elbo (BASELINE configs[3])"),
    "gpr_c5": (5, "4x GPR (RBF+Matern32)*Linear fp64 N=4096 D=32, sum of per-output LML (BASELINE configs[4])"),
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            burst = float(d.get("bf16_tflops", 1590.0))
            return {"hbm_gbs": float(d.get("hbm_gbs", 6650.0)), "bf16_burst": burst,
                    "bf16_sustained": float(d.get("bf16_tflops_sustained", 0.88 * burst)),
                    "source": "measured (MEASURED_PEAKS.json)"}
        except Exception:  # noqa: BLE001  (unreadable file: fall through to the documented fallback)
            pass
    return {"hbm_gbs": 6650.0, "bf16_burst": 1590.0, "bf16_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(gpu_index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:  # noqa: BLE001
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------
# workloads
# ------------------------------------------------------------------------------------------------------
def host_problem(name: str, rank: int):
    """Synthetic host-side inputs for one rank (rank r evaluates replica / minibatch r)."""
    from oracle import gp_oracle as O  # input generator only (shared with the tests); no oracle compute here

    c = WORKLOADS[name][0]
    if name == "gpr_c2":
        d = O.make_data(2, 8192, 8, 1)
        return dict(X=d["X"], Y=d["Y"], N=8192, D=8, P=1, dtype=np.float64)
    if name == "gpr_c1":
        d = O.make_data(1, 512, 2, 1)
        return dict(X=d["X"], Y=d["Y"], N=512, D=2, P=1, dtype=np.float64)
    if name == "sgpr_c3":
        d = O.make_data(3, 100000, 16, 1, M=1024, dtype=np.float32)
        return dict(X=d["X"], Y=d["Y"], Z=d["Z"], N=100000, D=16, P=1, M=1024, dtype=np.float32)
    if name == "svgp_c4":
        d = O.make_data(4, 1000000, 16, 8, M=2048, dtype=np.float32)
        q_mu, q_sqrt = O.make_q(4, 2048, 8, dtype=np.float32)
        perm = np.random.default_rng(99).permutation(1000000)
        return dict(X=d["X"], Y=d["Y"], Z=d["Z"], q_mu=q_mu, q_sqrt=q_sqrt, perm=perm, N=1000000, D=16, P=8, M=2048,
                    B=4096, dtype=np.float32)
    if name == "gpr_c5":
        d = O.make_data(5, 4096, 32, 4)
        return dict(X=d["X"], Y=d["Y"], N=4096, D=32, P=4, dtype=np.float64)
    raise ValueError(name)


def make_kernel(name: str, mod, D: int, p: int = 0):
    s = float(np.sqrt(D))
    if name in ("gpr_c2",):
        return mod.Matern52(variance=1.0, lengthscales=s)
    if name in ("gpr_c1", "sgpr_c3"):
        return mod.SquaredExponential(variance=1.0, lengthscales=s)
    if name == "svgp_c4":
        return mod.SquaredExponential(variance=1.0, lengthscales=s) + mod.White(variance=0.1)
    if name == "gpr_c5":
        return (mod.SquaredExponential(variance=1.0 + 0.1 * p, lengthscales=s * (1 + 0.05 * p))
                + mod.Matern32(variance=1.0, lengthscales=2 * s)) * mod.Linear(variance=1.0 / (1 + p))
    raise ValueError(name)


def algorithmic_work(name: str, hp: dict):
    """Algorithmic flops / bytes per evaluation (SURVEY.md 8(d)); stated in DESIGN.md."""
    N, D, P = hp["N"], hp["D"], hp["P"]
    T = 8 if hp["dtype"] == np.float64 else 4
    if name in ("gpr_c2", "gpr_c1"):
        return {"chol_flops": N ** 3 / 3.0, "kbuild_bytes_lower": T * (N * (N + 1) / 2 + N * D),
                "kbuild_bytes_full": T * (N * N + N * D)}
    if name == "gpr_c5":
        return {"chol_flops": P * N ** 3 / 3.0, "kbuild_bytes_lower": P * T * (N * (N + 1) / 2 + N * D),
                "kbuild_bytes_full": P * T * (N * N + N * D)}
    if name == "sgpr_c3":
        M = hp["M"]
        return {"chol_flops": 2.0 * M * M * N + 2 * M ** 3 / 3.0, "kbuild_bytes_lower": T * (M * N + (M + N) * D),
                "kbuild_bytes_full": T * (M * N + (M + N) * D)}
    M, B = hp["M"], hp["B"]
    return {"chol_flops": M ** 3 / 3.0 + 2.0 * M * M * B / 2 + P * M * M * B, "kbuild_bytes_lower": T * (M * M / 2 + M * B),
            "kbuild_bytes_full": T * (M * M + M * B)}


class OurArm:
    """Evaluations through the public API of gpflow_b200 (which calls the C ABI)."""

    def __init__(self, name: str, hp: dict, rank: int, world: int):
        import gpflow_b200 as gpf

        self.gpf, self.name, self.hp, self.rank, self.world = gpf, name, hp, rank, world
        gpf.config.set_default_float(hp["dtype"])
        if hp["dtype"] == np.float32:
            gpf.config.set_default_jitter(1e-4)  # SURVEY 8(d): explicit jitter for the fp32 configs
        self.models = None
        self.step_idx = 0

    def build_resident(self):
        """Models with inputs already resident in HBM (for `value`)."""
        gpf, hp, name = self.gpf, self.hp, self.name
        K = gpf.kernels
        if name in ("gpr_c2", "gpr_c1"):
            self.models = [gpf.models.GPR((hp["X"], hp["Y"]), make_kernel(name, K, hp["D"]), noise_variance=0.1)]
        elif name == "gpr_c5":
            Xd = gpf.ops.to_device(hp["X"])
            self.models = [gpf.models.GPR((Xd, hp["Y"][:, p:p + 1]), make_kernel(name, K, hp["D"], p), noise_variance=0.1)
                           for p in range(hp["P"])]
        elif name == "sgpr_c3":
            self.models = [gpf.models.SGPR((hp["X"], hp["Y"]), make_kernel(name, K, hp["D"]), hp["Z"], noise_variance=0.1)]
        elif name == "svgp_c4":
            m = gpf.models.SVGP(make_kernel(name, K, hp["D"]), gpf.likelihoods.Gaussian(0.1), hp["Z"], num_latent_gps=hp["P"],
                                q_mu=hp["q_mu"], q_sqrt=hp["q_sqrt"], whiten=True, num_data=hp["N"])
            self.models = [m]
            # minibatches = consecutive slices of a fixed permutation; keep a window of them resident
            self.batches = []
            for i in range(8):
                idx = hp["perm"][(self.rank * 8 + i) * hp["B"]:(self.rank * 8 + i + 1) * hp["B"]]
                self.batches.append((gpf.ops.to_device(hp["X"][idx]), gpf.ops.to_device(hp["Y"][idx])))

    def eval_resident(self):
        """One evaluation, inputs resident; returns a device fp64 scalar tensor."""
        ops = self.gpf.ops
        if self.name == "svgp_c4":
            xb, yb = self.batches[self.step_idx % len(self.batches)]
            self.step_idx += 1
            return self.models[0].elbo((xb, yb))
        if self.name == "sgpr_c3":
            return self.models[0].elbo()
        if len(self.models) == 1:
            return self.models[0].log_marginal_likelihood()
        # independent outputs: one CUDA stream per model so the (latency-bound) factorisations overlap
        T = ops.torch()
        if not hasattr(self, "_streams"):
            self._streams = [T.cuda.Stream() for _ in self.models]
        cur = T.cuda.current_stream()
        vals = []
        for m, s_ in zip(self.models, self._streams):
            s_.wait_stream(cur)
            with T.cuda.stream(s_):
                vals.append(m.log_marginal_likelihood())
        acc = ops.zeros_scalar(1)
        for v, s_ in zip(vals, self._streams):
            cur.wait_stream(s_)
            ops.axpby(1.0, v.reshape(1), 1.0, acc)
        return acc[0]

    def eval_e2e(self, pinned):
        """One evaluation from HOST buffers through the public API: H2D of this step's inputs, the fused
        evaluation, D2H of the scalar.  Returns (float value, h2d bytes, d2h bytes)."""
        gpf, hp, name = self.gpf, self.hp, self.name
        T = gpf.ops.torch()
        K = gpf.kernels
        dev = gpf.ops.require_cuda()
        if name in ("gpr_c2", "gpr_c1", "gpr_c5"):
            Xd = pinned["X"].to(dev, non_blocking=True)
            Yd = pinned["Y"].to(dev, non_blocking=True)
            h2d = pinned["X"].numel() * pinned["X"].element_size() + pinned["Y"].numel() * pinned["Y"].element_size()
            if name == "gpr_c5":
                # independent outputs: one stream per output (as in eval_resident), workspaces of the resident models
                if not hasattr(self, "_streams"):
                    self._streams = [T.cuda.Stream() for _ in self.models]
                cur = T.cuda.current_stream()
                vals = []
                for p, (m0, s_) in enumerate(zip(self.models, self._streams)):
                    s_.wait_stream(cur)
                    with T.cuda.stream(s_):
                        m = gpf.models.GPR((Xd, Yd[:, p:p + 1].contiguous()), m0.kernel, noise_variance=0.1)
                        m._ws, m._out = m0._ws, m0._out
                        vals.append(m.log_marginal_likelihood().reshape(1).clone())
                for s_ in self._streams:
                    cur.wait_stream(s_)
                tot = 0.0
                for v in vals:
                    tot += float(v.item())
                return tot, h2d, 8 * hp["P"]
            m = self._e2e_model(Xd, Yd)
            return float(m.log_marginal_likelihood().item()), h2d, 8
        if name == "sgpr_c3":
            Xd = pinned["X"].to(dev, non_blocking=True)
            Yd = pinned["Y"].to(dev, non_blocking=True)
            h2d = pinned["X"].numel() * 4 + pinned["Y"].numel() * 4
            m = gpf.models.SGPR((Xd, Yd), make_kernel(name, K, hp["D"]), self.models[0].inducing_variable, noise_variance=0.1)
            return float(m.elbo().item()), h2d, 8
        i = self.step_idx % pinned["nb"]
        self.step_idx += 1
        xb = pinned["Xb"][i].to(dev, non_blocking=True)
        yb = pinned["Yb"][i].to(dev, non_blocking=True)
        h2d = xb.numel() * 4 + yb.numel() * 4
        return float(self.models[0].elbo((xb, yb)).item()), h2d, 8

    def _e2e_model(self, Xd, Yd):
        # reuse the workspace of the resident model: a fresh 537 MB cudaMalloc per step is not part of the path
        m = self.gpf.models.GPR((Xd, Yd), self.models[0].kernel, noise_variance=0.1)
        m._ws, m._out = self.models[0]._ws, self.models[0]._out
        return m

    def pinned_inputs(self):
        T = self.gpf.ops.torch()
        hp = self.hp
        if self.name == "svgp_c4":
            nb = 8
            Xb, Yb = [], []
            for i in range(nb):
                idx = hp["perm"][(self.rank * 8 + i) * hp["B"]:(self.rank * 8 + i + 1) * hp["B"]]
                Xb.append(T.from_numpy(np.ascontiguousarray(hp["X"][idx])).pin_memory())
                Yb.append(T.from_numpy(np.ascontiguousarray(hp["Y"][idx])).pin_memory())
            return {"Xb": Xb, "Yb": Yb, "nb": nb}
        return {"X": T.from_numpy(np.ascontiguousarray(hp["X"])).pin_memory(),
                "Y": T.from_numpy(np.ascontiguousarray(hp["Y"])).pin_memory()}


def cpu_eval(name: str, hp: dict, threads: int):
    """The oracle port of the reference's algorithm on the host cores (CPU arm / cpu_baseline)."""
    from oracle import fast_cpu, gp_oracle as O

    # torchrun exports OMP_NUM_THREADS=1 to its children: give BLAS/LAPACK all the host threads back for this leg
    try:
        from threadpoolctl import threadpool_limits
        limit = threadpool_limits(limits=threads)
    except Exception:  # noqa: BLE001
        import contextlib
        limit = contextlib.nullcontext()
    with limit:
        return _cpu_eval(name, hp, threads, fast_cpu, O)


def _cpu_eval(name, hp, threads, fast_cpu, O):
    if name in ("gpr_c2", "gpr_c1"):
        return fast_cpu.gpr_lml_threaded(hp["X"], hp["Y"], make_kernel(name, O, hp["D"]), 0.1, threads)
    if name == "gpr_c5":
        return sum(fast_cpu.gpr_lml_threaded(hp["X"], hp["Y"][:, p:p + 1], make_kernel(name, O, hp["D"], p), 0.1, threads)
                   for p in range(hp["P"]))
    if name == "sgpr_c3":   # Kuf [1024 x 1e5] built in column blocks on all cores (bit-identical values)
        return O.sgpr_elbo(hp["X"], hp["Y"], fast_cpu.ThreadedKernel(make_kernel(name, O, hp["D"]), threads), hp["Z"], 0.1,
                           jitter=1e-4)
    idx = hp["perm"][:hp["B"]]
    return O.svgp_elbo(hp["X"][idx], hp["Y"][idx], hp["Z"], make_kernel(name, O, hp["D"]), hp["q_mu"], hp["q_sqrt"], 0.1,
                       whiten=True, num_data=hp["N"], jitter=1e-4)


# ------------------------------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    name = args.workload
    hp = host_problem(name, 0)
    threads = os.cpu_count() or 1
    for _ in range(args.warmup):
        cpu_eval(name, hp, threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        val = cpu_eval(name, hp, threads)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"objective": np.array([val], dtype=np.float64)})
    v = args.steps / dt
    line = {
        "impl": "reference", "metric": "objective_evals_per_sec", "value": v, "unit": "evals/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64" if hp["dtype"] == np.float64 else "f32",
        "data": "synthetic", "config": {"workload": WORKLOADS[name][1]}, "objective": float(val),
        "cpu_baseline": {"value": v, "unit": "evals/s", "cores": threads, "kind": "port",
                         "sample": f"{args.steps} full evaluations of the workload (NumPy/SciPy+OpenBLAS oracle port of "
                                   "the reference algorithm; TensorFlow not installable, see DESIGN.md)"},
        "e2e": {"value": v, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    return 0


def pin_to_gpu_numa_node(local: int):
    """Pins this rank's host threads to the CPUs NVML reports as local to its GPU (ranks of GPUs 4-7 sit on the
    second NUMA node of these boxes).  Returns the previous affinity so that the CPU-baseline leg can have all cores."""
    prev = None
    try:
        import pynvml
        import torch

        prev = os.sched_getaffinity(0)
        pr = torch.cuda.get_device_properties(local)
        bus = f"{pr.pci_domain_id:08x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
        pynvml.nvmlDeviceSetCpuAffinity(h)
    except Exception:  # noqa: BLE001  (best effort: an unpinned rank is still correct)
        pass
    return prev


def step_stats(per_rank_ms):
    """per_rank_ms [world, steps] -> summary that tells a one-off stall from a per-step cost."""
    a = np.asarray(per_rank_ms, dtype=np.float64)
    worst = a.max(axis=0)  # slowest rank of every step
    return {"median_ms": float(np.median(worst)), "min_ms": float(worst.min()), "max_ms": float(worst.max()),
            "p95_ms": float(np.percentile(worst, 95)), "per_rank_median_ms": [float(x) for x in np.median(a, axis=1)],
            "steps_over_1p5x_median": int((worst > 1.5 * np.median(worst)).sum())}


def timed_loop(torch, dist, steps, one_step, slots):
    """`steps` iterations of one_step(i) -> device fp64 scalar.  The scalar of step i goes to slots[i] and is summed over
    the ranks by an ASYNCHRONOUS all-reduce (its own NCCL stream): step i+1 does not consume it, so the collective is
    off the critical path; all of them are complete before the closing event.  Device-timed, barrier + synchronize on
    both sides.  Returns (total ms on this rank, per-step ms list)."""
    works = []
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    ev[0].record()
    for i in range(steps):
        v = one_step(i)
        slot = slots[i:i + 1]
        slot.copy_(v.reshape(1))
        if dist is not None:
            works.append(dist.all_reduce(slot, async_op=True))  # ONE scalar all-reduce per evaluation (SURVEY 8(e))
        ev[i + 1].record()
    for w in works:
        w.wait()
    end = torch.cuda.Event(enable_timing=True)
    end.record()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    per_step = [ev[i].elapsed_time(ev[i + 1]) for i in range(steps)]
    return ev[0].elapsed_time(end), per_step


def gather_ms(torch, dist, world, ms_total, per_step):
    """max over ranks of the region time + the [world, steps] table of per-step times."""
    if dist is None:
        return ms_total, [per_step]
    t = torch.tensor([ms_total], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    mine = torch.tensor(per_step, dtype=torch.float64, device="cuda")
    allv = torch.empty((world, len(per_step)), dtype=torch.float64, device="cuda")
    dist.all_gather_into_tensor(allv.view(-1), mine)
    return float(t.item()), allv.cpu().numpy().tolist()


def svgp_c4_modes(args, torch, dist, rank, world):
    """BASELINE configs[3] on the N GPUs of this run, in the sharding modes of SURVEY 8(e) (gpflow_b200/sharding.py):
    independent minibatches (throughput), rows of ONE minibatch, latent GPs of ONE minibatch with the column-sharded
    solve + all-gather.  Every mode: device-timed, max over ranks, the async scalar all-reduce inside the region."""
    import gpflow_b200 as gpf
    from gpflow_b200 import sharding

    prev_float, prev_jit = gpf.config.default_float(), gpf.config.default_jitter()
    hp = host_problem("svgp_c4", rank)
    arm = OurArm("svgp_c4", hp, rank, world)
    arm.build_resident()
    model = arm.models[0]
    steps = args.steps
    slots = torch.zeros(steps, dtype=torch.float64, device="cuda")
    # one SHARED minibatch sequence for the single-minibatch modes (every rank holds the same rows)
    shared = []
    for i in range(4):
        idx = hp["perm"][i * hp["B"]:(i + 1) * hp["B"]]
        shared.append((gpf.ops.to_device(hp["X"][idx]), gpf.ops.to_device(hp["Y"][idx])))
    modes = {
        "independent_minibatches": lambda i: arm.eval_resident(),
        "rows_of_one_minibatch": lambda i: sharding.svgp_elbo_row_sharded(model, shared[i % 4], rank, world)[0],
        "latents_of_one_minibatch": lambda i: sharding.svgp_elbo_latent_sharded(model, shared[i % 4], rank, world)[0],
        "latents_no_sharded_solve": lambda i: sharding.svgp_elbo_latent_sharded(model, shared[i % 4], rank, world,
                                                                                shard_solve=False)[0],
    }
    out = {}
    full = None
    for name, fn in modes.items():
        internal_reduce = name != "independent_minibatches"  # the sharded modes all-reduce inside (the share IS the step)
        for i in range(3):
            fn(i)
        ms, per = timed_loop(torch, None if internal_reduce else dist, steps, fn, slots)
        if internal_reduce and dist is not None:
            dist.barrier()
        ms, table = gather_ms(torch, dist, world, ms, per)
        evals = (world if name == "independent_minibatches" else 1) * steps / (ms * 1e-3)
        out[name] = {"evals_per_s": evals, "ms_per_step": ms / steps, "step_stats": step_stats(table)}
        if name != "independent_minibatches":
            val = float(fn(0).item())
            if full is None:
                full = float(model.elbo(shared[0]).item())
            out[name]["sum_of_shares_vs_full_rel_err"] = abs(val - full) / max(abs(full), 1e-300)
    out["config"] = WORKLOADS["svgp_c4"][1]
    out["n_gpus"] = world
    out["note"] = ("independent_minibatches = the throughput mode the north star's >= 6x refers to (weak scaling, one "
                   "minibatch per GPU per step); the one-minibatch modes are strong scaling and pay the replicated "
                   "chol(Kuu) of M = 2048 on every rank")
    gpf.config.set_default_float(prev_float)
    gpf.config.set_default_jitter(prev_jit)
    del arm, model, shared
    torch.cuda.empty_cache()
    return out


def run_ours(args):
    import ctypes

    import torch

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local)
    prev_affinity = pin_to_gpu_numa_node(local)
    dist = None
    if world > 1:
        import torch.distributed as dist_

        dist = dist_
        if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", ""):
            os.environ["NCCL_DEBUG"] = "WARN"  # NCCL prints its version banner on STDOUT; keep stdout = one JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from gpflow_b200 import _lib

    lib = _lib.load()
    name = args.workload
    hp = host_problem(name, rank)
    arm = OurArm(name, hp, rank, world)
    arm.build_resident()
    steps = args.steps
    warm = max(args.warmup, 3)
    slots = torch.zeros(steps, dtype=torch.float64, device="cuda")

    for i in range(warm):
        arm.eval_resident()
    sampler = ClockSampler(local) if rank == 0 else None
    lib.gpk_launch_count_reset()
    ms_total, per_step = timed_loop(torch, dist, steps, lambda i: arm.eval_resident(), slots)
    launches = int(lib.gpk_launch_count())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"objective": slots[-1:].cpu().numpy()})
    objective = float(slots[-1].item()) / world
    ms_total, table = gather_ms(torch, dist, world, ms_total, per_step)
    ms_step = ms_total / steps
    value = world / (ms_step * 1e-3)

    # value + gradient evaluations (training step of the Scipy optimiser contract), when the model has a device backward
    grad = None
    if name in ("gpr_c2", "gpr_c1") and hasattr(arm.models[0], "log_marginal_likelihood_and_grad"):
        m0 = arm.models[0]
        for _ in range(2):
            m0.log_marginal_likelihood_and_grad()
        gsteps = max(3, steps // 4)
        gms, _ = timed_loop(torch, None, gsteps, lambda i: m0.log_marginal_likelihood_and_grad()[0], slots)
        gms, _ = gather_ms(torch, dist, world, gms, [0.0])
        grad = {"value_and_grad_evals_per_s": world * gsteps / (gms * 1e-3), "ms_per_step": gms / gsteps, "steps": gsteps}

    # instrumented pass: the same K steps with CUDA events around every launch (per-kernel-class time and issued work)
    NC = 8
    lib.gpk_prof_enable(1)
    for _ in range(steps):
        arm.eval_resident()
    msv, cnt, wk = (ctypes.c_double * NC)(), (ctypes.c_int64 * NC)(), (ctypes.c_double * NC)()
    lib.gpk_prof_read2(msv, cnt, wk, NC)
    lib.gpk_prof_enable(0)
    cls_names = ["kbuild", "gemm_dmma_simt", "potrf_leaf", "gemm_skinny", "misc", "tcgen05", "panel_solve"]
    prof = {k: {"ms_per_step": msv[i] / steps, "launches_per_step": cnt[i] / steps, "issued_macs_per_step": wk[i] / steps}
            for i, k in enumerate(cls_names)}
    clocks = sampler.stop() if sampler is not None else None
    pk_probe = (ctypes.c_double * 4)()
    lib.gpk_peak_probe(pk_probe, None)

    # standalone K-build of the FULL symmetric matrix (the reference's `kernel(X)` op): CUDA events around
    # K launches of gpk_kbuild alone, output = 8*N^2 bytes > L2
    kfull = None
    if name in ("gpr_c2", "gpr_c1"):
        from gpflow_b200 import ops as _ops
        from gpflow_b200.kernels import compile_kernel as _ck
        Xd = arm.models[0].data[0]
        desc = _ck(arm.models[0].kernel, hp["D"])
        Kbuf = _ops.empty((hp["N"], hp["N"]), like=Xd)
        for _ in range(3):
            _ops.kbuild(desc, Xd, None, out=Kbuf)
        torch.cuda.synchronize()
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0.record()
        for _ in range(steps):
            _ops.kbuild(desc, Xd, None, out=Kbuf)
        k1.record()
        torch.cuda.synchronize()
        kfull = k0.elapsed_time(k1) / steps
        del Kbuf

    # end-to-end through the public API from pinned HOST buffers (H2D + evaluation + D2H every step)
    pinned = arm.pinned_inputs()
    for _ in range(3):
        arm.eval_e2e(pinned)
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        val, h2d, d2h = arm.eval_e2e(pinned)
    e1.record()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    e2e_ms = max(e0.elapsed_time(e1), 1e3 * (time.perf_counter() - t0)) / steps
    if dist is not None:
        t = torch.tensor([e2e_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    e2e_value = world / (e2e_ms * 1e-3)

    # BASELINE configs[2] names "posterior predict": SGPR.predict_f at Xnew [10000, D] (fused: Kuf/Kuu, two factorisations, the
    # conditional), timed the same way; serving-style throughput in predicted points per second
    predict = None
    if name == "sgpr_c3":
        from oracle import gp_oracle as _O
        Xn = arm.gpf.ops.to_device(_O.make_data(3, hp["N"], hp["D"], 1, M=hp["M"], n_new=10000, dtype=hp["dtype"])["Xnew"])
        m0 = arm.models[0]
        for _ in range(2):
            m0.predict_f(Xn)
        psteps = max(3, steps // 2)
        torch.cuda.synchronize()
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record()
        for _ in range(psteps):
            mean, var = m0.predict_f(Xn)
        p1.record()
        torch.cuda.synchronize()
        pms = p0.elapsed_time(p1) / psteps
        post = m0.posterior()
        for _ in range(2):
            post.predict_f(Xn)
        p0.record()
        for _ in range(psteps):
            post.predict_f(Xn)
        p1.record()
        torch.cuda.synchronize()
        cms = p0.elapsed_time(p1) / psteps
        predict = {"n_new": 10000, "fused_predict_f_ms": pms, "fused_points_per_s": 10000 / (pms * 1e-3),
                   "cached_posterior_predict_f_ms": cms, "cached_points_per_s": 10000 / (cms * 1e-3),
                   "note": "fused = SGPR.predict_f (factorisations redone per call, posteriors.py:520-551); cached = "
                           "model.posterior() once, then posterior.predict_f (PrecomputeCacheType.TENSOR)"}
        del Xn, mean, var, post

    # BASELINE configs[3] (SVGP, 8 latent GPs) on the same GPUs, every sharding mode: the multi-GPU row of the north star
    svgp = None
    if not args.no_svgp and name != "svgp_c4":
        del pinned
        svgp = svgp_c4_modes(args, torch, dist, rank, world)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0

    pk = peaks()
    work = algorithmic_work(name, hp)
    f64 = hp["dtype"] == np.float64
    tc_s, dm_s, pn_s = (prof[k]["ms_per_step"] * 1e-3 for k in ("tcgen05", "gemm_dmma_simt", "panel_solve"))
    kb_s = prof["kbuild"]["ms_per_step"] * 1e-3
    tc_macs = prof["tcgen05"]["issued_macs_per_step"]
    i8_peak, dmma_peak = float(pk_probe[0]), float(pk_probe[1])
    ncu = {}
    try:
        ncu = json.load(open(os.path.join(ROOT, "profiles", "r2_ncu_summary.json")))
    except Exception:  # noqa: BLE001
        pass
    if f64:
        ach = 2.0 * tc_macs / tc_s / 1e12 if tc_s > 0 else 0.0
        S = int(lib.gpk_potrf_last_slices()) or 7
        n_digit_mmas = S * (S + 1) // 2 + (1 if S == 6 else 0)   # + the (3,3) product at S = 6 (planes.cuh)
        roofline = {
            "bound": "tensor",
            "kernel": "syrk_i8_kernel (tcgen05 kind::i8: fp64 operands as S balanced base-256 digit planes, S(S+1)/2 "
                      "(+1 at S = 6) digit MMAs per 32-deep k-step, exact int32 accumulation in TMEM; tcgen05 has no f64 kind)",
            "achieved": ach, "peak": i8_peak, "unit": "TFLOP/s", "frac": ach / i8_peak if i8_peak else None,
            "ops": "int8 operations ISSUED by the launches of this kernel (2 per MAC, padding tiles included) / summed "
                   "duration of those launches (CUDA events on the launch stream)",
            "peak_source": "tcgen05 kind::i8 issue peak measured in this run on this GPU (gpk_peak_probe: 128x256x32 MMAs, "
                           "operands resident in shared memory, all SMs); MEASURED_PEAKS.json holds bf16 only",
            "peak_bf16_measured_for_context": {"tflops_sustained": pk["bf16_sustained"], "source": pk["source"],
                                               "frac_vs_2x_bf16": ach / (2.0 * pk["bf16_sustained"])},
            "slices": S, "digit_radix": 256, "digit_mmas_per_fp64_kstep": n_digit_mmas,
            "fp64_equivalent_tflops": (2.0 * tc_macs / n_digit_mmas) / tc_s / 1e12 if tc_s > 0 else 0.0,
            "kernel_ms_per_step": prof["tcgen05"]["ms_per_step"], "launches_per_step": prof["tcgen05"]["launches_per_step"],
            "share_of_step": prof["tcgen05"]["ms_per_step"] / ms_step,
            "traffic": ncu.get("syrk_i8_dram_bytes_per_launch"),
            "traffic_source": ncu.get("syrk_i8_source"),
            "dmma_class": {"kernels": "potrf_panel_kernel (panel solve + fused K = 128 update) + gemm_dmma_kernel (trailing updates "
                                      "below the tcgen05 threshold), mma.sync.m8n8k4.f64",
                           "achieved_tflops": 2.0 * (prof["gemm_dmma_simt"]["issued_macs_per_step"] + prof["panel_solve"]["issued_macs_per_step"])
                           / (dm_s + pn_s) / 1e12 if dm_s + pn_s > 0 else 0.0,
                           "peak_tflops": dmma_peak, "peak_source": "gpk_peak_probe (DMMA, registers only, all SMs)",
                           "ms_per_step": prof["gemm_dmma_simt"]["ms_per_step"], "panel_ms_per_step": prof["panel_solve"]["ms_per_step"]},
            "whole_factorisation": {"algorithmic_fp64_flops": work["chol_flops"],
                                    "fp64_equivalent_tflops_of_the_step": work["chol_flops"] / (ms_step * 1e-3) / 1e12,
                                    "frac_of_dmma_peak": work["chol_flops"] / (ms_step * 1e-3) / 1e12 / dmma_peak if dmma_peak else None},
        }
        if roofline["dmma_class"]["peak_tflops"]:
            roofline["dmma_class"]["frac"] = roofline["dmma_class"]["achieved_tflops"] / dmma_peak
    else:
        ach = 2.0 * tc_macs / tc_s / 1e12 if tc_s > 0 else 0.0
        tf32_peak = pk["bf16_sustained"] / 2.0
        roofline = {
            "bound": "tensor", "kernel": "gemm_tf32_kernel (tcgen05 kind::tf32, 3 MMAs per fp32 product: hi*hi + hi*lo + lo*hi)",
            "achieved": ach, "peak": tf32_peak, "unit": "TFLOP/s", "frac": ach / tf32_peak,
            "ops": "tf32 operations ISSUED (2 per MAC, 3 MACs per fp32 product) / summed duration of the launches",
            "peak_source": pk["source"] + ": half of the measured sustained bf16 rate (tf32 dense = bf16 / 2 on this part)",
            "fp32_equivalent_tflops": ach / 3.0, "kernel_ms_per_step": prof["tcgen05"]["ms_per_step"],
            "launches_per_step": prof["tcgen05"]["launches_per_step"], "share_of_step": prof["tcgen05"]["ms_per_step"] / ms_step,
            "traffic": ncu.get("gemm_tf32_dram_bytes_per_launch"), "traffic_source": ncu.get("gemm_tf32_source"),
        }
    if svgp is not None:
        roofline["svgp_c4"] = svgp
    kb_ach = work["kbuild_bytes_lower"] / kb_s / 1e9 if kb_s > 0 else 0.0
    kbuild = {"bound": "hbm", "achieved": kb_ach, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": kb_ach / pk["hbm_gbs"],
              "peak_source": pk["source"], "algorithmic_bytes_per_step": work["kbuild_bytes_lower"],
              "ms_per_step": prof["kbuild"]["ms_per_step"], "traffic": ncu.get("kbuild_dram_bytes_per_launch"),
              "note": "inside the LML: lower-triangle tiles only (GPK_LOWER); fp64 exp/sqrt make it fp64-pipe / issue bound"}
    if kfull:
        fa = work["kbuild_bytes_full"] / (kfull * 1e-3) / 1e9
        kbuild["full_matrix"] = {"ms": kfull, "achieved": fa, "frac": fa / pk["hbm_gbs"],
                                 "algorithmic_bytes": work["kbuild_bytes_full"],
                                 "note": "standalone kernel(X): lower tiles computed once, mirrored tile stored straight from registers"}

    # CPU baseline on this box's host cores (all of them again): bounded sample = full evaluations for ~10-30 s
    if prev_affinity is not None:
        try:
            os.sched_setaffinity(0, prev_affinity)
        except Exception:  # noqa: BLE001
            pass
    threads = os.cpu_count() or 1
    t0 = time.perf_counter()
    n_cpu = 0
    cpu_val = None
    while True:
        cpu_val = cpu_eval(name, hp, threads)
        n_cpu += 1
        if time.perf_counter() - t0 > 12.0 or n_cpu >= 8:
            break
    cpu_dt = (time.perf_counter() - t0) / n_cpu
    # parity of the objective against the CPU port ON THE SAME INPUTS: the SVGP steps cycle through minibatches,
    # the CPU port evaluates minibatch 0 of rank 0, so that one is re-evaluated here (outside the timed region)
    check = objective
    if name == "svgp_c4":
        arm.step_idx = 0
        check = float(arm.eval_resident().item())
    rel = abs(check - cpu_val) / max(abs(cpu_val), 1e-300)

    line = {
        "metric": "objective_evals_per_sec", "value": value, "unit": "evals/s", "n_gpus": world, "steps": steps,
        "warmup": warm, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64" if f64 else "f32", "data": "synthetic",
        "config": {"workload": WORKLOADS[name][1]},
        "parallelism": f"replicas x{world}, 1 asynchronous scalar all-reduce per evaluation" if world > 1 else "single GPU",
        "l2": "working set (K / Kuf matrix) exceeds the 126 MB L2, no flush between steps" if name not in ("gpr_c1",) else "fits L2 (plumbing config)",
        "objective": objective, "objective_vs_cpu_rel_err": rel, "step_stats": step_stats(table),
        "roofline": roofline, "kbuild_roofline": kbuild, "kernel_classes": prof,
        "pipe_peaks_probe": {"tcgen05_i8_tops": i8_peak, "dmma_fp64_tflops": dmma_peak, "sms": int(pk_probe[2])},
        "cpu_baseline": {"value": 1.0 / cpu_dt, "unit": "evals/s", "cores": threads, "kind": "port",
                         "sample": f"{n_cpu} full evaluation(s) of the same workload, NumPy/SciPy+OpenBLAS oracle port"},
        "e2e": {"value": e2e_value, "unit": "evals/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h},
        "gpu_launches": launches, "clocks": clocks,
    }
    if grad is not None:
        line["value_and_grad"] = grad
    if predict is not None:
        line["posterior_predict"] = predict
    if svgp is not None:
        line["svgp_c4"] = svgp
    emit(line)
    if dist is not None:
        dist.destroy_process_group()
    return 0


_REAL_STDOUT = None


def dump_outputs(out_dir: str, arrays: dict):
    """Writes what the timed path returned in its last step as out_dir/<name>.npy (float64). The inputs are seeded,
    so two builds run with the same arguments can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def emit(line: dict):
    """The ONE JSON line of the contract, on the process's original stdout."""
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    # stdout must carry exactly one JSON line: libraries (NCCL prints its version banner on stdout at some debug
    # levels) get stderr instead -- file descriptor 1 is re-pointed at stderr and the original kept for emit()
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="gpr_c2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-svgp", action="store_true", help="skip the SVGP C4 sharding-mode section")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the objective of the last timed step as DIR/objective.npy (float64, shape [1]; "
                         "summed over ranks under torchrun)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
