"""Times SGPR value-only elbo() against value + gradient elbo_and_grad() at BASELINE configs[2] (C3: N = 1e5, M = 1024,
D = 16, RBF, the bench's host_problem data), in float32 and float64, interleaved in one process with CUDA events, and
the per-class kernel times of both calls (gpk_prof_*).  Prints one JSON object and writes it to --out when given.

    python scripts/time_sgpr_grad.py [--steps 20] [--warmup 3] [--out profiles/sgpr_grad_c3.json]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import gpflow_b200 as gpf  # noqa: E402
from gpflow_b200 import _lib  # noqa: E402
from oracle import gp_oracle as O  # noqa: E402  (input generator only)

CLASSES = ["kbuild", "gemm", "leaf", "skinny", "misc", "tc", "panel"]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, check=False).stdout.strip()
    name, power, clock = (s.strip() for s in q.splitlines()[0].split(","))
    return {"device": name, "power_limit": power, "clocks_max_sm": clock}


def per_class(lib, fn, steps):
    lib.gpk_prof_enable(1)
    for _ in range(steps):
        fn()
    n = len(CLASSES)
    ms, cnt = (ctypes.c_double * n)(), (ctypes.c_int64 * n)()
    lib.gpk_prof_read(ms, cnt, n)
    lib.gpk_prof_enable(0)
    return {k: round(ms[i] / steps, 4) for i, k in enumerate(CLASSES)}


def run(dtype, steps, warmup):
    lib = _lib.load()
    d = O.make_data(3, 100000, 16, 1, M=1024, dtype=dtype)
    gpf.config.set_default_float(dtype)
    gpf.config.set_default_jitter(1e-4)      # the bench's jitter for C3
    m = gpf.models.SGPR((d["X"], d["Y"]), gpf.kernels.SquaredExponential(lengthscales=4.0), d["Z"], noise_variance=0.1)

    def value():
        v = m.elbo()
        torch.cuda.synchronize()
        return v

    def grad():
        return m.elbo_and_grad()

    for _ in range(warmup):
        value()
        grad()
    torch.cuda.synchronize()
    tv, tg = [], []
    for _ in range(steps):                    # interleaved: value, value + gradient, value, ...
        for fn, acc in ((value, tv), (grad, tg)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            acc.append(e0.elapsed_time(e1))
    ev = float(value())
    eg, g = grad()
    return {
        "dtype": np.dtype(dtype).name, "N": 100000, "M": 1024, "D": 16, "P": 1, "steps": steps, "warmup": warmup,
        "value_ms_median": round(float(np.median(tv)), 4), "value_ms_min": round(float(np.min(tv)), 4),
        "value_grad_ms_median": round(float(np.median(tg)), 4), "value_grad_ms_min": round(float(np.min(tg)), 4),
        "ratio_median": round(float(np.median(tg) / np.median(tv)), 3),
        "elbo_value": ev, "elbo_from_grad_call": float(eg),
        "grad_variance": float(g[m.kernel.variance]), "grad_lengthscale": float(g[m.kernel.lengthscales]),
        "grad_noise": float(g[m.likelihood.variance]),
        "value_class_ms": per_class(lib, value, 5), "value_grad_class_ms": per_class(lib, grad, 5),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "time_sgpr_grad.py needs a CUDA device"
    res = {"gpu": gpu_info(), "runs": [run(np.float32, a.steps, a.warmup), run(np.float64, a.steps, a.warmup)]}
    s = json.dumps(res, indent=1)
    print(s, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
