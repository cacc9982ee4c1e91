"""CPU-only tests: C-ABI library loads and exports every declared symbol, host-side descriptor
compilation, dispatch, parameters, config, argument errors (no compute without a GPU)."""
import ctypes
import os
import re

import numpy as np
import pytest

import gpflow_b200 as gpf
from gpflow_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_loads_and_exports_every_declared_symbol():
    lib = _lib.load()
    header = open(os.path.join(ROOT, "include", "gpk.h")).read()
    declared = set(re.findall(r"GPK_API\s+[\w\s\*]+?\b(gpk_\w+)\s*\(", header))
    assert len(declared) >= 25
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    for name in declared:
        assert getattr(lib, name) is not None
    assert lib.gpk_version() == 1


def test_knode_struct_matches_header_layout():
    # int32 op, n_children, child[8]; 3 doubles; 4 int32
    assert ctypes.sizeof(_lib.KNode) == 4 * 10 + 8 * 3 + 4 * 4
    assert _lib.KNode.variance.offset == 40 and _lib.KNode.n_dims.offset == 64


def test_compile_kernel_tree_and_flattening():
    k = gpf.kernels
    expr = (k.RBF(lengthscales=2.0) + k.Matern32(lengthscales=4.0)) * k.Linear()
    nodes, n, dims, ard = k.compile_kernel(expr, 5)
    assert n == 5
    assert [nd.op for nd in nodes] == [_lib.K_RBF, _lib.K_MATERN32, _lib.K_SUM, _lib.K_LINEAR, _lib.K_PRODUCT]
    assert list(nodes[2].child)[:2] == [0, 1] and list(nodes[4].child)[:2] == [2, 3]
    # same-class nesting is flattened (gpflow/kernels/base.py:246-254)
    s = (k.RBF() + k.Matern12()) + k.White()
    assert len(s.kernels) == 3
    p = (k.RBF() * k.Matern12()) * k.White()
    assert len(p.kernels) == 3
    assert len(((k.RBF() + k.Matern12()) * k.White()).kernels) == 2


def test_compile_kernel_active_dims_and_ard():
    k = gpf.kernels
    kern = k.RBF(lengthscales=[1.0, 2.0], active_dims=[0, 3]) + k.Linear(variance=[0.5, 0.25, 2.0], active_dims=slice(1, 4))
    nodes, n, dims, ard = k.compile_kernel(kern, 5)
    assert nodes[0].n_dims == 2 and list(dims)[:2] == [0, 3] and nodes[0].n_ard == 2
    assert nodes[1].n_dims == 3 and list(dims)[2:5] == [1, 2, 3] and list(ard)[2:5] == [0.5, 0.25, 2.0]
    with pytest.raises(ValueError):  # gpflow/kernels/base.py:164-168
        k.RBF(lengthscales=[1.0, 2.0, 3.0], active_dims=[0, 1])
    with pytest.raises(ValueError):
        k.compile_kernel(k.RBF(active_dims=[7]), 5)
    with pytest.raises(ValueError):
        k.compile_kernel(k.RBF(lengthscales=[1.0, 2.0]), 5)
    with pytest.raises(TypeError):  # stationaries.py:56-58
        k.RBF(foo=1)


def test_call_rejects_ambiguous_inputs():
    with pytest.raises(ValueError):  # gpflow/kernels/base.py:203-204
        gpf.kernels.RBF()(np.zeros((3, 2)), np.zeros((3, 2)), full_cov=False)


def test_kbuild_argument_errors_reported_through_status():
    lib = _lib.load()
    nodes = (_lib.KNode * 1)()
    nodes[0].op = 99
    st = lib.gpk_kbuild(nodes, 1, None, None, ctypes.c_void_p(16), 4, 2, None, 4, 2, 2, ctypes.c_void_p(16), 4,
                        _lib.GPK_F64, _lib.GPK_FULL, 0.0, None, None)
    assert st == -1 and b"unknown kernel op" in lib.gpk_last_error()
    with pytest.raises(ValueError):
        _lib.check(st, "gpk_kbuild")
    st = lib.gpk_potrf(None, 4, 4, 4, _lib.GPK_F64, None, None, None)
    assert st == -1
    st = lib.gpk_gemm(0, 0, 4, 4, 4, 1.0, ctypes.c_void_p(16), 4, ctypes.c_void_p(16), 4, 0.0, ctypes.c_void_p(16), 4,
                      7, 0, None)
    assert st == -1 and b"dtype" in lib.gpk_last_error()


def test_workspace_queries():
    lib = _lib.load()
    assert lib.gpk_potrf_ws(128, 128, _lib.GPK_F64) == 128 * 128 * 8 + 256
    assert lib.gpk_potrf_ws(129, 129, _lib.GPK_F32) == 2 * 128 * 128 * 4 + 256
    assert lib.gpk_potrf_ws(8192, 8193, _lib.GPK_F64) > 64 * 128 * 128 * 8 + 8193 * 4096 * 7  # + tcgen05 digit planes
    n, p = 8192, 1
    assert lib.gpk_gpr_lml_ws(n, p, _lib.GPK_F64) >= (n + p) * n * 8
    assert lib.gpk_sgpr_elbo_ws(1000, 100, 2, _lib.GPK_F32) > 1000 * 100 * 4
    assert lib.gpk_svgp_elbo_ws(64, 32, 2, _lib.GPK_F32) > 0


def test_dispatcher_plugin_mechanism():
    from gpflow_b200.utilities import Dispatcher

    d = Dispatcher("demo")

    class A: ...
    class B(A): ...

    @d.register(A, object)
    def _a(x, y):
        return "A"

    @d.register(B, int)
    def _b(x, y):
        return "B"

    assert d(A(), 1) == "A" and d(B(), 1) == "B" and d(B(), "s") == "A"
    with pytest.raises(NotImplementedError):
        d(1, 2)
    assert d.dispatch_or_raise(B, int) is _b
    # the reference registries exist with the same names
    from gpflow_b200 import covariances, kullback_leiblers, posteriors
    assert covariances.Kuu.dispatch(gpf.inducing_variables.InducingPoints, gpf.kernels.RBF) is not None
    assert covariances.Kuf.dispatch(gpf.inducing_variables.InducingPoints, gpf.kernels.RBF, np.ndarray) is not None
    assert posteriors.get_posterior_class(gpf.kernels.RBF(), gpf.inducing_variables.InducingPoints(np.zeros((2, 1)))) \
        is posteriors.IndependentPosteriorSingleOutput


def test_parameter_transforms_and_bounds():
    from gpflow_b200.base import Parameter, positive

    p = Parameter(0.3, transform=positive())
    assert np.isclose(np.logaddexp(0, p.unconstrained_variable), 0.3)
    with pytest.raises(ValueError):
        Parameter(-1.0, transform=positive())
    lik = gpf.likelihoods.Gaussian(0.1)
    with pytest.raises(ValueError):  # lower bound 1e-6, scalar_continuous.py:70-77
        lik.variance.assign(1e-7)
    m = gpf.kernels.RBF() + gpf.kernels.White()
    assert len(m.parameters) == 3 and len(m.trainable_parameters) == 3
    gpf.set_trainable(m.kernels[1], False)
    assert len(m.trainable_parameters) == 2


def test_config_defaults_and_context():
    c = gpf.config
    assert c.default_float() is np.float64 and c.default_jitter() == 1e-6
    with c.as_context(c.Config(float=np.float32, jitter=1e-4)):
        assert c.default_float() is np.float32 and c.default_jitter() == 1e-4
        assert gpf.Parameter(1.0).dtype == np.float32
    assert c.default_float() is np.float64
    with pytest.raises(TypeError):
        c.set_default_float(np.int32)


def test_model_constructors_defaults_without_gpu():
    # SVGP holds only host parameters until evaluated (gpflow/models/svgp.py:124-140)
    m = gpf.models.SVGP(gpf.kernels.RBF(), gpf.likelihoods.Gaussian(), np.zeros((7, 2)), num_latent_gps=3)
    assert m.q_mu.shape == (7, 3) and m.q_sqrt.shape == (3, 7, 7) and m.whiten
    assert np.array_equal(m.q_sqrt.numpy()[1], np.eye(7))
    m = gpf.models.SVGP(gpf.kernels.RBF(), gpf.likelihoods.Gaussian(), np.zeros((7, 2)), q_diag=True, num_latent_gps=2)
    assert m.q_sqrt.shape == (7, 2)


def test_product_has_no_cpu_fallback():
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(_lib.GpkError):
        gpf.kernels.RBF()(np.zeros((3, 2)))
    src = ""
    for root, _, files in os.walk(os.path.join(ROOT, "gpflow_b200")):
        for f in files:
            if f.endswith(".py"):
                src += open(os.path.join(root, f)).read()
    assert "oracle" not in src.replace("gp_oracle", "oracle") or "import oracle" not in src
    assert "from oracle" not in src and "import oracle" not in src


def test_bench_reference_arm_prints_one_json_line():
    """bench.py contract: exactly ONE JSON line on stdout (library banners must not leak into it)."""
    import json
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--workload", "gpr_c1",
                        "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "evals/s" and d["e2e"]["h2d_bytes_per_step"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["higher_is_better"] is True


def test_bench_dump_outputs_writes_the_last_step_objective(tmp_path):
    """--dump-outputs DIR: the objective of the last timed step as DIR/objective.npy, the value the JSON line reports."""
    import json
    import subprocess
    import sys

    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "gpr_c1",
                        "--steps", "1", "--warmup", "0", "--dump-outputs", str(tmp_path / "out")],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip())
    got = np.load(tmp_path / "out" / "objective.npy")
    assert got.dtype == np.float64 and got.shape == (1,)
    assert got[0] == d["objective"] and d["steps"] == 1


def test_kernel_expressions_pass_the_host_compile_path_without_gpu():
    """Every leaf op (incl. Polynomial, whose offset / degree ride in the lengthscale / alpha fields) must get past the
    C-ABI's argument and expression checks (status -1 -> ValueError); without a device the call then fails only at
    the CUDA launch (status -2)."""
    lib = _lib.load()
    K = gpf.kernels
    exprs = [K.Polynomial(3.0, 0.35, 0.8),
             K.Polynomial(2.0, [0.5, 0.7], 1.3, active_dims=[1, 2]) * K.RBF() + K.White(0.3),
             (K.RBF() + K.Matern32(lengthscales=2.0)) * K.Linear(0.5) + K.RationalQuadratic(alpha=0.7) + K.Constant(0.1)]
    buf = (ctypes.c_double * 64)()
    ptr = ctypes.cast(buf, ctypes.c_void_p)
    for k in exprs:
        nodes, n, dims, ard = gpf.kernels.compile_kernel(k, 4)
        st = lib.gpk_kbuild(nodes, n, dims, ard, ptr, 4, 4, None, 4, 0, 4, ptr, 4, _lib.GPK_F64, 0, 0.0, None, None)
        assert st in (0, -2), lib.gpk_last_error().decode()
    bad = gpf.kernels.compile_kernel(K.Polynomial(), 4)
    bad[0][0].op = 99
    assert lib.gpk_kbuild(bad[0], bad[1], bad[2], bad[3], ptr, 4, 4, None, 4, 0, 4, ptr, 4, _lib.GPK_F64, 0, 0.0, None, None) == -1
    assert b"unknown kernel op" in lib.gpk_last_error()


def test_product_kernel_error_behaviour_matches_reference_without_gpu():
    """Same exceptions as the reference, raised before any device work: full_cov=False with X2 (kernels/base.py:203-204,
    tests/gpflow/kernels/test_kernels.py:621-627), ARD size mismatch (base.py:164-168, test_kernels.py:471-491), unknown
    keyword (stationaries.py:56-58), on_separate_dimensions (base.py:256-278, test_kernels.py:607-618)."""
    K = gpf.kernels
    X, X2 = np.random.randn(4, 1), np.random.randn(5, 1)
    for k in (K.RBF(), K.Matern32() + K.White(), K.Linear() * K.Constant(), K.Polynomial()):
        with pytest.raises(ValueError):
            k(X, X2, full_cov=False)
    with pytest.raises(ValueError):
        K.RBF(lengthscales=[1.0, 2.0, 3.0], active_dims=[0, 1])
    with pytest.raises(TypeError):
        K.RBF(foo=1)
    k1, k2, k3 = K.Linear(active_dims=[1, 2, 3]), K.RBF(active_dims=[4, 5, 6]), K.RBF(active_dims=[3, 4, 5])
    assert (k1 + k2).on_separate_dimensions is True
    assert (k1 + k3).on_separate_dimensions is False
    assert (K.Linear() + K.RBF()).on_separate_dimensions is False
