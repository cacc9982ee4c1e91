"""CPU tests of the host-side logic added in round 2 (no device arithmetic): the triangular packing of the digit-plane
store, the choice of the number of digit planes, constructor / error behaviour of the widened kernel classes and the
multi-output plumbing, the bijector chain rule, heteroskedastic likelihood bookkeeping."""
import numpy as np
import pytest

import gpflow_b200 as gpf
from gpflow_b200.base import Parameter, positive
from gpflow_b200.inducing_variables import (InducingPoints, SeparateIndependentInducingVariables,
                                            SharedIndependentInducingVariables)

K = gpf.kernels


def plane_prefix(rb, nbk):  # mirror of csrc/planes.cuh::plane_prefix
    q = min(rb, nbk + 1)
    return 2 * q * (q - 1) + (rb - q) * 4 * nbk


def test_plane_store_packing_is_a_bijection_onto_a_dense_range():
    """Row block rb stores min(4 rb, 4 nbk) k-block tiles; the prefix sums give every (rb, kb) its own slot and leave no
    holes (csrc/planes.cuh).  Extra row blocks below the square part (rb > nbk) hold all 4 nbk k-blocks."""
    for nbk in (1, 2, 7, 64):
        for rbt in (nbk, nbk + 1, nbk + 3):
            slots = []
            for rb in range(rbt):
                nk = min(4 * rb, 4 * nbk)
                slots += [plane_prefix(rb, nbk) + kb for kb in range(nk)]
            assert slots == list(range(len(slots)))
            assert plane_prefix(rbt, nbk) == len(slots)
    # C2: 8192 + 1 rows -> 65 row blocks of 64 column blocks: 8320 + 256 tiles of S * 4096 bytes
    assert plane_prefix(66, 64) == 2 * 65 * 64 + 256


def pick_slices(cond):  # mirror of csrc/potrf.cu::pick_slices
    return 6 if 0 < cond <= 1e4 else 7


def test_digit_plane_count_follows_the_conditioning_bound():
    """Measured with static scales on numerically low-rank matrices (scripts/radix_study.py, base-256 digits): S = 6 (with
    the (3,3) product) moves L by ~1e-12 cond relative to max |L|; S = 7 is within ~3x of fp64 arithmetic itself at every
    conditioning, so nothing falls back to the DMMA engine any more.  The threshold keeps the S = 6 perturbation two
    orders inside the 1e-5 parity bar."""
    assert pick_slices((1.0 + 0.1) / 0.1) == 6          # BASELINE configs[1]
    assert pick_slices(1e4) == 6 and pick_slices(1.0001e4) == 7
    assert pick_slices((1 + 1e-6) / 1e-6) == 7           # likelihood variance at its lower bound, unit kernel variance
    assert pick_slices(1e9) == 7 and pick_slices(0.0) == 7
    assert 1e-12 * 1e4 < 1e-7


def test_widened_kernel_constructors_and_errors():
    with pytest.raises(TypeError):
        K.Periodic(K.Linear())                                          # periodic.py:66-67
    with pytest.raises(ValueError):
        K.ArcCosine(order=5)                                            # misc.py:67-68
    with pytest.raises(ValueError):
        K.ChangePoints([K.SquaredExponential()], [0.1, 0.2])            # changepoints.py:62-67
    with pytest.raises(ValueError):
        K.ChangePoints([K.SquaredExponential(), K.Matern12()], [0.1], steepness=[1.0, 2.0])
    with pytest.raises(ValueError):
        K.LinearCoregionalization([K.SquaredExponential()], np.ones((3, 2)))
    p = K.Periodic(K.Matern32(active_dims=[1, 2]), period=[1.0, 2.0])
    assert list(p.active_dims) == [1, 2]                                # uses the base kernel's active_dims
    c = K.Coregion(3, 2)
    assert c.output_covariance().shape == (3, 3) and np.allclose(c.output_variance(), np.diag(c.output_covariance()))
    assert not (K.Cosine() + K.SquaredExponential()).is_fusable() and (K.Matern12() * K.White()).is_fusable()
    cp = K.ChangePoints([K.SquaredExponential(), K.Matern12()], [0.3])
    assert len(cp.kernels) == 2 and not cp.is_fusable() and len(cp.parameters) >= 6
    lc = K.LinearCoregionalization([K.SquaredExponential(), K.Matern32()], np.ones((3, 2)))
    assert lc.num_latent_gps == 2 and len(lc.latent_kernels) == 2


def test_multioutput_inducing_variables_and_latent_pairing():
    from gpflow_b200.covariances import _latent_pairs

    Z = np.zeros((5, 2))
    sh = SharedIndependentInducingVariables(Z)
    se = SeparateIndependentInducingVariables([Z, Z + 1, Z + 2])
    assert sh.num_inducing == 5 and se.num_inducing == 5 and len(se.inducing_variables) == 3
    ks = [K.SquaredExponential(), K.Matern12(), K.Matern32()]
    assert len(_latent_pairs(sh, K.SeparateIndependent(ks))) == 3
    assert len(_latent_pairs(se, K.SharedIndependent(ks[0], 3))) == 3
    pairs = _latent_pairs(se, K.SeparateIndependent(ks))
    assert [type(k).__name__ for _, k in pairs] == ["SquaredExponential", "Matern12", "Matern32"]
    assert all(isinstance(iv, InducingPoints) for iv, _ in pairs)
    with pytest.raises(ValueError):
        _latent_pairs(se, K.SeparateIndependent(ks[:2]))


def test_bijector_chain_rule_and_unconstrained_assignment():
    for lower in (None, 1e-6):
        p = Parameter(0.7, transform=positive(lower=lower) if lower else positive())
        u = p.unconstrained_variable
        h = 1e-6
        fwd = p.transform.forward
        fd = (fwd(u + h) - fwd(u - h)) / (2 * h)
        np.testing.assert_allclose(p.unconstrained_gradient(2.0), 2.0 * fd, rtol=1e-8)
        p.assign_unconstrained(u + 0.3)
        np.testing.assert_allclose(p.numpy(), fwd(u + 0.3), rtol=1e-14)
    q = Parameter(np.array([1.0, -2.0]))
    np.testing.assert_allclose(q.unconstrained_gradient([3.0, 4.0]), [3.0, 4.0])


def test_heteroskedastic_gaussian_bookkeeping():
    lin = gpf.mean_functions.Linear(A=np.array([[0.1]]), b=np.array([0.2]))
    lik = gpf.likelihoods.Gaussian(variance=lin)
    assert lik.heteroskedastic and lik.scale is None
    with pytest.raises(NotImplementedError):
        lik._variance_value()
    lik2 = gpf.likelihoods.Gaussian(scale=lin)
    assert lik2.heteroskedastic and lik2.variance is None
    assert not gpf.likelihoods.Gaussian(0.3).heteroskedastic
    with pytest.raises(AssertionError):
        gpf.likelihoods.Gaussian(0.1, scale=0.2)


# ---- mirror of the launch sequence of csrc/potrf.cu (potrf_rec / potrf_block / trailing_update, slim fp64 path) -------------
def _potrf_schedule(n, rows, nb=128, tc_min_k=256):
    """Returns the launch list of one factorisation as tuples; `follow` is threaded through the recursion exactly as the
    (fk0, fK) arguments of potrf_rec: the k-range of the tcgen05 update that directly follows a sub-factorisation."""
    out = []

    def split_point(m):
        return ((m // nb + 1) // 2) * nb

    def eligible(m, nn, K):
        return K >= tc_min_k and K % 32 == 0 and nn <= m

    def block(n_, rows_, col0, fuse_cols, follow):
        out.append(("leaf", col0))
        if rows_ <= n_:
            return
        if fuse_cols > 0:
            out.append(("fused_panel", col0, fuse_cols))
            return
        dyn = None
        fk0, fK = follow
        if n_ == nb and fK > 0 and fk0 + fK == col0 + n_ and rows_ + col0 > n:   # extra rows below the square part exist
            dyn = (fk0, fK)
        out.append(("panel", col0, dyn))

    def rec(n_, rows_, col0, follow):
        if n_ <= nb:
            return block(n_, rows_, col0, 0, follow)
        n1 = split_point(n_)
        if n_ <= 2 * nb:
            block(n1, rows_, col0, n_ - n1, (-1, 0))
            return rec(n_ - n1, rows_ - n1, col0 + n1, follow)
        tc = eligible(rows_ - n1, n_ - n1, n1)
        rec(n1, rows_, col0, (col0, n1 if tc else 0))
        out.append(("update", col0, n1, tc))
        rec(n_ - n1, rows_ - n1, col0 + n1, follow)

    rec(n, rows, 0, (-1, 0))
    return out


@pytest.mark.parametrize("n,extra", [(8192, 1), (4096, 3), (1024, 0), (1536, 2), (8192 + 128, 1), (700, 1)])
def test_every_tcgen05_update_finds_its_extra_rows_sliced_by_the_panel_before_it(n, extra):
    sched = _potrf_schedule(n, n + extra)
    leaves = [e[1] for e in sched if e[0] == "leaf"]
    assert leaves == list(range(0, n, 128))                                   # one leaf per diagonal block, in order
    for i, e in enumerate(sched):
        if e[0] == "update" and e[3]:                                         # runs on tcgen05
            prev = sched[i - 1]
            assert prev[0] == "panel" and prev[1] + 128 == e[1] + e[2]        # a PLAIN panel, the block that ends the k-range
            if extra and prev[1] + 128 <= n:
                assert prev[2] == (e[1], e[2])                                # ... which sliced [col0, col0 + K) for it
        if e[0] == "panel" and e[2] is not None:
            nxt = sched[i + 1]
            assert nxt[0] == "update" and (nxt[1], nxt[2]) == e[2]            # never a stale k-range
        if e[0] == "fused_panel":
            assert sched[i + 1][0] == "leaf"                                  # the fused update plays the role of U
    if n == 8192:
        assert sum(e[0] == "update" for e in sched) == 31 and sum(e[0] == "fused_panel" for e in sched) == 32
