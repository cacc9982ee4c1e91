"""Multi-rank NCCL parity (needs >= 2 GPUs; skipped on a single-GPU box): the shares of the sharded SVGP evaluations --
rows of one minibatch, latent GPs with and without the column-sharded triangular solve + all-gather -- sum ON THE DEVICE
(one NCCL all-reduce) to the ELBO of the unsharded evaluation, and that matches the oracle.
Reference: gpflow/models/svgp.py:166-181, conditionals/util.py:125-164 (SURVEY.md 8(e))."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _worker(rank, world, port, q):
    import torch
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    import gpflow_b200 as gpf
    from gpflow_b200 import sharding
    from oracle import gp_oracle as O

    d = O.make_data(4, 4000, 6, 4, M=300)
    q_mu, q_sqrt = O.make_q(4, 300, 4)
    kp = gpf.kernels.SquaredExponential(lengthscales=2.0) + gpf.kernels.White(variance=0.1)
    ko = O.SquaredExponential(lengthscales=2.0) + O.White(variance=0.1)
    m = gpf.models.SVGP(kp, gpf.likelihoods.Gaussian(0.1), d["Z"], num_latent_gps=4, q_mu=q_mu, q_sqrt=q_sqrt,
                        whiten=True, num_data=4000)
    Xb, Yb = gpf.ops.to_device(d["X"][:512]), gpf.ops.to_device(d["Y"][:512])
    full = float(m.elbo((Xb, Yb)))
    rows = float(sharding.svgp_elbo_row_sharded(m, (Xb, Yb)).item())
    lat = float(sharding.svgp_elbo_latent_sharded(m, (Xb, Yb), shard_solve=False).item())
    lat_cs = float(sharding.svgp_elbo_latent_sharded(m, (Xb, Yb), shard_solve=True).item())
    ref = O.svgp_elbo(d["X"][:512], d["Y"][:512], d["Z"], ko, q_mu, q_sqrt, 0.1, whiten=True, num_data=4000)
    q.put((rank, full, rows, lat, lat_cs, ref))
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_svgp_elbo_sums_to_full_on_nccl(cuda_device):
    import torch
    import torch.multiprocessing as mp

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 33500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=300) for _ in procs]
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for rank, full, rows, lat, lat_cs, ref in res:
        np.testing.assert_allclose(full, ref, rtol=1e-8)      # fp64 parity bar of the models
        np.testing.assert_allclose(rows, full, rtol=1e-10)
        np.testing.assert_allclose(lat, full, rtol=1e-10)
        np.testing.assert_allclose(lat_cs, full, rtol=1e-10)
