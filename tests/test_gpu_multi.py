"""Multi-rank parity.  With >= 2 GPUs (`gpurun --gpus 2 -- python -m pytest tests/test_gpu_multi.py`)
every rank owns a GPU and torch.distributed runs on NCCL; on a ONE-GPU box the two ranks share
the device (CUDA IPC maps a buffer of another process on the same device just as well, so the
peer-memory exchange of trb_comm.cu is exercised unchanged) and torch.distributed falls back to
gloo, which NCCL's "one rank per GPU" rule requires.

BASELINE config 5 in miniature: ONE instance whose thin-SVD operators are row
sharded over the ranks; the two expansions per iteration are summed over the
ranks through peer memory (or, as a baseline, all-reduced by NCCL).  Every rank must reproduce the reference's golden sweep."""
import json
import os
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _init(rank, world, port):
    """One process per rank: its own GPU over NCCL when the box has one per rank, else a shared
    GPU over gloo."""
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    if torch.cuda.device_count() >= world:
        torch.cuda.set_device(rank)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    else:
        torch.cuda.set_device(0)
        dist.init_process_group("gloo", rank=rank, world_size=world)
    return dist


def _sum_over_ranks(dist, v):
    """Library all-reduce of a device tensor (the reference value for the peer-memory sum)."""
    if dist.get_backend() == "gloo":
        host = v.cpu()
        dist.all_reduce(host)
        return host.to(v.device)
    out = v.clone()
    dist.all_reduce(out)
    return out


def _worker(rank, world, port, golden_dir, name, out_path, backend):
    import torch
    from tests.golden import load_sweeps
    dist = _init(rank, world, port)
    from tramp_b200 import ops
    from tramp_b200.priors import get_prior
    from tramp_b200.likelihoods import get_likelihood
    from tramp_b200.channels import LinearChannel
    from tramp_b200.variables import SISOVariable as V
    from tramp_b200.algos import ExpectationPropagation, TrackErrors
    from tramp_b200.distributed import instance_shard
    sw = load_sweeps(golden_dir)
    cfg = [c for c in json.loads(str(sw["configs"])) if c["name"] == name][0]
    W = sw[name + "_W"]
    M, N = W.shape
    U, s, Vt = np.linalg.svd(W, full_matrices=False)
    r0, r1 = instance_shard(s.size, rank, world)          # contiguous block of singular triplets
    lin = LinearChannel.from_sharded_factors(
        ops.padded(U.T[r0:r1].copy())[None].contiguous(), ops.to_dev(s[None, r0:r1]),
        ops.padded(Vt[r0:r1].copy())[None].contiguous(), s, Nx=M, Nz=N, group=dist.group.WORLD)
    pk = {k: v for k, v in cfg["prior"].items() if k != "kind"}
    lk = {k: v for k, v in cfg["lik"].items() if k != "kind"}
    model = (get_prior(size=N, prior_type=cfg["prior"]["kind"], **pk) @ V("x") @ lin @ V("z")
             @ get_likelihood(y=sw[name + "_y"], likelihood_type=cfg["lik"]["kind"], **lk)).to_model()
    # the stand-alone sum over the same peer-memory protocol agrees with NCCL's
    v = torch.arange(64, dtype=torch.float64, device="cuda") * (rank + 1) + 0.25 * rank
    v_lib = _sum_over_ranks(dist, v)
    lin.exchange.all_reduce(v)
    assert torch.equal(v, v_lib) and int(lin.exchange.timeout.item()) == 0
    ep = ExpectationPropagation(model)
    ep.linear_backend = backend
    track = TrackErrors({"x": sw[name + "_x"]})
    ep.iterate(max_iter=cfg["n_iter"], callback=track, damping=cfg["damping"])
    assert ep.backend == backend
    d = ep.get_variables_data()
    np.savez(out_path % rank, rx=d["x"]["r"], rz=d["z"]["r"], vx=d["x"]["v"], vz=d["z"]["v"],
             mse=np.array([e["mse"] for e in track.errors]))
    dist.destroy_process_group()


@pytest.mark.parametrize("backend", ["sharded", "sharded_nccl"])
@pytest.mark.parametrize("name", ["cs_gb_gauss", "perceptron_gauss_sgn", "gb_sgn_damped"])
def test_row_sharded_instance_matches_reference(golden_dir, tmp_path, name, backend):
    """backend "sharded": expansions exchanged through peer memory inside the update
    kernels (trb_comm.cu), whole sweep in one trb_sweep_run; "sharded_nccl": the
    library baseline (local GEMVs + NCCL all-reduce, staged from Python)."""
    import torch
    import torch.multiprocessing as mp
    from tests.golden import load_sweeps
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    world = 2
    out = str(tmp_path / "rank%d.npz")
    mp.spawn(_worker, args=(world, 29600 + os.getpid() % 300, golden_dir, name, out, backend), nprocs=world,
             join=True)
    sw = load_sweeps(golden_dir)
    res = [np.load(out % r) for r in range(world)]
    for r in res:
        np.testing.assert_allclose(r["mse"], sw[name + "_mse"], rtol=1e-9)
        for key, ref in (("rx", sw[name + "_rx"]), ("rz", sw[name + "_rz"])):
            np.testing.assert_allclose(r[key], ref, rtol=1e-9, atol=1e-9 * np.abs(ref).max())
        np.testing.assert_allclose(r["vx"], sw[name + "_vx_final"], rtol=1e-9)
        np.testing.assert_allclose(r["vz"], sw[name + "_vz_final"], rtol=1e-9)
    # the replicated state is bit-identical across ranks (every rank adds the same vectors in rank order)
    assert np.array_equal(res[0]["rx"], res[1]["rx"]) and np.array_equal(res[0]["mse"], res[1]["mse"])


def _instances_worker(rank, world, port, out_path):
    dist = _init(rank, world, port)
    from tramp_b200.experiments import run_ep_sharded
    from tests.test_distributed_cpu import _ep_builders
    build_model, x_true, B = _ep_builders()
    res = run_ep_sharded(build_model, B, x_true=x_true, max_iter=40)
    np.savez(out_path % rank, rx=res["r"]["x"], vx=res["v"]["x"], n_iter=res["n_iter"], mse=res["mse"])
    dist.destroy_process_group()


def test_instances_sharded_over_two_gpus_match_the_oracle(tmp_path):
    """BASELINE config 3 in miniature: five independent instances as blocks of 3 and 2
    on two GPUs (run_ep_sharded, no data-path collective, results gathered over NCCL);
    every instance stops where its own oracle run stops, with the oracle's posterior."""
    import torch
    import torch.multiprocessing as mp
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from oracle import tramp_oracle as orc
    from tests.test_distributed_cpu import _ep_problem
    out = str(tmp_path / "inst_rank%d.npz")
    mp.spawn(_instances_worker, args=(2, 29650 + os.getpid() % 300, out), nprocs=2, join=True)
    r0, r1 = np.load(out % 0), np.load(out % 1)
    for k in r0.files:
        assert np.array_equal(r0[k], r1[k], equal_nan=True)
    W, x, y = _ep_problem()
    for b in range(W.shape[0]):
        ref = orc.ep_glm(dict(kind="gauss_bernoulli", rho=0.2), W[b], dict(kind="gaussian", var=1e-2, y=y[b]),
                         40, early_stopping=dict(tol=1e-6), x_true=x[b])
        assert r0["n_iter"][b] == ref["n_iter"]
        np.testing.assert_allclose(r0["rx"][b], ref["r_x"], rtol=1e-9, atol=1e-9 * np.abs(ref["r_x"]).max())
        np.testing.assert_allclose(r0["vx"][b], ref["v_x"], rtol=1e-9)
