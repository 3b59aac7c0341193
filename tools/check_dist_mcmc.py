"""Sharded stretch move == single-GPU stretch move, bit for bit, for both exchanges -- NVLink peer stores with
the flag barrier, and the packed all-gather over NCCL (developer check; also run by tests/test_sampler.py when
two GPUs are visible, and by bench.py --gpus N, which reports the result as extra.sharded_equals_single).
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tools/check_dist_mcmc.py
MOVES=mix runs emcee's recommended mix, 0.8 DEMove / 0.2 DESnookerMove, instead of the stretch move."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, ROOT)
import numpy as np, torch, torch.distributed as dist
from magprop_b200 import _capi as A
from magprop_b200.engine import Likelihood, time_grid
from magprop_b200.sampler import DEMove, DESnookerMove, DeviceEnsemble
from magprop_b200.synthetic.mcmc_eqns import lower, upper
from magprop_b200.synthetic.synth_mcmc import truths


def sharded_equals_single(lk, n, nsteps, seed=17, sigma=1e-2, moves=None):
    """{exchange: bool} on this rank: the chain of a sharded run equals the chain of an unsharded one."""
    p0 = truths["Humped"] + sigma * np.random.RandomState(4).randn(n, 6)
    single = DeviceEnsemble.from_likelihood(lk, n, 6, a=2.0, seed=seed, dist=None, moves=moves)
    single.initialise(p0)
    single.run(nsteps)
    out = {}
    for exchange in ("peer", "allgather"):
        ens = DeviceEnsemble.from_likelihood(lk, n, 6, a=2.0, seed=seed, dist=dist, exchange=exchange, moves=moves)
        ens.initialise(p0)
        ens.run(nsteps)
        torch.cuda.synchronize()
        ens.check_peers()
        same = torch.equal(ens.coords, single.coords) and torch.equal(ens.lnp, single.lnp)
        acc_same = torch.equal(ens.acceptance_fraction(), single.acceptance_fraction())
        out[f"{exchange}->{ens.exchange}"] = bool(same and acc_same)
        ens.close()
    return out


if __name__ == "__main__":
    rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    g = np.load(os.path.join(ROOT, "tests", "golden", "lnprob_script.npz"))
    lk = Likelihood(A.script_model_spec(), time_grid(None), g["Humped_x"], g["Humped_y"], g["Humped_yerr"], lower, upper, device=local)
    moves = [(DEMove(), 0.8), (DESnookerMove(), 0.2)] if os.environ.get("MOVES") == "mix" else None
    res = sharded_equals_single(lk, int(os.environ.get("NWALK", 4096)), 6, moves=moves)
    same = all(res.values())
    print(f"rank {rank}: sharded == single: {same} {res}; world {dist.get_world_size()}", flush=True)
    ok = torch.tensor([1 if same else 0], device="cuda")
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    lk.close()
    dist.destroy_process_group()
    sys.exit(0 if int(ok.item()) == 1 else 1)
