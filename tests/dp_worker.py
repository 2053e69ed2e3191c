"""Worker of tests/test_dp_gpu.py (one process per GPU under torch.distributed.run): a row-sharded minibatch trained
through drvae_b200.dp on `world` GPUs must follow the same trajectory as the unsharded minibatch on one GPU — same Philox
noise (keyed by global row), same global normalisers, gradients summed over NVLink peer memory (PeerBackend) or NCCL."""
import json
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from drvae_b200 import dp as dpm  # noqa: E402
from drvae_b200.init import init_state_dict  # noqa: E402
from drvae_b200.plan import Plan, anneal_coef  # noqa: E402
from drvae_b200.synth import synthetic_batch  # noqa: E402

ARCHS = dict(tiny=dict(dim_x=40, dim_y=2, dim_z1=12, dim_z3=10, enc_z1=[24], dec_x=[28], enc_z3=[20], dec_z1=[18]),
             readme=dict(dim_x=978, dim_y=2, dim_z1=100, dim_z3=100, enc_z1=[800], dec_x=[600], enc_z3=[200], dec_z1=[200]))
FIELDS = ("x1", "x2", "y", "has_x2", "has_y")


def main():
    backend, arch_name, N, steps = sys.argv[1], sys.argv[2], int(sys.argv[3]), int(sys.argv[4])
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
    dev = torch.device("cuda", int(os.environ["LOCAL_RANK"]))
    dist.init_process_group("nccl", device_id=dev)
    arch = ARCHS[arch_name]
    sd = init_state_dict("drvae", seed=123, **arch)
    full = synthetic_batch(N, arch["dim_x"], seed=3)
    lo, hi = dpm.shard_rows(N, world, rank)
    plan = Plan("drvae", L=2, max_batch=hi - lo, n_models=1, **arch)
    plan.load_state_dict(sd)
    be = dpm.PeerBackend(plan) if backend == "peer" else dpm.PlanBackend(plan)
    runner = dpm.DataParallel(be)
    shard = {k: full[k][lo:hi].contiguous().to(dev) for k in FIELDS}
    host = {k: full[k][lo:hi] for k in ("has_x2", "has_y")}
    losses = []
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        for it in range(steps):
            out = runner.step(shard, hp_kwargs=dict(beta_pert=anneal_coef(it, 1, 0)), seed=5, row_offset=lo, host_flags=host)
            losses.append(out.detach().float().cpu().clone())
    torch.cuda.synchronize()
    params = plan.params.cpu().clone()
    # every rank must hold the same parameters (replicated optimizer on identical sums)
    gathered = [torch.zeros_like(params) for _ in range(world)] if rank == 0 else None
    dist.gather(params.to(dev), [g.to(dev) for g in gathered] if rank == 0 else None, dst=0)
    res = None
    if rank == 0:
        # single-GPU run of the unsharded minibatch
        ref = Plan("drvae", L=2, max_batch=N, n_models=1, **arch)
        ref.load_state_dict(sd)
        fb = {k: full[k].to(dev) for k in FIELDS}
        ref_losses = []
        for it in range(steps):
            hp = ref.hparams(step=it, beta_pert=anneal_coef(it, 1, 0))
            ref_losses.append(ref.grad_step(fb, hp, seed=5).float().cpu().clone()[0])
            ref.adam_step(hp)
        torch.cuda.synchronize()
        worst = 0.0
        for a, b in zip(losses, ref_losses):
            for i in (0, 1, 2, 3, 5, 6):
                worst = max(worst, abs(float(a[i]) - float(b[i])) / (abs(float(b[i])) + 1e-12))
        pref = ref.params.cpu()
        res = {"backend": backend, "world": world, "worst_rel_loss_err": worst,
               "param_rel_l2": float((params - pref).norm() / pref.norm()),
               "max_param_abs_diff": float((params - pref).abs().max()),
               "ranks_identical": True, "graph_replays": plan.graph_replays(),
               "graph_failures": plan.graph_failures(),
               "multicast": bool(getattr(be, "multicast", False))}
    if rank == 0:
        print("DPRESULT " + json.dumps(res), flush=True)
    # rank-to-rank equality of the parameters
    t = plan.params.clone()
    dist.broadcast(t, src=0)
    same = bool(torch.equal(t, plan.params))
    flag = torch.tensor([1 if same else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("DPSAME %d" % int(flag.item()), flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
