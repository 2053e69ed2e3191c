"""Time of a sweep epoch's validation against its training, before and after drvae_eval_members.

For DrVAE README-shape ensembles of E = 32 and E = 80 members with L1000-shaped splits (validation of about 500 and
about 4 000 rows per member, training splits three times larger, as a 5-fold split gives), after warm-up, in one
process, alternating old and new:
  old     the per-member loop sweep.evaluate_members ran before drvae_eval_members: per member torch.nonzero, sklearn
          AUROC / AUPR on host copies, one or two drvae_eval_x_reconstruction calls with their own read backs,
          pair.any() (rebuilt here as it was)
  new     sweep.evaluate_members: the same chunked inference, one drvae_eval_members call, one [E, 11] read back
  infer   the chunked inference alone (part of both)
  train   one training epoch of graph-replayed steps, max_m floor(n_m / 200) steps, as sweep.fit_sweep runs it
Each time is a host clock around work that ends in a device synchronise; the median of --reps repetitions is printed.
Also the y group of drvae_eval_members alone (the ranking kernels) at D = 65 536, E = 80, by CUDA events.

    python tools/sweep_eval_bench.py [--reps 5] [--out FILE]
"""
import argparse
import os
import statistics
import subprocess
import sys
import time
import warnings
from collections import OrderedDict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from drvae_b200.init import init_state_dict  # noqa: E402
from drvae_b200.plan import Plan, anneal_coef  # noqa: E402
from drvae_b200.sweep import MODEL_CLASS, evaluate_members, steps_per_epoch  # noqa: E402
from drvae_b200.training import eval_members, eval_x_reconstruction, eval_y_prediction  # noqa: E402

ARCH = dict(dim_x=978, dim_y=2, dim_z1=100, dim_z3=100, enc_z1=[800], dec_x=[600], enc_z3=[200], dec_z1=[200])
BATCH = 200


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # the card name from torch is still printed
        q = "nvidia-smi unavailable (%s)" % e
    return "%s | nvidia-smi: %s" % (torch.cuda.get_device_name(), q)


def padded_split(E, sizes, gen):
    """L1000-shaped padded fields on the device: x1 ~ N(0, 1), half the rows paired (x2 = x1 + noise), 2/3 labeled,
    y from a linear signal.  -> (fields, mask)."""
    D, X = max(sizes), ARCH["dim_x"]
    dev = "cuda"
    mask = (torch.arange(D, device=dev)[None, :] < torch.tensor(sizes, device=dev)[:, None]).to(torch.int32)
    x1 = torch.randn(E, D, X, device=dev, generator=gen)
    has_x2 = (torch.rand(E, D, device=dev, generator=gen) < 0.5).to(torch.int32) * mask
    x2 = (x1 + 0.3 * torch.randn(E, D, X, device=dev, generator=gen)) * has_x2[..., None]
    has_y = (torch.arange(D, device=dev) % 3 != 0).to(torch.int32)[None, :] * mask
    y = ((x1[..., :8].sum(-1) + 0.5 * torch.randn(E, D, device=dev, generator=gen)) > 0).to(torch.int32)
    y = torch.where(has_y != 0, y, torch.full_like(y, -66))
    return dict(x1=x1 * mask[..., None], x2=x2, y=y, has_x2=has_x2, has_y=has_y), mask


def old_evaluate_members(plan, kind, fields, mask):
    """The per-member loop of sweep.evaluate_members before drvae_eval_members (y metrics through sklearn on host
    copies, as eval_y_prediction computed them for CUDA tensors then)."""
    D = fields["x1"].shape[1]
    outs = [plan.infer(fields["x1"][:, c0:c0 + plan.Ncap]) for c0 in range(0, D, plan.Ncap)]
    res = {k: torch.cat([o[k] for o in outs], 1) for k in outs[0]}
    perfs = []
    for m in range(plan.E):
        valid = mask[m] != 0
        perf = OrderedDict(losses=None)
        idx = torch.nonzero(valid & (fields["has_y"][m] != 0)).view(-1)
        y = eval_y_prediction(res["pred"][m][idx].long().cpu(), res["proba"][m][idx].cpu(), fields["y"][m][idx].cpu(), plan.dim_y)
        perf.update(("y_" + k, v) for k, v in y.items())
        x1 = eval_x_reconstruction(fields["x1"][m], res["px1_mu"][m], res["px1_sg"][m], mask=valid)
        perf.update(("x1_" + k, v) for k, v in x1.items())
        pair = valid & (fields["has_x2"][m] != 0)
        if bool(pair.any()):
            x2 = eval_x_reconstruction(fields["x2"][m], res["px2_mu"][m], res["px2_sg"][m], mask=pair)
            perf.update(("x2_" + k, v) for k, v in x2.items())
        else:
            perf.update(("x2_" + k, float("nan")) for k in ("rmse", "r2", "pearr", "ll"))
        perf["model_class"] = MODEL_CLASS[kind]
        perfs.append(perf)
    return perfs


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, r


def max_diff(a, b):
    d = 0.0
    for pa, pb in zip(a, b):
        assert list(pa) == list(pb)
        for k in pa:
            if k in ("losses", "model_class"):
                continue
            if pa[k] != pa[k] and pb[k] != pb[k]:
                continue
            d = max(d, abs(pa[k] - pb[k]))
    return d


def sweep_case(E, n_valid, reps, say):
    gen = torch.Generator(device="cuda").manual_seed(E * 7919 + n_valid)
    vsizes = [n_valid - 20 + (37 * m) % 41 for m in range(E)]  # unequal splits, as folds give
    tsizes = [3 * n for n in vsizes]
    valid, vmask = padded_split(E, vsizes, gen)
    train, tmask = padded_split(E, tsizes, gen)
    plan = Plan("drvae", L=1, max_batch=BATCH, n_models=E, **ARCH)
    for m in range(E):
        plan.load_state_dict(init_state_dict("drvae", seed=m + 1, **ARCH), model=m)
    plan.set_member_hparams([dict(yloss_rate=[1., 10., 50., 100.][m % 4], pertloss_rate=0.05, kl_qz2pz2_rate=1.0,
                                  noise_std=0.01, lr=5e-4, weight_decay=0.05, prior_y=[0.5, 0.5]) for m in range(E)])
    nsteps = steps_per_epoch(tsizes, BATCH)
    w = tmask.float()
    cur = torch.empty(E, BATCH, dtype=torch.int32, device="cuda")
    state = dict(step=0)

    def epoch():
        idx = torch.multinomial(w, tmask.shape[1], replacement=True, generator=gen).to(torch.int32)
        for b in range(nsteps):
            cur.copy_(idx[:, b * BATCH:(b + 1) * BATCH])
            hp = plan.hparams(step=state["step"], training=True, add_noise=True, beta_pert=anneal_coef(state["step"], 1, 0))
            plan.train_step(dict(train, row_index=cur), hp, seed=12345)
            state["step"] += 1

    def infer():
        D = valid["x1"].shape[1]
        return [plan.infer(valid["x1"][:, c0:c0 + plan.Ncap]) for c0 in range(0, D, plan.Ncap)]

    old = lambda: old_evaluate_members(plan, "drvae", valid, vmask)
    new = lambda: evaluate_members(plan, "drvae", valid, vmask)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for fn in (epoch, epoch, infer, old, new):  # warm-up: graph capture, module loads, sklearn imports
            timed(fn)
        t = dict(old=[], new=[], infer=[], train=[])
        diff = 0.0
        for _ in range(reps):
            dt, a = timed(old)
            t["old"].append(dt)
            dt, b = timed(new)
            t["new"].append(dt)
            diff = max(diff, max_diff(a, b))
            t["infer"].append(timed(infer)[0])
            t["train"].append(timed(epoch)[0])
    med = {k: statistics.median(v) * 1e3 for k, v in t.items()}
    spread = {k: (min(v) * 1e3, max(v) * 1e3) for k, v in t.items()}
    say("E=%d valid rows/member %d-%d (D=%d), train rows/member %d-%d, %d train steps/epoch" % (
        E, min(vsizes), max(vsizes), max(vsizes), min(tsizes), max(tsizes), nsteps))
    for k in ("old", "new", "infer", "train"):
        say("  %-5s %9.2f ms  (min %.2f, max %.2f over %d reps)" % (k, med[k], spread[k][0], spread[k][1], reps))
    say("  validation old / new: %.1fx; validation / training epoch: old %.2f, new %.2f; "
        "metrics part (minus inference): old %.2f ms, new %.2f ms; max |old - new| over all metrics %.3g" % (
            med["old"] / med["new"], med["old"] / med["train"], med["new"] / med["train"],
            med["old"] - med["infer"], med["new"] - med["infer"], diff))
    del plan, valid, train
    torch.cuda.empty_cache()


def ranking_alone(E, D, reps, say):
    gen = torch.Generator(device="cuda").manual_seed(3)
    valid = torch.ones(E, D, dtype=torch.int32, device="cuda")
    has_y = torch.ones_like(valid)
    y = (torch.rand(E, D, device="cuda", generator=gen) < 0.5).to(torch.int32)
    p1 = torch.rand(E, D, device="cuda", generator=gen)
    proba = torch.stack([1 - p1, p1], -1).contiguous()
    pred = (p1 > 0.5).to(torch.int32)
    run = lambda: eval_members(valid, proba=proba, pred=pred, y=y, has_y=has_y)
    run()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        run()
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / reps
    P = y.sum(1).double()
    cmp = float((P * D).sum())  # each positive against every labeled row
    say("ranking kernels alone (y group of drvae_eval_members, binary): E=%d D=%d: %.2f ms per call over %d calls; "
        "%.3g score comparisons -> %.3g comparisons/s" % (E, D, ms, reps, cmp, cmp / (ms * 1e-3)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sweep_eval_bench: needs a CUDA device")
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    say("card: " + card())
    say("torch %s, CUDA %s" % (torch.__version__, torch.version.cuda))
    for E in (32, 80):
        for n_valid in (500, 4000):
            sweep_case(E, n_valid, args.reps, say)
    ranking_alone(80, 65536, 10, say)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
