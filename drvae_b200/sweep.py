"""Hyperparameter sweeps as ONE ensemble plan: the reference's grid (src/scripts/submitVAE.sh: y-loss rates x folds x
seeds per model family, one CPU process per job) trained as E members of one launch sequence.

Each member has its own initial weights (init_state_dict(seed=...)), its own train / validation split and its own
per-member hyperparameters (Plan.set_member_hparams: loss rates, noise, lr, weight decay, class prior).  The splits
are padded to the largest one and kept on the device; every step reads them through row indices.
"""
import types
from collections import OrderedDict

import torch

from . import checkpoint
from .init import init_state_dict
from .plan import Plan, anneal_coef
from ._lib import EVAL_MEMBER_COLUMNS
from .training import SnapshotRule, eval_members, validation_objective

FIELDS = {"drvae": ("x1", "x2", "y", "has_x2", "has_y"), "pvae": ("x1", "x2", "has_x2"), "vfae": ("x1", "y", "has_y")}
MODEL_CLASS = {"drvae": "DrVAE", "pvae": "PVAE", "vfae": "VFAE"}


def pad_members(kind, datasets):
    """Stack one dataset per member (DrVAEDataset / VFAEDataset, any sizes) into [E, D, ...] tensors, D = the largest
    size, padding rows zero at the end.  -> (fields dict, mask int32 [E, D] with 1 on real rows, sizes list)."""
    sizes = [int(ds.x1.shape[0]) for ds in datasets]
    D = max(sizes)
    out = OrderedDict()
    for k in FIELDS[kind]:
        parts = []
        for ds, n in zip(datasets, sizes):
            t = getattr(ds, k)
            t = t.float() if t.is_floating_point() else t.to(torch.int32)
            parts.append(torch.cat([t, t.new_zeros((D - n,) + tuple(t.shape[1:]))]) if n < D else t)
        out[k] = torch.stack(parts)
    mask = torch.zeros(len(sizes), D, dtype=torch.int32)
    for m, n in enumerate(sizes):
        mask[m, :n] = 1
    return out, mask, sizes


def steps_per_epoch(sizes, batch_size):
    """max_m floor(n_m / batch): every member sees about one pass of its own split per epoch."""
    return max(1, max(n // batch_size for n in sizes))


def evaluate_members(plan, kind, fields, mask):
    """Per-member metrics of evaluate_performance (training.py) on padded device data: one ensemble inference in
    chunks of the plan's row capacity, one drvae_eval_members call over every member's real rows, and one [E, 11] read
    back.  -> [perf dict]."""
    D = fields["x1"].shape[1]
    outs = [plan.infer(fields["x1"][:, c0:c0 + plan.Ncap]) for c0 in range(0, D, plan.Ncap)]
    res = {k: torch.cat([o[k] for o in outs], 1) for k in outs[0]}
    groups = dict(x1=fields["x1"], px1_mu=res["px1_mu"], px1_sg=res["px1_sg"])
    keys = ["x1_rmse", "x1_r2", "x1_pearr", "x1_ll"]
    if kind != "pvae":
        groups.update(proba=res["proba"], pred=res["pred"], y=fields["y"], has_y=fields["has_y"])
        keys = ["y_acc", "y_auroc", "y_aupr"] + keys
    if kind != "vfae":
        groups.update(x2=fields["x2"], px2_mu=res["px2_mu"], px2_sg=res["px2_sg"], has_x2=fields["has_x2"])
        keys += ["x2_rmse", "x2_r2", "x2_pearr", "x2_ll"]
    table = eval_members(mask, **groups).cpu().tolist()
    perfs = []
    for row in table:
        v = dict(zip(EVAL_MEMBER_COLUMNS, row))
        perf = OrderedDict(losses=None)
        perf.update((k, v[k]) for k in keys)
        perf["model_class"] = MODEL_CLASS[kind]
        perfs.append(perf)
    return perfs


def fit_sweep(kind, arch, members, datasets, batch_size=200, L=1, epochs=300, early_stop=False, min_patience=None,
              add_noise=False, weight_norm=False, kl_min=2.0, anneal_perturb=(1, 0), sample_seed=0, noise_seed=None,
              weights=None, log=None):
    """Train E members in one plan.

    kind: "drvae" | "pvae" | "vfae"; arch: Plan's shape arguments (dim_x, dim_y, dim_z1, dim_z3, enc_z1, dec_x,
    enc_z3, dec_z1, clf_hidden) and optionally its activation ("elu" | "softplus"; init_state_dict ignores it).
    members: E dicts {"seed": int, "hparams": dict of Plan.MEMBER_KEYS}.  datasets: E pairs (train, valid) of
    DrVAEDataset / VFAEDataset.  anneal_perturb: (itermax, offset) of the perturbation-loss anneal, or None for a
    constant 1 (VFAE).  weights: optional E sampling-weight tensors over each training split.

    Per epoch one device multinomial over [E, D] weights (zero on padding rows) draws every member's minibatches;
    max_m floor(n_m / batch) steps follow, each one CUDA-graph replay.  After every epoch each member is validated and
    goes through training.SnapshotRule, the rule of training.fit; a snapshot is a device copy of the member's
    parameters.  Members cannot leave the shared launch sequence, so a member whose rule says stop is frozen: its
    snapshot is final while the others keep training.  The loop ends when every member has stopped or at the epoch cap.
    A member's snapshot is the one training.fit (early_stop) would have kept for the same sequence of validation
    objectives, but the trajectory differs from a single-model run: the sampler and the noise keys are not the same.

    -> dict: plan (holding the snapshots), best (the [E, P] snapshot buffer), snapshot_epoch, stopped_epoch and
    history ([E] lists of validation objectives)."""
    say = log or (lambda *a: None)
    E = len(members)
    if len(datasets) != E:
        raise ValueError("need one (train, valid) pair per member")
    plan = Plan(kind, L=L, max_batch=batch_size, n_models=E, weight_norm=weight_norm, **arch)
    dev = plan.device
    checkpoint.load_ensemble(plan, [init_state_dict(kind, seed=int(m["seed"]), weight_norm=weight_norm, **arch) for m in members])
    plan.set_member_hparams([m["hparams"] for m in members])

    train, tmask, tsizes = pad_members(kind, [d[0] for d in datasets])
    valid, vmask, _ = pad_members(kind, [d[1] for d in datasets])
    train = {k: v.to(dev).contiguous() for k, v in train.items()}
    valid = {k: v.to(dev).contiguous() for k, v in valid.items()}
    vmask = vmask.to(dev)
    D = train["x1"].shape[1]
    w = tmask.double()
    if weights is not None:
        for m, wm in enumerate(weights):
            w[m, :tsizes[m]] = torch.as_tensor(wm, dtype=torch.float64)
    w = w.to(dev)
    bs = min(int(batch_size), D)
    nsteps = steps_per_epoch(tsizes, bs)
    gen = torch.Generator(device=dev).manual_seed(int(sample_seed))
    cur = torch.empty(E, bs, dtype=torch.int32, device=dev)  # fixed address: every step replays one graph
    if noise_seed is None:
        noise_seed = (int(members[0]["seed"]) << 20) ^ 0x5DEECE66D

    rules = [SnapshotRule(kind, epochs, early_stop, min_patience) for _ in range(E)]
    best = plan.params.clone()
    snapshot_epoch, stopped_epoch = [0] * E, [0] * E
    history = [[] for _ in range(E)]
    step = 0
    for epoch in range(1, int(epochs) + 1):
        idx = torch.multinomial(w.float(), D, replacement=True, generator=gen).to(torch.int32)
        for b in range(nsteps):
            cur.copy_(idx[:, b * bs:(b + 1) * bs])
            beta = anneal_coef(step, *anneal_perturb) if anneal_perturb else 1.0
            hp = plan.hparams(step=step, training=True, add_noise=add_noise, beta_pert=beta, kl_min=kl_min)
            plan.train_step(dict(train, row_index=cur), hp, seed=noise_seed)
            step += 1
        perfs = evaluate_members(plan, kind, valid, vmask)
        model = types.SimpleNamespace(kind=kind)
        for m in range(E):
            if stopped_epoch[m]:
                continue
            vobj = validation_objective(model, perfs[m])
            history[m].append(vobj)
            snapshot, _, stop = rules[m].update(epoch, vobj)
            if snapshot:
                best[m].copy_(plan.params[m])
                snapshot_epoch[m] = epoch
            if stop:
                stopped_epoch[m] = epoch
        say("epoch %d: %d/%d members stopped" % (epoch, sum(1 for s in stopped_epoch if s), E))
        if all(stopped_epoch):
            break
    for m in range(E):
        if not snapshot_epoch[m]:  # like the single-model driver: no snapshot taken -> the final parameters
            best[m].copy_(plan.params[m])
    plan.params.copy_(best)
    plan.sync_shadows()
    return dict(plan=plan, best=best, snapshot_epoch=snapshot_epoch, stopped_epoch=stopped_epoch, history=history,
                steps=step)
