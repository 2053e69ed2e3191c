"""GPU tests of per-member hyperparameters (drvae_set_member_hparams / Plan.set_member_hparams) and of the sweep
driver built on them (`python -m drvae_b200.cli sweep`).

The yardstick is bit identity: a table that repeats the shared hyperparameters changes nothing, and member k of a plan
with distinct members equals member k of a table-less plan run with member k's values."""
import glob
import json
import math
import os

import numpy as np
import pytest
import torch

from helpers import ARCH, KINDS, L, SEED_TAPE, batch_fields, orc

from drvae_b200.init import init_state_dict
from drvae_b200.noise import eps_block_from_tape
from drvae_b200.plan import Plan, anneal_coef, losses_to_dict

pytestmark = pytest.mark.gpu

ODD = dict(dim_x=37, dim_y=3, dim_z1=13, dim_z3=7, enc_z1=[23], dec_x=[19, 21], enc_z3=[11], dec_z1=[9])
CASES = dict(readme=(ARCH["readme"], False, 150), odd=(ODD, False, 29), tiny_wn=(ARCH["tiny"], True, 24))
SHARED = dict(yloss_rate=3.0, pertloss_rate=0.05, kl_qz2pz2_rate=1.0, noise_std=0.02, lr=1e-3, weight_decay=0.05)


def _prior(dim_y, k=0):
    p = np.arange(1, dim_y + 1, dtype=np.float64) + k
    return list(p / p.sum())


def _hp(plan, step, m, training=True):
    """drvae_hparams_t carrying member dict m's values."""
    return plan.hparams(step=step, training=training, beta_pert=anneal_coef(step, 1, 0), yloss_rate=m["yloss_rate"],
                        pertloss_rate=m["pertloss_rate"], kl_qz2pz2_rate=m["kl_qz2pz2_rate"], noise_std=m["noise_std"],
                        lr=m["lr"], weight_decay=m["weight_decay"], prior_y=m["prior_y"])


def _members(E, dim_y):
    """Distinct values of every per-member field."""
    return [dict(yloss_rate=[1.0, 10.0, 50.0, 100.0][k % 4], pertloss_rate=0.02 + 0.03 * k, kl_qz2pz2_rate=0.5 + 0.25 * k,
                 noise_std=0.005 * (k + 1), lr=[5e-4, 1e-3, 2e-4, 3e-3][k % 4], weight_decay=0.01 * k,
                 prior_y=_prior(dim_y, k)) for k in range(E)]


def _batches(kind, arch, N, E, seed=5):
    parts = [orc.synthetic_batch(N, arch["dim_x"], seed=seed + m, dim_y=arch["dim_y"]) for m in range(E)]
    return {k: torch.stack([p[k] for p in parts]).cuda() for k in batch_fields(kind, parts[0])}


def _plan(kind, arch, wn, N, E, seeds):
    plan = Plan(kind, L=L, max_batch=N, n_models=E, weight_norm=wn, **arch)
    for m, s in enumerate(seeds):
        plan.load_state_dict(init_state_dict(kind, seed=s, weight_norm=wn, **arch), model=m)
    return plan


def _state(plan):
    torch.cuda.synchronize()
    return [t.clone() for t in (plan.params, plan.adam_m, plan.adam_v)]


def _sequence(plan, batch, hp_of, seed=11):
    """4 fused train steps (graph replays from the 3rd), grad_step + adam_step, loss_forward -> every output."""
    out = []
    for it in range(4):
        out.append(plan.train_step(batch, hp_of(it)).clone())
    out += _state(plan)
    out.append(plan.grad_step(batch, hp_of(4), seed=seed).clone())
    out.append(plan.grads.clone())
    plan.adam_step(hp_of(4))
    out += _state(plan)
    out.append(plan.loss_forward(batch, hp_of(5)).clone())
    return out


def _assert_same(a, b, what):
    for i, (x, y) in enumerate(zip(a, b)):
        assert torch.equal(x, y), "%s: output %d differs (max |d| %g)" % (what, i, (x - y).abs().max().item())


@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("kind", KINDS)
def test_uniform_table_changes_nothing(kind, case):
    arch, wn, N = CASES[case]
    E = 2
    shared = dict(SHARED, prior_y=_prior(arch["dim_y"]))
    batch = _batches(kind, arch, N, E)
    runs = []
    for table in (None, [shared] * E):
        plan = _plan(kind, arch, wn, N, E, [123, 456])
        if table:
            plan.set_member_hparams(table)
        runs.append(_sequence(plan, batch, lambda it: _hp(plan, it, shared)))
        assert plan.graph_replays() >= 2 and plan.graph_failures() == 0
    _assert_same(runs[0], runs[1], "%s/%s uniform table" % (kind, case))


def _distinct_vs_reference(kind, arch, wn, N, E=4, steps=3, configure=None):
    members = _members(E, arch["dim_y"])
    seeds = [100 + 7 * m for m in range(E)]
    batch = _batches(kind, arch, N, E)
    plan = _plan(kind, arch, wn, N, E, seeds)
    if configure:
        configure(plan)
    plan.set_member_hparams(members)
    losses = [plan.train_step(batch, _hp(plan, it, SHARED | dict(prior_y=_prior(arch["dim_y"])))).clone() for it in range(steps)]
    got = _state(plan)
    return members, seeds, batch, losses, got


@pytest.mark.parametrize("case", ("readme", "odd", "tiny_wn"))
@pytest.mark.parametrize("kind", KINDS)
def test_distinct_members_match_table_less_plans(kind, case):
    arch, wn, N = CASES[case]
    E, steps = 4, 3
    members, seeds, batch, losses, got = _distinct_vs_reference(kind, arch, wn, N, E, steps)
    for k in range(E):
        ref = _plan(kind, arch, wn, N, E, seeds)
        ref_losses = [ref.train_step(batch, _hp(ref, it, members[k])).clone() for it in range(steps)]
        want = _state(ref)
        for it in range(steps):
            assert torch.equal(losses[it][k], ref_losses[it][k]), "%s/%s member %d step %d losses" % (kind, case, k, it)
        for g, w in zip(got, want):
            assert torch.equal(g[k], w[k]), "%s/%s member %d state" % (kind, case, k)
    # the members did train differently
    assert not torch.equal(losses[-1][0], losses[-1][1])


@pytest.mark.parametrize("kind", KINDS)
def test_members_track_the_oracle(kind):
    """Tape noise, 3 train steps: each member's losses follow OracleModel run with that member's cfg (tolerance of
    test_step_gpu.py::test_train_steps_track_the_oracle)."""
    arch, N, E = ARCH["tiny"], 24, 4
    members = _members(E, arch["dim_y"])
    plan = _plan(kind, arch, False, N, E, [123 + m for m in range(E)])
    plan.set_member_hparams(members)
    batch = orc.synthetic_batch(N, arch["dim_x"])
    fields = {k: v.unsqueeze(0).expand(E, *v.shape).contiguous() for k, v in batch_fields(kind, batch).items()}
    for it in range(3):
        los, eps = [], []
        for m in range(E):
            cfg = orc.default_cfg(kind, L=L, noise_std=members[m]["noise_std"], yloss_rate=members[m]["yloss_rate"],
                                  pertloss_rate=members[m]["pertloss_rate"], kl_qz2pz2_rate=members[m]["kl_qz2pz2_rate"],
                                  prior_y_vec=members[m]["prior_y"])
            o = orc.OracleModel({k: v.cpu() for k, v in plan.state_dict(m).items()}, cfg)
            o.iters = it
            tape = orc.Tape(seed=SEED_TAPE + 10 * it + m)
            los.append(o.loss(batch, tape, train=True, emulate_bf16=True))
            eps.append(eps_block_from_tape(plan, tape.log, batch["has_x2"], batch["has_y"], noisy=True))
        out = plan.train_step(fields, _hp(plan, it, members[0]), eps=torch.stack(eps)).cpu()
        for m in range(E):
            got = {k: float(v) for k, v in losses_to_dict(kind, out[m]).items()}
            for k, ref in los[m].items():
                if k == "MMD":
                    continue
                ref = float(ref)
                assert abs(got[k] - ref) <= 2e-5 * abs(ref) + 1e-6, "member %d step %d %s: %.6f vs %.6f" % (m, it, k, got[k], ref)


def test_table_swap_replays_without_recapture_and_clear_restores():
    kind, (arch, wn, N) = "drvae", CASES["readme"]
    E = 4
    A = _members(E, 2)
    B = [dict(m, yloss_rate=m["yloss_rate"] * 2, lr=m["lr"] * 0.5) for m in A]
    shared = dict(SHARED, prior_y=_prior(2))
    batch = _batches(kind, arch, N, E)
    runs = []
    for graphs in (True, False):
        plan = _plan(kind, arch, wn, N, E, [1, 2, 3, 4])
        plan.set_graph(graphs)
        plan.set_member_hparams(A)
        out = [plan.train_step(batch, _hp(plan, it, shared)).clone() for it in range(3)]
        replays = plan.graph_replays()
        plan.set_member_hparams(B)
        out.append(plan.train_step(batch, _hp(plan, 3, shared)).clone())
        if graphs:
            assert plan.graph_replays() == replays + 1, "table B did not run as a replay of the captured graph"
        out += _state(plan)
        plan.set_member_hparams(None)
        out += [plan.train_step(batch, _hp(plan, it, shared)).clone() for it in (4, 5, 6)]
        out += _state(plan)
        assert plan.graph_failures() == 0
        runs.append(out)
    _assert_same(runs[0], runs[1], "graph replay vs plain launches")
    # after clearing, the step is the table-less step: same bits as a plan that never had a table, from the same state
    ref = _plan(kind, arch, wn, N, E, [1, 2, 3, 4])
    plan = _plan(kind, arch, wn, N, E, [1, 2, 3, 4])
    plan.set_member_hparams(A)
    plan.train_step(batch, _hp(plan, 0, shared))
    plan.set_member_hparams(None)
    for p in (ref, plan):
        p.params.copy_(runs[0][4]), p.adam_m.copy_(runs[0][5]), p.adam_v.copy_(runs[0][6])
        p.sync_shadows()
    a = [ref.train_step(batch, _hp(ref, it, shared)).clone() for it in (4, 5, 6)] + _state(ref)
    b = [plan.train_step(batch, _hp(plan, it, shared)).clone() for it in (4, 5, 6)] + _state(plan)
    _assert_same(a, b, "cleared table vs no table")


@pytest.mark.parametrize("schedule", ("step_kernel",))
def test_table_under_other_schedules(schedule):
    kind, (arch, wn, N) = "drvae", CASES["readme"]
    base = _distinct_vs_reference(kind, arch, wn, N)
    other = _distinct_vs_reference(kind, arch, wn, N, configure=lambda p: p.set_step_kernel(True))
    _assert_same(base[3] + base[4], other[3] + other[4], schedule)


def test_errors_are_status_codes():
    arch = ARCH["tiny"]
    plan = _plan("drvae", arch, False, 24, 2, [1, 2])
    good = _members(2, 2)
    lib, h, stream = plan.lib, plan.h, plan._stream()
    from drvae_b200 import _lib
    table = (_lib.MemberHParams * 2)()
    for m, d in zip(table, good):
        for k in Plan.MEMBER_KEYS[:-1]:
            setattr(m, k, d[k])
    assert lib.drvae_set_member_hparams(h, table, 2, stream) == 0
    assert lib.drvae_set_member_hparams(h, table, 1, stream) != 0  # wrong count
    assert lib.drvae_set_member_hparams(h, None, 2, stream) != 0
    table[1].noise_std = float("nan")
    assert lib.drvae_set_member_hparams(h, table, 2, stream) != 0
    table[1].noise_std, table[0].lr = 0.01, -1e-3
    assert lib.drvae_set_member_hparams(h, table, 2, stream) != 0
    assert b"lr" in lib.drvae_last_error()
    table[0].lr, table[0].log_prior_y[0] = 1e-3, float("-inf")
    assert lib.drvae_set_member_hparams(h, table, 2, stream) != 0
    assert lib.drvae_set_member_hparams(h, None, 0, stream) == 0
    # the Python surface validates before the library does
    for bad in (good[:1], [dict(good[0], lr=-1.0), good[1]], [dict(good[0], prior_y=[1.0, 0.0]), good[1]],
                [{k: v for k, v in good[0].items() if k != "lr"}, good[1]]):
        with pytest.raises(ValueError):
            plan.set_member_hparams(bad)
    # data-parallel plans take no table, in either order
    for order in ("attach_first", "table_first"):
        dp = _plan("drvae", arch, False, 24, 1, [1])
        grads = torch.zeros(dp.dp_grad_floats(), device="cuda")
        ctl = torch.zeros(128, dtype=torch.int64, device="cuda")
        if order == "attach_first":
            dp.dp_attach(0, 1, [grads.data_ptr()], [ctl.data_ptr()])
            with pytest.raises(RuntimeError, match="data-parallel"):
                dp.set_member_hparams(good[:1])
        else:
            dp.set_member_hparams(good[:1])
            with pytest.raises(RuntimeError, match="member table"):
                dp.dp_attach(0, 1, [grads.data_ptr()], [ctl.data_ptr()])
    # a failed call changes nothing: the plan still trains
    plan.set_member_hparams(good)
    batch = _batches("drvae", arch, 24, 2)
    assert torch.isfinite(plan.train_step(batch, _hp(plan, 0, good[0]))).all()


def test_cli_sweep_end_to_end(tmp_path):
    from drvae_b200 import DrVAE, cli
    flags = ("--datafile synthetic:300 --rseeds 1 2 --folds 1 2 --yloss-rates 10 50 --epochs 3 --batch-size 32 "
             "--dim-z1 8 --enc-z1 16 --dec-x 16 --dim-z3 6 --enc-z3 12 --dec-z1 12 --train-w-noise --clf-dataprior "
             "--outdir %s" % tmp_path).split()
    cli.main(["sweep", "drvae"] + flags)
    pths = sorted(glob.glob(str(tmp_path / "models" / "*.pth")))
    jsons = sorted(glob.glob(str(tmp_path / "results" / "*.json")))
    assert len(pths) == 8 and len(jsons) == 8
    assert os.path.basename(pths[0]) == "DrVAE_SD_RS1_L1_YR10.0_FOLD1_26.pth"
    sds = {}
    for p in pths:
        m = DrVAE(dim_x=978, dim_s=1, dim_y=2, dim_h_en_z1=[16], dim_h_de_z1=[12], dim_h_en_z2Fz1=[], dim_h_en_z3=[12],
                  dim_h_de_x=[16], dim_h_clf=[], dim_z1=8, dim_z3=6, type_rec='diag_gaussian', clf_z1z2=True,
                  type_y='discrete', prior_y='uniform', batch_size=32, nonlinearity='elu', learning_rate=0.0005, L=1,
                  weight_decay=0.05, use_MMD=False, random_seed=1, log_txt=None)
        m.load_params_from_file(p)
        sds[os.path.basename(p)] = {k: v.detach().clone() for k, v in m.state_dict().items()}
    a, b = sds["DrVAE_SD_RS1_L1_YR10.0_FOLD1_26.pth"], sds["DrVAE_SD_RS1_L1_YR50.0_FOLD1_26.pth"]
    assert any(not torch.equal(a[k], b[k]) for k in a), "members that differ only in the y-loss rate ended equal"
    for j in jsons:
        res = json.load(open(j))["26"]
        for split in ("train", "valid", "test"):
            assert res[split]["losses"] is None
            for k in ("y_acc", "y_auroc", "y_aupr", "x1_rmse", "x1_r2", "x1_pearr", "x1_ll", "x2_rmse", "x2_pearr"):
                assert math.isfinite(res[split][k]), (j, split, k)
            assert res[split]["model_class"] == "DrVAE"
