"""Classifier hidden layers (dim_h_clf, --class-y) on the B200: u -> [Linear -> ELU] x k -> linear_p -> clamp(softmax).

Parity against the float64 oracle that emulates the kernels' bf16 rounding points (losses, every gradient row and
column, eval losses, fp32 inference), the fused optimizer against gradient + Adam, bit identity of the schedule variants,
the fall-back of the classifier fusions, and the model / CLI surface.  The oracle evaluates the classifier through
test_clf_hidden_host.classifier_oracle (its own mlp + linear_p); that composition is not pinned by a reference golden
file (each piece is, elsewhere): parity with the reference for --class-y is inferred."""
import glob

import pytest
import torch

from helpers import SEED_MODEL, assert_grad_close, batch_fields, orc, rel_l2
from test_clf_hidden_host import classifier_oracle

from drvae_b200.init import init_state_dict
from drvae_b200.noise import eps_block_from_tape, tape_shapes
from drvae_b200.plan import Plan, losses_to_dict

pytestmark = pytest.mark.gpu

README = dict(dim_x=978, dim_y=2, dim_z1=100, dim_z3=100, enc_z1=[800], dec_x=[600], enc_z3=[200], dec_z1=[200])
Z256 = dict(README, dim_z1=256, dim_z3=256)
SMALL = dict(dim_x=40, dim_y=2, dim_z1=128, dim_z3=9, enc_z1=[48], dec_x=[48], enc_z3=[48], dec_z1=[48])
DEEP4 = dict(dim_x=40, dim_y=2, dim_z1=16, dim_z3=9, enc_z1=[48, 32, 24, 40], dec_x=[32, 48, 40, 24], enc_z3=[24, 32, 16, 48],
             dec_z1=[40, 16, 32, 24])
CLF = {"c16": [16], "c200": [200], "c64_32": [64, 32], "c4l": [24, 48, 16, 40], "c256": [256]}
# id -> (kind, arch, class_y, weight_norm, N, L)
CASES = {"%s-readme-%s" % (k, c): (k, README, w, False, 150, 2) for k in ("drvae", "vfae") for c, w in CLF.items()}
CASES["drvae-readme-c200-wn"] = ("drvae", README, [200], True, 150, 2)
for k in ("drvae", "vfae"):
    CASES["%s-z256-c200" % k] = (k, Z256, [200], False, 150, 2)
    CASES["%s-z256-c64_32" % k] = (k, Z256, [64, 32], False, 150, 2)
SEED_BATCH, SEED_TAPE, SEED_EVAL = 5, 901, 902
TOL_EMU_LOSS, TOL_REF_LOSS = 5e-5, 1e-3
# Weight norm: the kernels round g v / ||v|| computed in fp32 to bf16, the oracle the float64 value, so single shadow
# entries can round the other way.  The project's weight-norm tests hold losses to 1e-4 of the emulating oracle and
# gradients to a per-tensor relative L2 (2e-2 against the reference golden); here 3e-2, because linear_p's bias gradient
# over two classes is a difference of near-equal sums (measured 2.2e-2 for this case, every other tensor within 2e-2).
TOL_WN_LOSS, TOL_WN_GRAD = 1e-4, 3e-2


def make_plan(kind, arch, clf, wn=False, N=150, L=2, n_models=1, sds=None):
    plan = Plan(kind, L=L, max_batch=N, n_models=n_models, weight_norm=wn, clf_hidden=clf, **arch)
    for m in range(n_models):
        sd = sds[m] if sds is not None else init_state_dict(kind, seed=SEED_MODEL + m, weight_norm=wn, clf_hidden=clf, **arch)
        plan.load_state_dict(sd, model=m)
    return plan


def loss_dict(kind, losses, model=0):
    return {k: float(v) for k, v in losses_to_dict(kind, losses[model].cpu()).items()}


def check_losses(got, want, tol, tag):
    for k, ref in want.items():
        if k == "MMD":
            continue
        ref = float(ref)
        assert abs(got[k] - ref) <= tol * abs(ref) + 1e-6, "%s %s: gpu %.7g ref %.7g" % (tag, k, got[k], ref)


class OracleRun:
    def __init__(self, case):
        kind, arch, clf, wn, N, L = CASES[case]
        self.sd = init_state_dict(kind, seed=SEED_MODEL, weight_norm=wn, clf_hidden=clf, **arch)
        self.batch = orc.synthetic_batch(N, arch["dim_x"], seed=SEED_BATCH, dim_y=arch["dim_y"])
        om = orc.OracleModel(self.sd, orc.default_cfg(kind, L=L, dim_y=arch["dim_y"]), dtype=torch.float64)
        om.iters = 1
        tape = orc.Tape(seed=SEED_TAPE)
        with classifier_oracle(True):
            self.lo_emu, self.g_emu = om.grads(self.batch, tape, emulate_bf16=True)
        self.tape = tape.log
        with classifier_oracle(False):
            self.lo_plain = om.loss(self.batch, orc.Tape(recorded=self.tape), train=True)
        etape = orc.Tape(seed=SEED_EVAL)
        with classifier_oracle(True):
            self.lo_eval = om.loss(self.batch, etape, train=False, emulate_bf16=True)
        self.eval_tape = etape.log
        with classifier_oracle(False):
            self.fwd = om.forward(self.batch["x1"])


@pytest.fixture(scope="module")
def oracle():
    cache = {}

    def get(case):
        if case not in cache:
            cache[case] = OracleRun(case)
        return cache[case]

    return get


@pytest.mark.parametrize("case", list(CASES))
def test_grad_step_matches_the_float64_oracle(oracle, case):
    kind, arch, clf, wn, N, L = CASES[case]
    o = oracle(case)
    plan = make_plan(kind, arch, clf, wn, N, L, sds=[o.sd])
    names = [t[0] for t in plan.tensors]
    assert [n for n in names if n.startswith("encoder_y")] == [n for n in o.sd if n.startswith("encoder_y")]
    eps = eps_block_from_tape(plan, o.tape, o.batch["has_x2"], o.batch["has_y"], noisy=True)
    got = loss_dict(kind, plan.grad_step(batch_fields(kind, o.batch), plan.hparams(step=1), eps=eps))
    check_losses(got, o.lo_emu, TOL_WN_LOSS if wn else TOL_EMU_LOSS, "%s vs emulating float64 oracle" % case)
    check_losses(got, o.lo_plain, TOL_REF_LOSS, "%s vs float64 oracle" % case)
    gv = plan.tensor_views(plan.grads, 0)
    for name, g in o.g_emu.items():
        if float(g.norm()) == 0:
            assert float(gv[name].norm()) == 0, name
            continue
        if wn:
            assert rel_l2(gv[name], g) <= TOL_WN_GRAD, "%s grad %s relL2 %.3e" % (case, name, rel_l2(gv[name], g))
        else:
            assert_grad_close(gv[name], g, "%s grad %s" % (case, name))


@pytest.mark.parametrize("case", list(CASES))
def test_eval_loss_and_inference_match_the_float64_oracle(oracle, case):
    kind, arch, clf, wn, N, L = CASES[case]
    o = oracle(case)
    plan = make_plan(kind, arch, clf, wn, N, L, sds=[o.sd])
    eps = eps_block_from_tape(plan, o.eval_tape, o.batch["has_x2"], o.batch["has_y"], noisy=False)
    got = loss_dict(kind, plan.loss_forward(batch_fields(kind, o.batch), plan.hparams(step=1, training=False), eps=eps))
    check_losses(got, o.lo_eval, TOL_WN_LOSS if wn else TOL_EMU_LOSS, "%s eval" % case)
    res = plan.infer(o.batch["x1"])  # fp32 path (weight norm: the bf16 tensor-core path)
    ref = o.fwd["proba"]
    a = res["proba"][0].cpu().double()
    tol = (2e-6 + 2e-5 * ref.abs()) if not wn else (2e-3 + 0 * ref)
    bad = (a - ref).abs() > tol
    assert not bool(bad.any()), "%s proba: %d off, max %.3e" % (case, int(bad.sum()), float((a - ref).abs().max()))
    p = torch.sort(ref, dim=1, descending=True)[0]
    sure = (p[:, 0] - p[:, 1]) > (1e-5 if not wn else 1e-2)
    assert torch.equal(res["pred"][0].cpu().long()[sure], o.fwd["pred"][sure]), "%s: thresholded predictions differ" % case


def test_bf16_inference_path_matches_the_oracle():
    for kind in ("drvae", "vfae"):
        clf = [64, 32]
        sd = init_state_dict(kind, seed=SEED_MODEL, clf_hidden=clf, **README)
        plan = make_plan(kind, README, clf, sds=[sd])
        plan.set_infer_precision(False)
        x1 = orc.synthetic_batch(150, README["dim_x"], seed=3)["x1"]
        res = plan.infer(x1)
        om = orc.OracleModel(sd, orc.default_cfg(kind, L=2), dtype=torch.float64)
        with classifier_oracle(True):
            ref = om.forward(x1, emulate_bf16=True)["proba"]
        assert float((res["proba"][0].cpu().double() - ref).abs().max()) < 2e-3, kind


# Inputs of the fused-optimizer checks: (architecture, classifier hidden layers).  deep4 has 4 hidden layers in every MLP
# and in the classifier: 25 weight layers for DrVAE, one more than the grouped dW+Adam launch takes (its train step runs
# gradient + stand-alone Adam), and 24 for VFAE, the most the grouped launch takes.
STEP_CASES = {"readme": (README, [64, 32]), "deep4": (DEEP4, [8, 8, 8, 8])}


def _split_vs_fused(kind, arch, clf, N, L):
    fields = batch_fields(kind, orc.synthetic_batch(N, arch["dim_x"], seed=SEED_BATCH))
    res = {}
    for mode in ("fused", "split"):
        plan = make_plan(kind, arch, clf, N=N, L=L)
        out = []
        for it in range(2):
            hp = plan.hparams(step=it)
            if mode == "fused":
                out.append(plan.train_step(fields, hp, seed=17).cpu().clone())
            else:
                out.append(plan.grad_step(fields, hp, seed=17).cpu().clone())
                plan.adam_step(hp)
        torch.cuda.synchronize()
        res[mode] = (out, plan.params.cpu().clone(), plan.adam_m.cpu().clone(), plan.adam_v.cpu().clone())
    f, s = res["fused"], res["split"]
    assert torch.equal(f[0][0], s[0][0]), "first-step losses differ"
    for i, name in ((1, "params"), (2, "adam_m"), (3, "adam_v")):
        bad = ~torch.isclose(f[i], s[i], rtol=1e-6, atol=1e-9)
        assert not bool(bad.any()), "%s: %d %s entries differ" % (kind, int(bad.sum()), name)
    assert torch.allclose(f[0][1], s[0][1], rtol=1e-5, atol=1e-6), "second-step losses differ"


@pytest.mark.parametrize("case", list(STEP_CASES))
@pytest.mark.parametrize("kind", ("drvae", "vfae"))
def test_fused_adam_equals_grad_then_adam(kind, case):
    arch, clf = STEP_CASES[case]
    _split_vs_fused(kind, arch, clf, 150, 2)


@pytest.mark.parametrize("case", list(STEP_CASES))
@pytest.mark.parametrize("kind", ("drvae", "vfae"))
def test_train_steps_track_the_oracle(kind, case):
    arch, clf = STEP_CASES[case]
    N, L = 150, 2
    batch = orc.synthetic_batch(N, arch["dim_x"], seed=SEED_BATCH)
    plan = make_plan(kind, arch, clf, N=N, L=L)
    for it in range(3):
        cur = plan.state_dict()
        o = orc.OracleModel({k: v.cpu() for k, v in cur.items()}, orc.default_cfg(kind, L=L), dtype=torch.float64)
        o.iters = it
        tape = orc.Tape(seed=SEED_TAPE + it)
        with classifier_oracle(True):
            lo = o.loss(batch, tape, train=True, emulate_bf16=True)
        eps = eps_block_from_tape(plan, tape.log, batch["has_x2"], batch["has_y"], noisy=True)
        hp = plan.hparams(step=it, beta_pert=orc.anneal(it, 1, 0))
        got = loss_dict(kind, plan.train_step(batch_fields(kind, batch), hp, eps=eps))
        check_losses(got, lo, TOL_EMU_LOSS, "%s step %d" % (kind, it))
        new = plan.state_dict()
        for name in new:
            if name.startswith("encoder_y.nnet"):
                assert 0 < float((new[name] - cur[name]).abs().max()) <= 2.5 * 5e-4, name


def _ens(kind, clf, E=3, N=64, arch=SMALL, L=2):
    batches = [batch_fields(kind, orc.synthetic_batch(N, arch["dim_x"], seed=20 + m)) for m in range(E)]
    return {k: torch.stack([b[k] for b in batches]).contiguous().cuda() for k in batches[0]}, batches


def _run(plan, big, steps=3):
    losses = [plan.train_step(big, plan.hparams(step=it), seed=9).cpu().clone() for it in range(steps)]
    g = plan.grad_step(big, plan.hparams(step=steps), seed=9).cpu().clone()
    grads = plan.grads.cpu().clone()
    plan.adam_step(plan.hparams(step=steps))
    ev = plan.loss_forward(big, plan.hparams(step=steps + 1, training=False), seed=9).cpu().clone()
    torch.cuda.synchronize()
    return [torch.stack(losses), plan.params.cpu().clone(), g, grads, ev]


@pytest.mark.parametrize("kind", ("drvae", "vfae"))
def test_graph_replay_and_step_kernel_are_bit_identical(kind):
    """graph replay = plain launches, persistent step kernel = one launch per operation."""
    clf, E = [64, 32], 3
    big, _ = _ens(kind, clf, E)
    base = _run(make_plan(kind, SMALL, clf, N=64, n_models=E), big)
    variants = {}
    p = make_plan(kind, SMALL, clf, N=64, n_models=E)
    p.set_graph(False)
    variants["no_graph"] = (_run(p, big), None)
    p = make_plan(kind, SMALL, clf, N=64, n_models=E)
    p.set_step_kernel(True)
    variants["step_kernel"] = (_run(p, big), p)
    assert variants["step_kernel"][1].step_kernel_launches() >= 1
    for name, (res, _) in variants.items():
        for a, b in zip(base, res):
            assert torch.equal(a, b), name


@pytest.mark.parametrize("kind", ("drvae", "vfae"))
def test_ensemble_member_equals_a_single_model_plan(kind):
    clf, N = [200], 64
    sds = [init_state_dict(kind, seed=SEED_MODEL + m, clf_hidden=clf, **SMALL) for m in range(2)]
    batches = [orc.synthetic_batch(N, SMALL["dim_x"], seed=30 + m) for m in range(2)]
    plan = make_plan(kind, SMALL, clf, N=N, n_models=2, sds=sds)
    epss = []
    for m in range(2):
        b = batches[m]
        draws = [torch.randn(*sh, generator=torch.Generator().manual_seed(70 + m)) for sh in tape_shapes(
            kind, b["has_x2"], b["has_y"], SMALL["dim_x"], SMALL["dim_z1"], SMALL["dim_z3"], SMALL["dim_y"], 2, noisy=True)]
        epss.append(eps_block_from_tape(plan, draws, b["has_x2"], b["has_y"], noisy=True))
    fields = [batch_fields(kind, b) for b in batches]
    big = {k: torch.stack([f[k] for f in fields]).contiguous() for k in fields[0]}
    losses = plan.grad_step(big, plan.hparams(step=1), eps=torch.stack(epss)).cpu().clone()
    grads = plan.grads.cpu().clone()
    single = make_plan(kind, SMALL, clf, N=N, sds=[sds[1]])
    l1 = single.grad_step(fields[1], single.hparams(step=1), eps=epss[1]).cpu()
    assert not torch.equal(losses[0], losses[1])
    assert torch.equal(l1[0], losses[1])
    assert torch.equal(single.grads[0].cpu(), grads[1])


@pytest.mark.parametrize("kind", ("drvae", "vfae"))
def test_member_table_equals_a_table_less_plan_with_the_members_values(kind):
    clf, E, N = [64, 32], 3, 64
    big, _ = _ens(kind, clf, E, N)
    shared = dict(yloss_rate=1.0, pertloss_rate=0.05, kl_qz2pz2_rate=1.0, noise_std=0.01, lr=5e-4, weight_decay=0.05,
                  prior_y=[0.5, 0.5])  # the defaults of Plan.hparams
    members = [dict(shared, yloss_rate=10.0 * (m + 1), lr=5e-4 * (m + 1)) for m in range(E)]
    ens = make_plan(kind, SMALL, clf, N=N, n_models=E)
    ens.set_member_hparams(members)
    out = [ens.train_step(big, ens.hparams(step=it), seed=4).cpu().clone() for it in range(3)]
    torch.cuda.synchronize()
    for m in range(E):
        ref = make_plan(kind, SMALL, clf, N=N, n_models=E)
        got = [ref.train_step(big, ref.hparams(step=it, yloss_rate=members[m]["yloss_rate"], lr=members[m]["lr"]), seed=4)
               .cpu().clone() for it in range(3)]
        torch.cuda.synchronize()
        for it in range(3):
            assert torch.equal(got[it][m], out[it][m]), (m, it)
        assert torch.equal(ref.params[m].cpu(), ens.params[m].cpu()), m


def _steady_launches(plan, fields):
    plan.set_graph(False)
    plan.train_step(fields, plan.hparams(step=0), seed=3)
    n0 = plan.launch_count()
    plan.train_step(fields, plan.hparams(step=1), seed=3)
    torch.cuda.synchronize()
    return plan.launch_count() - n0


def test_one_hidden_layer_adds_five_launches_to_the_step():
    """One hidden layer adds clf_u, its forward GEMM, clf_fwd (T_post no longer computes the classifier), its dX GEMM
    and clf_du to the DrVAE step; its dW + Adam joins the grouped launch."""
    kind = "drvae"
    fields = batch_fields(kind, orc.synthetic_batch(64, SMALL["dim_x"], seed=1))
    counts = [_steady_launches(make_plan(kind, SMALL, clf, N=64), fields) for clf in ([], [64])]
    assert counts[1] == counts[0] + 5, counts


def test_readme_step_without_hidden_layers_issues_35_launches():
    kind, E = "drvae", 32
    big, _ = _ens(kind, [], E, 150, README)
    assert _steady_launches(make_plan(kind, README, [], N=150, L=1, n_models=E), big) == 35


def test_pth_round_trip_and_reference_state_dict(tmp_path):
    from drvae_b200 import DrVAE
    kw = dict(dim_x=40, dim_s=1, dim_y=2, dim_h_en_z1=[32], dim_h_de_z1=[16], dim_h_en_z2Fz1=[], dim_h_en_z3=[16],
              dim_h_de_x=[32], dim_h_clf=[200], dim_z1=8, dim_z3=6, type_rec='diag_gaussian', clf_z1z2=True,
              nonlinearity='elu', batch_size=32, random_seed=3)
    m = DrVAE(**kw)
    keys = list(m.state_dict())
    i = keys.index("encoder_y.nnet.model.linear1.weight")
    assert keys[i:i + 4] == ["encoder_y.nnet.model.linear1.weight", "encoder_y.nnet.model.linear1.bias",
                             "encoder_y.decoder_p.linear_p.weight", "encoder_y.decoder_p.linear_p.bias"]
    assert m.state_dict()["encoder_y.nnet.model.linear1.weight"].shape == (200, 16)
    assert m.state_dict()["encoder_y.decoder_p.linear_p.weight"].shape == (2, 200)
    f = str(tmp_path / "m.pth")
    m.save_to_file(f)
    m2 = DrVAE(**dict(kw, random_seed=4))
    m2.load_params_from_file(f)
    for k, v in m.state_dict().items():
        assert torch.equal(v.cpu(), m2.state_dict()[k].cpu()), k
    x = torch.randn(16, 40)
    assert torch.equal(m.forward(x1=x)["proba"].cpu(), m2.forward(x1=x)["proba"].cpu())


def test_cli_drvae_with_class_y_runs(tmp_path):
    from drvae_b200 import cli
    argv = ["drvae", "--modelid", "auto", "--datafile", "synthetic:300", "--outdir", str(tmp_path), "--epochs", "2",
            "--batch-size", "40", "--dim-z1", "8", "--enc-z1", "16", "--dec-x", "16", "--dim-z3", "6", "--enc-z3", "12",
            "--dec-z1", "12", "--yloss-rate", "1", "--class-y", "200"]
    res = cli.main(argv)
    assert 0.0 <= res["test"]["y_acc"] <= 1.0
    pths = glob.glob(str(tmp_path / "models" / "*.pth"))
    assert len(pths) == 1
    sd = torch.load(pths[0])
    assert sd["encoder_y.nnet.model.linear1.weight"].shape == (200, 16)


def test_cli_sweep_vfae_with_class_y_runs(tmp_path):
    from drvae_b200 import cli
    flags = ("--datafile synthetic:300 --rseeds 1 2 --folds 1 --epochs 2 --batch-size 32 --dim-z1 8 --enc-z1 16 "
             "--dec-x 16 --dim-z2 6 --enc-z2 12 --dec-z1 12 --class-y 50 50 --outdir %s" % tmp_path).split()
    cli.main(["sweep", "vfae"] + flags)
    pths = sorted(glob.glob(str(tmp_path / "models" / "*.pth")))
    assert len(pths) == 2
    sd = torch.load(pths[0])
    assert sd["encoder_y.nnet.model.linear2.weight"].shape == (50, 50)
    assert sd["encoder_y.decoder_p.linear_p.weight"].shape == (2, 50)
