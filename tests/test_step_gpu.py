"""GPU parity tests of the training step, through the C ABI (drvae_b200.plan.Plan is a ctypes
shim over include/drvae_b200.h).

Two yardsticks:
  * the bf16-emulating oracle (oracle/drvae_oracle.py, emulate_bf16=True) reproduces the CUDA
    path's rounding points, so kernel LOGIC is held to a tight tolerance: losses 2e-5 relative,
    gradients 1e-2 relative L2 per tensor (bf16 rounding flips on stored activations);
  * the fp32 reference values recorded in tests/golden (from the reference itself): losses
    within 1e-3 relative — the tolerance BASELINE.json's north_star states for the bf16 path.
"""
import numpy as np
import pytest
import torch

from helpers import ARCH, KINDS, L, NROWS, SEED_MODEL, SEED_TAPE, batch_fields, golden, orc, rel_l2

from drvae_b200.init import init_state_dict
from drvae_b200.noise import eps_block_from_tape
from drvae_b200.plan import LOSS_KEYS, Plan, anneal_coef, losses_to_dict

pytestmark = pytest.mark.gpu

CASES = ("tiny", "deep", "readme")
TOL_EMU_LOSS = 2e-5
TOL_EMU_GRAD = 1e-2
TOL_REF_LOSS = 1e-3  # north_star: "within 1e-3 relative for bf16"


def loss_dict(kind, losses, model=0):
    return {k: float(v) for k, v in losses_to_dict(kind, losses[model].cpu()).items()}


def check_losses(got, want, tol, tag):
    for k, ref in want.items():
        if k == "MMD":
            continue
        ref = float(ref)
        assert abs(got[k] - ref) <= tol * abs(ref) + 1e-6, "%s %s: gpu %.6f ref %.6f" % (tag, k, got[k], ref)


def setup(kind, case, step=0, impl="tc", n_models=1):
    arch, N = ARCH[case], NROWS[case]
    sd = init_state_dict(kind, seed=SEED_MODEL, **arch)
    batch = orc.synthetic_batch(N, arch["dim_x"])
    om = orc.OracleModel(sd, orc.default_cfg(kind, L=L))
    om.iters = step
    plan = Plan(kind, L=L, max_batch=N, n_models=n_models, **arch)
    plan.set_gemm_impl(impl)
    for m in range(n_models):
        plan.load_state_dict(sd, model=m)
    return arch, N, sd, batch, om, plan


@pytest.mark.parametrize("step", (0, 1))
@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("kind", KINDS)
def test_forward_backward_parity(kind, case, step):
    arch, N, sd, batch, om, plan = setup(kind, case, step)
    tape = orc.Tape(seed=SEED_TAPE + step)
    lo_emu, g_emu = om.grads(batch, tape, emulate_bf16=True)
    eps = eps_block_from_tape(plan, tape.log, batch["has_x2"], batch["has_y"], noisy=True)
    hp = plan.hparams(step=step, beta_pert=anneal_coef(step, 1, 0))
    got = loss_dict(kind, plan.grad_step(batch_fields(kind, batch), hp, eps=eps))
    check_losses(got, lo_emu, TOL_EMU_LOSS, "vs emulating oracle")
    gv = plan.tensor_views(plan.grads, 0)
    for name, g in g_emu.items():
        assert rel_l2(gv[name], g) <= TOL_EMU_GRAD, "grad %s relL2 %.3e" % (name, rel_l2(gv[name], g))
    if step == 0:
        g = golden(kind, case)
        ref = {k[len("loss_train0/"):]: float(g[k]) for k in g.files if k.startswith("loss_train0/")}
        check_losses(got, ref, TOL_REF_LOSS, "vs reference golden")
        # gradient direction agrees with the fp32 reference (bf16 budget: 2e-2 relative L2)
        for name in g_emu:
            gn = float(g["gradnorm0/" + name])
            assert abs(float(gv[name].double().norm()) - gn) <= 2e-2 * gn + 1e-9, name


@pytest.mark.parametrize("kind", KINDS)
def test_second_step_against_reference_weights(kind):
    """Golden step 1 (beta_pert = 1) starts from the reference's own post-step-0 weights."""
    case = "tiny"
    g = golden(kind, case)
    arch, N, _, batch, _, plan = setup(kind, case)
    sd1 = {k[len("sd_after1/"):]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd_after1/")}
    plan.load_state_dict(sd1)
    om = orc.OracleModel(sd1, orc.default_cfg(kind, L=L))
    om.iters = 1
    tape = orc.Tape(seed=SEED_TAPE + 1)
    om.loss(batch, tape, train=True)
    eps = eps_block_from_tape(plan, tape.log, batch["has_x2"], batch["has_y"], noisy=True)
    got = loss_dict(kind, plan.grad_step(batch_fields(kind, batch), plan.hparams(step=1, beta_pert=1.0), eps=eps))
    ref = {k[len("loss_train1/"):]: float(g[k]) for k in g.files if k.startswith("loss_train1/")}
    check_losses(got, ref, TOL_REF_LOSS, "vs reference golden step 1")


@pytest.mark.parametrize("kind", KINDS)
def test_simt_and_tensor_core_mainloops_agree(kind):
    res = {}
    for impl in ("simt", "tc"):
        arch, N, sd, batch, om, plan = setup(kind, "tiny", impl=impl)
        tape = orc.Tape(seed=SEED_TAPE)
        om.loss(batch, tape, train=True)
        eps = eps_block_from_tape(plan, tape.log, batch["has_x2"], batch["has_y"], noisy=True)
        losses = plan.grad_step(batch_fields(kind, batch), plan.hparams(step=0, beta_pert=0.01), eps=eps)
        res[impl] = (losses[0].cpu().clone(), plan.grads[0].cpu().clone())
    assert torch.allclose(res["simt"][0], res["tc"][0], rtol=1e-5, atol=1e-6)
    assert rel_l2(res["tc"][1], res["simt"][1]) < 5e-3


@pytest.mark.parametrize("kind", KINDS)
def test_eval_mode_loss(kind):
    for case in ("tiny", "readme"):
        arch, N, sd, batch, om, plan = setup(kind, case)
        tape = orc.Tape(seed=SEED_TAPE + 100)
        lo = om.loss(batch, tape, train=False, emulate_bf16=True)
        eps = eps_block_from_tape(plan, tape.log, batch["has_x2"], batch["has_y"], noisy=False)
        hp = plan.hparams(step=0, training=False, beta_pert=0.01)
        got = loss_dict(kind, plan.loss_forward(batch_fields(kind, batch), hp, eps=eps))
        check_losses(got, lo, TOL_EMU_LOSS, "eval vs emulating oracle")
        g = golden(kind, case)
        ref = {k[len("loss_eval/"):]: float(g[k]) for k in g.files if k.startswith("loss_eval/")}
        check_losses(got, ref, TOL_REF_LOSS, "eval vs reference golden")


def test_adam_kernel_matches_torch_adam():
    """Same gradients in -> same update out as torch.optim.Adam (lr 5e-4, wd 0.05 coupled)."""
    arch, N, sd, batch, om, plan = setup("drvae", "tiny")
    g = torch.Generator().manual_seed(3)
    params = [p for p in om.sd.values()]
    for t in range(3):
        views = plan.tensor_views(plan.grads, 0)
        for (name, p) in om.sd.items():
            gr = torch.randn(p.shape, generator=g) * 0.1
            p.grad = gr.clone()
            views[name].copy_(gr)
        om.opt.step()
        plan.adam_step(plan.hparams(step=t))
        torch.cuda.synchronize()
        pv = plan.tensor_views(plan.params, 0)
        for name, p in om.sd.items():
            assert torch.allclose(pv[name].cpu(), p.detach(), rtol=2e-5, atol=2e-7), (t, name)


@pytest.mark.parametrize("kind", KINDS)
def test_train_steps_track_the_oracle(kind):
    """Three fused steps (fwd+bwd+Adam).  After each step the GPU's own parameters are read back
    and the oracle evaluates the NEXT loss from them: this checks Adam -> shadow refresh -> next
    forward without accumulating the sign-sensitivity of Adam's first updates."""
    arch, N, sd, batch, om, plan = setup(kind, "tiny")
    for it in range(3):
        cur = plan.state_dict()
        o = orc.OracleModel({k: v.cpu() for k, v in cur.items()}, orc.default_cfg(kind, L=L))
        o.iters = it
        tape = orc.Tape(seed=SEED_TAPE + it)
        lo = o.loss(batch, tape, train=True, emulate_bf16=True)
        eps = eps_block_from_tape(plan, tape.log, batch["has_x2"], batch["has_y"], noisy=True)
        hp = plan.hparams(step=it, beta_pert=anneal_coef(it, 1, 0))
        got = loss_dict(kind, plan.train_step(batch_fields(kind, batch), hp, eps=eps))
        check_losses(got, lo, TOL_EMU_LOSS, "step %d" % it)
        new = plan.state_dict()
        moved = max((new[k] - cur[k]).abs().max().item() for k in new)
        assert 0 < moved <= 2.5 * 5e-4, "Adam step size out of range: %g" % moved


def _margin_ok(proba_ref, pred_gpu, pred_ref, margin):
    p = np.sort(proba_ref, axis=1)
    sure = (p[:, -1] - p[:, -2]) > margin
    return np.array_equal(pred_gpu[sure], pred_ref[sure]), int(sure.sum())


@pytest.mark.parametrize("case", ("tiny", "readme"))
@pytest.mark.parametrize("kind", KINDS)
def test_inference_matches_oracle_and_reference(kind, case):
    """drvae_infer, both arithmetic modes.  Default fp32 path: every output within fp32 rounding of the reference's
    forward() and thresholded predictions IDENTICAL on every row (no margin mask).  bf16 tensor-core path: within the
    bf16 budget of the oracle that emulates its rounding points."""
    arch, N, sd, batch, om, plan = setup(kind, case)
    fr = om.forward(batch["x1"], emulate_bf16=False)
    g = golden(kind, case)
    # ---- fp32 path (default) ----
    res = plan.infer(batch["x1"])
    t32 = dict(rtol=2e-5, atol=2e-6)
    assert torch.allclose(res["z1_mu"][0].cpu(), fr["z1"], **t32)
    assert torch.allclose(res["z1_lv"][0].cpu(), fr["qz1"][1], **t32)
    assert torch.allclose(res["px1_mu"][0].cpu(), fr["x1_rec"], **t32)
    assert torch.allclose(res["px1_sg"][0].cpu(), fr["px1"][1], **t32)
    if kind != "vfae":
        assert torch.allclose(res["z2_mu"][0].cpu(), fr["z2"], **t32)
        assert torch.allclose(res["z2_lv"][0].cpu(), fr["pz2"][1], **t32)
        assert torch.allclose(res["px2_mu"][0].cpu(), fr["x2_pert"], **t32)
        assert torch.allclose(res["px2_sg"][0].cpu(), fr["px2"][1], **t32)
    if kind != "pvae":
        assert (res["proba"][0].cpu() - fr["proba"]).abs().max() < 2e-6
        assert np.array_equal(res["pred"][0].cpu().numpy(), fr["pred"].numpy())
        assert np.array_equal(res["pred"][0].cpu().numpy(), g["fwd/pred"]), "thresholded predictions differ from the reference"
        assert np.abs(res["proba"][0].cpu().numpy() - g["fwd/proba"]).max() < 2e-6
    # ---- bf16 tensor-core path ----
    plan.set_infer_precision(False)
    res = plan.infer(batch["x1"])
    fo = om.forward(batch["x1"], emulate_bf16=True)
    # vs the oracle with the same rounding points: only accumulation order and rare bf16 rounding
    # flips of stored activations differ (one flip of a hidden unit moves an output by ~1e-4)
    tz = dict(rtol=1e-3, atol=5e-4)
    tx = dict(rtol=2e-3, atol=2e-3)
    assert torch.allclose(res["z1_mu"][0].cpu(), fo["z1"], **tz)
    assert torch.allclose(res["z1_lv"][0].cpu(), fo["qz1"][1], **tz)
    assert torch.allclose(res["px1_mu"][0].cpu(), fo["x1_rec"], **tx)
    assert torch.allclose(res["px1_sg"][0].cpu(), fo["px1"][1], **tx)
    if kind != "vfae":
        assert torch.allclose(res["z2_mu"][0].cpu(), fo["z2"], **tz)
        assert torch.allclose(res["px2_mu"][0].cpu(), fo["x2_pert"], **tx)
    if kind != "pvae":
        assert torch.allclose(res["proba"][0].cpu(), fo["proba"], rtol=1e-3, atol=2e-4)
        same, n_sure = _margin_ok(fo["proba"].numpy(), res["pred"][0].cpu().numpy(), fo["pred"].numpy(), 1e-3)
        assert same and n_sure > 0
        assert (res["proba"][0].cpu() - fr["proba"]).abs().max() < 5e-3


def test_ensemble_members_are_independent():
    """Three models with different weights, batches and group mixes in ONE launch sequence give
    exactly what three single-model plans give."""
    kind, case = "drvae", "tiny"
    arch, N = ARCH[case], NROWS[case]
    E = 3
    plan = Plan(kind, L=L, max_batch=N, n_models=E, **arch)
    sds, batches, epss = [], [], []
    x1, x2, y, hx, hy = [], [], [], [], []
    for m in range(E):
        sd = init_state_dict(kind, seed=SEED_MODEL + m, **arch)
        b = orc.synthetic_batch(N, arch["dim_x"], seed=m)
        if m == 1:
            b["has_x2"][:] = 0  # no pairs at all
            b["x2"][:] = 0
        if m == 2:
            b["has_y"][:] = 1  # fully labeled
        plan.load_state_dict(sd, model=m)
        tape = orc.Tape(seed=50 + m)
        orc.OracleModel(sd, orc.default_cfg(kind, L=L)).loss(b, tape, train=True)
        epss.append(eps_block_from_tape(plan, tape.log, b["has_x2"], b["has_y"], noisy=True))
        sds.append(sd)
        batches.append(b)
        for lst, key in ((x1, "x1"), (x2, "x2"), (y, "y"), (hx, "has_x2"), (hy, "has_y")):
            lst.append(b[key])
    hp = plan.hparams(step=1)
    big = dict(x1=torch.stack(x1), x2=torch.stack(x2), y=torch.stack(y), has_x2=torch.stack(hx), has_y=torch.stack(hy))
    losses = plan.grad_step(big, hp, eps=torch.stack(epss)).cpu().clone()
    grads = plan.grads.cpu().clone()
    for m in range(E):
        single = Plan(kind, L=L, max_batch=N, n_models=1, **arch)
        single.load_state_dict(sds[m])
        l1 = single.grad_step(batch_fields(kind, batches[m]), single.hparams(step=1), eps=epss[m]).cpu()
        assert torch.equal(l1[0], losses[m]), m
        assert torch.equal(single.grads[0].cpu(), grads[m]), m
        om = orc.OracleModel(sds[m], orc.default_cfg(kind, L=L))
        om.iters = 1
        tape = orc.Tape(seed=50 + m)
        lo, _ = om.grads(batches[m], tape, emulate_bf16=True)
        check_losses(loss_dict(kind, losses, m), lo, TOL_EMU_LOSS, "ensemble member %d" % m)


EDGE = [
    ("single row", 1, lambda b: None),
    ("no pairs, no labels", 17, lambda b: (b["has_x2"].zero_(), b["has_y"].zero_(), b["x2"].zero_())),
    ("all pairs, all labels", 17, lambda b: (b["has_x2"].fill_(1), b["has_y"].fill_(1))),
    ("one pair only", 9, lambda b: (b["has_x2"].zero_(), b["has_x2"].__setitem__(4, 1))),
    ("ragged 131 rows", 131, lambda b: None),
]


@pytest.mark.parametrize("name,N,edit", EDGE, ids=[e[0] for e in EDGE])
@pytest.mark.parametrize("kind", KINDS)
def test_edge_case_row_groups(kind, name, N, edit):
    arch = ARCH["tiny"]
    sd = init_state_dict(kind, seed=SEED_MODEL, **arch)
    batch = orc.synthetic_batch(N, arch["dim_x"], seed=7)
    edit(batch)
    if kind == "vfae" and int(batch["has_y"].sum()) == 0:
        pytest.skip("the reference divides by Nl = 0 here (VFAE.py:443)")
    om = orc.OracleModel(sd, orc.default_cfg(kind, L=L))
    om.iters = 1
    plan = Plan(kind, L=L, max_batch=160, n_models=1, **arch)  # capacity larger than the batch
    plan.load_state_dict(sd)
    tape = orc.Tape(seed=11)
    lo, g_emu = om.grads(batch, tape, emulate_bf16=True)
    eps = eps_block_from_tape(plan, tape.log, batch["has_x2"], batch["has_y"], noisy=True)
    got = loss_dict(kind, plan.grad_step(batch_fields(kind, batch), plan.hparams(step=1), eps=eps))
    check_losses(got, lo, 5e-5, name)
    gv = plan.tensor_views(plan.grads, 0)
    for k, g in g_emu.items():
        if float(g.norm()) == 0:
            assert float(gv[k].norm()) == 0, k
        else:
            assert rel_l2(gv[k], g) <= 2e-2, "%s grad %s relL2 %.3e" % (name, k, rel_l2(gv[k], g))


def test_philox_noise_statistics_and_determinism():
    arch, N = ARCH["tiny"], 64
    kind = "drvae"
    sd = init_state_dict(kind, seed=SEED_MODEL, **arch)
    batch = orc.synthetic_batch(N, arch["dim_x"])
    plan = Plan(kind, L=L, max_batch=N, n_models=2, **arch)
    for m in range(2):
        plan.load_state_dict(sd, model=m)
    big = {k: torch.stack([v, v]) for k, v in batch_fields(kind, batch).items()}
    l1 = plan.loss_forward(big, plan.hparams(step=3), seed=99).cpu().clone()
    eps, _, _ = plan.debug_buffer("eps")
    # latent draws live in the eps block; the input noise of x1 / x2 is drawn inside prep_kernel (same generator, never
    # stored) and is recovered here from the noisy fp32 targets: tgt = x + noise_std * eps
    e_lat = eps[:, plan.eps_layout.off_z1:].cpu().clone()
    tg, _, _ = plan.debug_buffer("tgt4")
    Xc = (arch["dim_x"] + 1 + 15) // 16 * 16
    R0cap = tg.shape[1] // Xc
    t = tg.reshape(2, Xc // 4, R0cap, 4).permute(0, 2, 1, 3).reshape(2, R0cap, Xc)[:, :N, :arch["dim_x"]].cpu()
    e_x = (t - batch["x1"][None]) / 0.01
    assert not torch.equal(e_x[0], e_x[1])
    assert abs(float(e_x.mean())) < 0.03 and abs(float(e_x.std()) - 1.0) < 0.03, (float(e_x.mean()), float(e_x.std()))
    e = e_lat
    l2 = plan.loss_forward(big, plan.hparams(step=3), seed=99).cpu().clone()
    assert torch.equal(l1, l2), "same (seed, step) must give the same noise"
    l3 = plan.loss_forward(big, plan.hparams(step=4), seed=99).cpu().clone()
    assert not torch.equal(l1, l3)
    assert not torch.equal(l1[0], l1[1]), "ensemble members draw different noise"
    assert abs(float(e.mean())) < 0.01 and abs(float(e.std()) - 1.0) < 0.01
    assert float(e.abs().max()) < 7.0
    k = float(((e - e.mean()) ** 4).mean() / e.var() ** 2)
    assert abs(k - 3.0) < 0.1, "kurtosis %g" % k


def test_model_class_surface():
    """The reference-facing classes: state_dict keys/order, run_on_batch dictionary, save/load."""
    import os
    import tempfile

    from drvae_b200 import DrVAE, PVAE, VFAE
    a = ARCH["tiny"]
    common = dict(type_rec="diag_gaussian", nonlinearity="elu", L=L, batch_size=24, learning_rate=5e-4, weight_decay=0.05,
                  add_noise_var=0.01, use_MMD=False, random_seed=SEED_MODEL)
    models = {
        "drvae": DrVAE(dim_x=a["dim_x"], dim_s=1, dim_y=2, dim_h_en_z1=a["enc_z1"], dim_h_de_z1=a["dec_z1"], dim_h_en_z2Fz1=[],
                       dim_h_en_z3=a["enc_z3"], dim_h_de_x=a["dec_x"], dim_h_clf=[], dim_z1=a["dim_z1"], dim_z3=a["dim_z3"],
                       pertloss_rate=0.05, **common),
        "pvae": PVAE(dim_x=a["dim_x"], dim_s=1, dim_y=2, dim_h_en_z1=a["enc_z1"], dim_h_en_z2Fz1=[], dim_h_de_x=a["dec_x"],
                     dim_z1=a["dim_z1"], pertloss_rate=0.05, **common),
        "vfae": VFAE(dim_x=a["dim_x"], dim_s=1, dim_y=2, dim_h_en_z1=a["enc_z1"], dim_h_de_z1=a["dec_z1"], dim_h_en_z2=a["enc_z3"],
                     dim_h_de_x=a["dec_x"], dim_h_clf=[], dim_z1=a["dim_z1"], dim_z2=a["dim_z3"], semi_supervised=True, **common),
    }
    batch = orc.synthetic_batch(24, a["dim_x"])
    for kind, model in models.items():
        g = golden(kind, "tiny")
        ref_keys = [k[3:] for k in g.files if k.startswith("sd/")]
        sd = model.state_dict()
        assert list(sd.keys()) == ref_keys
        for k in ref_keys:  # same seed -> same initial weights as the reference
            assert np.array_equal(sd[k].cpu().numpy(), g["sd/" + k]), k
        kw = dict(x1=batch["x1"], s=batch["s"])
        if kind != "vfae":
            kw.update(x2=batch["x2"], has_x2=batch["has_x2"])
        if kind != "pvae":
            kw.update(y=batch["y"], has_y=batch["has_y"])
        model.add_noise = True
        # parity through the public API with an injected tape (golden step 0 of the reference)
        draws = [torch.from_numpy(g[k]) for k in sorted(f for f in g.files if f.startswith("tape0/"))]
        model.set_eps_tape(draws)
        losses = model.run_on_batch(train_mode=True, **kw)
        want = [k for k in LOSS_KEYS if not (kind == "pvae" and k == "YL") and not (kind == "vfae" and k == "PERT")]
        assert list(losses.keys()) == want
        for k in want:
            if k != "MMD":
                ref = float(g["loss_train0/" + k])
                assert abs(float(losses[k]) - ref) <= TOL_REF_LOSS * abs(ref) + 1e-6, (kind, k)
        assert model.finished_training_iters == 1
        ev = model.run_on_batch(train_mode=False, **kw)
        assert set(ev.keys()) == set(want) and all(np.isfinite(float(v)) for v in ev.values())
        out = model.forward(batch["x1"])
        assert out["x1_rec"].shape == (24, a["dim_x"])
        with tempfile.TemporaryDirectory() as d:
            f = os.path.join(d, "m.pth")
            model.save_to_file(f)
            before = {k: v.clone() for k, v in model.state_dict().items()}
            model.run_on_batch(train_mode=True, **kw)
            model.load_params_from_file(f)
            for k, v in model.state_dict().items():
                assert torch.equal(v, before[k])
            ev2 = model.run_on_batch(train_mode=False, **kw)
            assert np.isfinite(float(ev2["CMPL"]))


@pytest.mark.parametrize("case", ("tiny", "deep", "readme"))
@pytest.mark.parametrize("kind", KINDS)
def test_fused_adam_equals_grad_then_adam(kind, case):
    """drvae_train_step applies Adam inside the grouped weight-gradient launch (the gradient never reaches
    HBM); drvae_grad_step + drvae_adam_step materialise it and run the stand-alone optimizer kernel.
    Same gradients, same formula: parameters, moments and the refreshed bf16 shadows must agree."""
    res = {}
    for mode in ("fused", "split"):
        arch, N, sd, batch, om, plan = setup(kind, case)
        out = []
        for it in range(2):
            tape = orc.Tape(seed=SEED_TAPE + it)
            om.iters = it
            om.loss(batch, tape, train=True)
            eps = eps_block_from_tape(plan, tape.log, batch["has_x2"], batch["has_y"], noisy=True)
            hp = plan.hparams(step=it, beta_pert=anneal_coef(it, 1, 0))
            if mode == "fused":
                lo = plan.train_step(batch_fields(kind, batch), hp, eps=eps).cpu().clone()
            else:
                lo = plan.grad_step(batch_fields(kind, batch), hp, eps=eps).cpu().clone()
                plan.adam_step(hp)
            out.append(lo)
        sh, _, _ = plan.debug_buffer("shadow", torch.bfloat16)
        dv, _, _ = plan.debug_buffer("derived")
        res[mode] = (out, plan.params.cpu().clone(), plan.adam_m.cpu().clone(), plan.adam_v.cpu().clone(),
                     sh.float().cpu().clone(), dv.cpu().clone())
    f, s = res["fused"], res["split"]
    assert torch.equal(f[0][0], s[0][0]), "first-step losses differ"
    for i, name in ((1, "params"), (2, "adam_m"), (3, "adam_v")):
        assert torch.allclose(f[i], s[i], rtol=1e-6, atol=1e-9), name
    assert rel_l2(f[4], s[4]) < 1e-4 and rel_l2(f[5], s[5]) < 1e-6, "shadow / derived copies differ"
    assert torch.allclose(f[0][1], s[0][1], rtol=1e-5, atol=1e-6), "second-step losses differ"


@pytest.mark.parametrize("kind", KINDS)
def test_weight_norm_parity(kind):
    """layers.WeightNormLinear (reference layers.py:25-41): parameters (v, g, b), effective weight
    g v / ||v||.  Golden recorded from the reference built with wn=True and perturbed g."""
    case = "tiny_wn"
    g = golden(kind, case)
    arch, N = ARCH[case], NROWS[case]
    sd = {k[3:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd/")}
    assert any(k.endswith(".g") for k in sd)
    batch = orc.synthetic_batch(N, arch["dim_x"])
    plan = Plan(kind, L=L, max_batch=N, n_models=1, weight_norm=True, **arch)
    assert [t[0] for t in plan.tensors] == list(sd.keys())
    plan.load_state_dict(sd)
    om = orc.OracleModel(sd, orc.default_cfg(kind, L=L))
    tape = orc.Tape(seed=SEED_TAPE)
    lo_emu, g_emu = om.grads(batch, tape, emulate_bf16=True)
    eps = eps_block_from_tape(plan, tape.log, batch["has_x2"], batch["has_y"], noisy=True)
    hp = plan.hparams(step=0, beta_pert=anneal_coef(0, 1, 0))
    got = loss_dict(kind, plan.grad_step(batch_fields(kind, batch), hp, eps=eps))
    check_losses(got, lo_emu, TOL_EMU_LOSS, "wn vs emulating oracle")
    ref = {k[len("loss_train0/"):]: float(g[k]) for k in g.files if k.startswith("loss_train0/")}
    # this tiny model with randomly perturbed g is not a BASELINE config: its KL terms are more sensitive to the
    # bf16 rounding of the (rescaled) weights than the 1e-3 budget of the shipped configs; the emulating oracle above
    # holds the kernel logic to 2e-5
    check_losses(got, ref, 5e-3, "wn vs reference golden")
    gv = plan.tensor_views(plan.grads, 0)
    for name, gr in g_emu.items():
        assert rel_l2(gv[name], gr) <= 2e-2, "wn grad %s relL2 %.3e" % (name, rel_l2(gv[name], gr))
        gn = float(g["gradnorm0/" + name])
        assert abs(float(gv[name].double().norm()) - gn) <= 3e-2 * gn + 1e-9, name
    # optimizer steps act on (v, g, b); the next forward must see the refreshed effective weights
    for it in range(2):
        cur = plan.state_dict()
        o = orc.OracleModel({k: v.cpu() for k, v in cur.items()}, orc.default_cfg(kind, L=L))
        o.iters = it
        tape = orc.Tape(seed=SEED_TAPE + 10 + it)
        lo = o.loss(batch, tape, train=True, emulate_bf16=True)
        eps = eps_block_from_tape(plan, tape.log, batch["has_x2"], batch["has_y"], noisy=True)
        got = loss_dict(kind, plan.train_step(batch_fields(kind, batch), plan.hparams(step=it, beta_pert=anneal_coef(it, 1, 0)), eps=eps))
        check_losses(got, lo, TOL_EMU_LOSS, "wn step %d" % it)
        new = plan.state_dict()
        assert all(torch.isfinite(v).all() for v in new.values())
        assert max((new[k] - cur[k]).abs().max().item() for k in new if k.endswith(".g")) > 0
    res = plan.infer(batch["x1"])
    fo = orc.OracleModel({k: v.cpu() for k, v in plan.state_dict().items()}, orc.default_cfg(kind, L=L)).forward(batch["x1"], emulate_bf16=True)
    assert torch.allclose(res["z1_mu"][0].cpu(), fo["z1"], rtol=1e-3, atol=5e-4)
    if kind != "pvae":
        assert torch.allclose(res["proba"][0].cpu(), fo["proba"], rtol=1e-3, atol=2e-4)


@pytest.mark.parametrize("kind", KINDS)
def test_row_shards_with_global_counts_add_up(kind):
    """Data-parallel contract (SURVEY.md 8(e)): a minibatch split into row shards, each given the GLOBAL
    normalisers and the global index of its first row (Philox noise is keyed by global row), produces additive
    shares of every loss term and of the gradient — independent of how many shards there are."""
    from drvae_b200.dp import local_counts, shard_rows
    arch, N = ARCH["tiny"], 48
    sd = init_state_dict(kind, seed=SEED_MODEL, **arch)
    batch = orc.synthetic_batch(N, arch["dim_x"], seed=3)
    fields = batch_fields(kind, batch)
    full = Plan(kind, L=L, max_batch=N, n_models=1, **arch)
    full.load_state_dict(sd)
    lf = full.grad_step(fields, full.hparams(step=2), seed=1234).cpu().clone()
    gf = full.grads[0].cpu().clone()
    counts = local_counts(N, batch.get("has_x2") if kind != "vfae" else None, batch.get("has_y") if kind != "pvae" else None)
    for world in (2, 3):
        lsum, gsum = torch.zeros(8), torch.zeros_like(gf)
        for r in range(world):
            lo, hi = shard_rows(N, world, r)
            shard = {k: v[lo:hi].contiguous() for k, v in fields.items()}
            p = Plan(kind, L=L, max_batch=hi - lo, n_models=1, **arch)
            p.load_state_dict(sd)
            l = p.grad_step(shard, p.hparams(step=2, global_counts=counts), seed=1234, row_offset=lo).cpu()
            lsum += l[0]
            gsum += p.grads[0].cpu()
            if r == 0:
                # the same normalisers handed over in device memory (what dp.py's all-reduce leaves behind): bit-identical
                dev_counts = torch.tensor(counts, dtype=torch.int64, device="cuda")
                l2 = p.grad_step(shard, p.hparams(step=2, global_counts=dev_counts), seed=1234, row_offset=lo).cpu()
                assert torch.equal(l2, l)
                assert torch.equal(p.grads[0].cpu(), gsum)
        for i, k in enumerate(LOSS_KEYS):
            assert abs(float(lsum[i]) - float(lf[0, i])) <= 2e-5 * abs(float(lf[0, i])) + 1e-5, (world, k, float(lsum[i]), float(lf[0, i]))
        assert rel_l2(gsum, gf) < 2e-3, (world, rel_l2(gsum, gf))


@pytest.mark.parametrize("kind", KINDS)
def test_large_batch_split_k_matches_oracle(kind):
    """Single model, large minibatch (BASELINE configs[3] regime): weight gradients run split-K with atomic
    accumulation into a zeroed gradient buffer; train_step falls back from the fused epilogue to gradient +
    stand-alone Adam.  Checked against the emulating oracle and against two fused-regime half batches."""
    arch, N = ARCH["tiny"], 1536
    sd = init_state_dict(kind, seed=SEED_MODEL, **arch)
    batch = orc.synthetic_batch(N, arch["dim_x"], seed=5)
    om = orc.OracleModel(sd, orc.default_cfg(kind, L=L))
    om.iters = 1
    tape = orc.Tape(seed=21)
    lo_emu, g_emu = om.grads(batch, tape, emulate_bf16=True)
    plan = Plan(kind, L=L, max_batch=N, n_models=1, **arch)
    plan.load_state_dict(sd)
    eps = eps_block_from_tape(plan, tape.log, batch["has_x2"], batch["has_y"], noisy=True)
    got = loss_dict(kind, plan.grad_step(batch_fields(kind, batch), plan.hparams(step=1), eps=eps))
    check_losses(got, lo_emu, 5e-5, "large batch")
    gv = plan.tensor_views(plan.grads, 0)
    for name, g in g_emu.items():
        assert rel_l2(gv[name], g) <= 1e-2, "grad %s relL2 %.3e" % (name, rel_l2(gv[name], g))
    # a second call must not accumulate on top of the first (the buffer is re-zeroed)
    g1 = plan.grads.clone()
    plan.grad_step(batch_fields(kind, batch), plan.hparams(step=1), eps=eps)
    assert rel_l2(plan.grads, g1) < 1e-5
    before = plan.params.clone()
    out = loss_dict(kind, plan.train_step(batch_fields(kind, batch), plan.hparams(step=1), eps=eps))
    check_losses(out, lo_emu, 5e-5, "large batch train_step")
    moved = (plan.params - before).abs().max().item()
    assert 0 < moved <= 2.5 * 5e-4


@pytest.mark.parametrize("kind,dim_y,Lmc", [("drvae", 3, 1), ("vfae", 4, 3), ("drvae", 2, 3), ("pvae", 2, 1)])
def test_other_class_counts_and_sample_counts(kind, dim_y, Lmc):
    """dim_y > 2 (unlabeled rows are marginalised over every class, DrVAE.py:516-526) and L != 2."""
    arch = dict(ARCH["tiny"], dim_y=dim_y)
    N = 30
    sd = init_state_dict(kind, seed=SEED_MODEL, **arch)
    batch = orc.synthetic_batch(N, arch["dim_x"], seed=11, dim_y=dim_y)
    cfg = orc.default_cfg(kind, L=Lmc, dim_y=dim_y)
    om = orc.OracleModel(sd, cfg)
    om.iters = 1
    tape = orc.Tape(seed=31)
    lo_emu, g_emu = om.grads(batch, tape, emulate_bf16=True)
    plan = Plan(kind, L=Lmc, max_batch=N, n_models=1, **arch)
    plan.load_state_dict(sd)
    eps = eps_block_from_tape(plan, tape.log, batch["has_x2"], batch["has_y"], noisy=True)
    got = loss_dict(kind, plan.grad_step(batch_fields(kind, batch), plan.hparams(step=1), eps=eps))
    check_losses(got, lo_emu, 5e-5, "dim_y=%d L=%d" % (dim_y, Lmc))
    gv = plan.tensor_views(plan.grads, 0)
    for name, g in g_emu.items():
        assert rel_l2(gv[name], g) <= 2e-2, "grad %s relL2 %.3e" % (name, rel_l2(gv[name], g))
    if kind != "pvae":
        res = plan.infer(batch["x1"])
        fr = om.forward(batch["x1"], emulate_bf16=False)
        assert res["proba"].shape[-1] == dim_y
        assert torch.allclose(res["proba"][0].cpu(), fr["proba"], rtol=1e-4, atol=2e-6)
        assert np.array_equal(res["pred"][0].cpu().numpy(), fr["pred"].numpy())


def test_argument_errors_are_reported_not_crashed():
    """Error convention of the C ABI: non-zero status + message, surfaced as RuntimeError / ValueError."""
    arch, N = ARCH["tiny"], 8
    plan = Plan("drvae", L=1, max_batch=N, n_models=1, **arch)
    b = orc.synthetic_batch(N + 1, arch["dim_x"])
    with pytest.raises(RuntimeError, match="max_batch"):
        plan.grad_step(batch_fields("drvae", b), plan.hparams(step=0))
    b = orc.synthetic_batch(N, arch["dim_x"] + 1)
    with pytest.raises(ValueError):
        plan.grad_step(batch_fields("drvae", b), plan.hparams(step=0))
    with pytest.raises(RuntimeError):
        Plan("drvae", L=1, max_batch=N, n_models=1, **dict(arch, dim_y=9))
    from drvae_b200 import DrVAE
    with pytest.raises(ValueError, match="use_s"):
        DrVAE(dim_x=10, dim_s=1, dim_y=2, type_rec="diag_gaussian", nonlinearity="elu", use_s=True)


@pytest.mark.parametrize("kind", KINDS)
def test_graph_replay_equals_plain_launches(kind):
    """drvae_train_step replays its launch sequence as a CUDA graph from the third call on (per-step scalars live
    in device memory).  Same seeds, same batches: parameters after 6 steps must be identical to the plan that
    launches kernel by kernel, and both must equal the oracle-tracked behaviour checked elsewhere."""
    arch, N = ARCH["tiny"], 40
    sd = init_state_dict(kind, seed=SEED_MODEL, **arch)
    batch = {k: v.cuda() for k, v in batch_fields(kind, orc.synthetic_batch(N, arch["dim_x"], seed=2)).items()}
    res = {}
    for mode in ("graph", "plain"):
        plan = Plan(kind, L=L, max_batch=N, n_models=2, **arch)
        plan.set_graph(mode == "graph")
        for m in range(2):
            plan.load_state_dict(sd, model=m)
        big = {k: torch.stack([v, v]).contiguous() for k, v in batch.items()}
        losses = []
        for it in range(6):
            out = plan.train_step(big, plan.hparams(step=it, beta_pert=anneal_coef(it, 1, 0)), seed=5)
            losses.append(out.cpu().clone())
        ev = plan.loss_forward(big, plan.hparams(step=6, training=False), seed=5).cpu().clone()
        ev2 = plan.loss_forward(big, plan.hparams(step=7, training=False), seed=5).cpu().clone()
        ev3 = plan.loss_forward(big, plan.hparams(step=7, training=False), seed=5).cpu().clone()
        assert torch.equal(ev2, ev3)
        res[mode] = (losses, plan.params.cpu().clone(), ev, plan.graph_replays())
    assert res["graph"][3] >= 4 and res["plain"][3] == 0, (res["graph"][3], res["plain"][3])
    assert plan.graph_failures() == 0
    for a, b in zip(res["graph"][0], res["plain"][0]):
        assert torch.equal(a, b)
    assert torch.equal(res["graph"][1], res["plain"][1])
    assert torch.equal(res["graph"][2], res["plain"][2])
    # steps differ (noise, Adam bias correction): the dynamic scalars really are updated under replay
    assert not torch.equal(res["graph"][0][3], res["graph"][0][4])


@pytest.mark.parametrize("kind", KINDS)
def test_odd_dimensions(kind):
    """Nothing in the layouts may assume even / multiple-of-4 feature counts (978 = 2 * 489 is even, but the
    reference accepts any --dim-z1 / --enc-z1 ...): odd sizes everywhere, Philox noise and tape noise."""
    arch = dict(dim_x=37, dim_y=3, dim_z1=13, dim_z3=7, enc_z1=[23], dec_x=[19, 21], enc_z3=[11], dec_z1=[9])
    N = 29
    sd = init_state_dict(kind, seed=SEED_MODEL, **arch)
    batch = orc.synthetic_batch(N, arch["dim_x"], seed=13, dim_y=3)
    om = orc.OracleModel(sd, orc.default_cfg(kind, L=L, dim_y=3))
    om.iters = 1
    tape = orc.Tape(seed=41)
    lo_emu, g_emu = om.grads(batch, tape, emulate_bf16=True)
    plan = Plan(kind, L=L, max_batch=N + 3, n_models=1, **arch)
    plan.load_state_dict(sd)
    eps = eps_block_from_tape(plan, tape.log, batch["has_x2"], batch["has_y"], noisy=True)
    got = loss_dict(kind, plan.grad_step(batch_fields(kind, batch), plan.hparams(step=1), eps=eps))
    check_losses(got, lo_emu, 5e-5, "odd dims")
    gv = plan.tensor_views(plan.grads, 0)
    for name, g in g_emu.items():
        assert rel_l2(gv[name], g) <= 2e-2, "grad %s relL2 %.3e" % (name, rel_l2(gv[name], g))
    # Philox path: finite, deterministic, and training moves the loss
    fields = {k: v.cuda() for k, v in batch_fields(kind, batch).items()}
    first = None
    for it in range(8):
        out = plan.train_step(fields, plan.hparams(step=it, beta_pert=anneal_coef(it, 1, 0), lr=2e-3), seed=3).cpu()
        assert torch.isfinite(out).all()
        first = out.clone() if it == 1 else first
    assert float(out[0, 6]) < float(first[0, 6])


@pytest.mark.gpu
def test_data_parallel_graph_replay_equals_eager():
    """On one rank drvae_b200.dp runs drvae_dp_train_step, which the plan captures as one CUDA graph and replays with the
    per-step scalars updated in its set_dyn node.  Same trajectory as launching kernel by kernel."""
    from drvae_b200 import dp as dpm
    arch, N = ARCH["tiny"], 64
    sd = init_state_dict("drvae", seed=SEED_MODEL, **arch)
    batch = orc.synthetic_batch(N, arch["dim_x"], seed=9)
    fields = {k: v.cuda() for k, v in batch_fields("drvae", batch).items()}
    host = {k: batch[k] for k in ("has_x2", "has_y")}
    out = {}
    for mode in (False, True):
        plan = Plan("drvae", L=L, max_batch=N, n_models=1, **arch)
        plan.load_state_dict(sd)
        plan.set_graph(mode)
        runner = dpm.DataParallel(dpm.PlanBackend(plan))
        losses = []
        for it in range(7):
            res = runner.step(fields, hp_kwargs=dict(beta_pert=anneal_coef(it, 1, 0)), seed=5, host_flags=host)
            losses.append(res.detach().cpu().clone())
        out[mode] = (torch.stack(losses), plan.params.cpu().clone())
        if mode:
            assert plan.graph_replays() > 0 and plan.graph_failures() == 0  # captured on the second step, replayed afterwards
    assert torch.equal(out[False][0], out[True][0])
    assert torch.equal(out[False][1], out[True][1])
    assert not torch.equal(out[True][0][3], out[True][0][4])  # the pushed scalars really change between replays


@pytest.mark.parametrize("kind", ("drvae", "vfae"))
def test_side_stream_delay_does_not_change_results(kind):
    """The label-dependent branch runs on the plan's side stream.  clf_back (main stream) consumes the per-class KL
    terms pz1_post (side stream) writes; holding the side stream for ~1.5 ms in front of pz1_post must not change a
    single bit of the result — a missing cross-stream dependency would (round-1 ADVICE, plan.cu clf_bwd)."""
    arch, N = ARCH["tiny"], 40
    sd = init_state_dict(kind, seed=SEED_MODEL, **arch)
    batch = {k: v.cuda() for k, v in batch_fields(kind, orc.synthetic_batch(N, arch["dim_x"], seed=4)).items()}
    res = {}
    for delay in (0, 3_000_000):
        plan = Plan(kind, L=L, max_batch=N, n_models=2, **arch)
        plan.debug_side_delay(delay)
        for m in range(2):
            plan.load_state_dict(sd, model=m)
        big = {k: torch.stack([v, v]).contiguous() for k, v in batch.items()}
        out = []
        for it in range(4):  # plain launches, then (from the third call) the captured graph
            out.append(plan.train_step(big, plan.hparams(step=it, beta_pert=anneal_coef(it, 1, 0)), seed=7).cpu().clone())
        res[delay] = (torch.stack(out), plan.params.cpu().clone())
    assert torch.equal(res[0][0], res[3_000_000][0])
    assert torch.equal(res[0][1], res[3_000_000][1])


@pytest.mark.parametrize("path", ("fused", "split"))
def test_pvae_without_pairs_leaves_the_perturbation_block_untouched(path):
    """PVAE uses p(z2|z1) only for pair rows (PVAE.py:313-330).  On a batch without pairs the reference's gradient of
    decoder_z2Fz1 is None, so torch.optim.Adam skips those tensors entirely (no weight decay, no moment update);
    every other tensor takes a normal step.  Both optimizer paths must do the same."""
    kind, arch, N = "pvae", ARCH["tiny"], 20
    sd = init_state_dict(kind, seed=SEED_MODEL, **arch)
    batch = orc.synthetic_batch(N, arch["dim_x"], seed=6)
    batch["has_x2"].zero_()
    batch["x2"].zero_()
    plan = Plan(kind, L=L, max_batch=N, n_models=1, **arch)
    plan.load_state_dict(sd)
    om = orc.OracleModel(sd, orc.default_cfg(kind, L=L))
    for it in range(2):
        tape = orc.Tape(seed=60 + it)
        om.step(batch, tape)
        eps = eps_block_from_tape(plan, tape.log, batch["has_x2"], None, noisy=True)
        hp = plan.hparams(step=it, beta_pert=anneal_coef(it, 1, 0))
        if path == "fused":
            plan.train_step(batch_fields(kind, batch), hp, eps=eps)
        else:
            plan.grad_step(batch_fields(kind, batch), hp, eps=eps)
            plan.adam_step(hp)
    new, ref = plan.state_dict(), om.state_dict()
    mv, vv = plan.tensor_views(plan.adam_m, 0), plan.tensor_views(plan.adam_v, 0)
    for k in new:
        if k.startswith("decoder_z2Fz1"):
            assert torch.equal(ref[k], sd[k]), "oracle moved %s" % k
            assert torch.equal(new[k].cpu(), sd[k]), k
            assert float(mv[k].abs().max()) == 0 and float(vv[k].abs().max()) == 0, k
        else:
            assert not torch.equal(new[k].cpu(), sd[k]), k
            assert (new[k].cpu() - ref[k]).abs().max() <= 2.2 * 5e-4, k  # two Adam steps of lr 5e-4, signs may differ


@pytest.mark.parametrize("kind", KINDS)
def test_device_resident_dataset_indexing_equals_gathered_batches(kind):
    """drvae_batch_t.row_index: the minibatch as indices into datasets that stay on the device (what the reference's
    fit() does on the host with a sampler + DataLoader) gives bit-identical steps to passing the gathered rows."""
    arch, D, N, E = ARCH["tiny"], 90, 24, 2
    sd = init_state_dict(kind, seed=SEED_MODEL, **arch)
    data = [batch_fields(kind, orc.synthetic_batch(D, arch["dim_x"], seed=30 + m)) for m in range(E)]
    dataset = {k: torch.stack([d[k] for d in data]).contiguous().cuda() for k in data[0]}
    gen = torch.Generator().manual_seed(1)
    res = {}
    for mode in ("indexed", "gathered"):
        plan = Plan(kind, L=L, max_batch=N, n_models=E, **arch)
        for m in range(E):
            plan.load_state_dict(sd, model=m)
        gen.manual_seed(1)
        idx_buf = torch.zeros(E, N, dtype=torch.int32, device="cuda")
        out = []
        for it in range(5):
            idx = torch.stack([torch.randperm(D, generator=gen)[:N] for _ in range(E)]).int()
            hp = plan.hparams(step=it, beta_pert=anneal_coef(it, 1, 0))
            if mode == "indexed":
                idx_buf.copy_(idx)  # same device buffer every step: the captured graph is replayed
                out.append(plan.train_step(dict(dataset, row_index=idx_buf), hp, seed=3).cpu().clone())
            else:
                b = {k: torch.stack([v[m][idx[m].long().cuda()] for m in range(E)]).contiguous() for k, v in dataset.items()}
                out.append(plan.train_step(b, hp, seed=3).cpu().clone())
        res[mode] = (torch.stack(out), plan.params.cpu().clone())
        if mode == "indexed":
            assert plan.graph_replays() >= 2
    assert torch.equal(res["indexed"][0], res["gathered"][0])
    assert torch.equal(res["indexed"][1], res["gathered"][1])


@pytest.mark.parametrize("N", (511, 512))
def test_both_sides_of_the_fused_optimizer_threshold(N):
    """drvae_train_step fuses Adam into the weight-gradient launch below N * L = 1024 rows (single model) and switches to
    split-K gradients + the stand-alone optimizer from there on (plan.cu train_is_fused).  One row below and exactly at
    the threshold: same losses as the emulating oracle, and after the step the parameters of the two regimes agree
    with what gradient + drvae_adam_step gives."""
    kind, arch = "drvae", ARCH["tiny"]
    sd = init_state_dict(kind, seed=SEED_MODEL, **arch)
    batch = orc.synthetic_batch(N, arch["dim_x"], seed=8)
    om = orc.OracleModel(sd, orc.default_cfg(kind, L=L))
    om.iters = 1
    tape = orc.Tape(seed=17)
    lo_emu, _ = om.grads(batch, tape, emulate_bf16=True)
    res = []
    for mode in ("train", "split"):
        plan = Plan(kind, L=L, max_batch=N, n_models=1, **arch)
        plan.load_state_dict(sd)
        eps = eps_block_from_tape(plan, tape.log, batch["has_x2"], batch["has_y"], noisy=True)
        hp = plan.hparams(step=1)
        if mode == "train":
            out = plan.train_step(batch_fields(kind, batch), hp, eps=eps)
        else:
            out = plan.grad_step(batch_fields(kind, batch), hp, eps=eps)
            plan.adam_step(hp)
        check_losses(loss_dict(kind, out), lo_emu, 5e-5, "N=%d %s" % (N, mode))
        res.append(plan.params.cpu().clone())
    assert torch.allclose(res[0], res[1], rtol=1e-5, atol=2e-7)
    assert not torch.equal(res[0], torch.zeros_like(res[0]))


@pytest.mark.parametrize("arch_name", ("tiny", "deep"))
@pytest.mark.parametrize("kind", KINDS)
def test_step_kernel_equals_one_launch_per_operation(kind, arch_name):
    """The persistent step kernel (stepk.cuh) runs the recorded forward + input-gradient chain as one cooperative launch
    with grid barriers between dependent levels.  Same device code per item, so: bit-identical losses, parameters and
    eval-mode losses to the schedule that launches every GEMM / row operation separately — for the fused train step,
    the gradient + stand-alone optimizer path (split-K weight gradients inside the chain) and the loss-only pass."""
    arch, N, E = ARCH[arch_name], 40, 3
    sds = [init_state_dict(kind, seed=SEED_MODEL + m, **arch) for m in range(E)]
    batches = [batch_fields(kind, orc.synthetic_batch(N, arch["dim_x"], seed=20 + m)) for m in range(E)]
    big = {k: torch.stack([b[k] for b in batches]).contiguous().cuda() for k in batches[0]}
    res = {}
    for mode in (True, False):
        plan = Plan(kind, L=L, max_batch=N, n_models=E, **arch)
        plan.set_step_kernel(mode)
        for m in range(E):
            plan.load_state_dict(sds[m], model=m)
        losses = []
        for it in range(5):
            losses.append(plan.train_step(big, plan.hparams(step=it, beta_pert=anneal_coef(it, 1, 0)), seed=9).cpu().clone())
        g = plan.grad_step(big, plan.hparams(step=5), seed=9).cpu().clone()
        grads = plan.grads.cpu().clone()
        plan.adam_step(plan.hparams(step=5))
        ev = plan.loss_forward(big, plan.hparams(step=6, training=False), seed=9).cpu().clone()
        torch.cuda.synchronize()
        res[mode] = (losses, plan.params.cpu().clone(), g, grads, ev, plan.step_kernel_launches())
    assert res[True][5] >= 1 and res[False][5] == 0, (res[True][5], res[False][5])  # (graph replays are not counted; the deep gradient path exceeds the op table and falls back)
    for a, b in zip(res[True][0], res[False][0]):
        assert torch.equal(a, b)
    assert torch.equal(res[True][1], res[False][1])
    assert torch.equal(res[True][2], res[False][2])
    assert torch.equal(res[True][3], res[False][3])
    assert torch.equal(res[True][4], res[False][4])
    assert bool(torch.isfinite(res[True][1]).all())


@pytest.mark.parametrize("kind", ("drvae", "vfae"))
def test_early_part_of_the_grouped_optimizer_launch_changes_nothing(kind, monkeypatch):
    """The decoder heads' weight-gradient + Adam tiles start right after the decoder dX GEMM on a subset of the SMs,
    next to the rest of the backward chain, whose persistent GEMMs are capped to the other SMs (plan.cu, dwa_early).
    Same tiles, different launch grids and timing: losses and parameters must be bit-identical to the single launch at the
    end of backward (DRVAE_B200_DWA_EARLY_SMS=0), under graph replay as well."""
    arch, N, E = ARCH["tiny"], 40, 4
    sds = [init_state_dict(kind, seed=SEED_MODEL + m, **arch) for m in range(E)]
    batches = [batch_fields(kind, orc.synthetic_batch(N, arch["dim_x"], seed=30 + m)) for m in range(E)]
    big = {k: torch.stack([b[k] for b in batches]).contiguous().cuda() for k in batches[0]}
    res = {}
    for sms in ("0", "92", "16"):
        monkeypatch.setenv("DRVAE_B200_DWA_EARLY_SMS", sms)
        plan = Plan(kind, L=L, max_batch=N, n_models=E, **arch)
        for m in range(E):
            plan.load_state_dict(sds[m], model=m)
        l0 = plan.launch_count()
        losses = [plan.train_step(big, plan.hparams(step=it, beta_pert=anneal_coef(it, 1, 0)), seed=4).cpu().clone() for it in range(6)]
        torch.cuda.synchronize()
        res[sms] = (losses, plan.params.cpu().clone(), plan.adam_v.cpu().clone(), (plan.launch_count() - l0) // 6, plan.graph_replays())
    assert res["92"][3] == res["0"][3] + 1  # one more launch per step: the early part
    assert res["92"][4] >= 3
    for sms in ("92", "16"):
        for a, b in zip(res["0"][0], res[sms][0]):
            assert torch.equal(a, b)
        assert torch.equal(res["0"][1], res[sms][1]) and torch.equal(res["0"][2], res[sms][2])
