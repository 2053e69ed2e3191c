"""CPU: classifier hidden layers (dim_h_clf, --class-y) — the C entry point and its argument checks, the parameter
layout, the restated classifier against an independent torch composition, the model classes and the CLI.

The oracle restates the classifier without hidden layers only.  `categorical` below is the classifier with them,
composed from the oracle's own pieces (`mlp` for blocks.MLP, then linear_p in fp32), and `classifier_oracle` runs the
oracle with it in place of its own; the GPU tests (test_clf_hidden_gpu.py) take both from here.  Without hidden layers
it is the oracle's classifier exactly.  The composition is not pinned by a reference golden file (each piece is,
elsewhere): parity with the reference for --class-y is inferred."""
import contextlib
import ctypes
import os
import re

import pytest
import torch
import torch.nn.functional as F

from helpers import ROOT, orc

from drvae_b200 import _lib, cli
from drvae_b200.init import init_state_dict

ARCH = dict(dim_x=40, dim_y=2, dim_z1=12, dim_z3=10, enc_z1=[24], dec_x=[28], enc_z3=[20], dec_z1=[18])


def categorical(ops, sd, prefix, u):
    """CategoricalDecoder (blocks.py:456-463): blocks.MLP (dim_h_clf, ELU) then linear_p, softmax, clamp.  linear_p is
    fp32 in both modes, as in the oracle.  The hidden layers go through `ops` like every other MLP of the oracle, so
    with emulate_bf16 they round where the kernels store: u at the first GEMM, the activations H and the pre-activation
    gradients.  Without hidden layers the MLP is the identity and nothing is rounded."""
    h = orc.mlp(ops, sd, prefix, u)
    name = prefix + ".decoder_p.linear_p"
    W, b = sd[name + ".weight"], sd[name + ".bias"]
    s = orc._wn_scale(sd, name)
    if s is not None:
        W = W * s[:, None]
    ps = F.softmax(F.linear(h, W, b), dim=-1)
    return torch.clamp(ps, min=1e-10, max=1.0 - 1e-10)


@contextlib.contextmanager
def classifier_oracle(emulate_bf16):
    """Oracle calls inside this block evaluate q(y|.) with `categorical` above; pass the emulate_bf16 of those calls."""
    own = orc.categorical
    ops = orc.Ops(emulate_bf16)
    orc.categorical = lambda sd, prefix, u: categorical(ops, sd, prefix, u)
    try:
        yield
    finally:
        orc.categorical = own


def test_new_entry_point_is_declared_and_exported():
    hdr = open(os.path.join(ROOT, "include", "drvae_b200.h")).read()
    assert re.search(r"^int drvae_plan_create_clf\(const drvae_arch_t\* arch, int n_clf, const int\* clf_hidden, int n_models,",
                     hdr, re.M)
    assert "drvae_plan_create_clf" in _lib.EXPORTS
    assert hasattr(_lib.load(), "drvae_plan_create_clf")


def _create(kind="drvae", widths=()):
    a = _lib.Arch()
    a.kind = dict(drvae=0, pvae=1, vfae=2)[kind]
    a.dim_x, a.dim_y, a.dim_z1, a.dim_z3, a.L, a.max_batch = 40, 2, 12, 10, 1, 16
    for name in ("enc_z1", "dec_x", "enc_z3", "dec_z1"):
        setattr(a, "n_" + name, 1)
        getattr(a, name)[0] = 32
    lib = _lib.load()
    arr = (ctypes.c_int * max(1, len(widths)))(*widths)
    h = ctypes.c_void_p()
    rc = lib.drvae_plan_create_clf(ctypes.byref(a), len(widths), arr, 1, ctypes.byref(h))
    if rc == 0:
        lib.drvae_plan_destroy(h)
    return rc, (lib.drvae_last_error() or b"").decode()


@pytest.mark.parametrize("kind,widths,limit", [
    ("drvae", [8] * 5, "[0, 4]"),
    ("vfae", [8, 0], "[1, 4096]"),
    ("drvae", [4097], "[1, 4096]"),
    ("pvae", [8], "PVAE has no classifier"),
], ids=["n5", "width0", "width4097", "pvae"])
def test_arguments_beyond_the_limits_are_rejected(kind, widths, limit):
    rc, msg = _create(kind, widths)
    assert rc != 0
    assert limit in msg, msg


@pytest.mark.parametrize("kind", ("drvae", "vfae"))
def test_accepted_arguments_pass_the_checks(kind):
    """Without a device the call gets past the argument checks and fails at the first allocation."""
    rc, msg = _create(kind, [8, 16, 24, 4096])
    assert rc == 0 or "cudaMalloc" in msg, msg


def _plan_layout(kind, clf, wn=False):
    """The plan's tensor table (plan.cu add_tensor order, 16-byte aligned rows), restated for the classifier."""
    sd = init_state_dict(kind, seed=1, weight_norm=wn, clf_hidden=clf, **ARCH)
    P = 0
    for name, t in sd.items():
        P = (P + 3) // 4 * 4
        rows, cols = (t.shape[0], t.shape[1]) if t.dim() == 2 else (t.shape[0], 0)
        P += rows * ((cols + 3) // 4 * 4 if cols else 1)
    return sd, (P + 3) // 4 * 4


@pytest.mark.parametrize("kind", ("drvae", "vfae"))
@pytest.mark.parametrize("wn", (False, True))
def test_init_state_dict_order_and_shapes(kind, wn):
    clf = [64, 32]
    sd = init_state_dict(kind, seed=1, weight_norm=wn, clf_hidden=clf, **ARCH)
    keys = [k for k in sd if k.startswith("encoder_y")]
    want = []
    for i in (1, 2):
        want += ["encoder_y.nnet.model.linear%d.%s" % (i, p) for p in (("weight", "bias", "g") if wn else ("weight", "bias"))]
    want += ["encoder_y.decoder_p.linear_p.%s" % p for p in (("weight", "bias", "g") if wn else ("weight", "bias"))]
    assert keys == want
    u = 2 * ARCH["dim_z1"] if kind == "drvae" else ARCH["dim_z1"]
    assert sd["encoder_y.nnet.model.linear1.weight"].shape == (64, u)
    assert sd["encoder_y.nnet.model.linear2.weight"].shape == (32, 64)
    assert sd["encoder_y.decoder_p.linear_p.weight"].shape == (2, 32)
    # the classifier block sits where linear_p sat: the other tensors are unchanged, in the same order
    base = init_state_dict(kind, seed=1, weight_norm=wn, **ARCH)
    assert [k for k in sd if not k.startswith("encoder_y")] == [k for k in base if not k.startswith("encoder_y")]
    # the hidden linears consume the generator before linear_p, as nn.Linear modules created in that order
    torch.manual_seed(1)
    ref = {}
    seen = False
    for k, t in base.items():
        if k.startswith("encoder_y") and not seen:
            seen = True
            for i, (o, n) in enumerate(((64, u), (32, 64))):
                m = torch.nn.Linear(n, o)
                ref["encoder_y.nnet.model.linear%d.weight" % (i + 1)] = m.weight.detach()
                ref["encoder_y.nnet.model.linear%d.bias" % (i + 1)] = m.bias.detach()
            m = torch.nn.Linear(32, 2)
            ref["encoder_y.decoder_p.linear_p.weight"] = m.weight.detach()
            break
        if k.endswith(".weight") and k.replace(".weight", ".bias") in base:
            torch.nn.Linear(t.shape[1], t.shape[0])
        elif k.endswith("W_mu") or k.endswith("bias_mu"):
            torch.Tensor(*t.shape).uniform_(-0.0001, 0.0001)
    for k, t in ref.items():
        assert torch.equal(sd[k], t), k


@pytest.mark.parametrize("kind", ("drvae", "vfae"))
def test_parameter_count_of_the_tensor_table(kind):
    """Parameter count the plan reports for this architecture, restated from its tensor table rules."""
    _, P0 = _plan_layout(kind, [])
    _, P = _plan_layout(kind, [64, 32])
    u = 2 * ARCH["dim_z1"] if kind == "drvae" else ARCH["dim_z1"]
    assert P - P0 == 64 * u + 64 + 32 * 64 + 32 + 2 * 32 - 2 * u


def _reference_classifier(sd, u, wn):
    """nn.Sequential(Linear, ELU, ..., Linear) + softmax + clamp from the same state dict."""
    layers = []
    i = 1
    while "encoder_y.nnet.model.linear%d.weight" % i in sd:
        layers.append(("encoder_y.nnet.model.linear%d" % i, True))
        i += 1
    layers.append(("encoder_y.decoder_p.linear_p", False))
    mods = []
    for name, act in layers:
        W = sd[name + ".weight"]
        if wn:
            W = W * (sd[name + ".g"] / torch.norm(W, 2, 1))[:, None]
        lin = torch.nn.Linear(W.shape[1], W.shape[0]).to(u.dtype)
        with torch.no_grad():
            lin.weight.copy_(W)
            lin.bias.copy_(sd[name + ".bias"])
        mods.append(lin)
        if act:
            mods.append(torch.nn.ELU())
    net = torch.nn.Sequential(*mods)
    return torch.clamp(F.softmax(net(u), dim=-1), 1e-10, 1 - 1e-10), net


@pytest.mark.parametrize("dtype", (torch.float32, torch.float64))
@pytest.mark.parametrize("clf", ([], [16], [64, 32], [8, 16, 24, 8]))
@pytest.mark.parametrize("wn", (False, True))
def test_oracle_classifier_equals_an_independent_composition(dtype, clf, wn):
    sd = {k: v.to(dtype) for k, v in init_state_dict("drvae", seed=3, weight_norm=wn, clf_hidden=clf, **ARCH).items()}
    if wn:
        for k in sd:
            if k.endswith(".g"):
                sd[k] = sd[k] * 1.3
    u = torch.randn(20, 2 * ARCH["dim_z1"], dtype=dtype, generator=torch.Generator().manual_seed(0))
    ref, net = _reference_classifier(sd, u, wn)
    # values
    got = categorical(orc.Ops(False), sd, "encoder_y", u)
    tol = dict(rtol=1e-6, atol=1e-7) if dtype == torch.float32 else dict(rtol=1e-12, atol=1e-14)
    assert torch.allclose(got, ref.detach(), **tol)
    # autograd gradients w.r.t. the input and the parameters (the same upstream gradient through both)
    w = torch.randn(20, 2, dtype=dtype, generator=torch.Generator().manual_seed(1))
    u1 = u.clone().requires_grad_(True)
    sd1 = {k: v.clone().requires_grad_(True) for k, v in sd.items() if k.startswith("encoder_y")}
    (categorical(orc.Ops(False), sd1, "encoder_y", u1) * w).sum().backward()
    u2 = u.clone().requires_grad_(True)
    sd2 = {k: v.clone().requires_grad_(True) for k, v in sd.items() if k.startswith("encoder_y")}
    (_reference_classifier(sd2, u2, wn)[0] * w).sum().backward()
    # the reference net copies W into its modules: its parameter gradients are w.r.t. the effective weights, so compare
    # the input gradient and, without weight norm, the parameter gradients through the same graph
    assert torch.allclose(u1.grad, u2.grad, **tol)
    if not wn:
        _, net2 = _reference_classifier(sd, u, False)
        (torch.clamp(F.softmax(net2(u), -1), 1e-10, 1 - 1e-10) * w).sum().backward()
        lins = [m for m in net2 if isinstance(m, torch.nn.Linear)]
        names = ["encoder_y.nnet.model.linear%d" % (i + 1) for i in range(len(clf))] + ["encoder_y.decoder_p.linear_p"]
        for n, m in zip(names, lins):
            assert torch.allclose(sd1[n + ".weight"].grad, m.weight.grad, **tol), n
            assert torch.allclose(sd1[n + ".bias"].grad, m.bias.grad, **tol), n


def test_the_emulating_oracle_rounds_nothing_without_hidden_layers():
    sd = init_state_dict("vfae", seed=3, **ARCH)
    u = torch.randn(20, ARCH["dim_z1"], generator=torch.Generator().manual_seed(0))
    fn = orc.categorical
    own = fn(sd, "encoder_y", u)
    assert torch.equal(categorical(orc.Ops(True), sd, "encoder_y", u), own)
    assert torch.equal(categorical(orc.Ops(False), sd, "encoder_y", u), own)
    with classifier_oracle(True):
        assert torch.equal(orc.categorical(sd, "encoder_y", u), own)
    assert orc.categorical is fn  # the oracle's own function is back


def test_the_oracle_runs_with_hidden_layers_only_inside_the_block():
    kind, clf = "drvae", [16]
    sd = init_state_dict(kind, seed=3, clf_hidden=clf, **ARCH)
    batch = orc.synthetic_batch(12, ARCH["dim_x"], seed=1)
    om = orc.OracleModel(sd, orc.default_cfg(kind, L=1))
    with pytest.raises(ValueError, match="not restated"):
        om.loss(batch, orc.Tape(seed=1), train=True)
    with classifier_oracle(False):
        lo = om.loss(batch, orc.Tape(seed=1), train=True)
    assert all(bool(torch.isfinite(torch.as_tensor(v)).all()) for v in lo.values())


def test_model_classes_accept_dim_h_clf_and_still_refuse_clf_1sig(monkeypatch):
    from drvae_b200 import models
    built = {}

    def fake_build(self):
        built[type(self).__name__] = True

    monkeypatch.setattr(models._B200Model, "_build_blocks", fake_build)
    kw = dict(dim_x=40, dim_s=1, dim_y=2, dim_h_en_z1=[32], dim_h_de_z1=[16], dim_h_de_x=[32], dim_h_clf=[200], dim_z1=8,
              type_rec='diag_gaussian', nonlinearity='elu', batch_size=32)
    models.DrVAE(dim_h_en_z2Fz1=[], dim_h_en_z3=[16], dim_z3=6, clf_z1z2=True, **kw)
    models.VFAE(dim_h_en_z2=[16], dim_z2=6, semi_supervised=True, **kw)
    assert built == {"DrVAE": True, "VFAE": True}
    with pytest.raises(ValueError, match="clf_1sig"):
        models.DrVAE(dim_h_en_z2Fz1=[], dim_h_en_z3=[16], dim_z3=6, clf_z1z2=True, clf_1sig=True, **kw)


@pytest.mark.parametrize("kind", ("drvae", "vfae"))
def test_cli_class_y_reaches_the_arch(kind):
    args = cli.build_parser(kind).parse_args(["--modelid", "x", "--datafile", "synthetic", "--class-y", "64", "32"])
    assert args.class_y == [64, 32]
    sargs = cli.build_sweep_parser(kind).parse_args(["--datafile", "synthetic", "--rseeds", "1", "--folds", "1", "--class-y", "64", "32"])
    arch = cli.sweep_arch(kind, sargs, 978)
    assert arch["clf_hidden"] == [64, 32]
    assert "clf_hidden" not in cli.sweep_arch("pvae", cli.build_sweep_parser("pvae").parse_args(
        ["--datafile", "synthetic", "--rseeds", "1", "--folds", "1"]), 978)
