"""CPU: softplus hidden layers (the reference constructors' default `nonlinearity='softplus'`, nn.Softplus in the
reference's table, src/blocks.py:21-24) — the restated softplus MLP against an independent torch composition, its
bf16-emulating backward, the model classes' argument check, the C entry point and the Python surface.

The oracle restates the 'elu' nonlinearity only.  `SoftplusOps` below is its Ops with the activation replaced:
F.softplus in fp32 / fp64, and with emulate_bf16 `_SoftplusBF16`, which stores h = rb(softplus(x)) and recovers the
derivative from the stored h as -expm1(-h) (1 beyond the threshold 20), the rule the kernels apply.  `softplus_oracle`
runs the oracle with it in place of its own Ops; the GPU tests (test_activation_gpu.py) take it from here.  The
composition is not pinned by a reference golden file (the oracle's other pieces are, elsewhere): parity with the
reference for softplus is inferred."""
import contextlib
import os
import re
import types

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from helpers import ARCH, ROOT, orc

from drvae_b200 import _lib
from drvae_b200.init import init_state_dict


class _SoftplusBF16(torch.autograd.Function):
    """h = rb(softplus(x)); the derivative is recovered from the stored h: -expm1(-h), 1 for h > 20."""

    @staticmethod
    def forward(ctx, x):
        h = orc.rb(F.softplus(x))
        ctx.save_for_backward(h)
        return h

    @staticmethod
    def backward(ctx, g):
        (h,) = ctx.saved_tensors
        return g * torch.where(h > 20, torch.ones_like(h), -torch.expm1(-h))


class SoftplusOps(orc.Ops):
    def __init__(self, emulate_bf16=False, nonlin="softplus"):
        if nonlin != "softplus":
            raise ValueError("SoftplusOps restates the 'softplus' nonlinearity only")
        super().__init__(emulate_bf16)

    def act(self, x):
        return _SoftplusBF16.apply(x) if self.emu else F.softplus(x)


@contextlib.contextmanager
def softplus_oracle():
    """Oracle calls inside this block use softplus hidden layers.  Enter it before test_clf_hidden_host's
    classifier_oracle, which takes its Ops when it is entered."""
    own = orc.Ops
    orc.Ops = SoftplusOps
    try:
        yield
    finally:
        orc.Ops = own


def _block_sequential(sd, prefix):
    """nn.Sequential(Linear, Softplus, Linear, Softplus, ...) of a block's hidden layers, loaded from the state dict."""
    mods = []
    for name in orc._hidden(sd, prefix):
        W = sd[name + ".weight"]
        lin = nn.Linear(W.shape[1], W.shape[0]).to(W.dtype)
        with torch.no_grad():
            lin.weight.copy_(W)
            lin.bias.copy_(sd[name + ".bias"])
        mods += [lin, nn.Softplus()]
    return nn.Sequential(*mods)


@pytest.mark.parametrize("dtype", (torch.float32, torch.float64))
@pytest.mark.parametrize("kind", ("drvae", "vfae"))
def test_oracle_softplus_mlp_equals_an_nn_sequential(kind, dtype):
    sd = {k: v.to(dtype) for k, v in init_state_dict(kind, seed=4, clf_hidden=[16, 8], **ARCH["deep"]).items()}
    g = torch.Generator().manual_seed(0)
    with softplus_oracle():
        ops = orc.Ops(False)
        for prefix, width in (("encoder_z1", 40), ("decoder_x", 12), ("encoder_y", 24 if kind == "drvae" else 12)):
            x = 6.0 * torch.randn(33, width, generator=g, dtype=dtype)  # every regime, the threshold 20 included
            got = orc.mlp(ops, sd, prefix, x)
            want = _block_sequential(sd, prefix)(x)
            assert len(orc._hidden(sd, prefix)) == 2
            assert torch.equal(got, want.detach()), prefix
    assert orc.Ops is not SoftplusOps  # restored


def test_emulated_backward_is_recovered_from_the_stored_activation():
    x = torch.tensor([-80.0, -40.0, -20.5, -19.5, -8.0, -2.0, -1e-3, 0.0, 0.5, 3.0, 19.9, 20.0, 20.5, 40.0],
                     dtype=torch.float64, requires_grad=True)
    gy = torch.linspace(0.5, 2.0, x.numel(), dtype=torch.float64)
    with softplus_oracle():
        h = orc.Ops(True).act(x)
    h.backward(gy)
    sp = F.softplus(x.detach())
    assert torch.equal(h.detach(), orc.rb(sp))
    # bf16 keeps relative precision down to x << 0, where softplus(x) ~ exp(x)
    assert bool(((h.detach() - sp).abs() <= 2.0 ** -8 * sp).all())
    hd = h.detach()
    want = gy * torch.where(hd > 20, torch.ones_like(hd), -torch.expm1(-hd))
    assert torch.equal(x.grad, want)
    # ... which is sigmoid(x) to bf16 precision in every regime: no cancellation for tiny h, exactly 1 beyond 20
    assert bool(((x.grad / gy - torch.sigmoid(x.detach())).abs() <= 2.0 ** -7 * torch.sigmoid(x.detach())).all())
    assert bool((x.grad[x.detach() > 20] == gy[x.detach() > 20]).all())
    # the plain mode is torch's own softplus and its autograd
    x2 = x.detach().clone().requires_grad_(True)
    with softplus_oracle():
        orc.Ops(False).act(x2).backward(gy)
    assert torch.allclose(x2.grad, gy * torch.sigmoid(x.detach()) * (x.detach() <= 20) + gy * (x.detach() > 20))


def _cfg(kind, nonlinearity):
    return types.SimpleNamespace(kind=kind, type_rec='diag_gaussian', nonlinearity=nonlinearity, use_s=False, dropout_rate=0.,
                                 input_x_dropout=0., optim_alg='adam', type_y='discrete', clf_1sig=False, clf_z1z2=True,
                                 semi_supervised=True, prior_y='uniform')


@pytest.mark.parametrize("kind", ("drvae", "pvae", "vfae"))
def test_check_supported_accepts_softplus_and_refuses_the_rest(kind):
    from drvae_b200.models import _B200Model
    for nl in ("elu", "softplus"):
        _B200Model._check_supported(_cfg(kind, nl))
    for nl in ("relu", "sigmoid"):
        with pytest.raises(ValueError, match="nonlinearity=%r.*not supported by the B200 hot path" % nl):
            _B200Model._check_supported(_cfg(kind, nl))


def test_model_constructor_refuses_relu_before_touching_the_device():
    from drvae_b200 import DrVAE
    with pytest.raises(ValueError, match="nonlinearity='relu'"):
        DrVAE(dim_x=10, dim_s=1, dim_y=2, type_rec='diag_gaussian', nonlinearity='relu')


def test_setter_is_declared_and_exported():
    hdr = open(os.path.join(ROOT, "include", "drvae_b200.h")).read()
    assert re.search(r"^#define DRVAE_ACT_ELU 0$", hdr, re.M)
    assert re.search(r"^#define DRVAE_ACT_SOFTPLUS 1$", hdr, re.M)
    assert re.search(r"^int drvae_set_activation\(drvae_plan_t\* plan, int act\);", hdr, re.M)
    assert "drvae_set_activation" in _lib.EXPORTS
    assert _lib.ACTIVATION == {"elu": 0, "softplus": 1}
    lib = _lib.load()
    assert hasattr(lib, "drvae_set_activation")
    assert lib.drvae_set_activation(None, 1) != 0
    assert b"null plan" in lib.drvae_last_error()


def test_plan_refuses_other_activations_before_touching_the_device():
    from drvae_b200.plan import Plan
    with pytest.raises(ValueError, match="activation must be one of"):
        Plan("drvae", activation="relu", **ARCH["tiny"])


def test_initial_weights_do_not_depend_on_the_activation():
    a = init_state_dict("drvae", seed=9, clf_hidden=[8], **ARCH["tiny"])
    b = init_state_dict("drvae", seed=9, clf_hidden=[8], activation="softplus", **ARCH["tiny"])
    assert list(a) == list(b) and all(torch.equal(a[k], b[k]) for k in a)
