"""CPU oracle for the DrVAE / PertVAE / VFAE training step.  TEST INFRASTRUCTURE ONLY.

This is a restatement (closed forms of SURVEY.md Appendix A, written from scratch) of what the
reference computes in one `run_on_batch(train_mode=True)`:
    /root/reference/src/DGMMixin.py:91-126   run_on_batch (zero_grad, loss, backward, Adam step)
    /root/reference/src/DrVAE.py:333-626     _fprop, _compute_losses, loss_function
    /root/reference/src/PVAE.py:265-467      _compute_losses, loss_function
    /root/reference/src/VFAE.py:234-460      _fprop, _compute_losses, loss_function
    /root/reference/src/blocks.py:166-486    Gaussian mixins, encoder/decoder blocks, classifier
The arithmetic itself lives in PyTorch (the reference pins 0.3.1; parity is defined against the
torch in this image, SURVEY.md Appendix D), so the oracle is written with torch CPU ops and
autograd + torch.optim.Adam, exactly the third-party pieces the reference calls.

Pinning: the reference ships no tests or golden vectors (SURVEY.md §4), so the oracle is pinned
against the reference ITSELF, run in the build container through oracle/ref_harness.py with
identical weights and an identical ε tape; oracle/make_golden.py asserts agreement (<= 1e-5
relative on every loss term, gradients and post-Adam parameters) and commits the reference's
outputs under tests/golden/.  tests/test_oracle.py re-checks the oracle against those files.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module.  The product (drvae_b200/) never does.

`emulate_bf16=True` reproduces the rounding points of the CUDA path (GEMM operands and stored
activations / pre-activation gradients rounded to bf16, fp32 accumulation) so that kernel logic
can be checked at a much tighter tolerance than the bf16-vs-fp32 budget of 1e-3.

`OracleModel(..., dtype=torch.float64)` runs the same restatement in float64: parameters, Adam state, batch and tape
draws are cast on entry.  With `emulate_bf16=True` that keeps the kernels' bf16 rounding points and makes every other
operation (accumulation, transcendentals, reductions) exact to fp32 precision, so what is left of a difference is the
kernel's own fp32 arithmetic.  float32 (the default) is what tests/golden pins.
"""
from collections import OrderedDict

import numpy as np
import torch
import torch.nn.functional as F

LOG2PI = float(np.log(2 * np.pi))  # blocks.py:196,234 use float(np.log(2*np.pi))


# ------------------------------------------------------------------------------------------------
# ε tape: normal draws in the exact order the reference consumes them (SURVEY.md Appendix B)
# ------------------------------------------------------------------------------------------------
class Tape:
    """Sequential source of standard normals.  Either replays a recorded list of tensors or draws
    from a seeded CPU generator (recording what it drew)."""

    def __init__(self, seed=None, recorded=None):
        self.gen = torch.Generator().manual_seed(seed) if seed is not None else None
        self.recorded = list(recorded) if recorded is not None else None
        self.pos = 0
        self.log = []

    def draw(self, *shape):
        if self.recorded is not None:
            t = self.recorded[self.pos]
            assert tuple(t.shape) == tuple(shape), "tape shape mismatch at draw %d: %s vs %s" % (
                self.pos, tuple(t.shape), shape)
            self.pos += 1
        else:
            t = torch.randn(*shape, generator=self.gen)
        self.log.append(t)
        return t


# ------------------------------------------------------------------------------------------------
# bf16 emulation of the CUDA path's rounding points
# ------------------------------------------------------------------------------------------------
def rb(t):
    return t.to(torch.bfloat16).to(t.dtype)


class _LinearBF16(torch.autograd.Function):
    """y = rb(x) rb(W)^T + b with fp32 accumulation; backward uses rb(dy) for dX, dW and db."""

    @staticmethod
    def forward(ctx, x, W, b):
        xr, Wr = rb(x), rb(W)
        ctx.save_for_backward(xr, Wr)
        ctx.has_b = b is not None
        y = xr @ Wr.t()
        return y + b if b is not None else y

    @staticmethod
    def backward(ctx, gy):
        xr, Wr = ctx.saved_tensors
        g = rb(gy)
        return g @ Wr, g.t() @ xr, (g.sum(0) if ctx.has_b else None)


class _EluBF16(torch.autograd.Function):
    """h = rb(elu(x)); the derivative is recovered from the stored h: 1 if h > 0 else h + 1."""

    @staticmethod
    def forward(ctx, x):
        h = rb(F.elu(x))
        ctx.save_for_backward(h)
        return h

    @staticmethod
    def backward(ctx, g):
        (h,) = ctx.saved_tensors
        return g * torch.where(h > 0, torch.ones_like(h), h + 1.0)


class Ops:
    def __init__(self, emulate_bf16=False, nonlin="elu"):
        self.emu = emulate_bf16
        if nonlin != "elu":
            raise ValueError("oracle: only the 'elu' nonlinearity of the shipped configs is restated")

    def lin(self, x, W, b):
        return _LinearBF16.apply(x, W, b) if self.emu else F.linear(x, W, b)

    def act(self, x):
        return _EluBF16.apply(x) if self.emu else F.elu(x)

    def lin_cat_onehot(self, z, yhot, W, b):
        """Linear on cat([z, onehot(y)]) (blocks.py:161).  The CUDA path folds the one-hot columns
        into a per-class fp32 bias, which the emulation mirrors."""
        if not self.emu:
            return F.linear(torch.cat([z, yhot], 1), W, b)
        dz = z.shape[1]
        return _LinearBF16.apply(z, W[:, :dz].contiguous(), b) + yhot @ W[:, dz:].t()


# ------------------------------------------------------------------------------------------------
# blocks (SURVEY.md Appendix A.1)
# ------------------------------------------------------------------------------------------------
def _hidden(sd, prefix):
    i, names = 1, []
    while "%s.nnet.model.linear%d.weight" % (prefix, i) in sd:
        names.append("%s.nnet.model.linear%d" % (prefix, i))
        i += 1
    return names


def _wn_scale(sd, name):
    """WeightNormLinear (layers.py:38-40): per-output scale g/||v||, present iff a `.g` key exists."""
    if name + ".g" in sd:
        return sd[name + ".g"] / torch.norm(sd[name + ".weight"], 2, 1)
    return None


def _linear(ops, sd, name, x, yhot=None):
    W, b = sd[name + ".weight"], sd[name + ".bias"]
    s = _wn_scale(sd, name)
    if s is not None:
        W = W * s[:, None]  # (g/||v||) (x v^T) + b  ==  x (g v/||v||)^T + b
    if yhot is not None:
        return ops.lin_cat_onehot(x, yhot, W, b)
    return ops.lin(x, W, b)


def mlp(ops, sd, prefix, x, yhot=None):
    """blocks.MLP with bn off and dropout 0 (blocks.py:95-164)."""
    h = x
    first = True
    for name in _hidden(sd, prefix):
        h = ops.act(_linear(ops, sd, name, h, yhot if first else None))
        first = False
    if first and yhot is not None:  # no hidden layer: the concat itself is the feature vector
        h = torch.cat([x, yhot], 1)
    return h


def gauss_lv(ops, sd, prefix, x, yhot=None):
    """DiagGaussianModule (blocks.py:291-301): (mu, logvar - 2)."""
    h = mlp(ops, sd, prefix, x, yhot)
    mu = _linear(ops, sd, prefix + ".encoder_mu.linear_mu", h)
    lv = _linear(ops, sd, prefix + ".encoder_lv.linear_lv", h) - 2.0
    return mu, lv


def gauss_linear(ops, sd, prefix, z):
    """DiagGaussianModuleLinear (blocks.py:349-361): mu = z + z W_mu^T + bias_mu."""
    if ops.emu:  # the CUDA path treats bias_mu as the GEMM's bias: its gradient sums the bf16-rounded output gradient
        mu = z + ops.lin(z, sd[prefix + ".W_mu"], sd[prefix + ".bias_mu"])
    else:
        mu = z + ops.lin(z, sd[prefix + ".W_mu"], None) + sd[prefix + ".bias_mu"]
    lv = ops.lin(z, sd[prefix + ".encoder_lv.linear_lv.weight"], sd[prefix + ".encoder_lv.linear_lv.bias"]) - 2.0
    return mu, lv


def gauss_sigma(ops, sd, prefix, z):
    """DiagGaussianSigmaModule (blocks.py:410-416): (mu, softplus(.) + 1e-3)."""
    h = mlp(ops, sd, prefix, z)
    mu = _linear(ops, sd, prefix + ".encoder_mu.linear_mu", h)
    sg = F.softplus(_linear(ops, sd, prefix + ".encoder_sg.linear_sg", h)) + 1e-3
    return mu, sg


def categorical(sd, prefix, u):
    """CategoricalDecoder without hidden layers (blocks.py:456-463); fp32 in both modes."""
    if _hidden(sd, prefix):
        raise ValueError("oracle: classifier hidden layers (--class-y) are not restated")
    name = prefix + ".decoder_p.linear_p"
    W, b = sd[name + ".weight"], sd[name + ".bias"]
    s = _wn_scale(sd, name)
    if s is not None:
        W = W * s[:, None]
    ps = F.softmax(F.linear(u, W, b), dim=-1)
    return torch.clamp(ps, min=1e-10, max=1.0 - 1e-10)


def sample(mu, lv, eps):
    return eps * (lv * 0.5).exp() + mu  # blocks.py:170-174


def kl_perx(mu_q, lv_q, mu_p, lv_p):
    return -0.5 * torch.sum(1 - lv_p + lv_q - ((mu_q - mu_p) ** 2 + lv_q.exp()) / lv_p.exp(), dim=1)  # blocks.py:182


def kl_prior_perx(mu, lv):
    return kl_perx(mu, lv, torch.zeros(1), torch.zeros(1))  # prior_mu=0, prior_lv=log(1)


def logn_sigma(x, mu, sg):
    return (-0.5 * torch.sum(LOG2PI + torch.log(sg ** 2) + ((x - mu) ** 2) / (sg ** 2), dim=1)).sum()  # blocks.py:234


def one_hot(y, k, dtype=torch.float32):
    return F.one_hot(y.long().view(-1), k).to(dtype)


def free_bits(kl, kl_min):
    return torch.max(kl, torch.full_like(kl, kl_min))  # DGMMixin.py:68-75


def anneal(it, it_max, off):
    return min(1.0, 0.01 + (it - off) / (1.0 * it_max)) if it - off > 0 else 0.01  # DGMMixin.py:77-89


# ------------------------------------------------------------------------------------------------
# group losses
# ------------------------------------------------------------------------------------------------
def _fprop(ops, sd, cfg, enc, z1, q1, yhot, tape):
    """DrVAE._fprop / VFAE._fprop: fb(KL(q(z_top|z1,y) || N(0,I))) + fb(KL(q1 || p(z1|z_top,y)))."""
    q3 = gauss_lv(ops, sd, enc, z1, yhot)
    z3 = sample(q3[0], q3[1], tape.draw(*q3[0].shape))
    k = free_bits(kl_prior_perx(*q3), cfg["kl_min"])
    pz1 = gauss_lv(ops, sd, "decoder_z1", z3, yhot)
    return k + free_bits(kl_perx(q1[0], q1[1], pz1[0], pz1[1]), cfg["kl_min"])


def _y_terms(ops, sd, cfg, enc, z1, q1, qy, y, tape, n, L):
    """Label-dependent part shared by DrVAE (DrVAE.py:502-534) and VFAE (VFAE.py:332-391)."""
    dim_y = cfg["dim_y"]
    YL = 0.0
    if y is not None:
        YL = torch.log(qy).gather(1, y.long().view(-1, 1)).sum() / L  # -nll_loss(log ps, y) summed
        k = _fprop(ops, sd, cfg, enc, z1, q1, one_hot(y, dim_y, z1.dtype), tape)
    else:
        k = 0.0
        for j in range(dim_y):
            yj = one_hot(torch.full((n,), j), dim_y, z1.dtype)
            k = k + qy[:, j] * _fprop(ops, sd, cfg, enc, z1, q1, yj, tape)
        prior = cfg.get("prior_y_vec")
        pr = (torch.full((n, dim_y), 1.0 / dim_y, dtype=qy.dtype) if prior is None
              else torch.tensor(prior).float().to(qy.dtype).expand(n, dim_y))
        k = k + (-qy * (torch.log(pr) - torch.log(qy))).sum(1)  # blocks.py:479-480
    return YL, k.sum() / L


def drvae_group(ops, sd, cfg, x1, x2, y, tape, beta_pert):
    """Appendix A.2.  x2 is None for singletons, y is None for unlabeled rows."""
    L, n = cfg["L"], x1.shape[0]
    pair = x2 is not None
    a1 = x1 + cfg["noise_std"] * tape.draw(*x1.shape) if cfg["noisy"] else x1
    q1 = gauss_lv(ops, sd, "encoder_z1", a1)
    if pair:
        a2 = x2 + cfg["noise_std"] * tape.draw(*x2.shape) if cfg["noisy"] else x2
        q2 = gauss_lv(ops, sd, "encoder_z1", a2)
    RECL = KLD = PERT = YL = 0.0
    for _ in range(L):
        z1 = sample(q1[0], q1[1], tape.draw(*q1[0].shape))
        if pair:
            z2 = sample(q1[0], q1[1], tape.draw(*q1[0].shape))  # sic: q(z1|x1), DrVAE.py:427
        pz2 = gauss_linear(ops, sd, "decoder_z2Fz1", z1)
        z2f = sample(pz2[0], pz2[1], tape.draw(*pz2[0].shape))
        RECL = RECL + logn_sigma(a1, *gauss_sigma(ops, sd, "decoder_x", z1)) / L
        if pair:
            RECL = RECL + logn_sigma(a2, *gauss_sigma(ops, sd, "decoder_x", z2)) / L
            PERT = PERT + logn_sigma(a2, *gauss_sigma(ops, sd, "decoder_x", z2f)) / L
            klz2 = free_bits(kl_perx(q2[0], q2[1], pz2[0], pz2[1]), cfg["kl_min"])
            KLD = KLD + beta_pert * (cfg["kl_qz2pz2_rate"] * klz2.sum() / L)
        qy = categorical(sd, "encoder_y", torch.cat([z1, z2f - z1], 1))
        yl, k = _y_terms(ops, sd, cfg, "encoder_z3", z1, q1, qy, y, tape, n, L)
        YL = YL + yl
        KLD = KLD + k
    return dict(RECL=RECL, KLD=KLD, PERT=PERT, YL=YL)


def pvae_group(ops, sd, cfg, x1, x2, tape, beta_pert):
    """Appendix A.4."""
    L = cfg["L"]
    pair = x2 is not None
    a1 = x1 + cfg["noise_std"] * tape.draw(*x1.shape) if cfg["noisy"] else x1
    q1 = gauss_lv(ops, sd, "encoder_z1", a1)
    if pair:
        a2 = x2 + cfg["noise_std"] * tape.draw(*x2.shape) if cfg["noisy"] else x2
        q2 = gauss_lv(ops, sd, "encoder_z1", a2)
    RECL = KLD = PERT = 0.0
    for _ in range(L):
        z1 = sample(q1[0], q1[1], tape.draw(*q1[0].shape))
        if pair:
            z2 = sample(q1[0], q1[1], tape.draw(*q1[0].shape))  # sic, PVAE.py:313
        pz2 = gauss_linear(ops, sd, "decoder_z2Fz1", z1)
        z2f = sample(pz2[0], pz2[1], tape.draw(*pz2[0].shape))
        RECL = RECL + logn_sigma(a1, *gauss_sigma(ops, sd, "decoder_x", z1)) / L
        KLD = KLD + free_bits(kl_prior_perx(*q1), cfg["kl_min"]).sum() / L
        if pair:
            RECL = RECL + logn_sigma(a2, *gauss_sigma(ops, sd, "decoder_x", z2)) / L
            PERT = PERT + logn_sigma(a2, *gauss_sigma(ops, sd, "decoder_x", z2f)) / L
            KLD = KLD + free_bits(kl_prior_perx(*q2), cfg["kl_min"]).sum() / L
            klz2 = free_bits(kl_perx(q2[0], q2[1], pz2[0], pz2[1]), cfg["kl_min"])
            KLD = KLD + beta_pert * (cfg["kl_qz2pz2_rate"] * klz2.sum() / L)
    return dict(RECL=RECL, KLD=KLD, PERT=PERT)


def vfae_group(ops, sd, cfg, x1, y, tape):
    """Appendix A.5 (SSVAE mode, use_s=False)."""
    L, n = cfg["L"], x1.shape[0]
    a1 = x1 + cfg["noise_std"] * tape.draw(*x1.shape) if cfg["noisy"] else x1
    q1 = gauss_lv(ops, sd, "encoder_z1", a1)
    RECL = KLD = YL = 0.0
    for _ in range(L):
        z1 = sample(q1[0], q1[1], tape.draw(*q1[0].shape))
        RECL = RECL + logn_sigma(a1, *gauss_sigma(ops, sd, "decoder_x", z1)) / L
        qy = categorical(sd, "encoder_y", z1)
        yl, k = _y_terms(ops, sd, cfg, "encoder_z2", z1, q1, qy, y, tape, n, L)
        YL = YL + yl
        KLD = KLD + k
    return dict(RECL=RECL, KLD=KLD, YL=YL)


# ------------------------------------------------------------------------------------------------
# batch losses (Appendix A.3-A.5) — groups in the reference's fixed order
# ------------------------------------------------------------------------------------------------
def default_cfg(kind, **kw):
    cfg = dict(kind=kind, L=1, dim_y=2, noisy=True, noise_std=0.01, yloss_rate=1.0, pertloss_rate=0.05,
               kl_qz2pz2_rate=1.0, kl_min=2.0, anneal_perturb_rate_itermax=1, anneal_perturb_rate_offset=0,
               lr=5e-4, weight_decay=0.05, prior_y_vec=None, counts=None)
    cfg.update(kw)
    return cfg


def _idx(mask):
    return torch.nonzero(mask).view(-1)


class _CastTape:
    """Hands out a tape's draws in the oracle's dtype (the tape itself keeps what it drew, for the ε block)."""

    def __init__(self, tape, dtype):
        self.tape, self.dtype = tape, dtype

    def draw(self, *shape):
        return self.tape.draw(*shape).to(self.dtype)


def _cast_batch(batch, dtype):
    return {k: (v.to(dtype) if k in ("x1", "x2") else v) for k, v in batch.items()}


def loss_function(sd, batch, tape, cfg, iters, train=True, emulate_bf16=False, dtype=torch.float32):
    """Returns OrderedDict of 0-dim tensors with the reference's keys for cfg['kind'].  `dtype` is the arithmetic
    type: `sd` must hold it; the batch and the tape draws are cast to it."""
    ops = Ops(emulate_bf16)
    batch = _cast_batch(batch, dtype)
    tape = _CastTape(tape, dtype)
    cfg = dict(cfg)
    cfg["noisy"] = bool(cfg["noisy"] and train)  # noise only when self.training and self.add_noise
    kind = cfg["kind"]
    beta_pert = 1.0
    if cfg["anneal_perturb_rate_itermax"] > 0:
        beta_pert = anneal(iters, cfg["anneal_perturb_rate_itermax"], cfg["anneal_perturb_rate_offset"])
    x1 = batch["x1"]
    N = x1.shape[0]
    cnt = cfg.get("counts")  # optional global normalisers for data-parallel shards
    out = OrderedDict()
    if kind == "drvae":
        hx, hy = batch["has_x2"].bool(), batch["has_y"].bool()
        groups = [(_idx(hy & ~hx), False, True), (_idx(~hy & ~hx), False, False),
                  (_idx(hy & hx), True, True), (_idx(~hy & hx), True, False)]  # LS, US, LP, UP
        tot = dict(RECL=0.0, KLD=0.0, PERT=0.0, YL=0.0)
        for idx, pair, lab in groups:
            if len(idx) == 0:
                continue
            g = drvae_group(ops, sd, cfg, x1[idx].clone(), batch["x2"][idx].clone() if pair else None,
                            batch["y"][idx] if lab else None, tape, beta_pert)
            for k in tot:
                tot[k] = tot[k] + g[k]
        Np = int(hx.sum())
        Nl = int(hy.sum())
        if cnt is not None:
            N, Np, Nl = cnt["N"], cnt["Np"], cnt["Nlab"]
        out["RECL"] = tot["RECL"] / N
        out["KLD"] = tot["KLD"] / N
        out["PERT"] = tot["PERT"] / max(1.0, Np)
        out["YL"] = tot["YL"] / max(1.0, Nl)
        out["MMD"] = torch.zeros((), dtype=dtype)
        out["ELBO"] = out["RECL"] + beta_pert * cfg["pertloss_rate"] * out["PERT"] - out["KLD"]
        out["CMPL"] = -out["ELBO"] - cfg["yloss_rate"] * out["YL"]
    elif kind == "pvae":
        hx = batch["has_x2"].bool()
        tot = dict(RECL=0.0, KLD=0.0, PERT=0.0)
        for idx, pair in [(_idx(~hx), False), (_idx(hx), True)]:
            if len(idx) == 0:
                continue
            g = pvae_group(ops, sd, cfg, x1[idx].clone(), batch["x2"][idx].clone() if pair else None, tape, beta_pert)
            for k in tot:
                tot[k] = tot[k] + g[k]
        Np = int(hx.sum())
        if cnt is not None:
            N, Np = cnt["N"], cnt["Np"]
        out["RECL"] = tot["RECL"] / N
        out["KLD"] = tot["KLD"] / N
        out["PERT"] = tot["PERT"] / max(1.0, Np)
        out["MMD"] = torch.zeros((), dtype=dtype)
        out["ELBO"] = out["RECL"] + beta_pert * cfg["pertloss_rate"] * out["PERT"] - out["KLD"]
        out["CMPL"] = -out["ELBO"]
    elif kind == "vfae":
        hy = batch["has_y"].bool()
        tot = dict(RECL=0.0, KLD=0.0, YL=0.0)
        for idx, lab in [(_idx(hy), True), (_idx(~hy), False)]:
            if len(idx) == 0:
                continue
            g = vfae_group(ops, sd, cfg, x1[idx].clone(), batch["y"][idx] if lab else None, tape)
            for k in tot:
                tot[k] = tot[k] + g[k]
        Nl = int(hy.sum())
        if cnt is not None:
            N, Nl = cnt["N"], cnt["Nlab"]
        out["RECL"] = tot["RECL"] / N
        out["KLD"] = tot["KLD"] / N
        out["YL"] = tot["YL"] / Nl  # no max(1, .) guard in the reference (VFAE.py:443)
        out["MMD"] = torch.zeros((), dtype=dtype)
        out["ELBO"] = out["RECL"] - out["KLD"]
        out["CMPL"] = -out["ELBO"] - cfg["yloss_rate"] * out["YL"]
    else:
        raise ValueError(kind)
    for k in out:
        if not torch.is_tensor(out[k]):
            out[k] = torch.tensor(float(out[k]), dtype=dtype)
    return out


class OracleModel:
    """Parameters + torch.optim.Adam, stepping like DGMMixin.run_on_batch (DGMMixin.py:91-126)."""

    def __init__(self, state_dict, cfg, dtype=torch.float32):
        self.cfg = dict(cfg)
        self.dtype = dtype
        self.sd = OrderedDict((k, v.detach().clone().to(dtype).requires_grad_(True)) for k, v in state_dict.items())
        self.opt = torch.optim.Adam(list(self.sd.values()), lr=cfg["lr"], weight_decay=cfg["weight_decay"])
        self.iters = 0

    def loss(self, batch, tape, train=False, emulate_bf16=False):
        with torch.no_grad():
            return loss_function(self.sd, batch, tape, self.cfg, self.iters, train=train, emulate_bf16=emulate_bf16,
                                 dtype=self.dtype)

    def grads(self, batch, tape, emulate_bf16=False):
        """forward + backward only; returns (losses, {name: grad}) without touching the optimizer."""
        for p in self.sd.values():
            p.grad = None
        losses = loss_function(self.sd, batch, tape, self.cfg, self.iters, train=True, emulate_bf16=emulate_bf16,
                               dtype=self.dtype)
        losses["CMPL"].backward()
        g = OrderedDict((k, (p.grad.detach().clone() if p.grad is not None else torch.zeros_like(p)))
                        for k, p in self.sd.items())
        return OrderedDict((k, v.detach()) for k, v in losses.items()), g

    def step(self, batch, tape, emulate_bf16=False, grad_hook=None):
        self.opt.zero_grad()
        losses = loss_function(self.sd, batch, tape, self.cfg, self.iters, train=True, emulate_bf16=emulate_bf16,
                               dtype=self.dtype)
        losses["CMPL"].backward()
        if grad_hook is not None:
            grad_hook(self.sd)
        self.opt.step()
        self.iters += 1
        return OrderedDict((k, v.detach()) for k, v in losses.items())

    def state_dict(self):
        return OrderedDict((k, v.detach().clone()) for k, v in self.sd.items())

    # ---- deterministic inference (DrVAE.py:253-311, PVAE.py:206-246, VFAE.py:178-215) ----
    def forward(self, x1, emulate_bf16=False):
        ops = Ops(emulate_bf16)
        sd, kind = self.sd, self.cfg["kind"]
        x1 = x1.to(self.dtype)
        with torch.no_grad():
            q1 = gauss_lv(ops, sd, "encoder_z1", x1)
            res = {"z1": q1[0], "qz1": q1}
            res["px1"] = gauss_sigma(ops, sd, "decoder_x", q1[0])
            res["x1_rec"] = res["px1"][0]
            if kind in ("drvae", "pvae"):
                pz2 = gauss_linear(ops, sd, "decoder_z2Fz1", q1[0])
                res["z2"], res["pz2"] = pz2[0], pz2
                res["px2"] = gauss_sigma(ops, sd, "decoder_x", pz2[0])
                res["x2_pert"] = res["px2"][0]
            if kind == "drvae":
                res["proba"] = categorical(sd, "encoder_y", torch.cat([q1[0], pz2[0] - q1[0]], 1))
            elif kind == "vfae":
                res["proba"] = categorical(sd, "encoder_y", q1[0])
            if "proba" in res:
                res["pred"] = torch.max(res["proba"], dim=1)[1]
        return res


# ------------------------------------------------------------------------------------------------
# synthetic inputs of SURVEY.md §8(d)
# ------------------------------------------------------------------------------------------------
def synthetic_batch(N, dim_x=978, seed=0, dim_y=2):
    g = torch.Generator().manual_seed(seed)
    x1 = torch.randn(N, dim_x, generator=g)
    x2 = x1 + 0.3 * torch.randn(N, dim_x, generator=g)
    s = torch.zeros(N, dtype=torch.int32)
    y = torch.randint(0, dim_y, (N,), generator=g).int()
    i = torch.arange(N)
    has_x2 = (i % 2 == 0).int()
    has_y = (i % 3 != 0).int()
    x2[has_x2 == 0] = 0
    return dict(x1=x1, x2=x2, s=s, y=y, has_x2=has_x2, has_y=has_y)
