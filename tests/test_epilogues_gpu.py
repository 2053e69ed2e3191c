"""The step's GEMM epilogues element by element, recomputed in float64 from the operands the step itself stored, and the
saturated regimes of a trained model end to end against the float64 oracle.

Part 1 runs one grad_step kernel by kernel (no graph, no step kernel, tensor-core mainloop) and reads the workspace it
leaves behind.  Every GEMM whose output lands in a readable buffer is recomputed in float64 from the bf16 operand it
read (exact in float64), the bf16 weight shadow (checked once against round-to-nearest of the parameters) and the fp32
derived bias / class-bias copies (checked against the parameters plus the folded constants), then the epilogue's
formula is applied and every element compared.

Part 2 edits an initial state dict into a trained-like one (decoder sigma in every softplus regime, targets hundreds of
sigmas from mu, saturated ELUs, confident classifier rows, free bits on both sides of kl_min) and checks losses,
gradients, eval losses, inference and the fused optimizer against the oracle, plus the part-1 element checks.

Tolerances (see the functions that compute them): every check allows, per element, a bound built from
  * u = 2^-24, the unit roundoff of fp32: one rounding per fp32 operation;
  * K u sum_k |a_k| |b_k|: fp32 accumulation of K exact bf16 products (tcgen05 accumulates in fp32), the standard
    gamma_K bound of a recursively summed dot product (Higham, Accuracy and Stability, 3.1);
  * the PTX ISA's error bounds of the flush-to-zero approximations the decoder-loss epilogue uses: ex2.approx.ftz.f32
    relative 2^-22, lg2.approx.ftz.f32 absolute 2^-22 (the ISA states 2^-22.6), rcp.approx.ftz.f32 1 ulp = 2^-23
    relative, each propagated to the outputs to first order (torch.autograd of the float64 reference with respect to
    one perturbation per intermediate) and doubled for the neglected second-order terms;
  * __expf of ELU: the CUDA C Programming Guide bounds __expf(x) by 2 + floor(|1.173 x|) ulp; for x <= 0 the value is
    at most 1, so the absolute error is at most (3 + 1.173 |x|) 2^-24 (one more ulp for the subtraction of 1);
  * bf16 output rounding, round to nearest even: bf16 keeps 8 significant bits, so |rn(v) - v| <= 2^-8 |v|; a stored
    value may differ from the float64 reference r by 2^-8 (|r| + d) + d, where d bounds the fp32 value before rounding.
No bound is fitted to an observed error.  Each check prints its worst ratio of error to allowance."""
import math

import numpy as np
import pytest
import torch

from helpers import ARCH, KINDS, SEED_MODEL, assert_grad_close, batch_fields, orc

from drvae_b200.init import init_state_dict
from drvae_b200.noise import eps_block_from_tape, tape_shapes
from drvae_b200.plan import Plan, losses_to_dict

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
BF16_REL = 2.0 ** -8
EX2_REL, LG2_ABS, RCP_REL = 2.0 ** -22, 2.0 ** -22, 2.0 ** -23
CNT = dict(N=0, NP=1, NLAB=2, R0=3, LN=4, RD=5, F=6, FL=7)
COEF_RECL, COEF_PERT, COEF_KLD, COEF_YL = 0, 1, 3, 4
F32_1E10 = float(np.float32(1e-10))  # the clamp's lower bound as the kernels store it (1.00000001e-10)


def round_up(x, m):
    return (x + m - 1) // m * m


def cdiv(a, b):
    return (a + b - 1) // b


def tile_cap(n):
    n16 = round_up(n, 16)
    tiles = cdiv(n16, 256)
    return round_up(cdiv(n16, tiles), 16), tiles


# ---- the plan's weight shadows, in plan.cu's make_shadow order ------------------------------------------------------
class ShadowSpec:
    """One GEMM weight as the kernels see it: bf16 [rcap, kc] (shadow row s = stacked / interleaved output feature,
    column k < kin), fp32 derived bias [rcap] (constant folded in) and class bias [Y][rcap]."""

    def __init__(self, w, b, rows, kin, cc, ilv_block, ilv_stride, BN, tiles, bconst=(0.0, 0.0)):
        self.w, self.b, self.rows, self.kin, self.cc = w, b, rows, kin, cc
        self.kaug = kin + 1 + cc
        self.kc = round_up(self.kaug, 16)
        self.rcap = BN * tiles
        self.ilv_block, self.ilv_stride, self.bconst = ilv_block, ilv_stride, bconst

    def srow(self, which, n):
        return (n // self.ilv_block) * self.ilv_stride + which * self.ilv_block + n % self.ilv_block


def shadow_specs(kind, arch):
    """{block: (hidden specs, head spec)}; offsets into the shadow and derived arenas are assigned in creation order."""
    X, Z, Y, Z3 = arch["dim_x"], arch["dim_z1"], arch["dim_y"], arch["dim_z3"]
    big = 1 << 30
    out = {}

    def hidden(prefix, kin, cc, widths):
        specs, prev = [], kin
        for i, w in enumerate(widths):
            nm = "%s.nnet.model.linear%d" % (prefix, i + 1)
            bn, t = tile_cap(w + 1)
            specs.append(ShadowSpec([nm + ".weight"], [nm + ".bias"], w, prev, cc if i == 0 else 0, big, big, bn, t))
            prev = w
        return specs, prev

    def gauss(prefix, kin, cc, widths, outd, sigma):
        hs, prev = hidden(prefix, kin, cc, widths)
        sec = "sg" if sigma else "lv"
        w = [prefix + ".encoder_mu.linear_mu.weight", "%s.encoder_%s.linear_%s.weight" % (prefix, sec, sec)]
        b = [n[:-len("weight")] + "bias" for n in w]
        if sigma:
            hb = min(128, round_up(outd, 16))
            head = ShadowSpec(w, b, outd, prev, 0, hb, 2 * hb, 2 * hb, cdiv(outd, hb))
        else:
            os_ = round_up(outd, 16)
            bn, t = tile_cap(2 * os_)
            head = ShadowSpec(w, b, outd, prev, 0, os_, 2 * os_, bn, t, (0.0, -2.0))
        return hs, head

    out["enc"] = gauss("encoder_z1", X, 0, arch["enc_z1"], Z, False)
    if kind != "vfae":
        zs = round_up(Z, 16)
        bn, t = tile_cap(2 * zs)
        out["T"] = ([], ShadowSpec(["decoder_z2Fz1.W_mu", "decoder_z2Fz1.encoder_lv.linear_lv.weight"],
                                   ["decoder_z2Fz1.bias_mu", "decoder_z2Fz1.encoder_lv.linear_lv.bias"], Z, Z, 0, zs, 2 * zs,
                                   bn, t, (0.0, -2.0)))
    if kind != "pvae":
        out["z3"] = gauss("encoder_z3" if kind == "drvae" else "encoder_z2", Z, Y, arch["enc_z3"], Z3, False)
        out["dz1"] = gauss("decoder_z1", Z3, Y, arch["dec_z1"], Z, False)
    out["dec"] = gauss("decoder_x", Z, 0, arch["dec_x"], X, True)
    sh = dv = 0
    for blk in out.values():
        for s in blk[0] + [blk[1]]:
            s.sh_off, s.bias_off = sh, dv
            sh += s.kc * s.rcap
            dv += s.rcap
            if s.cc:
                s.clsb_off = dv
                dv += s.cc * s.rcap
    return out


def bf16_rn(t):
    return t.to(torch.bfloat16).to(torch.float64)


def read_weights(plan, specs, sd, m):
    """bf16 shadow [rcap, kc], derived bias [rcap] and class bias [cc, rcap] of every spec, as float64; checks that the
    shadow is round-to-nearest of the parameters (zero in the ones / class columns and padding rows) and that the
    derived copies are the fp32 parameters plus the folded constants."""
    shadow, _, _ = plan.debug_buffer("shadow", torch.bfloat16)
    derived, _, _ = plan.debug_buffer("derived")
    dev = plan.device
    for blk in specs.values():
        for s in blk[0] + [blk[1]]:
            S = shadow[m, s.sh_off:s.sh_off + s.kc * s.rcap].view(s.kc // 8, s.rcap, 8).permute(1, 0, 2).reshape(s.rcap, s.kc)
            s.S = S.to(torch.float64)
            s.bias = derived[m, s.bias_off:s.bias_off + s.rcap].to(torch.float64)
            want = torch.zeros(s.rcap, s.kc, dtype=torch.float64, device=dev)
            wb = torch.zeros(s.rcap, dtype=torch.float64, device=dev)
            wc = torch.zeros(max(s.cc, 1), s.rcap, dtype=torch.float64, device=dev)
            for which, (wn, bn) in enumerate(zip(s.w, s.b)):
                rows = torch.tensor([s.srow(which, n) for n in range(s.rows)], device=dev)
                W = sd[wn].to(dev, torch.float32)
                want[rows, :s.kin] = bf16_rn(W[:, :s.kin])
                wb[rows] = (sd[bn].to(dev, torch.float32) + torch.tensor(s.bconst[which], dtype=torch.float32, device=dev)).double()
                if s.cc:
                    wc[:, rows] = W[:, s.kin:].t().double()
            assert torch.equal(s.S, want), "shadow of %s is not round-to-nearest bf16 of the parameters" % s.w[0]
            assert torch.equal(s.bias, wb), "derived bias of %s" % s.b[0]
            if s.cc:
                s.clsb = derived[m, s.clsb_off:s.clsb_off + s.cc * s.rcap].view(s.cc, s.rcap).to(torch.float64)
                assert torch.equal(s.clsb, wc), "class bias of %s" % s.w[0]


# ---- tolerances -----------------------------------------------------------------------------------------------------
def acc_bound(A, B):
    """fp32 accumulation of exact bf16 products: K u sum_k |a_k| |b_k| for D = A B^T (A [M, K], B [N, K])."""
    return A.shape[1] * U * (A.abs() @ B.abs().t())


def bf16_allow(ref, d):
    return BF16_REL * (ref.abs() + d) + d


class Worst:
    def __init__(self):
        self.r = {}

    def check(self, tag, got, ref, allow):
        err = (got - ref).abs()
        ratio = err / allow.clamp_min(1e-300)
        worst = float(ratio.max()) if ratio.numel() else 0.0
        self.r[tag] = max(worst, self.r.get(tag, 0.0))
        if worst > 1.0:
            i = np.unravel_index(int(ratio.argmax()), tuple(ratio.shape))
            bad = int((ratio > 1).sum())
            raise AssertionError("%s: %d elements outside the bound, worst at %s: got %.8g ref %.8g |err| %.3e allowed %.3e" % (
                tag, bad, i, float(got[i]), float(ref[i]), float(err[i]), float(allow[i])))

    def report(self, title):
        print("\n%s: worst |err| / allowance per check" % title)
        for k, v in sorted(self.r.items()):
            print("  %-34s %.3f" % (k, v))


# ---- float64 references of the epilogues ----------------------------------------------------------------------------
def elu_ref(x, ex):
    """ELU in float64 and the bound on the kernel's fp32 value before bf16 rounding: the pre-activation bound `ex`
    times |ELU'| plus, for x <= 0, the __expf error (3 + 1.173 |x|) 2^-24 (module docstring)."""
    y = torch.where(x > 0, x, torch.expm1(x))
    d = torch.where(x > 0, ex, ex * torch.exp(torch.clamp(x, max=0.0)) + (3.0 + 1.173 * x.abs()) * U)
    return y, d


def decloss_ref(mu, s, tgt, coef, e_mu, e_s):
    """gemm.cuh decloss_pair in float64: (lp, d/dmu, d/dsigma-pre-activation) of -coef log N(tgt; mu, softplus(s)+1e-3),
    and first-order bounds of the kernel's fp32 values.  Every intermediate the kernel rounds or approximates gets one
    perturbation; autograd gives each output's sensitivity to it; bound = 2 sum |sensitivity| x (its error bound)."""
    LOG2E, LN2, HL2PI = 1.4426950408889634, 0.6931471805599453, 0.9189385332046727
    names = ("mu", "s", "x", "ex", "exa", "one", "l1p", "l1pm", "tiny", "soft", "sg", "sgm", "sig", "inv", "diff", "t", "lg", "inner",
             "lp", "c1", "dmu", "tt", "dsg")
    d = {k: torch.zeros_like(mu, requires_grad=True) for k in names}
    big = s > 20.0
    m = mu + d["mu"]
    sp = s + d["s"]
    x = torch.clamp(sp, max=20.0) * LOG2E * (1 + d["x"])
    ex = torch.exp2(x) * (1 + d["ex"]) + d["exa"]  # relative error, and the flush of results below 2^-126
    one = (ex + 1) * (1 + d["one"])
    l1p = (torch.log2(one) + d["l1p"]) * LN2 * (1 + d["l1pm"])
    tiny = ex * (1 - 0.5 * ex) + d["tiny"]
    small = ex.detach() < 1e-3
    soft = torch.where(big, sp, torch.where(small, tiny, l1p)) + d["soft"]
    sg = (soft + 1e-3) * (1 + d["sg"])
    sgm = ex / one * (1 + d["sgm"])
    sig = torch.where(big, torch.ones_like(sgm), sgm) + d["sig"]
    inv = 1 / sg * (1 + d["inv"])
    diff = (tgt - m) * (1 + d["diff"])
    t = diff * inv * (1 + d["t"])
    lg = torch.log2(sg) + d["lg"]
    inner = -LN2 * lg - HL2PI + d["inner"]
    lp = (-0.5 * t * t + inner) * (1 + d["lp"])
    c1 = -coef * inv * (1 + d["c1"])
    dmu = c1 * t * (1 + d["dmu"])
    tt = (t * t - 1) * (1 + d["tt"])
    dsg = c1 * tt * sig * (1 + d["dsg"])
    with torch.no_grad():
        exv = torch.exp2(torch.clamp(s, max=20.0) * LOG2E)
        tail = torch.exp(-torch.clamp(s, min=20.0))  # softplus(s) - s and 1 - sigmoid(s) beyond the threshold
        lgv = torch.log2(torch.where(big, s, torch.log1p(exv)) + 1e-3)
        B = dict(mu=e_mu, s=e_s, x=torch.full_like(mu, 2 * U), ex=torch.full_like(mu, EX2_REL),
                 exa=torch.full_like(mu, 2.0 ** -126), one=torch.full_like(mu, U), l1p=torch.full_like(mu, LG2_ABS),
                 l1pm=torch.full_like(mu, 2 * U), tiny=exv ** 3 / 3 + 2 * U * exv,
                 soft=torch.where(big, tail, torch.zeros_like(mu)), sg=torch.full_like(mu, 2 * U),
                 sgm=torch.full_like(mu, RCP_REL + U), sig=torch.where(big, tail, torch.zeros_like(mu)),
                 inv=torch.full_like(mu, RCP_REL), diff=torch.full_like(mu, U), t=torch.full_like(mu, U),
                 lg=torch.full_like(mu, LG2_ABS), inner=2 * U * (LN2 * lgv.abs() + HL2PI), lp=torch.full_like(mu, U),
                 c1=torch.full_like(mu, 2 * U), dmu=torch.full_like(mu, U), tt=torch.full_like(mu, U),
                 dsg=torch.full_like(mu, 2 * U))
    bounds = []
    for out in (lp, dmu, dsg):
        gs = torch.autograd.grad(out.sum(), [d[k] for k in names], retain_graph=True, allow_unused=True)
        tot = torch.zeros_like(mu)
        for k, g in zip(names, gs):
            if g is not None:
                tot = tot + g.abs() * B[k]
        bounds.append(2 * tot)
    return lp.detach(), dmu.detach(), dsg.detach(), bounds[0], bounds[1], bounds[2]


def dlogit_ref(q, lab, ycls, ke, coef_yl, coef_kld, log_prior):
    """rowops.cuh clf_dlogit_row in float64, with PyTorch's float32 clamp semantics: q = clamp(softmax, 1e-10,
    1 - 1e-10) in float32, whose upper bound rounds to 1.0, so only a class clamped at 1e-10 loses its gradient.
    (Rows with a logit gap above ln(1e10) = 23.03 are kept: the float64 oracle would also zero the dominant class
    there, a difference of 1e-10 x the coefficient that this check decides in favour of float32 semantics.)"""
    clamped = q <= F32_1E10
    g = torch.where(lab[:, None], torch.zeros_like(q), coef_kld * (ke + torch.log(q) - log_prior + 1.0))
    onehot = torch.zeros_like(q, dtype=torch.bool)
    onehot[torch.arange(q.shape[0]), ycls.long()] = True
    g = torch.where(lab[:, None] & onehot, -coef_yl / q, g)
    g = torch.where(clamped, torch.zeros_like(g), g)
    dot = (q * g).sum(1, keepdim=True)
    dl = q * (g - dot)
    # fp32: the unlabelled g is 4 additions and a logf (2 ulp), the labelled one a division; dot sums Y products
    dg = torch.where(lab[:, None], 2 * U * g.abs(), 8 * U * coef_kld * (ke.abs() + torch.log(q).abs() + abs(log_prior) + 1))
    dg = torch.where(clamped, torch.zeros_like(dg), dg)
    ddot = (q * dg).sum(1, keepdim=True) + q.shape[1] * 2 * U * (q * g).abs().sum(1, keepdim=True)
    allow = q * (dg + ddot) + 4 * U * q * (g.abs() + dot.abs())
    return dl, allow


# ---- one step, read back --------------------------------------------------------------------------------------------
def fp32_rows(plan, name, m, rows, ld):
    t, _, _ = plan.debug_buffer(name)
    return t[m, :rows * ld].view(rows, ld).to(torch.float64)


def c8(plan, name, m, rows, feats=None):
    t, rcap, fcap = plan.debug_buffer(name, torch.bfloat16)
    x = t[m].view(fcap // 8, rcap, 8).permute(1, 0, 2).reshape(rcap, fcap)
    return x[:rows, :feats].to(torch.float64)


BLOCKS = dict(enc=("Ain", "R0", "dY2", "Q"), T=("Zdec", "LN", "dYT", "PT"), z3=("Z1e", "F", "dY7", "Q3"),
              dz1=("Z3b", "F", "dY9", "PZ1"), dec=("Zdec", "RD", "dY5", None))


def check_step_elements(plan, kind, arch, sd, m, W, regimes=None):
    """Every epilogue of one grad_step of model m against float64 (see the module docstring)."""
    specs = shadow_specs(kind, arch)
    read_weights(plan, specs, sd, m)
    cnt = plan.debug_buffer("counts", torch.int32)[0][m].cpu().tolist()
    X = arch["dim_x"]
    gv = plan.tensor_views(plan.grads, m)
    dec_pre = None
    for blk, (hs, head) in specs.items():
        src_name, rkey, dyname, outname = BLOCKS[blk]
        R = cnt[CNT[rkey]]
        Rt = round_up(R, 128)
        ins = [c8(plan, src_name, m, Rt)]
        cls = None
        if blk in ("z3", "dz1"):
            cls = plan.debug_buffer("e_cls_full", torch.int32)[0][m, :R].long()
            # the stored input carries the one-hot of that class after its ones column
            kin = hs[0].kin
            assert torch.equal(ins[0][:R, kin], torch.ones(R, dtype=torch.float64, device=plan.device))
            assert torch.equal(ins[0][torch.arange(R, device=plan.device), kin + 1 + cls],
                               torch.ones(R, dtype=torch.float64, device=plan.device))
        # ---- EPI_ELU_C8: hidden layers ----
        for i, s in enumerate(hs):
            A = ins[-1][:R, :s.kc]
            acc = A @ s.S.t()
            bias = s.bias[None, :].expand(R, -1)
            if s.cc:
                bias = bias + s.clsb[cls]
            x = acc + bias
            ex = acc_bound(A, s.S) + U * (acc.abs() + bias.abs()) * 2
            y, d = elu_ref(x, ex)
            w = s.rows
            H = c8(plan, "%s.H%d" % (blk, i), m, Rt)
            fc = H.shape[1]
            W.check("ELU_C8 %s.H%d" % (blk, i), H[:R, :w], y[:, :w], bf16_allow(y[:, :w], d[:, :w]))
            assert torch.equal(H[:R, w], torch.ones(R, dtype=torch.float64, device=plan.device)), "%s.H%d ones column" % (blk, i)
            assert not bool(H[:R, w + 1:].any()), "%s.H%d: nonzero beyond the ones column" % (blk, i)
            assert not bool(H[R:Rt].any()), "%s.H%d: nonzero rows beyond the dynamic count %d" % (blk, i, R)
            if regimes is not None and i == 0:
                regimes.setdefault("elu_saturated", 0)
                regimes["elu_saturated"] += int((H[:R, :w] == -1).sum())
            ins.append(H)
        # ---- head forward: EPI_STORE_F32 with the derived bias, or the decoder's EPI_DECLOSS ----
        A = ins[-1][:R, :head.kc]
        acc = A @ head.S.t()
        ea = acc_bound(A, head.S)
        if outname is not None:
            ld = 2 * head.ilv_block  # (mu | logvar) rows, the logvar half at round_up(out, 16), the -2 in the derived bias
            got = fp32_rows(plan, outname, m, R, ld)
            ref = (acc + head.bias[None, :])[:, :ld]
            allow = (ea + U * (acc.abs() + head.bias.abs()[None, :]))[:, :ld]
            if blk == "T":
                # T_post then adds z1 to the mu half in place (blocks.py:349-361, mu = z + z W_mu^T + bias_mu): one more
                # fp32 addition
                Zd = arch["dim_z1"]
                ref = ref.clone()
                ref[:, :Zd] += fp32_rows(plan, "Z1f", m, R, Zd)
                allow = allow.clone()
                allow[:, :Zd] += U * ref[:, :Zd].abs()
            W.check("STORE_F32 %s" % outname, got, ref, allow)
        else:
            dec_pre = (A, acc, ea)
            check_decloss(plan, head, A, acc, ea, cnt, X, m, W, regimes)
        # ---- head input gradient: EPI_DACT_C8 into dPre of the last hidden layer ----
        dY = c8(plan, dyname, m, Rt)
        if hs:
            for i in range(len(hs) - 1, -1, -1):
                Wl = head if i == len(hs) - 1 else hs[i + 1]
                G = dY[:R, :Wl.rcap] if i == len(hs) - 1 else c8(plan, "%s.dPre%d" % (blk, i + 1), m, Rt)[:R, :Wl.rcap]
                Sl = Wl.S[:G.shape[1]]
                acc_d = G @ Sl
                ed = G.shape[1] * U * (G.abs() @ Sl.abs())
                h = ins[i + 1][:R, :Sl.shape[1]]
                fac = torch.where(h > 0, torch.ones_like(h), h + 1)
                ref = acc_d * fac
                w = hs[i].rows
                d = ed * fac + 2 * U * acc_d.abs()
                D = c8(plan, "%s.dPre%d" % (blk, i), m, Rt)
                W.check("DACT_C8 %s.dPre%d" % (blk, i), D[:R, :w], ref[:, :w], bf16_allow(ref[:, :w], d[:, :w]))
                assert not bool(D[:R, w:].any()) and not bool(D[R:Rt].any()), "%s.dPre%d padding" % (blk, i)
        # ---- EPI_GRAD: weight, bias and class-column gradients of every GEMM layer ----
        layers = [(ins[i][:R], s, dY[:R, :s.rcap] if s is head else None, i) for i, s in enumerate(hs + [head])]
        for Xin, s, G, i in layers:
            if G is None:
                G = c8(plan, "%s.dPre%d" % (blk, i), m, Rt)[:R, :s.rcap]
            Xa = Xin[:, :s.kaug]
            ref = Xa.t() @ G  # [kaug, rcap]
            allow = R * U * (Xa.abs().t() @ G.abs()) + 1e-30
            for which, (wn, bn) in enumerate(zip(s.w, s.b)):
                rows = torch.tensor([s.srow(which, n) for n in range(s.rows)], device=plan.device)
                gw = gv[wn].to(torch.float64)
                r = ref[:, rows].t()  # [rows, kaug]: columns kin (ones) -> bias, kin+1.. -> class columns
                a = allow[:, rows].t()
                W.check("GRAD weight", gw[:, :s.kin], r[:, :s.kin], a[:, :s.kin])
                W.check("GRAD bias", gv[bn].to(torch.float64), r[:, s.kin], a[:, s.kin])
                if s.cc:
                    W.check("GRAD class column", gw[:, s.kin:], r[:, s.kin + 1:], a[:, s.kin + 1:])
    return cnt, dec_pre


def check_decloss(plan, head, A, acc, ea, cnt, X, m, W, regimes):
    """dY5 (both halves) and the dec_part row partials of EPI_DECLOSS.  Row -> target / coefficient as epi_begin maps
    them: L N reconstruction rows, L Np pair-reconstruction rows, L Np perturbation rows."""
    R = A.shape[0]
    N, Np, L = cnt[CNT["N"]], cnt[CNT["NP"]], plan.L
    hb = head.ilv_block
    f = torch.arange(X, device=plan.device)
    cmu = (f // hb) * 2 * hb + f % hb
    csg = cmu + hb
    coefs = plan.debug_buffer("coefs")[0][m].to(torch.float64)
    r = torch.arange(R, device=plan.device)
    LN, LNp = L * N, L * Np
    trow = torch.where(r < LN, r % N, N + (r - LN) % max(Np, 1))
    coef = torch.where(r < LN + LNp, coefs[COEF_RECL], coefs[COEF_PERT])
    tg, _, _ = plan.debug_buffer("tgt4")
    R0cap = plan.debug_buffer("Ain", torch.bfloat16)[1]
    Xc = round_up(X + 1, 16)
    tg = tg[m, :Xc * R0cap].view(Xc // 4, R0cap, 4).permute(1, 0, 2).reshape(R0cap, Xc)
    tgt = tg[trow, :X].to(torch.float64)
    mu = acc[:, cmu] + head.bias[cmu]
    s = acc[:, csg] + head.bias[csg]
    e_mu = ea[:, cmu] + U * (acc[:, cmu].abs() + head.bias[cmu].abs())
    e_s = ea[:, csg] + U * (acc[:, csg].abs() + head.bias[csg].abs())
    lp, dmu, dsg, blp, bmu, bsg = decloss_ref(mu, s, tgt, coef[:, None].expand(-1, X), e_mu, e_s)
    dY5 = c8(plan, "dY5", m, R)
    W.check("DECLOSS dY5 d/dmu", dY5[:, cmu], dmu, bf16_allow(dmu, bmu))
    W.check("DECLOSS dY5 d/dsigma-pre", dY5[:, csg], dsg, bf16_allow(dsg, bsg))
    part, _, _ = plan.debug_buffer("dec_part")
    Rdcap = plan.debug_buffer("Zdec", torch.bfloat16)[1]
    nparts = (head.rcap // (2 * hb)) * 4
    P = part[m, :nparts * Rdcap].view(nparts, Rdcap)[:, :R].to(torch.float64).sum(0)
    allow = blp.sum(1) + X * U * lp.abs().sum(1) + nparts * U * P.abs()
    W.check("DECLOSS dec_part row sums", P, lp.sum(1), allow)
    if regimes is not None:
        sv = s.detach()
        for name, lo, hi in (("s<-20", -1e30, -20), ("series s<-6.91", -20, math.log(1e-3)),
                             ("general", math.log(1e-3), 20), ("s>20", 20, 1e30)):
            regimes[name] = regimes.get(name, 0) + int(((sv >= lo) & (sv < hi)).sum())
        near = (sv - math.log(1e-3)).abs() < 0.5
        regimes["series side of ex=1e-3"] = regimes.get("series side of ex=1e-3", 0) + int((near & (sv < math.log(1e-3))).sum())
        regimes["lg2 side of ex=1e-3"] = regimes.get("lg2 side of ex=1e-3", 0) + int((near & (sv >= math.log(1e-3))).sum())
        regimes["lg2 path, 1e-2 <= ex < 1e-1"] = regimes.get("lg2 path, 1e-2 <= ex < 1e-1", 0) + int(
            ((sv >= math.log(1e-2)) & (sv < math.log(1e-1))).sum())
        regimes["|t|>100"] = regimes.get("|t|>100", 0) + int(((tgt - mu).abs() / (torch.nn.functional.softplus(s) + 1e-3) > 100).sum())


def check_dlogit(plan, kind, m, W, regimes=None):
    if kind == "pvae":
        return
    cnt = plan.debug_buffer("counts", torch.int32)[0][m].cpu().tolist()
    N, LN, Fl, Y = cnt[CNT["N"]], cnt[CNT["LN"]], cnt[CNT["FL"]], plan.dim_y
    q = fp32_rows(plan, "QY", m, LN, Y)
    got = fp32_rows(plan, "dlogit", m, LN, Y)
    i32 = lambda n: plan.debug_buffer(n, torch.int32)[0][m]
    lab, ycls, ebase = i32("lab")[:N].bool(), i32("ycls")[:N], i32("ebase")[:N].long()
    kfp = plan.debug_buffer("kfp_row")[0][m].to(torch.float64)
    coefs = plan.debug_buffer("coefs")[0][m].to(torch.float64)
    r = torch.arange(LN, device=plan.device)
    l, i = r // N, r % N
    idx = (l * Fl)[:, None] + ebase[i][:, None] + torch.arange(Y, device=plan.device)[None, :]
    ke = kfp[idx.clamp_max(kfp.numel() - 1)]
    dl, allow = dlogit_ref(q, lab[i], ycls[i], ke, coefs[COEF_YL], coefs[COEF_KLD], math.log(1.0 / Y))
    W.check("dlogit (float32 clamp semantics)", got, dl, allow + 1e-45)
    if regimes is not None:
        regimes["rows q == 1.0f"] = regimes.get("rows q == 1.0f", 0) + int((q == 1.0).any(1).sum())
        regimes["rows q == 1.0f, none clamped"] = regimes.get("rows q == 1.0f, none clamped", 0) + int(
            ((q == 1.0).any(1) & (q > F32_1E10).all(1)).sum())
        regimes["rows clamped at 1e-10"] = regimes.get("rows clamped at 1e-10", 0) + int((q <= F32_1E10).any(1).sum())


def check_decout(plan, kind, arch, sd, x1, m, W, regimes=None):
    """EPI_DECOUT: bf16 inference's px1_mu / px1_sg from the decoder activation the inference left behind."""
    specs = shadow_specs(kind, arch)
    read_weights(plan, specs, sd, m)
    head = specs["dec"][1]
    X, N = arch["dim_x"], x1.shape[-2]
    plan.set_infer_precision(False)
    res = plan.infer(x1)
    plan.set_infer_precision(True)
    torch.cuda.synchronize()
    nh = len(arch["dec_x"])
    A = c8(plan, "dec.H%d" % (nh - 1), m, N)[:, :head.kc]
    acc = A @ head.S.t()
    ea = acc_bound(A, head.S)
    hb = head.ilv_block
    f = torch.arange(X, device=plan.device)
    cmu = (f // hb) * 2 * hb + f % hb
    csg = cmu + hb
    mu = acc[:, cmu] + head.bias[cmu]
    s = acc[:, csg] + head.bias[csg]
    W.check("DECOUT px1_mu", res["px1_mu"][m].double(), mu, ea[:, cmu] + U * (acc[:, cmu].abs() + head.bias[cmu].abs()))
    sg = torch.nn.functional.softplus(s, threshold=20.0) + 1e-3
    es = ea[:, csg] + U * (acc[:, csg].abs() + head.bias[csg].abs())
    # expf / log1pf: 2 ulp each (CUDA C Programming Guide); the softplus slope is at most 1; + the 1e-3 addition
    W.check("DECOUT px1_sg", res["px1_sg"][m].double(), sg, es + 8 * U * sg)


# ---- part 1: architectures, batches ----------------------------------------------------------------------------------
def _arch(dim_x, z1, z3, h, dim_y=2):
    return dict(dim_x=dim_x, dim_y=dim_y, dim_z1=z1, dim_z3=z3, enc_z1=[h], dec_x=[h], enc_z3=[h], dec_z1=[h])


# id -> (architecture, N, L, members)
CASES = {
    "readme": (ARCH["readme"], 150, 2, 1),        # X = 978: the last decoder tile (978 = 7 x 128 + 82) takes the masked path
    "x16": (_arch(96, 12, 10, 40), 24, 2, 1),     # X = 96: one decoder tile, every chunk on the unmasked fast path
    "ragged": (dict(ARCH["deep"]), 37, 2, 1),    # N = 37 rows and two hidden layers per block (dPre chain, H1 from H0)
    "ens2": (ARCH["tiny"], 24, 2, 2),             # two members, different parameters and batches
}


def make_batch(kind, arch, N, seed):
    return orc.synthetic_batch(N, arch["dim_x"], seed=seed, dim_y=arch["dim_y"])


def random_draws(kind, batch, arch, L, seed):
    g = torch.Generator().manual_seed(seed)
    shapes = tape_shapes(kind, batch["has_x2"], batch["has_y"], arch["dim_x"], arch["dim_z1"], arch["dim_z3"],
                         arch["dim_y"], L, noisy=True)
    return [torch.randn(*s, generator=g) for s in shapes]


def plain_plan(kind, arch, N, L, E):
    plan = Plan(kind, L=L, max_batch=N, n_models=E, **arch)
    plan.set_graph(False)
    plan.set_step_kernel(False)
    plan.set_gemm_impl("tc")
    return plan


def run_grad_step(plan, kind, arch, sds, batches, L, hp_kw=None, tapes=None):
    E = len(sds)
    for m in range(E):
        plan.load_state_dict(sds[m], model=m)
    epss = []
    for m in range(E):
        draws = tapes[m] if tapes is not None else random_draws(kind, batches[m], arch, L, seed=50 + m)
        epss.append(eps_block_from_tape(plan, draws, batches[m]["has_x2"], batches[m]["has_y"], noisy=True))
    if E == 1:
        fields, eps = batch_fields(kind, batches[0]), epss[0]
    else:
        fl = [batch_fields(kind, b) for b in batches]
        fields = {k: torch.stack([f[k] for f in fl]).contiguous() for k in fl[0]}
        eps = torch.stack(epss)
    losses = plan.grad_step(fields, plan.hparams(step=1, **(hp_kw or {})), eps=eps)
    torch.cuda.synchronize()
    return losses


P1 = [(c, k) for c in CASES for k in KINDS]


@pytest.mark.parametrize("case,kind", P1, ids=["%s-%s" % ck for ck in P1])
def test_every_epilogue_element_matches_float64(case, kind):
    arch, N, L, E = CASES[case]
    plan = plain_plan(kind, arch, N, L, E)
    sds = [init_state_dict(kind, seed=SEED_MODEL + m, **arch) for m in range(E)]
    batches = [make_batch(kind, arch, N, seed=5 + m) for m in range(E)]
    run_grad_step(plan, kind, arch, sds, batches, L)
    W = Worst()
    for m in range(E):
        check_step_elements(plan, kind, arch, sds[m], m, W)
        check_dlogit(plan, kind, m, W)
    x1 = torch.stack([b["x1"] for b in batches]) if E > 1 else batches[0]["x1"]
    for m in range(E):
        check_decout(plan, kind, arch, sds[m], x1, m, W)
    W.report("%s %s" % (case, kind))
    if case == "readme":
        assert arch["dim_x"] % 16 != 0  # the masked last chunk ran
    if case == "x16":
        assert arch["dim_x"] % 16 == 0


# ---- part 2: a trained-like parameter set ----------------------------------------------------------------------------
# decoder sigma pre-activations, cycled over the features: ex = e^s vanishes against 1 (and sigma sits at its 1e-3
# floor); the log1p series (ex < 1e-3) far from and just below its cutoff; just above it; ex = 0.08, where the series
# would be off by 2e-3 relative and the lg2 path must be taken; the general path; both sides of the softplus threshold
SIGMA_PRE = (-40.0, -12.0, -7.2, -6.6, -2.5, -2.0, 0.0, 5.0, 19.5, 20.5, 35.0)
T_ARCH, T_N, T_L = ARCH["readme"], 150, 2


def trained_like(kind, arch, batch):
    """init_state_dict edited into the regimes of a trained model (module docstring)."""
    sd = init_state_dict(kind, seed=SEED_MODEL, **arch)
    X = arch["dim_x"]
    # decoder sigma: pre-activation = bias (per feature, cycling through SIGMA_PRE) + a small weight term
    sd["decoder_x.encoder_sg.linear_sg.weight"] *= 1e-3
    sd["decoder_x.encoder_sg.linear_sg.bias"] = torch.tensor([SIGMA_PRE[f % len(SIGMA_PRE)] for f in range(X)])
    # decoder mu pulled away from the targets: t = (x - mu) / sigma in the hundreds where sigma sits at its floor
    sd["decoder_x.encoder_mu.linear_mu.bias"] += 0.5
    # every third unit of the decoder's first hidden layer saturates its ELU at -1
    b = sd["decoder_x.nnet.model.linear1.bias"]
    b[::3] = -30.0
    if kind != "pvae":
        # classifier: logit gap of class 1 over class 0 = c (u_0 - mean) + small: spread over [0, > 30]
        om = orc.OracleModel(sd, orc.default_cfg(kind, L=T_L), dtype=torch.float64)
        z = om.forward(batch["x1"])["z1"][:, 0]
        spread = math.sqrt(float(z.var()) + math.exp(-2.0))
        W = sd["encoder_y.decoder_p.linear_p.weight"]
        W[1] = W[0]
        W[1, 0] += 16.0 / spread
        sd["encoder_y.decoder_p.linear_p.bias"][1] = sd["encoder_y.decoder_p.linear_p.bias"][0] - 16.0 / spread * float(z.mean())
    return sd


def trained_batch(kind, arch):
    return orc.synthetic_batch(T_N, arch["dim_x"], seed=5, dim_y=arch["dim_y"])


class TrainedRun:
    def __init__(self, kind, kl_min):
        arch = T_ARCH
        self.batch = trained_batch(kind, arch)
        self.sd = trained_like(kind, arch, self.batch)
        cfg = orc.default_cfg(kind, L=T_L, dim_y=arch["dim_y"], kl_min=kl_min)
        om = orc.OracleModel(self.sd, cfg, dtype=torch.float64)
        om.iters = 1
        tape = orc.Tape(seed=901)
        self.lo_emu, self.g_emu = om.grads(self.batch, tape, emulate_bf16=True)
        self.tape = tape.log
        etape = orc.Tape(seed=902)
        self.lo_eval = om.loss(self.batch, etape, train=False, emulate_bf16=True)
        self.eval_tape = etape.log
        self.fwd = om.forward(self.batch["x1"])


_KL_MEDIAN = {}


def kl_values(plan, kind, batch):
    """Per-row values a free-bits mask decides, as the step stored them, and the multiple of kl_min that means
    "floored": klz2_row (max(KL(q(z2|x2) || p(z2|z1)), kl_min) of the pair rows, rows l N + i), or for VFAE kfp_row
    (per evaluation max(KL3, kl_min) + max(KL1, kl_min): 2 kl_min exactly when both terms are floored)."""
    cnt = plan.debug_buffer("counts", torch.int32)[0][0].cpu().tolist()
    if kind == "vfae":
        return plan.debug_buffer("kfp_row")[0][0, :cnt[CNT["F"]]].double().cpu(), 2.0
    v = plan.debug_buffer("klz2_row")[0][0, :cnt[CNT["LN"]]].double().cpu()
    return v[batch["has_x2"].bool().repeat(plan.L)], 1.0


def kl_terms_vfae(plan):
    """max(KL(q(z2|z1,y) || N(0, I)), KL(q(z1|x1) || p(z1|z2,y))) per evaluation, in float64 from the heads the step
    stored (Q3, Q, PZ1): an evaluation is fully floored exactly when kl_min is at least this value."""
    cnt = plan.debug_buffer("counts", torch.int32)[0][0].cpu().tolist()
    F, Fl = cnt[CNT["F"]], cnt[CNT["FL"]]
    Z, Z3 = plan.dim_z1, plan.dim_z3
    Zs, Z3s = round_up(Z, 16), round_up(Z3, 16)
    q3 = fp32_rows(plan, "Q3", 0, F, 2 * Z3s)
    pz = fp32_rows(plan, "PZ1", 0, F, 2 * Zs)
    q1 = fp32_rows(plan, "Q", 0, cnt[CNT["R0"]], 2 * Zs)
    i = plan.debug_buffer("e_row", torch.int32)[0][0, :Fl].long().repeat(F // Fl)
    mu3, lv3 = q3[:, :Z3], q3[:, Z3s:Z3s + Z3]
    k3 = -0.5 * (1 + lv3 - mu3 ** 2 - lv3.exp()).sum(1)
    m1, l1, mp, lp = q1[i, :Z], q1[i, Zs:Zs + Z], pz[:, :Z], pz[:, Zs:Zs + Z]
    k1 = -0.5 * (1 - lp + l1 - ((m1 - mp) ** 2 + l1.exp()) / lp.exp()).sum(1)
    return torch.maximum(k3, k1).cpu()


def kl_min_value(kind, which):
    """kl_min of a parametrisation: 0, 1e4 (every row floored), or the median over the rows of what the mask decides,
    read from a kl_min = 0 step (for VFAE the larger of an evaluation's two KLs, so that half the evaluations have
    both terms floored and half do not)."""
    if which == "zero":
        return 0.0
    if which == "all":
        return 1e4
    if kind not in _KL_MEDIAN:
        arch = T_ARCH
        plan = plain_plan(kind, arch, T_N, T_L, 1)
        b = trained_batch(kind, arch)
        sd = trained_like(kind, arch, b)
        run_grad_step(plan, kind, arch, [sd], [b], T_L, hp_kw=dict(kl_min=0.0))
        v = kl_terms_vfae(plan) if kind == "vfae" else kl_values(plan, kind, b)[0]
        _KL_MEDIAN[kind] = float(np.float32(v.median()))
    return _KL_MEDIAN[kind]


P2 = [(k, w) for k in KINDS for w in ("zero", "median", "all")]


@pytest.mark.parametrize("kind,klm", P2, ids=["%s-klmin_%s" % p for p in P2])
def test_trained_regimes_match_the_float64_oracle(kind, klm):
    kl_min = kl_min_value(kind, klm)
    o = TrainedRun(kind, kl_min)
    arch = T_ARCH
    plan = plain_plan(kind, arch, T_N, T_L, 1)
    losses = run_grad_step(plan, kind, arch, [o.sd], [o.batch], T_L, hp_kw=dict(kl_min=kl_min), tapes=[o.tape])
    got = {k: float(v) for k, v in losses_to_dict(kind, losses[0].cpu()).items()}
    for k, ref in o.lo_emu.items():
        if k == "MMD":
            continue
        ref = float(ref)
        assert abs(got[k] - ref) <= 5e-5 * abs(ref) + 1e-6, "%s %s: gpu %.7g oracle %.7g" % (kind, k, got[k], ref)
    gv = plan.tensor_views(plan.grads, 0)
    for name, g in o.g_emu.items():
        if float(g.norm()) == 0:
            assert float(gv[name].norm()) == 0, name
            continue
        assert_grad_close(gv[name], g, "%s kl_min=%g grad %s" % (kind, kl_min, name))
    # the element checks at this parameter set, and the regimes they claim to cover
    W = Worst()
    regimes = {}
    check_step_elements(plan, kind, arch, o.sd, 0, W, regimes)
    check_dlogit(plan, kind, 0, W, regimes)
    # free bits on both sides of kl_min
    v, scale = kl_values(plan, kind, o.batch)
    floor = scale * float(np.float32(kl_min))  # (the step compares with kl_min as a float32)
    n_floor, n_above = int((v <= floor).sum()), int((v > floor).sum())
    regimes["KL rows floored"], regimes["KL rows above kl_min"] = n_floor, n_above
    W.report("trained %s kl_min=%g" % (kind, kl_min))
    print("  regimes: %s" % regimes)
    for r in ("s<-20", "series s<-6.91", "general", "s>20", "lg2 path, 1e-2 <= ex < 1e-1", "|t|>100", "elu_saturated"):
        assert regimes[r] > 0, "regime %s not reached" % r
    # both sides of ex = 1e-3 (s = ln 1e-3 = -6.91), where the log1p series hands over to lg2
    assert regimes["series side of ex=1e-3"] > 0 and regimes["lg2 side of ex=1e-3"] > 0
    if kind != "pvae":
        assert regimes["rows q == 1.0f, none clamped"] > 0, "no row with a logit gap in (16.6, 23.03)"
        assert regimes["rows clamped at 1e-10"] > 0, "no row with a logit gap beyond 23.03"
    if klm == "zero":
        assert n_above > 0
    elif klm == "median":
        assert n_floor > 0 and n_above > 0, (n_floor, n_above)
    else:
        assert n_above == 0 and n_floor > 0


@pytest.mark.parametrize("kind", KINDS)
def test_trained_regimes_eval_inference_and_fused_optimizer(kind):
    arch = T_ARCH
    kl_min = kl_min_value(kind, "median")
    o = TrainedRun(kind, kl_min)
    plan = plain_plan(kind, arch, T_N, T_L, 1)
    plan.load_state_dict(o.sd)
    eps = eps_block_from_tape(plan, o.eval_tape, o.batch["has_x2"], o.batch["has_y"], noisy=False)
    got = plan.loss_forward(batch_fields(kind, o.batch), plan.hparams(step=1, training=False, kl_min=kl_min), eps=eps)
    got = {k: float(v) for k, v in losses_to_dict(kind, got[0].cpu()).items()}
    for k, ref in o.lo_eval.items():
        if k != "MMD":
            assert abs(got[k] - float(ref)) <= 5e-5 * abs(float(ref)) + 1e-6, "eval %s %s: %.7g vs %.7g" % (kind, k, got[k], float(ref))
    res = plan.infer(o.batch["x1"])
    fr = o.fwd
    want = dict(z1_mu=fr["z1"], z1_lv=fr["qz1"][1], px1_mu=fr["x1_rec"], px1_sg=fr["px1"][1])
    if kind != "vfae":
        want.update(z2_mu=fr["z2"], z2_lv=fr["pz2"][1], px2_mu=fr["x2_pert"], px2_sg=fr["px2"][1])
    if kind != "pvae":
        want["proba"] = fr["proba"]
    for k, ref in want.items():
        a = res[k][0].cpu().double()
        bad = (a - ref).abs() > 2e-6 + 2e-5 * ref.abs()
        if k == "proba":
            # the float64 oracle clamps at 1 - 1e-10, which float32 rounds to 1.0: compare at float32 resolution
            bad = (a - ref.float().double()).abs() > 2e-6 + 2e-5 * ref.abs()
        assert not bool(bad.any()), "%s infer %s: %d elements off" % (kind, k, int(bad.sum()))
    # the fused optimizer against gradient + stand-alone Adam in this regime: the same losses bit for bit; parameters and
    # moments to the criterion of test_arch_envelope_gpu.py (the grouped dW+Adam launch sums the weight gradient in its
    # own order)
    fields = batch_fields(kind, o.batch)
    out = {}
    for mode in ("fused", "split"):
        p = plain_plan(kind, arch, T_N, T_L, 1)
        p.load_state_dict(o.sd)
        hp = p.hparams(step=0, kl_min=kl_min)
        if mode == "fused":
            lo = p.train_step(fields, hp, seed=17).cpu().clone()
        else:
            lo = p.grad_step(fields, hp, seed=17).cpu().clone()
            p.adam_step(hp)
        torch.cuda.synchronize()
        out[mode] = (lo, p.params.cpu().clone(), p.adam_m.cpu().clone(), p.adam_v.cpu().clone())
    assert torch.equal(out["fused"][0], out["split"][0]), "%s: fused step losses differ" % kind
    for a, b, name in zip(out["fused"][1:], out["split"][1:], ("params", "adam_m", "adam_v")):
        bad = ~torch.isclose(a, b, rtol=1e-6, atol=1e-9)
        assert not bool(bad.any()), "%s: %d fused %s entries differ from grad_step + adam_step" % (kind, int(bad.sum()), name)
