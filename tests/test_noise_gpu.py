"""The step's own noise (drvae_noise_t.eps == NULL) element by element against the host reference (tests/philox_ref.py).

philox_normal_kernel writes the latent draws (z1, z2, z2f, z3) to the plan's ε block; prep_kernel draws the input noise
of x1 / x2 itself and only its sum with the input is stored, in the fp32 reconstruction targets (tgt4).  Both are
recomputed here for every (model, MC sample, row, position): the Philox integers exactly, Box-Muller in float64 with a
per-element allowance built from the PTX ISA bounds of lg2.approx / sqrt.approx / sin.approx / cos.approx, the fp32
argument reduction of sin / cos for angles beyond pi, and one fp32 rounding per multiply (philox_ref.normals).  No bound is fitted to an observed error; each check prints its worst ratio
of error to allowance.  Negative controls move one key field by one and require the allowance to reject the result.

Then: nothing outside the written region changes and no consumer reads it; default launches, graph replay and the
persistent step kernel draw the same bits, replays take each call's keys; eval mode and add_noise=False; and the
generator's block, fed back as a caller's block and as an oracle tape, gives the same step."""
import math

import numpy as np
import pytest
import torch

from helpers import ARCH, assert_grad_close, batch_fields, orc
from philox_ref import U32, normals
from test_step_gpu import TOL_EMU_LOSS, check_losses, loss_dict

from drvae_b200.init import init_state_dict
from drvae_b200.noise import group_indices
from drvae_b200.plan import Plan, anneal_coef

pytestmark = pytest.mark.gpu

SEG = dict(x1=0, x2=1, z1=2, z2=3, z2f=4, z3=5)  # draw kind = segment index of the eps layout
LATENT = ("z1", "z2", "z2f", "z3")
SEED_A = 0x0123456789ABCDEF  # both 32-bit halves non-zero


def _arch(dim_x, dim_y, dim_z1, dim_z3):
    return dict(dim_x=dim_x, dim_y=dim_y, dim_z1=dim_z1, dim_z3=dim_z3, enc_z1=[24], dec_x=[20], enc_z3=[16], dec_z1=[12])


# store: the branch philox_normal_kernel takes per drawn segment, "f2" (even width at an even offset: float2 pairs) or
# "scalar"; asserted against the plan's eps_layout
CASES = dict(
    # odd widths everywhere; L Ncap Z = 3 * 45 * 13 is odd, so z2 and z3 start at odd offsets; Y Z3 = 21 odd
    drvae_odd=dict(kind="drvae", arch=_arch(37, 3, 13, 7), L=3, Ncap=45, N=41, E=3, noise_std=(0.01, 0.05, 0.2),
                   seed=SEED_A, step=2 ** 31 - 1, row_offset=2 ** 32 + 3,
                   store=dict(z1="scalar", z2="scalar", z2f="scalar", z3="scalar")),
    # an even z3 width (Y Z3 = 18) at an odd offset: the scalar branch although the width is even
    vfae_odd_offset=dict(kind="vfae", arch=_arch(41, 3, 13, 6), L=3, Ncap=45, N=37, E=1, noise_std=None,
                         seed=0, step=0, row_offset=1000, store=dict(z1="scalar", z3="scalar")),
    # widths = 2 mod 4 (the last quad stores half a float2); dim_x 300 crosses prep's 256-feature slab; 3 blocks
    # per latent segment
    drvae_half_quad=dict(kind="drvae", arch=_arch(300, 3, 14, 6), L=3, Ncap=64, N=64, E=1, noise_std=None,
                         seed=(7 << 32) | 9, step=5, row_offset=2 ** 32 + 3,
                         store=dict(z1="f2", z2="f2", z2f="f2", z3="f2")),
    # widths multiple of 4; L = 256 reaches the top bits of the sample index; one row
    drvae_L256=dict(kind="drvae", arch=_arch(40, 2, 16, 10), L=256, Ncap=4, N=1, E=1, noise_std=None,
                    seed=0xFFFFFFFF00000001, step=3, row_offset=0, store=dict(z1="f2", z2="f2", z2f="f2", z3="f2")),
    pvae=dict(kind="pvae", arch=_arch(41, 2, 12, 10), L=2, Ncap=96, N=70, E=2, noise_std=(0.03, 0.01),
              seed=SEED_A, step=2 ** 31 - 1, row_offset=1000, store=dict(z1="f2", z2="f2", z2f="f2")),
)
PRODUCTION = dict(
    readme_8192=dict(kind="drvae", arch=ARCH["readme"], L=2, Ncap=8192, N=8192, E=1, noise_std=None,
                     seed=SEED_A, step=17, row_offset=2 ** 32 + 3),
    readme_150x32=dict(kind="drvae", arch=ARCH["readme"], L=2, Ncap=150, N=150, E=32, noise_std=None,
                       seed=12345, step=3, row_offset=0),
)
# key fields a wrong kernel could confuse; each must make the reference disagree almost everywhere
CONTROLS = ("row", "sample", "model", "kind", "step", "seed_lo", "seed_hi", "row_offset", "quad")


# ---- shapes ---------------------------------------------------------------------------------------------------------
def eps_widths(kind, arch):
    """Floats per row of each latent segment in the layout, and whether the kind draws it (plan.cu launch_noise)."""
    Z = arch["dim_z1"]
    Y, Z3 = (1, 1) if kind == "pvae" else (arch["dim_y"], arch["dim_z3"])
    return dict(z1=(Z, True), z2=(Z, kind != "vfae"), z2f=(Z, kind != "vfae"), z3=(Y * Z3, kind != "pvae"))


def eps_offsets(kind, arch, L, Ncap):
    """drvae_eps_layout_t as plan.cu builds it."""
    w = eps_widths(kind, arch)
    off = dict(x1=0, x2=Ncap * arch["dim_x"])
    off["z1"] = 2 * Ncap * arch["dim_x"]
    off["z2"] = off["z1"] + L * Ncap * w["z1"][0]
    off["z2f"] = off["z2"] + L * Ncap * w["z2"][0]
    off["z3"] = off["z2f"] + L * Ncap * w["z2f"][0]
    off["total"] = off["z3"] + L * Ncap * w["z3"][0]
    return off


def store_branch(width, offset):
    return "f2" if width % 2 == 0 and offset % 2 == 0 else "scalar"


# ---- plans and batches ----------------------------------------------------------------------------------------------
def make_plan(c, seed_model=123):
    plan = Plan(c["kind"], L=c["L"], max_batch=c["Ncap"], n_models=c["E"], **c["arch"])
    sd = init_state_dict(c["kind"], seed=seed_model, **c["arch"])
    for m in range(c["E"]):
        plan.load_state_dict(sd, model=m)
    if c["noise_std"] is not None:
        ny = max(1, c["arch"]["dim_y"])
        plan.set_member_hparams([dict(yloss_rate=1.0, pertloss_rate=0.05, kl_qz2pz2_rate=1.0, noise_std=s, lr=5e-4,
                                      weight_decay=0.05, prior_y=[1.0 / ny] * ny) for s in c["noise_std"]])
    return plan


def noise_std(c, m):
    """The fp32 std prep_kernel multiplies by: the member table's value, else drvae_hparams_t.noise_std (0.01)."""
    return float(np.float32(c["noise_std"][m] if c["noise_std"] is not None else 0.01))


def make_batch(c, seed=5):
    """Device batch [E, N, ...]; pairs in an irregular pattern so that the pair rows' order is visible."""
    parts = []
    for m in range(c["E"]):
        b = orc.synthetic_batch(c["N"], c["arch"]["dim_x"], seed=seed + m, dim_y=max(2, c["arch"]["dim_y"]))
        g = torch.Generator().manual_seed(100 + seed + m)
        b["has_x2"] = (torch.rand(c["N"], generator=g) < 0.6).int()
        b["x2"][b["has_x2"] == 0] = 0
        parts.append(b)
    cpu = {k: torch.stack([p[k] for p in parts]) for k in parts[0]}
    dev = {k: v.cuda() for k, v in batch_fields(c["kind"], cpu).items()}
    return cpu, dev


# ---- references -----------------------------------------------------------------------------------------------------
def _keys(seed, step, row_offset, control):
    """(seed, step, row_offset, d_model, d_sample, d_kind, row_xor, d_quad) with one field moved by one."""
    d = dict(model=0, sample=0, kind=0, row=0, quad=0)
    if control == "step":
        step = (step + 1) % 2 ** 32
    elif control == "seed_lo":
        seed = (seed & ~0xFFFFFFFF) | ((seed + 1) & 0xFFFFFFFF)
    elif control == "seed_hi":
        seed = (seed + (1 << 32)) % 2 ** 64
    elif control == "row_offset":
        row_offset += 1
    elif control is not None:
        d[control] = 1
    return seed, step, row_offset, d


def latent_reference(c, seg, width, seed, step, row_offset, control=None):
    """-> (z, allowance), each [E, L, N, width]."""
    seed, step, row_offset, d = _keys(seed, step, row_offset, control)
    E, L, N = c["E"], c["L"], c["N"]
    Q = (width + 3) // 4
    m = np.arange(E).reshape(E, 1, 1, 1) + d["model"]
    l = np.arange(L).reshape(1, L, 1, 1) + d["sample"]
    grow = row_offset + (np.arange(N) ^ d["row"]).reshape(1, 1, N, 1)
    q = np.arange(Q).reshape(1, 1, 1, Q) + d["quad"]
    z, a = normals(seed, step, m, SEG[seg] + d["kind"], l, grow, q)
    return z.reshape(E, L, N, 4 * Q)[..., :width], a.reshape(E, L, N, 4 * Q)[..., :width]


def input_reference(X, seed, step, model, kind, rows, row_offset, control=None):
    """Input noise of the rows `rows` (key rows row_offset + rows) of one model -> (z, allowance) [len(rows), X]."""
    seed, step, row_offset, d = _keys(seed, step, row_offset, control)
    Q = (X + 3) // 4
    grow = row_offset + (np.asarray(rows, dtype=np.int64) ^ d["row"])[:, None]
    q = np.arange(Q)[None, :] + d["quad"]
    z, a = normals(seed, step, model + d["model"], kind + d["kind"], d["sample"], grow, q)
    return z.reshape(len(rows), 4 * Q)[:, :X], a.reshape(len(rows), 4 * Q)[:, :X]


def noisy_input(x, s, z, a):
    """fl32(x + fl32(s z)) and its allowance: s times the normal's, one rounding each for the product and the sum in
    the kernel (fused or not) and in this reference; (1 + 4u) covers the second-order terms."""
    ref = (x + (s * z).astype(np.float32)).astype(np.float64)
    sz = s * (np.abs(z) + a)
    return ref, (s * a + 2 * U32 * sz + 2 * U32 * (np.abs(x.astype(np.float64)) + sz)) * (1 + 4 * U32)


def _assert_within(got, ref, allow, tag, where):
    err = np.abs(got - ref)
    ratio = np.where(err <= allow, err / allow, np.inf)  # NaN in got -> inf
    worst = float(ratio.max()) if ratio.size else 0.0
    if not worst <= 1.0:
        i = np.unravel_index(int(np.argmax(ratio)), ratio.shape)
        raise AssertionError("%s: element %s (%s): got %r, reference %r, allowance %.3e" % (
            tag, i, where, float(got[i]), float(ref[i]), float(allow[i])))
    return worst


def read_eps(plan):
    return plan.debug_buffer("eps")[0].double().cpu().numpy()


def read_targets(plan, X):
    tg = plan.debug_buffer("tgt4")[0]
    Xc = (X + 1 + 15) // 16 * 16
    R0cap = tg.shape[1] // Xc
    return tg.reshape(plan.E, Xc // 4, R0cap, 4).permute(0, 2, 1, 3).reshape(plan.E, R0cap, Xc)[:, :, :X].cpu().numpy()


def latent_view(eps, c, seg):
    off = eps_offsets(c["kind"], c["arch"], c["L"], c["Ncap"])
    w = eps_widths(c["kind"], c["arch"])[seg][0]
    return eps[:, off[seg]:off[seg] + c["L"] * c["Ncap"] * w].reshape(c["E"], c["L"], c["Ncap"], w)


def check_latents(eps, c, seed, step, row_offset, tag, controls=False):
    worst = 0.0
    for seg in LATENT:
        w, drawn = eps_widths(c["kind"], c["arch"])[seg]
        if not drawn:
            continue
        got = latent_view(eps, c, seg)[:, :, :c["N"]]
        ref, allow = latent_reference(c, seg, w, seed, step, row_offset)
        worst = max(worst, _assert_within(got, ref, allow, "%s %s" % (tag, seg), "model, sample, row, position"))
        if controls:
            for ctl in CONTROLS:
                bad, _ = latent_reference(c, seg, w, seed, step, row_offset, control=ctl)
                agree = float(np.mean(np.abs(got - bad) <= allow))
                print("  control %-10s %-3s agreement %.4f" % (ctl, seg, agree))
                assert agree < 0.01, "%s %s: the reference with %s moved by one matches %.1f%% of the elements" % (
                    tag, seg, ctl, 100 * agree)
    print("noise %s latent: worst error / allowance %.3f" % (tag, worst))
    return worst


def input_rows(c, cpu, m):
    """(kind, key rows, fp32 inputs) of the stacked encoder rows of model m: x1 rows 0..N, then the pairs' x2 rows in
    row order (the order rowmap's row_of_pair lists them)."""
    N = c["N"]
    out = [(SEG["x1"], np.arange(N), cpu["x1"][m].numpy())]
    if c["kind"] != "vfae":
        pr = np.nonzero(cpu["has_x2"][m].numpy())[0]
        out.append((SEG["x2"], pr, cpu["x2"][m].numpy()[pr]))
    return out


def check_inputs(tgt, c, cpu, seed, step, row_offset, noisy, tag, controls=False):
    X, N, worst = c["arch"]["dim_x"], c["N"], 0.0
    for m in range(c["E"]):
        r0 = 0
        for kind, rows, x in input_rows(c, cpu, m):
            got = tgt[m, r0:r0 + len(rows)]
            r0 += len(rows)
            if not noisy:
                assert np.array_equal(got, x), "%s: model %d kind %d rows are not the inputs bit for bit" % (tag, m, kind)
                continue
            s = noise_std(c, m)
            z, a = input_reference(X, seed, step, m, kind, rows, row_offset)
            ref, allow = noisy_input(x, np.float32(s), z, a)
            worst = max(worst, _assert_within(got.astype(np.float64), ref, allow, "%s model %d kind %d" % (tag, m, kind),
                                              "row, feature"))
            if controls and m == 0:
                for ctl in CONTROLS:
                    if ctl == "sample":  # the input draws have no sample index (l = 0)
                        continue
                    zb, _ = input_reference(X, seed, step, m, kind, rows, row_offset, control=ctl)
                    bad, _ = noisy_input(x, np.float32(s), zb, a)
                    agree = float(np.mean(np.abs(got - bad) <= allow))
                    assert agree < 0.01, "%s kind %d: the reference with %s moved by one matches %.1f%% of the elements" % (
                        tag, kind, ctl, 100 * agree)
        assert r0 == (N if c["kind"] == "vfae" else N + int(cpu["has_x2"][m].sum()))
    if noisy:
        print("noise %s input: worst error / allowance %.3f" % (tag, worst))
    return worst


def written(eps, tgt, c, cpu):
    """Everything the generator writes: the drawn latent rows < N and the stacked encoder input rows < R0."""
    out = [latent_view(eps, c, s)[:, :, :c["N"]] for s in LATENT if eps_widths(c["kind"], c["arch"])[s][1]]
    for m in range(c["E"]):
        R0 = sum(len(rows) for _, rows, _ in input_rows(c, cpu, m))
        out.append(tgt[m, :R0])
    return out


def same_bits(a, b):
    return all(x.shape == y.shape and np.array_equal(x.view(np.int64 if x.dtype == np.float64 else np.int32),
                                                     y.view(np.int64 if y.dtype == np.float64 else np.int32))
               for x, y in zip(a, b))


def run_and_read(plan, c, dev, seed, step, row_offset, fn="loss_forward", **hp):
    getattr(plan, fn)(dev, plan.hparams(step=step, **hp), seed=seed, row_offset=row_offset)
    torch.cuda.synchronize()
    return read_eps(plan), read_targets(plan, c["arch"]["dim_x"])


# ---- tests ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(CASES))
def test_own_noise_element_by_element(name):
    c = CASES[name]
    plan = make_plan(c)
    el = plan.eps_layout
    off = eps_offsets(c["kind"], c["arch"], c["L"], c["Ncap"])
    assert [el.off_x1, el.off_x2, el.off_z1, el.off_z2, el.off_z2f, el.off_z3, el.total] == [
        off[k] for k in ("x1", "x2", "z1", "z2", "z2f", "z3", "total")]
    widths = eps_widths(c["kind"], c["arch"])
    assert {s: store_branch(widths[s][0], off[s]) for s in LATENT if widths[s][1]} == c["store"]
    cpu, dev = make_batch(c)
    eps, tgt = run_and_read(plan, c, dev, c["seed"], c["step"], c["row_offset"], fn="train_step")
    check_latents(eps, c, c["seed"], c["step"], c["row_offset"], name, controls=True)
    check_inputs(tgt, c, cpu, c["seed"], c["step"], c["row_offset"], True, name, controls=True)


@pytest.mark.parametrize("name", list(PRODUCTION))
def test_own_noise_production_shapes(name):
    c = PRODUCTION[name]
    plan = make_plan(c)
    cpu, dev = make_batch(c)
    eps, tgt = run_and_read(plan, c, dev, c["seed"], c["step"], c["row_offset"])
    check_latents(eps, c, c["seed"], c["step"], c["row_offset"], name)
    check_inputs(tgt, c, cpu, c["seed"], c["step"], c["row_offset"], True, name)


@pytest.mark.parametrize("name", ("drvae_odd", "vfae_odd_offset", "pvae"))
def test_own_noise_writes_only_its_region_and_nothing_reads_past_it(name):
    """The ε block is filled with NaN before a step with N < max_batch: afterwards everything the generator does not
    draw is still NaN (rows >= N of every sample, the input-noise segments, the segments the kind has no use for), and
    the step's losses and gradients equal those of the same step on a fresh plan."""
    c = CASES[name]
    assert c["N"] < c["Ncap"]
    cpu, dev = make_batch(c)
    keys = (c["seed"], c["step"], c["row_offset"])
    fresh = make_plan(c)
    run_and_read(fresh, c, dev, *keys, fn="grad_step")
    want = (fresh.losses.clone(), fresh.grads.clone())
    plan = make_plan(c)
    plan.debug_buffer("eps")[0].fill_(float("nan"))
    eps, _ = run_and_read(plan, c, dev, *keys, fn="grad_step")
    assert torch.equal(plan.losses, want[0]), "losses depend on ε rows past N"
    assert torch.equal(plan.grads, want[1]), "gradients depend on ε rows past N"
    off = eps_offsets(c["kind"], c["arch"], c["L"], c["Ncap"])
    assert np.isnan(eps[:, off["x1"]:off["z1"]]).all(), "input-noise segments written"
    for seg in LATENT:
        blk = latent_view(eps, c, seg)
        if eps_widths(c["kind"], c["arch"])[seg][1]:
            assert not np.isnan(blk[:, :, :c["N"]]).any(), "%s: a row < N left unwritten" % seg
            assert np.isnan(blk[:, :, c["N"]:]).all(), "%s: rows >= N written" % seg
        else:
            assert np.isnan(blk).all(), "%s: segment %s is not drawn by %s but was written" % (name, seg, c["kind"])
    check_latents(eps, c, *keys, tag=name + " after NaN fill")


def test_schedules_draw_the_same_bits_and_replays_take_each_calls_keys():
    c = CASES["drvae_odd"]
    cpu, dev = make_batch(c)
    k0 = (c["seed"], c["step"], c["row_offset"])
    plan = make_plan(c)
    plan.set_graph(False)
    eps0, tgt0 = run_and_read(plan, c, dev, *k0)
    check_latents(eps0, c, *k0, tag="kernel by kernel")
    check_inputs(tgt0, c, cpu, *k0, noisy=True, tag="kernel by kernel")

    plan = make_plan(c)
    replays = plan.graph_replays()
    keys = [(SEED_A + 17 * i, 2 ** 31 - 1 - i, 1000 * i + (2 ** 32 + 3 if i % 2 else 0)) for i in range(5)] + [k0]
    for i, k in enumerate(keys):
        eps, tgt = run_and_read(plan, c, dev, *k)
        check_latents(eps, c, *k, tag="graph call %d" % i)
        check_inputs(tgt, c, cpu, *k, noisy=True, tag="graph call %d" % i)
    assert plan.graph_replays() - replays >= 4, "the calls did not replay a graph"
    want = written(eps0, tgt0, c, cpu)
    assert same_bits(written(eps, tgt, c, cpu), want), "graph replay drew other bits than launches kernel by kernel"

    plan = make_plan(c)
    plan.set_graph(False)
    plan.set_step_kernel(True)
    eps, tgt = run_and_read(plan, c, dev, *k0)
    assert plan.step_kernel_launches() > 0, "the persistent step kernel did not run"
    assert same_bits(written(eps, tgt, c, cpu), want), "the step kernel drew other bits than launches kernel by kernel"


@pytest.mark.parametrize("mode", ("eval", "no_input_noise"))
def test_latent_noise_without_input_noise(mode):
    c = CASES["drvae_odd"]
    cpu, dev = make_batch(c)
    plan = make_plan(c)
    hp = dict(training=False) if mode == "eval" else dict(add_noise=False)
    eps, tgt = run_and_read(plan, c, dev, c["seed"], c["step"], c["row_offset"], **hp)
    check_latents(eps, c, c["seed"], c["step"], c["row_offset"], mode)
    check_inputs(tgt, c, cpu, c["seed"], c["step"], c["row_offset"], False, mode)


def test_row_offset_range_is_enforced():
    c = CASES["drvae_L256"]
    cpu, dev = make_batch(c)
    plan = make_plan(c)
    top = 2 ** 40 - c["N"]
    for bad in (-1, top + 1, 2 ** 62):
        with pytest.raises(RuntimeError, match="row_offset"):
            plan.loss_forward(dev, plan.hparams(step=0), seed=1, row_offset=bad)
    eps, _ = run_and_read(plan, c, dev, 1, 0, top)  # the last accepted row: every bit of the 40-bit row key set
    check_latents(eps, c, 1, 0, top, "row_offset 2^40 - N")
    # a caller's block carries no keys: any row_offset is accepted
    plan.loss_forward(dev, plan.hparams(step=0), eps=torch.zeros(plan.E, plan.eps_layout.total), row_offset=-1)


# ---- end to end -----------------------------------------------------------------------------------------------------
def tape_from_eps_block(plan, blk, has_x2, has_y):
    """Inverse of noise.eps_block_from_tape without input noise: one model's ε block -> the reference-order draws."""
    kind, L, Ncap, el = plan.kind, plan.L, plan.Ncap, plan.eps_layout
    Z, Z3, Y = plan.dim_z1, max(1, plan.dim_z3), max(1, plan.dim_y)
    if kind == "pvae":
        Z3, Y = 1, 1
    z1 = blk[el.off_z1:el.off_z1 + L * Ncap * Z].view(L, Ncap, Z)
    z2 = blk[el.off_z2:el.off_z2 + L * Ncap * Z].view(L, Ncap, Z)
    z2f = blk[el.off_z2f:el.off_z2f + L * Ncap * Z].view(L, Ncap, Z)
    z3 = blk[el.off_z3:el.off_z3 + L * Ncap * Y * Z3].view(L, Ncap, Y, Z3)
    draws = []
    for idx, pair, lab in group_indices(kind, has_x2, has_y):
        if len(idx) == 0:
            continue
        for l in range(L):
            draws.append(z1[l, idx].clone())
            if kind != "vfae":
                if pair:
                    draws.append(z2[l, idx].clone())
                draws.append(z2f[l, idx].clone())
            if kind != "pvae":
                for jj in range(1 if lab else Y):
                    draws.append(z3[l, idx, jj].clone())
    return draws


@pytest.mark.parametrize("kind", ("drvae", "pvae", "vfae"))
def test_generated_block_read_back_gives_the_same_step_and_matches_the_oracle(kind):
    """add_noise=False and 3 L N < 2048 rows (no split-K): the gradient is deterministic.  The block the generator
    wrote, passed back as a caller's block, gives the same losses and gradients bit for bit (the consumers read it with
    a caller block's Ncap stride, model stride and row indexing); as an oracle tape it gives the float64 oracle's
    step."""
    arch, N, L = ARCH["tiny"], 24, 2
    assert 3 * L * N < 2048
    sd = init_state_dict(kind, seed=123, **arch)
    batch = orc.synthetic_batch(N, arch["dim_x"], seed=3)
    fields = batch_fields(kind, batch)
    hp_kw = dict(step=0, add_noise=False, beta_pert=anneal_coef(0, 1, 0))
    own = Plan(kind, L=L, max_batch=32, n_models=1, **arch)
    own.load_state_dict(sd)
    lo_own = own.grad_step(fields, own.hparams(**hp_kw), seed=SEED_A, row_offset=2 ** 32 + 3).clone()
    g_own = own.grads.clone()
    blk = own.debug_buffer("eps")[0][0].clone()
    caller = Plan(kind, L=L, max_batch=32, n_models=1, **arch)
    caller.load_state_dict(sd)
    lo_caller = caller.grad_step(fields, caller.hparams(**hp_kw), eps=blk).clone()
    assert torch.equal(lo_own, lo_caller)
    assert torch.equal(g_own, caller.grads)

    draws = tape_from_eps_block(own, blk.cpu(), batch["has_x2"], batch["has_y"])
    om = orc.OracleModel(sd, orc.default_cfg(kind, L=L, noisy=False))
    om.iters = 0
    lo, g_ref = om.grads(batch, orc.Tape(recorded=draws), emulate_bf16=True)
    check_losses(loss_dict(kind, lo_own), lo, TOL_EMU_LOSS, "own noise vs emulating oracle")
    gv = own.tensor_views(g_own, 0)
    for name, g in g_ref.items():
        assert_grad_close(gv[name], g, "%s grad %s" % (kind, name))
    assert math.isfinite(float(lo_own[0, 6]))
