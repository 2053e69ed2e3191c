"""GPU tests of drvae_eval_members (csrc/evalmetrics.cu), the one-call metrics of every ensemble member.

y metrics are checked against the sklearn branch of training.eval_y_prediction on CPU copies of each member's labeled
rows (accuracy exactly, AUROC / AUPR within 1e-12); reconstruction metrics bit for bit against
drvae_eval_x_reconstruction on each member's slice; sweep.evaluate_members against the per-member loop it replaces."""
import math
import warnings
from collections import OrderedDict

import numpy as np
import pytest
import torch

from helpers import ARCH

from drvae_b200 import _lib
from drvae_b200.init import init_state_dict
from drvae_b200.plan import Plan
from drvae_b200.sweep import MODEL_CLASS, evaluate_members, pad_members
from drvae_b200.training import DrVAEDataset, VFAEDataset, eval_members, eval_x_reconstruction, eval_y_prediction

pytestmark = pytest.mark.gpu
COL = {k: i for i, k in enumerate(_lib.EVAL_MEMBER_COLUMNS)}
EXTREME = np.array([np.nan, np.inf, -np.inf, 1e30, -1e30, 0.5], dtype=np.float32)


def _same(a, b, tol=1e-12):
    return (math.isnan(a) and math.isnan(b)) or abs(a - b) <= tol


def _sk_y(pred, proba, y, dim_y):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return eval_y_prediction(pred.cpu().long(), proba.cpu(), y.cpu(), dim_y)


def _ref_y(valid, has_y, pred, proba, y, dim_y):
    """The per-member loop: each member's labeled rows through eval_y_prediction's sklearn branch."""
    out = []
    for m in range(valid.shape[0]):
        idx = torch.nonzero((valid[m] != 0) & (has_y[m] != 0)).view(-1).cpu()
        r = _sk_y(pred[m].cpu()[idx], proba[m].cpu()[idx], y[m].cpu()[idx], dim_y)
        out.append((r["acc"], r["auroc"], r["aupr"]))
    return out


def _assert_y(got, want, what=""):
    for m, (g, w) in enumerate(zip(got, want)):
        assert _same(g[0], w[0], 0.0), (what, m, "acc", g[0], w[0])
        assert _same(g[1], w[1]) and _same(g[2], w[2]), (what, m, g, w)


def _pad(members, D, dim_y, rng):
    """members: [(y, proba, has_y)] of any lengths -> padded [E, D] device tensors.  Padding rows (valid == 0) hold
    extreme scores, labels out of range and has_y = 1, so that only `valid` keeps them out."""
    E = len(members)
    valid = np.zeros((E, D), np.int32)
    y = rng.choice([-66, dim_y + 7], size=(E, D)).astype(np.int32)
    has_y = np.ones((E, D), np.int32)
    proba = rng.choice(EXTREME, size=(E, D, dim_y))
    pred = rng.randint(0, dim_y, size=(E, D)).astype(np.int32)
    for m, (ym, pm, hm) in enumerate(members):
        n = len(ym)
        valid[m, :n] = 1
        y[m, :n], proba[m, :n], has_y[m, :n] = ym, pm, hm
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return t(valid), t(has_y), t(pred), t(proba.astype(np.float32)), t(y)


def _member(rng, n, dim_y, mode):
    y = rng.randint(0, dim_y, size=n)
    p = rng.rand(n, dim_y) if mode == "random" else rng.randint(0, 4, size=(n, dim_y)) / 4.0
    has_y = (rng.rand(n) < 0.8).astype(np.int32)
    # unlabeled rows carry the reference's y = -66 and scores that would change the result if they counted
    y = np.where(has_y != 0, y, -66)
    p[has_y == 0] = rng.choice(EXTREME, size=(int((has_y == 0).sum()), dim_y))
    return y, p.astype(np.float32), has_y


def _y_out(valid, has_y, pred, proba, y):
    out = eval_members(valid, proba=proba, pred=pred, y=y, has_y=has_y).cpu()
    return out, [tuple(r[:3]) for r in out.tolist()]


@pytest.mark.parametrize("mode", ["random", "quantised"])
@pytest.mark.parametrize("dim_y", [2, 3, 5])
def test_y_metrics_match_sklearn(dim_y, mode):
    rng = np.random.RandomState(dim_y * 10 + len(mode))
    sizes = [300, 17, 256, 1, 129, 300, 2, 77]
    D = max(sizes) + 11
    members = [_member(rng, n, dim_y, mode) for n in sizes]
    valid, has_y, pred, proba, y = _pad(members, D, dim_y, rng)
    pred[:, ::3] = y[:, ::3].clamp(0, dim_y - 1)  # some correct predictions
    out, got = _y_out(valid, has_y, pred, proba, y)
    _assert_y(got, _ref_y(valid, has_y, pred, proba, y, dim_y), (dim_y, mode))
    assert torch.isnan(out[:, 3:]).all()  # no x group given
    # the single-model path: eval_y_prediction on CUDA tensors equals its sklearn branch
    idx = torch.nonzero((valid[0] != 0) & (has_y[0] != 0)).view(-1)
    dev = eval_y_prediction(pred[0][idx], proba[0][idx], y[0][idx], dim_y)
    host = _sk_y(pred[0][idx], proba[0][idx], y[0][idx], dim_y)
    assert list(dev) == ["acc", "auroc", "aupr"]
    _assert_y([tuple(dev.values())], [tuple(host.values())], "eval_y_prediction")
    empty = eval_y_prediction(pred[0][:0], proba[0][:0], y[0][:0], dim_y)
    assert all(math.isnan(v) for v in empty.values())


@pytest.mark.parametrize("dim_y", [2, 3])
def test_y_degenerate_cases(dim_y):
    rng = np.random.RandomState(5)
    n = 40
    base = rng.randint(0, dim_y, size=n)
    p = rng.rand(n, dim_y).astype(np.float32)
    ones = np.ones(n, np.int32)
    cases = OrderedDict()
    cases["no labeled row"] = (base, p, np.zeros(n, np.int32))
    if dim_y == 2:
        cases["all positive"] = (np.ones(n, int), p, ones)
        cases["all negative"] = (np.zeros(n, int), p, ones)
        q = p.copy()
        q[7, 0] = np.inf
        cases["non-finite unscored column"] = (base, q, ones)
    else:
        cases["a class absent"] = (base % (dim_y - 1), p, ones)
        cases["one class only"] = (np.zeros(n, int), p, ones)
        q = p.copy()
        q[7, 0] = np.inf
        cases["inf in column 0"] = (base, q, ones)
    q = p.copy()
    q[3, 1] = np.nan
    cases["nan score"] = (base, q, ones)
    q = p.copy()
    q[3, 1] = -np.inf
    cases["-inf score"] = (base, q, ones)
    q = p.copy()
    q[3, 1] = np.nan
    cases["nan score on an unlabeled row"] = (base, q, np.where(np.arange(n) == 3, 0, 1).astype(np.int32))
    cases["label out of range"] = (np.where(np.arange(n) == 9, dim_y, base), p, ones)
    cases["negative label"] = (np.where(np.arange(n) == 9, -1, base), p, ones)
    names = list(cases)
    valid, has_y, pred, proba, y = _pad(list(cases.values()), n + 5, dim_y, rng)
    _, got = _y_out(valid, has_y, pred, proba, y)
    for m, name in enumerate(names):
        if name in ("label out of range", "negative label") and dim_y > 2:
            # eval_y_prediction's one-hot encoding cannot take such a label; the device path gives nan
            lab = (valid[m] != 0) & (has_y[m] != 0)
            acc = float((pred[m][lab] == y[m][lab]).double().mean())
            assert got[m][0] == acc and math.isnan(got[m][1]) and math.isnan(got[m][2]), name
            continue
        want = _ref_y(valid[m:m + 1], has_y[m:m + 1], pred[m:m + 1], proba[m:m + 1], y[m:m + 1], dim_y)
        _assert_y([got[m]], want, name)
    g = dict(zip(names, got))
    assert math.isnan(g["no labeled row"][0])
    assert all(math.isnan(v) for v in g["nan score"][1:]) and all(math.isnan(v) for v in g["label out of range"][1:])
    assert not math.isnan(g["nan score on an unlabeled row"][1])
    if dim_y == 2:
        assert g["all positive"][2] == 1.0 and g["all negative"][2] == 0.0 and math.isnan(g["all positive"][1])
        assert not math.isnan(g["non-finite unscored column"][1])
    else:
        assert math.isnan(g["one class only"][1]) and abs(g["one class only"][2] - 1.0 / dim_y) < 1e-15


@pytest.mark.parametrize("dim_y", [2, 3])
def test_large_inputs_and_determinism(dim_y):
    """D = 65 536: rows span many shared-memory tiles and the positives of a column span many blocks."""
    rng = np.random.RandomState(11)
    D = 65536
    sizes = [D, 65000, 40000, D]
    members = [_member(rng, n, dim_y, "quantised" if m % 2 else "random") for m, n in enumerate(sizes)]
    valid, has_y, pred, proba, y = _pad(members, D, dim_y, rng)
    out, got = _y_out(valid, has_y, pred, proba, y)
    _assert_y(got, _ref_y(valid, has_y, pred, proba, y, dim_y), "large")
    again, _ = _y_out(valid, has_y, pred, proba, y)
    assert torch.equal(out.view(torch.int64), again.view(torch.int64))


def _x_members(rng, E, D, X, sizes, no_x2=()):
    valid = torch.zeros(E, D, dtype=torch.int32)
    for m, n in enumerate(sizes):
        valid[m, :n] = 1
    g = torch.Generator().manual_seed(int(rng.randint(1 << 30)))
    x1, x2 = torch.randn(E, D, X, generator=g), torch.randn(E, D, X, generator=g)
    r1, r2 = x1 + 0.5 * torch.randn(E, D, X, generator=g), x2 + 0.3 * torch.randn(E, D, X, generator=g)
    s1, s2 = torch.rand(E, D, X, generator=g) + 0.1, torch.rand(E, D, X, generator=g) + 0.1
    pad = valid == 0
    for t in (x1, x2, r1, r2):
        t[pad] = 1e6  # padding rows must not enter any sum
    has_x2 = (torch.rand(E, D, generator=g) < 0.5).to(torch.int32)
    for m in no_x2:
        has_x2[m] = 0
    return [t.cuda() for t in (valid, x1, r1, s1, x2, r2, s2, has_x2)]


def _assert_bitwise(a, b, what):
    na, nb = torch.isnan(a), torch.isnan(b)
    assert torch.equal(na, nb) and torch.equal(a[~na], b[~nb]), (what, a, b)


@pytest.mark.parametrize("layout", ["drvae", "no_sigma", "vfae"])
def test_reconstruction_equals_the_single_member_kernel(layout):
    rng = np.random.RandomState(2)
    E, D, X = 6, 300, 97
    sizes = [300, 120, 1, 0, 299, 57]
    valid, x1, r1, s1, x2, r2, s2, has_x2 = _x_members(rng, E, D, X, sizes, no_x2=(1,))
    if layout == "no_sigma":
        s1 = s2 = None
    kw = dict(x1=x1, px1_mu=r1, px1_sg=s1)
    if layout != "vfae":
        kw.update(x2=x2, px2_mu=r2, px2_sg=s2, has_x2=has_x2)
    else:  # VFAE: x1 and y, no x2 group
        dim_y = 2
        members = [_member(rng, n, dim_y, "random") for n in sizes]
        _, has_y, pred, proba, y = _pad(members, D, dim_y, rng)
        kw.update(proba=proba, pred=pred, y=y, has_y=has_y)
    out = eval_members(valid, **kw).cpu()
    for m in range(E):
        one = lambda x, r, s, mask: torch.tensor(list(eval_x_reconstruction(x[m], r[m], None if s is None else s[m],
                                                                            mask=mask).values()), dtype=torch.float64)
        _assert_bitwise(out[m, 3:7], one(x1, r1, s1, valid[m]), (layout, m, "x1"))
        if layout != "vfae":
            _assert_bitwise(out[m, 7:11], one(x2, r2, s2, valid[m] * has_x2[m]), (layout, m, "x2"))
        else:
            assert torch.isnan(out[m, 7:]).all()
    assert torch.isnan(out[3, 3:]).all()  # the member without rows
    if layout != "vfae":
        assert torch.isnan(out[1, 7:]).all()  # the member without x2 rows
    if layout == "no_sigma":
        assert torch.isnan(out[:, COL["x1_ll"]]).all() and not torch.isnan(out[0, COL["x1_rmse"]])
    if layout == "vfae":
        _assert_y([tuple(r[:3]) for r in out.tolist()], _ref_y(valid, has_y, pred, proba, y, 2), "vfae")
    again = eval_members(valid, **kw).cpu()
    assert torch.equal(out.view(torch.int64), again.view(torch.int64))


def _datasets(kind, sizes, dim_x, seed):
    out = []
    for k, n in enumerate(sizes):
        g = torch.Generator().manual_seed(seed + k)
        x1 = torch.randn(n, dim_x, generator=g)
        y = (x1[:, :8].sum(1) + 0.5 * torch.randn(n, generator=g) > 0).long()
        has_y = (torch.rand(n, generator=g) < 0.7).to(torch.int32)
        y = torch.where(has_y != 0, y, torch.full_like(y, -66))
        s = torch.zeros(n, dtype=torch.int32)
        if kind == "vfae":
            out.append(VFAEDataset(x1=x1, s=s, y=y, has_y=has_y))
        else:
            has_x2 = (torch.rand(n, generator=g) < 0.5).to(torch.int32)
            if k == 2:
                has_x2.zero_()  # one member without paired rows
            x2 = torch.where(has_x2[:, None] != 0, x1 + 0.3 * torch.randn(n, dim_x, generator=g), torch.zeros(n, dim_x))
            out.append(DrVAEDataset(x1=x1, x2=x2, s=s, y=y, has_x2=has_x2, has_y=has_y))
    return out


def _old_evaluate_members(plan, kind, fields, mask):
    """The per-member loop evaluate_members replaced, with the y metrics through sklearn on CPU copies."""
    D = fields["x1"].shape[1]
    outs = [plan.infer(fields["x1"][:, c0:c0 + plan.Ncap]) for c0 in range(0, D, plan.Ncap)]
    res = {k: torch.cat([o[k] for o in outs], 1) for k in outs[0]}
    perfs = []
    for m in range(plan.E):
        valid = mask[m] != 0
        perf = OrderedDict(losses=None)
        if kind != "pvae":
            idx = torch.nonzero(valid & (fields["has_y"][m] != 0)).view(-1)
            y = _sk_y(res["pred"][m][idx], res["proba"][m][idx], fields["y"][m][idx], plan.dim_y)
            perf.update(("y_" + k, v) for k, v in y.items())
        x1 = eval_x_reconstruction(fields["x1"][m], res["px1_mu"][m], res["px1_sg"][m], mask=valid)
        perf.update(("x1_" + k, v) for k, v in x1.items())
        if kind != "vfae":
            pair = valid & (fields["has_x2"][m] != 0)
            if bool(pair.any()):
                x2 = eval_x_reconstruction(fields["x2"][m], res["px2_mu"][m], res["px2_sg"][m], mask=pair)
                perf.update(("x2_" + k, v) for k, v in x2.items())
            else:
                perf.update(("x2_" + k, float("nan")) for k in ("rmse", "r2", "pearr", "ll"))
        perf["model_class"] = MODEL_CLASS[kind]
        perfs.append(perf)
    return perfs


@pytest.mark.parametrize("kind,sizes", [("drvae", [150, 97, 201, 64, 180, 33]), ("vfae", [120, 250, 71, 199])])
def test_evaluate_members_equals_the_per_member_loop(kind, sizes):
    arch = ARCH["readme"]
    E = len(sizes)
    plan = Plan(kind, L=1, max_batch=64, n_models=E, **arch)
    for m in range(E):
        plan.load_state_dict(init_state_dict(kind, seed=100 + m, **arch), model=m)
    fields, mask, _ = pad_members(kind, _datasets(kind, sizes, arch["dim_x"], seed=3))
    fields = {k: v.cuda() for k, v in fields.items()}
    mask = mask.cuda()
    got = evaluate_members(plan, kind, fields, mask)
    want = _old_evaluate_members(plan, kind, fields, mask)
    for m, (g, w) in enumerate(zip(got, want)):
        assert list(g) == list(w), m
        for k in g:
            if k in ("losses", "model_class"):
                assert g[k] == w[k]
            else:
                assert _same(g[k], w[k]), (m, k, g[k], w[k])
    if kind == "drvae":
        assert all(math.isnan(got[2][k]) for k in ("x2_rmse", "x2_r2", "x2_pearr", "x2_ll"))
    # the metrics need one synchronisation: the final [E, 11] copy
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        torch.cuda.set_sync_debug_mode("warn")
        try:
            evaluate_members(plan, kind, fields, mask)
        finally:
            torch.cuda.set_sync_debug_mode(0)
    syncs = [w for w in caught if "called a synchronizing CUDA operation" in str(w.message)]
    assert len(syncs) == 1, [str(w.message) for w in caught]
