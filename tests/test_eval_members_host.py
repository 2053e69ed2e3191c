"""Host-side checks of drvae_eval_members (csrc/evalmetrics.cu): the counting form of AUROC / average precision the
ranking kernels implement, written in float64 numpy, against sklearn (the sklearn branch of
training.eval_y_prediction), including the degenerate cases; the argument checks of the C entry point, which return
before any launch; and the output column order against the header."""
import ctypes
import os
import re
import warnings

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAN = float("nan")


def counting_metrics(y, p, dim_y):
    """(auroc, aupr) by the counting form: for each positive i, nlt / neq = negatives with score < / == s_i,
    tp / fp = positives / negatives with score >= s_i; AUROC = sum(nlt + neq / 2) / (P Nn), AP = mean(tp / (tp + fp)).
    Binary: column 1; more classes: one-vs-rest per column, macro average."""
    y = np.asarray(y, dtype=np.int64)
    p = np.asarray(p, dtype=np.float64)
    cols = [1] if dim_y == 2 else list(range(dim_y))
    if len(y) == 0 or (y < 0).any() or (y >= dim_y).any() or not np.isfinite(p[:, cols]).all():
        return NAN, NAN
    aurocs, aps = [], []
    for c in cols:
        s = p[:, c]
        sp, sn = s[y == c], s[y != c]
        P, Nn = len(sp), len(sn)
        nlt = (sn[None, :] < sp[:, None]).sum(1)
        neq = (sn[None, :] == sp[:, None]).sum(1)
        tp = P - (sp[None, :] < sp[:, None]).sum(1)
        fp = Nn - nlt
        aurocs.append((nlt + 0.5 * neq).sum() / (P * Nn) if P and Nn else NAN)
        aps.append((tp / (tp + fp)).sum() / P if P else 0.0)
    return float(np.mean(aurocs)), float(np.mean(aps))


def sklearn_metrics(y, p, dim_y):
    from drvae_b200.training import eval_y_prediction
    n = len(y)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        r = eval_y_prediction(torch.zeros(n, dtype=torch.long), torch.from_numpy(np.asarray(p, np.float32)),
                              torch.as_tensor(np.asarray(y, np.int64)), dim_y)
    return r["auroc"], r["aupr"]


def _same(a, b, tol=1e-12):
    return (np.isnan(a) and np.isnan(b)) or abs(a - b) <= tol


def _scores(rng, n, dim_y, mode):
    if mode == "random":
        p = rng.rand(n, dim_y)
    elif mode == "tied":
        p = rng.randint(0, 4, size=(n, dim_y)) / 4.0
    else:
        p = np.full((n, dim_y), 0.5)
    return p.astype(np.float32)


@pytest.mark.parametrize("mode", ["random", "tied", "equal"])
@pytest.mark.parametrize("dim_y", [2, 3, 5])
def test_counting_form_matches_sklearn(dim_y, mode):
    rng = np.random.RandomState(7 + dim_y)
    for n in (2, 7, 60, 333):
        for _ in range(6):
            y = rng.randint(0, dim_y, size=n)
            p = _scores(rng, n, dim_y, mode)
            got, want = counting_metrics(y, p, dim_y), sklearn_metrics(y, p, dim_y)
            assert _same(got[0], want[0]) and _same(got[1], want[1]), (n, got, want)


@pytest.mark.parametrize("dim_y", [2, 3, 5])
def test_counting_form_reproduces_the_degenerate_cases(dim_y):
    rng = np.random.RandomState(1)
    n = 12
    p = _scores(rng, n, dim_y, "random")
    y = np.arange(n) % dim_y
    cases = {"none": (y[:0], p[:0])}
    if dim_y == 2:
        cases["all positive"] = (np.ones(n, int), p)
        cases["all negative"] = (np.zeros(n, int), p)
        q = p.copy()
        q[3, 0] = np.inf  # column 0 is not scored in the binary case
        cases["non-finite unscored column"] = (y, q)
    else:
        cases["a class absent"] = (y % (dim_y - 1), p)
        cases["one class only"] = (np.zeros(n, int), p)
    for bad in (np.nan, np.inf, -np.inf):
        q = p.copy()
        q[5, 1] = bad
        cases["score %s" % bad] = (y, q)
    cases["label out of range"] = (np.where(np.arange(n) == 4, dim_y, y), p)
    for name, (yy, pp) in cases.items():
        got = counting_metrics(yy, pp, dim_y)
        if name == "label out of range" and dim_y > 2:
            # eval_y_prediction's one-hot encoding cannot take the label (IndexError); the device path defines nan
            assert np.isnan(got[0]) and np.isnan(got[1])
            continue
        want = sklearn_metrics(yy, pp, dim_y)
        assert _same(got[0], want[0]) and _same(got[1], want[1]), (name, got, want)
    # the degenerate values the header documents for drvae_eval_members
    if dim_y == 2:
        assert np.isnan(counting_metrics(np.ones(n, int), p, 2)[0])
        assert counting_metrics(np.ones(n, int), p, 2)[1] == 1.0 and counting_metrics(np.zeros(n, int), p, 2)[1] == 0.0
    else:
        auroc, aupr = counting_metrics(np.zeros(n, int), p, dim_y)
        assert np.isnan(auroc) and abs(aupr - 1.0 / dim_y) < 1e-15


def _fake(n=1):
    """Non-NULL addresses that are never dereferenced: every call below is rejected before a launch."""
    return ctypes.c_void_p(0x1000 * n)


def _full_input():
    from drvae_b200 import _lib
    a = _lib.EvalMembersIn()
    for k, (name, _) in enumerate(_lib.EvalMembersIn._fields_):
        setattr(a, name, 0x1000 * (k + 1))
    return a


def _with(a, **changes):
    from drvae_b200 import _lib
    b = _lib.EvalMembersIn()
    ctypes.pointer(b)[0] = a
    for k, v in changes.items():
        setattr(b, k, v)
    return b


def test_eval_members_rejects_bad_arguments():
    from drvae_b200 import _lib
    lib = _lib.load()
    E, D, X, Y = 3, 10, 5, 2

    def call(a, e=E, d=D, x=X, y=Y, out=_fake(50), ws=_fake(60), by_ref=True):
        return lib.drvae_eval_members(ctypes.byref(a) if by_ref else None, e, d, x, y, out, ws, None)

    cases = []
    a = _full_input()
    cases.append(("valid", lambda: call(_with(a, valid=None))))
    cases.append(("out", lambda: call(a, out=None)))
    cases.append(("workspace", lambda: call(a, ws=None)))
    cases.append(("in", lambda: call(a, by_ref=False)))
    cases.append(("E", lambda: call(a, e=0)))
    cases.append(("D", lambda: call(a, d=0)))
    cases.append(("X", lambda: call(a, x=0)))
    cases.append(("Y", lambda: call(a, y=1)))
    for group, names in (("x1", ("x1", "px1_mu")), ("x2", ("x2", "px2_mu", "has_x2")),
                         ("y", ("proba", "pred", "y", "has_y"))):
        for n in names:
            cases.append((group, lambda n=n: call(_with(a, **{n: None}))))
    for word, fn in cases:
        assert fn() != 0, word
        msg = lib.drvae_last_error().decode()
        assert "drvae_eval_members" in msg and word in msg, (word, msg)
    assert lib.drvae_eval_members_workspace_bytes(0, D, X, Y) < 0
    assert lib.drvae_eval_members_workspace_bytes(E, 0, X, Y) < 0
    assert lib.drvae_eval_members_workspace_bytes(E, D, 0, Y) < 0
    # without the y group (Y < 2) the workspace is the reconstruction part alone
    assert lib.drvae_eval_members_workspace_bytes(E, D, X, 0) == 8 * E * (4 * D + 2 * X)
    assert lib.drvae_eval_members_workspace_bytes(E, D, X, 2) > lib.drvae_eval_members_workspace_bytes(E, D, X, 0)
    assert {"drvae_eval_members", "drvae_eval_members_workspace_bytes"} <= set(_lib.EXPORTS)


def test_column_order_and_struct_match_the_header():
    from drvae_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "drvae_b200.h")).read()
    cols = re.search(r"columns in this fixed order:\s*\n\s*\*\s*([^\n]*)", hdr).group(1)
    assert tuple(re.findall(r"\d+ (\w+)", cols)) == _lib.EVAL_MEMBER_COLUMNS
    body = hdr.split("} drvae_eval_members_in_t;")[0].rsplit("typedef struct {", 1)[1]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = re.findall(r"\*\s*(\w+)\s*;", body)
    assert [f[0] for f in _lib.EvalMembersIn._fields_] == names
