"""Shared fixtures for the parity tests: architectures, synthetic batches, oracle runs."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import drvae_oracle as orc  # noqa: E402  (tests are allowed to use the oracle)

GOLDEN = os.path.join(ROOT, "tests", "golden")
ARCH = dict(
    readme=dict(dim_x=978, dim_y=2, dim_z1=100, dim_z3=100, enc_z1=[800], dec_x=[600], enc_z3=[200], dec_z1=[200]),
    tiny=dict(dim_x=40, dim_y=2, dim_z1=12, dim_z3=10, enc_z1=[24], dec_x=[28], enc_z3=[20], dec_z1=[18]),
    deep=dict(dim_x=40, dim_y=2, dim_z1=12, dim_z3=10, enc_z1=[24, 20], dec_x=[16, 28], enc_z3=[20, 12], dec_z1=[18, 14]),
)
ARCH["tiny_wn"] = ARCH["tiny"]  # same dims, built from layers.WeightNormLinear (golden recorded with wn=True)
NROWS = dict(readme=150, tiny=24, deep=24, tiny_wn=24)
KINDS = ("drvae", "pvae", "vfae")
SEED_MODEL, SEED_TAPE, L = 123, 777, 2


def golden(kind, case):
    return np.load(os.path.join(GOLDEN, "%s_%s.npz" % (kind, case)))


def batch_fields(kind, batch):
    """Subset of the synthetic batch a model kind consumes (as keyword arguments of Plan calls)."""
    b = dict(x1=batch["x1"])
    if kind in ("drvae", "pvae"):
        b.update(x2=batch["x2"], has_x2=batch["has_x2"])
    if kind in ("drvae", "vfae"):
        b.update(y=batch["y"], has_y=batch["has_y"])
    return b


def oracle_batch(kind, batch):
    return batch


def rel_err(a, b):
    a = a.detach().float().cpu()
    b = b.detach().float().cpu()
    return ((a - b).abs().max() / (b.abs().max() + 1e-12)).item()


def rel_l2(a, b):
    a = a.detach().double().cpu()
    b = b.detach().double().cpu()
    return ((a - b).norm() / (b.norm() + 1e-30)).item()


def _worst_line(d, r, dim):
    """Largest ||d_i|| / (||r_i|| + 0.1 ||r|| / sqrt(lines)) over the lines i of `dim` (0: rows, 1: columns)."""
    other = 1 - dim
    lines = r.shape[dim]
    allowed = r.norm(dim=other) + 0.1 * r.norm() / np.sqrt(lines)
    ratio = d.norm(dim=other) / allowed.clamp_min(1e-300)
    i = int(ratio.argmax())
    return float(ratio[i]), i, float(d.norm(dim=other)[i]), float(allowed[i])


def grad_errors(got, ref):
    """Relative L2 of the whole tensor and, per output row / input column, the worst ||got_i - ref_i|| divided by
    (||ref_i|| + 0.1 ||ref|| / sqrt(lines)).  A vector is checked element by element (its rows have one column).
    The floor keeps rows whose reference is near zero from failing on rounding noise."""
    g = got.detach().double().cpu()
    r = ref.detach().double().cpu()
    assert g.shape == r.shape, (tuple(g.shape), tuple(r.shape))
    out = dict(l2=((g - r).norm() / (r.norm() + 1e-300)).item())
    if r.norm() == 0:
        out["l2"] = 0.0 if g.norm() == 0 else float("inf")
    d = g - r
    if r.dim() == 1:
        d, r = d[:, None], r[:, None]
    out["row"] = _worst_line(d, r, 0)
    if r.shape[1] > 1:
        out["col"] = _worst_line(d, r, 1)
    return out


def assert_grad_close(got, ref, tag, tol_l2=1e-2, tol_line=3e-2):
    """Tensor-wide relative L2 <= tol_l2, and every row and every column within tol_line of its own reference norm
    (see grad_errors).  A fault confined to one tile, row or column of a large matrix hides in the tensor-wide norm;
    the line checks name where it is.  Returns the errors for reporting."""
    e = grad_errors(got, ref)
    assert e["l2"] <= tol_l2, "%s: relative L2 %.3e > %.1e" % (tag, e["l2"], tol_l2)
    for what in ("row", "col"):
        if what in e:
            ratio, i, err, allowed = e[what]
            assert ratio <= tol_line, "%s: %s %d of %s: |got - ref| = %.4e is %.3e of its reference scale %.4e (> %.1e)" % (
                tag, what, i, tuple(ref.shape), err, ratio, allowed, tol_line)
    return e
