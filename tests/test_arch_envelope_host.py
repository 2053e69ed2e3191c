"""CPU: the architecture-envelope cases of test_arch_envelope_gpu.py still straddle every shape threshold of plan.cu,
and drvae_plan_create rejects what lies beyond its limits before it touches the device."""
import ctypes

import pytest

from helpers import KINDS
from test_arch_envelope_gpu import CASES, geometry, tile_cap

from drvae_b200 import _lib

GEO = {(c, k): geometry(c, k) for c in CASES for k in KINDS}


def _where(pred):
    return sorted({"%s-%s" % ck for ck, g in GEO.items() if pred(g)})


def _covers(pred, what):
    hits = _where(pred)
    assert hits, "no case covers: " + what
    return hits


def test_tile_cap_matches_plan_cu():
    assert tile_cap(256) == (256, 1)
    assert tile_cap(257) == (144, 2)
    assert tile_cap(512) == (256, 2)
    assert tile_cap(33) == (48, 1)


def test_row_kernel_width_on_both_sides():
    _covers(lambda g: g["Zc"] == 128 and not g["maxj"], "Zc = 128 with the <4> row kernels")
    _covers(lambda g: g["Zc"] == 144 and g["maxj"], "the first <MAXJ> width, Zc = 144")
    _covers(lambda g: g["maxj"] and g["Zc"] > 256, "<MAXJ> with every lane slot populated (dim_z1 = 256)")
    _covers(lambda g: g["Z3c"] > 128, "<MAXJ> chosen by Z3c (z3_post / z3_back)")


def test_grouped_and_split_optimizer_on_both_sides():
    _covers(lambda g: g["split_optimizer"] and g["Y"] == 2, "gradient + stand-alone Adam with two classes (126 + 1 + 2 = 129)")
    _covers(lambda g: g["split_optimizer"] and g["Y"] == 8, "gradient + stand-alone Adam with eight classes (120 + 1 + 8 = 129)")
    # the grouped launch is still used when the class columns end exactly at row 128
    _covers(lambda g: not g["split_optimizer"] and g["Zc"] == 128 and g["Y"] == 2, "class columns ending at row 128")
    _covers(lambda g: g["dwa_layers"] == 21, "21 layers in the grouped dW+Adam table")
    assert max(g["dwa_layers"] for g in GEO.values()) <= 24


def test_head_tiles():
    _covers(lambda g: g["enc_head"] == (256, 1), "a (mu | logvar) head in one tile exactly 256 wide")
    _covers(lambda g: g["enc_head"][1] == 2, "a (mu | logvar) head over two N tiles")
    _covers(lambda g: g["dec_tiles"] >= 2 and g["dec_last"] == 1, "a decoder-head tile holding one feature")
    _covers(lambda g: g["dec_tiles"] == 2 and g["dec_last"] == 128 and g["Xc"] == 272, "two full decoder-head tiles")
    _covers(lambda g: g["dec_tiles"] == 8 and g["hb"] == 128, "the README decoder head (978 = 7 x 128 + 82)")


def test_hidden_layer_tiles():
    _covers(lambda g: (256, 1) in g["hidden"], "a hidden layer in one tile 256 wide (width 255)")
    _covers(lambda g: (144, 2) in g["hidden"], "a hidden layer in two tiles 144 wide (width 256)")
    _covers(lambda g: (256, 2) in g["hidden"], "a hidden layer in two tiles 256 wide (width 511)")
    _covers(lambda g: g["n_hidden"] == 4, "four hidden layers in an MLP")


def test_classes():
    _covers(lambda g: g["Y"] == 8, "eight classes")
    _covers(lambda g: g["Y"] == 3, "an odd class count")
    _covers(lambda g: g["Y"] == 8 and g["rows"]["F"] == 8 * g["rows"]["LN"] == 528, "F = 8 L N = 528 marginalised rows")


def test_stacked_row_counts_on_the_128_row_tile():
    """Counts of the batches the GPU tests run (runtime_rows), not the plan's capacities."""
    for buf in ("R0", "LN", "F"):
        _covers(lambda g: g["rows"][buf] == 128, "%s exactly on the 128-row tile" % buf)
    _covers(lambda g: g["rows"]["Rd"] == 384, "Rd on the tile")
    _covers(lambda g: g["rows"]["LN"] % 128 == 1, "LN one row past the tile")
    _covers(lambda g: g["rows"]["LN"] % 128 == 2, "LN two rows past the tile")
    _covers(lambda g: g["rows"]["R0"] % 128 == 1, "R0 one row past the tile")


def _create(**kw):
    a = _lib.Arch()
    a.kind = _lib.KIND[kw.pop("kind", "drvae")]
    a.dim_x, a.dim_y, a.dim_z1, a.dim_z3 = 40, 2, 16, 16
    a.L, a.max_batch = 1, 8
    for name in ("enc_z1", "dec_x", "enc_z3", "dec_z1"):
        setattr(a, "n_" + name, 1)
        getattr(a, name)[0] = 32
    for k, v in kw.items():
        setattr(a, k, v)
    lib = _lib.load()
    h = ctypes.c_void_p()
    rc = lib.drvae_plan_create(ctypes.byref(a), 1, ctypes.byref(h))
    if rc == 0:
        lib.drvae_plan_destroy(h)
    return rc, (lib.drvae_last_error() or b"").decode()


@pytest.mark.parametrize("kw,limit", [
    (dict(dim_z1=257), "256"),
    (dict(dim_z3=257), "256"),
    (dict(kind="vfae", dim_z3=257), "256"),
    (dict(dim_y=9), "[2, 8]"),
    (dict(dim_y=1), "[2, 8]"),
    (dict(n_enc_z1=5), "between 1 and 4"),
    (dict(n_dec_x=0), "between 1 and 4"),
    (dict(n_enc_z3=5), "between 1 and 4"),
    (dict(n_dec_z1=0), "between 1 and 4"),
    (dict(kind="pvae", n_enc_z1=0), "between 1 and 4"),
], ids=["z1_257", "z3_257", "vfae_z3_257", "y9", "y1", "enc5", "dec0", "encz3_5", "decz1_0", "pvae_enc0"])
def test_arguments_beyond_the_limits_are_rejected(kw, limit):
    rc, msg = _create(**kw)
    assert rc != 0
    assert limit in msg, msg


def test_pvae_ignores_the_label_dimensions():
    """PVAE has no classes and no top latent: dim_y / dim_z3 / enc_z3 / dec_z1 are not checked.  Without a device the
    call gets past the argument checks and fails at the first allocation."""
    rc, msg = _create(kind="pvae", dim_y=0, dim_z3=0, n_enc_z3=0, n_dec_z1=0)
    assert rc == 0 or "cudaMalloc" in msg, msg
