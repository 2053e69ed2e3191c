"""CPU: the host reference of the step's own noise (tests/philox_ref.py) against the published Philox4x32-10 answers,
the key ranges inside which the counter packing gives every draw its own numbers, and drvae_plan_create's rejection of
plans that would leave them."""
import ctypes

import numpy as np
import pytest
import torch

from philox_ref import counter, normals, philox4x32_10

from drvae_b200 import _lib

# Random123 known-answer vectors of philox4x32-10: counter c0..c3, key k0 k1 -> output
KAT = [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff, 0xffffffff), (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
]


@pytest.mark.parametrize("ctr,key,want", KAT, ids=["zeros", "ones", "pi"])
def test_philox_known_answers(ctr, key, want):
    got = philox4x32_10(*ctr, *key)
    assert tuple(int(w) for w in got) == want, ["%08x" % int(w) for w in got]


def test_philox_vectorised_matches_scalar():
    rng = np.random.default_rng(0)
    c = rng.integers(0, 2 ** 32, size=(4, 64), dtype=np.uint64)
    k = rng.integers(0, 2 ** 32, size=2, dtype=np.uint64)
    vec = np.stack(philox4x32_10(*c, *k))
    for i in range(64):
        assert np.array_equal(np.stack(philox4x32_10(*c[:, i], *k)), vec[:, i])


def test_counter_keys_are_distinct_inside_the_accepted_ranges():
    """The packing {q | (row >> 32) << 24, row, step, model | kind << 20 | l << 24} is injective for model < 2^20,
    l < 256 and row < 2^40, and the first value past each range lands on an accepted key."""
    base = dict(q=3, grow=(1 << 40) - 1, step=7, model=(1 << 20) - 1, seg=5, l=255)

    def ctr(**kw):
        d = dict(base, **kw)
        return tuple(int(c) for c in counter(d["q"], d["grow"], d["step"], d["model"], d["seg"], d["l"]))

    top = ctr()
    for field, value in (("grow", (1 << 40) - 2), ("model", (1 << 20) - 2), ("l", 254), ("seg", 4), ("q", 2), ("step", 6)):
        assert ctr(**{field: value}) != top, field
    # one past the range collides
    assert ctr(l=256) == ctr(l=0)
    assert ctr(grow=1 << 40) == ctr(grow=0)
    assert ctr(model=1 << 20, seg=0) == ctr(model=0, seg=1)


def test_reference_normals_edges():
    """u0 = 1 (counter word 0xffffffff, or any word that rounds to 2^32) gives radius 0 exactly; the smallest
    u0 = 2^-32 gives the largest radius sqrt(64 ln 2)."""
    z, allow = normals(seed=0, step=0, model=0, seg=0, l=0, grow=np.arange(4096), q=0)
    assert z.shape == allow.shape == (4096, 4)
    assert np.all(allow > 0) and np.all(allow < 1e-3)
    assert abs(z.mean()) < 0.05 and abs(z.std() - 1) < 0.05
    assert float(np.abs(z).max()) <= np.sqrt(64 * np.log(2.0))


def test_gpu_cases_cover_every_store_branch():
    """test_noise_gpu.py's cases reach each store branch of philox_normal_kernel: scalar for an odd width and for an
    even width at an odd offset, float2 for widths 2 mod 4 (half a quad) and 0 mod 4; every kind; the input widths."""
    from test_noise_gpu import CASES, LATENT, eps_offsets, eps_widths, store_branch
    seen = set()
    for c in CASES.values():
        off, w = eps_offsets(c["kind"], c["arch"], c["L"], c["Ncap"]), eps_widths(c["kind"], c["arch"])
        for s in LATENT:
            if w[s][1]:
                seen.add((store_branch(w[s][0], off[s]), w[s][0] % 4, off[s] % 2))
    assert {b for b in seen if b[0] == "scalar" and b[1] % 2 == 1}
    assert ("scalar", 2, 1) in seen or ("scalar", 0, 1) in seen
    assert ("f2", 2, 0) in seen and ("f2", 0, 0) in seen
    assert {c["kind"] for c in CASES.values()} == {"drvae", "pvae", "vfae"}
    xs = [c["arch"]["dim_x"] for c in CASES.values()]
    assert any(x > 256 for x in xs) and any(x % 4 == 1 for x in xs)
    assert any(c["N"] == 1 for c in CASES.values()) and any(c["L"] == 256 for c in CASES.values())


def _create(n_models=1, **kw):
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
    rc = lib.drvae_plan_create_clf(ctypes.byref(a), 0, None, n_models, ctypes.byref(h))
    if rc == 0:
        lib.drvae_plan_destroy(h)
    return rc, (lib.drvae_last_error() or b"").decode()


@pytest.mark.parametrize("kw,limit", [
    (dict(L=257), "256"),
    (dict(kind="pvae", L=257), "256"),
    (dict(kind="vfae", L=1000), "256"),
    (dict(n_models=(1 << 20) + 1), "2^20"),
], ids=["L257", "pvae_L257", "vfae_L1000", "models_2p20_plus1"])
def test_noise_key_ranges_are_enforced_at_plan_creation(kw, limit):
    rc, msg = _create(**kw)
    assert rc != 0
    assert limit in msg, msg


def test_L_256_passes_the_argument_checks():
    """Without a device the call gets past the argument checks and fails at the first allocation."""
    rc, msg = _create(L=256, max_batch=2)
    assert rc == 0 or "cudaMalloc" in msg, msg


@pytest.mark.skipif(torch.cuda.is_available(), reason="on a device this would allocate the workspace of 2^20 models")
def test_2p20_models_pass_the_argument_checks():
    rc, msg = _create(n_models=1 << 20)
    assert rc != 0 and "cudaMalloc" in msg, msg
