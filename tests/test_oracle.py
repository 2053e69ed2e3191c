"""CPU: the oracle (oracle/drvae_oracle.py) against the golden vectors recorded from the
reference itself (tests/golden/*.npz, written by oracle/make_golden.py)."""
import os

import numpy as np
import pytest
import torch

from helpers import ARCH, GOLDEN, KINDS, L, NROWS, SEED_MODEL, SEED_TAPE, golden, orc

from drvae_b200.init import init_state_dict

CASES = ("tiny", "deep", "readme", "tiny_wn")


def _sd(kind, case, g):
    if any(k.startswith("sd/") for k in g.files):
        return {k[3:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd/")}
    return init_state_dict(kind, seed=SEED_MODEL, **ARCH[case])


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("kind", KINDS)
def test_oracle_matches_reference_golden(kind, case):
    torch.set_num_threads(4)
    g = golden(kind, case)
    arch, N = ARCH[case], NROWS[case]
    sd = _sd(kind, case, g)
    batch = orc.synthetic_batch(N, arch["dim_x"])
    om = orc.OracleModel(sd, orc.default_cfg(kind, L=L))
    # eval-mode loss
    le = om.loss(batch, orc.Tape(seed=SEED_TAPE + 100), train=False)
    for k, v in le.items():
        ref = float(g["loss_eval/" + k])
        assert abs(float(v) - ref) <= 1e-5 * abs(ref) + 1e-7, (k, float(v), ref)
    # two training steps, gradients of the first
    for it in range(2):
        tape = orc.Tape(seed=SEED_TAPE + it)
        lo = om.step(batch, tape)
        assert [len(tape.log), sum(t.numel() for t in tape.log)] == list(g["meta/draws%d" % it])
        for k, v in lo.items():
            ref = float(g["loss_train%d/%s" % (it, k)])
            assert abs(float(v) - ref) <= 1e-5 * abs(ref) + 1e-7, (it, k, float(v), ref)
        if it == 0:
            for name, p in om.sd.items():
                gn = float(g["gradnorm0/" + name])
                assert abs(float(p.grad.double().norm()) - gn) <= 1e-4 * gn + 1e-9, name
                if "grad0/" + name in g.files:
                    ref = torch.from_numpy(g["grad0/" + name])
                    assert (p.grad - ref).abs().max() <= 1e-4 * ref.abs().max() + 1e-9, name
                else:
                    stride = int(g["gradstride0/" + name])
                    ref = torch.from_numpy(g["gradsample0/" + name])
                    got = p.grad.reshape(-1)[::stride][:ref.numel()]
                    assert (got - ref).abs().max() <= 1e-4 * ref.abs().max() + 1e-9, name


@pytest.mark.parametrize("kind", KINDS)
def test_oracle_forward_matches_reference_golden(kind):
    g = golden(kind, "tiny")
    arch = ARCH["tiny"]
    om = orc.OracleModel(_sd(kind, "tiny", g), orc.default_cfg(kind, L=L))
    fo = om.forward(torch.from_numpy(g["batch/x1"]))
    for key in ("pred", "proba", "z1", "z2", "x1_rec", "x2_pert"):
        if "fwd/" + key in g.files:
            assert np.allclose(fo[key].numpy(), g["fwd/" + key], rtol=1e-4, atol=1e-5), key


def test_golden_files_stay_small():
    for f in os.listdir(GOLDEN):
        assert os.path.getsize(os.path.join(GOLDEN, f)) <= 1 << 20, f


def test_bf16_emulation_is_close_to_fp32():
    """The emulated rounding must stay inside the 1e-3 budget north_star gives the bf16 path."""
    arch, N = ARCH["tiny"], NROWS["tiny"]
    sd = init_state_dict("drvae", seed=SEED_MODEL, **arch)
    batch = orc.synthetic_batch(N, arch["dim_x"])
    om = orc.OracleModel(sd, orc.default_cfg("drvae", L=L))
    tape = orc.Tape(seed=SEED_TAPE)
    a, _ = om.grads(batch, tape, emulate_bf16=False)
    b, _ = om.grads(batch, orc.Tape(recorded=tape.log), emulate_bf16=True)
    for k in ("RECL", "KLD", "PERT", "YL", "ELBO", "CMPL"):
        assert abs(float(a[k]) - float(b[k])) <= 1e-3 * abs(float(a[k])), k
