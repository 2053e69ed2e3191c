"""CPU: the gradient comparison of tests/helpers.py (assert_grad_close) passes bf16-sized noise and catches the
localised faults a tensor-wide relative L2 lets through."""
import pytest
import torch

from helpers import assert_grad_close, grad_errors, rel_l2

ROWS, COLS = 300, 978  # a decoder-head-like weight gradient: 978 inputs, a partial 128-row block at the end


def _reference(seed=0):
    """Gradient-like matrix: rows and columns of very different scales, plus its bias vector."""
    g = torch.Generator().manual_seed(seed)
    rs = torch.exp(torch.randn(ROWS, 1, generator=g, dtype=torch.float64))
    cs = torch.exp(0.5 * torch.randn(1, COLS, generator=g, dtype=torch.float64))
    W = torch.randn(ROWS, COLS, generator=g, dtype=torch.float64) * rs * cs
    b = torch.randn(ROWS, generator=g, dtype=torch.float64) * rs[:, 0]
    return W, b


def _noisy(t, seed=1, rel=4e-3):
    g = torch.Generator().manual_seed(seed)
    return t * (1 + rel * torch.randn(t.shape, generator=g, dtype=torch.float64))


def test_bf16_sized_noise_passes():
    W, b = _reference()
    e = assert_grad_close(_noisy(W), W, "W")
    assert e["row"][0] < 1e-2 and e["col"][0] < 1e-2, e  # a third of the default line tolerance
    assert_grad_close(_noisy(b, 2), b, "b")
    # a row whose reference is ~0 is held to the floor of the tensor's scale, not to its own rounding noise
    W0 = W.clone()
    W0[7] *= 1e-9
    got = _noisy(W0)
    got[7] += 1e-4 * W.norm() / ROWS ** 0.5 / COLS ** 0.5 * torch.randn(COLS, dtype=torch.float64)
    assert_grad_close(got, W0, "W with a near-zero row")


def _zero_col(W):
    W[:, 517] = 0


def _zero_row(W):
    W[211] = 0


def _block(W):
    W[128:144, 496:512] *= 1.3


def _col_30(W):
    W[:, 517] *= 1.3


def _lost_tile(W):
    W[:, 256:] = 0


FAULTS = [("one zeroed column", _zero_col), ("one zeroed row", _zero_row), ("one 16x16 block x1.3", _block),
          ("one column x1.3", _col_30)]
HIDDEN_FROM_L2 = ("one 16x16 block x1.3", "one column x1.3")


@pytest.mark.parametrize("name,fault", FAULTS, ids=[f[0] for f in FAULTS])
def test_localised_faults_fail(name, fault):
    W, _ = _reference()
    got = _noisy(W)
    fault(got)
    if name in HIDDEN_FROM_L2:
        assert rel_l2(got, W) <= 1e-2, "this fault should be invisible to the tensor-wide check alone"
    with pytest.raises(AssertionError):
        assert_grad_close(got, W, name)
    e = grad_errors(got, W)
    assert max(e["row"][0], e["col"][0]) > 3e-2, e


def test_error_message_names_the_line():
    W, _ = _reference()
    got = _noisy(W)
    _col_30(got)
    with pytest.raises(AssertionError, match="col 517 of"):
        assert_grad_close(got, W, "W")
    got = _noisy(W)
    got[211] *= 0.8
    with pytest.raises(AssertionError, match="row 211 of"):
        assert_grad_close(got, W, "W", tol_l2=1.0)


def test_lost_partial_n_tile_fails():
    """Everything past column 256 zeroed: the last of four N tiles 256 wide never written."""
    W, _ = _reference()
    got = _noisy(W)
    _lost_tile(got)
    with pytest.raises(AssertionError):
        assert_grad_close(got, W, "W")
    assert grad_errors(got, W)["col"][1] >= 256


def test_swapped_bias_block_fails():
    """The bias entries of one 128-row block permuted (adjacent pairs swapped): the tensor norm is unchanged."""
    _, b = _reference()
    got = _noisy(b)
    blk = got[128:256].clone().view(64, 2).flip(1).reshape(-1)
    got[128:256] = blk
    assert abs(float(got.norm() / b.norm()) - 1) < 1e-2
    with pytest.raises(AssertionError):
        assert_grad_close(got, b, "bias")
    assert 128 <= grad_errors(got, b)["row"][1] < 256
