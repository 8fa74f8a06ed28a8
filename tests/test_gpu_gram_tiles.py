"""The exact Gram kernel at row counts on both sides of its tile edges (64-row tiles, paired into 128-row super tiles,
with an odd last tile), on data whose products and sums are exact in float64: every element must equal numpy's
product bit for bit, whatever the summation order, so a misplaced, missing or mirrored block shows as an error."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return torch


def _exact(N, p, seed):
    # multiples of 1/8 below 8 in magnitude: products are multiples of 1/64 below 64, and a sum over a few thousand
    # voxels stays far inside the 53-bit significand
    return np.random.RandomState(seed).randint(-64, 64, size=(N, p)).astype(np.float64) / 8.0


@pytest.mark.parametrize("N", [1, 63, 64, 65, 127, 128, 129, 192, 193, 257, 312, 385])
@pytest.mark.parametrize("p", [1000, 997])
def test_gram_tiles_exact(torch_cuda, N, p):
    from plspy_b200.engine import Engine
    X = _exact(N, p, N + p)
    G = Engine(X).G.cpu().numpy()
    assert np.array_equal(G, X @ X.T)


@pytest.mark.parametrize("N", [65, 193])
def test_gram_tiles_x32_exact(torch_cuda, N):
    from plspy_b200.engine import Engine
    X = _exact(N, 2000, N).astype(np.float32)
    G = Engine(X, x_storage="fp32").G.cpu().numpy()
    Xw = X.astype(np.float64)
    assert np.array_equal(G, Xw @ Xw.T)


@pytest.mark.parametrize("N,K,fuses", [(300, 12, True), (250, 12, False), (128, 1, False), (120, 8, True)])
def test_gram_stack_tiles(torch_cuda, N, K, fuses):
    """The stack [X; Z] against numpy, and its X block against gram_of(X) bit for bit when the stack adds no tile."""
    import torch
    from plspy_b200._lib import lib
    from plspy_b200.engine import Engine
    X = _exact(N, 1500, N)
    Z = _exact(K, 1500, N + 1)
    assert bool(lib.plsb200_gram_stack_fuses(N, K)) == fuses
    eng = Engine(X)
    Gs = eng.gram_stacked(eng.X, torch.from_numpy(Z).to(eng.X.device)).cpu().numpy()
    S = np.vstack([X, Z])
    assert np.array_equal(Gs, S @ S.T)
    if fuses:
        assert np.array_equal(Gs[:N, :N], eng.gram_of(eng.X).cpu().numpy())
