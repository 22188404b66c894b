"""CPU: known answers of the completion's restatement (tests/completion_oracle.py).
  * an all-observed mask returns x, whatever the number of iterations;
  * with nothing observed, one iteration is the reconstruction (or the intervention) of x;
  * `iters` = T is T single steps chained, each from the previous step's composite;
  * observed pixels never change and the others are the last step's decode."""
import pytest
import torch

import completion_oracle as CO
import generation_oracle as GO
from test_oracle_walk import _setup

DTYPES = [torch.float64, torch.float32]


def _mask(B, seed=3):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(B, 64, 64, generator=g) < 0.6


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("labels", [False, True])
def test_all_observed_returns_x(dtype, labels):
    p, x, y, noise, c = _setup(dtype)
    y_new = (1 - y) if labels else None
    out, z, _ = CO.complete(p, x, torch.ones(x.shape[0], 64, 64, dtype=torch.bool), 3, y_new=y_new, c=c)
    assert torch.equal(out, x)
    _, z_r = GO.reconstruct(p, x)
    if not labels:     # every iteration encodes x itself: z is its posterior mean
        assert torch.equal(z, z_r)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("sample", [False, True])
def test_nothing_observed_one_iteration_is_reconstruct_or_intervene(dtype, sample):
    p, x, y, noise, c = _setup(dtype)
    eps = noise["eps"] if sample else None
    none = torch.zeros(x.shape[0], 64, 64, dtype=torch.bool)
    out, z, _ = CO.complete(p, x, none, 1, eps=None if eps is None else eps[None])
    img_r, z_r = GO.reconstruct(p, x, eps)
    assert torch.equal(out, img_r) and torch.equal(z, z_r)
    y_new = 1 - y
    out, z, y_src = CO.complete(p, x, none, 1, y_new=y_new, c=c, y=y, eps=None if eps is None else eps[None])
    img_i, z_i, y_i = GO.intervene(p, x, y_new, c, y=y, eps=eps)
    assert torch.equal(out, img_i) and torch.equal(z, z_i) and torch.equal(y_src, y_i)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("labels", [False, True])
def test_iterations_chain_single_steps(dtype, labels):
    p, x, y, noise, c = _setup(dtype)
    B, T = x.shape[0], 3
    m = _mask(B)
    eps = torch.randn(T, B, 45, generator=torch.Generator().manual_seed(7), dtype=dtype)
    y_new = (1 - y) if labels else None
    out, z, y_src = CO.complete(p, x, m, T, y_new=y_new, c=c, eps=eps)
    comp = x
    for t in range(T):
        comp, img, z_t, y_t = CO.step(p, comp, x, m, y_new=y_new, c=c, eps=eps[t])
    assert torch.equal(out, comp) and torch.equal(z, z_t)
    assert (y_src is None) == (not labels) and (y_src is None or torch.equal(y_src, y_t))
    mm = m.unsqueeze(-1).expand_as(x)
    assert torch.equal(out[mm], x[mm]) and torch.equal(out[~mm], img[~mm])
    # T = 2 from x is T = 1 from the first composite (with the observed pixels of x)
    c1, _, _ = CO.complete(p, x, m, 1, y_new=y_new, c=c, eps=eps[:1])
    two, _, _ = CO.complete(p, x, m, 2, y_new=y_new, c=c, eps=eps[:2])
    comp2, _, _, _ = CO.step(p, c1, x, m, y_new=y_new, c=c, eps=eps[1])
    assert torch.equal(two, comp2)
