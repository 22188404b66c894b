"""CPU: known answers of the importance-weighted log-likelihood restated in tests/likelihood_oracle.py (fp64), and its
relation to the ELBO terms of the unchanged oracle's unsup_loss."""
import math
import os

import numpy as np
import pytest
import torch

import gccvae_oracle as O
import likelihood_oracle as LO
from helpers import GOLDEN


def _setup(B, K, seed=3):
    p = O.init_params(0, dtype=torch.float64, trained_like=True)
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(B, 64, 64, 3, generator=g, dtype=torch.float64)
    y = (torch.rand(B, 18, generator=g) < 0.5).to(torch.int64)
    eps = torch.randn(K, B, 45, generator=g, dtype=torch.float64)
    U_y = torch.rand(K, B, 18, generator=g, dtype=torch.float64)
    mu = torch.as_tensor(np.load(os.path.join(GOLDEN, "data", "gating_matrix_0.2.npy")))
    U1 = torch.rand(18, 18, generator=g, dtype=torch.float64)
    U2 = torch.rand(18, 18, generator=g, dtype=torch.float64)
    c = O.sample_gating_parameter(mu, 0.3, U1, U2)
    return p, x, y, eps, U_y, c, (mu, U1, U2)


@pytest.mark.parametrize("labelled", [True, False])
def test_one_sample_is_its_log_weight(labelled):
    p, x, y, eps, U_y, c, _ = _setup(4, 1)
    est, ess, lw = LO.log_likelihood(p, x, c, eps, y if labelled else None, U_y)
    assert torch.equal(est, lw[0]) and torch.equal(ess, torch.ones(4, dtype=torch.float64))


@pytest.mark.parametrize("labelled", [True, False])
def test_identical_samples_cancel_ln_k(labelled):
    p, x, y, eps, U_y, c, _ = _setup(4, 1)
    K = 7
    est, ess, lw = LO.log_likelihood(p, x, c, eps.repeat(K, 1, 1), y if labelled else None, U_y.repeat(K, 1, 1))
    one = LO.log_weight_terms(p, x, c, eps, y if labelled else None, U_y)["log_w"][0]
    assert float(((est - one) / one).abs().max()) <= 1e-12
    assert float((ess - K).abs().max()) <= 1e-9


def _scalar_log_w(p, x, c, e, y, u):
    """log w of one image and one sample, term by term with Python floats (no tensor algebra except the networks)."""
    locs, scale = O.encoder(p, x.unsqueeze(0))
    locs, scale = locs[0].tolist(), scale[0].tolist()
    e = e.tolist()
    z = [locs[d] + scale[d] * e[d] for d in range(45)]
    h = 0.5 * math.log(2.0 * math.pi)
    log_q = sum(-0.5 * e[d] * e[d] - math.log(scale[d]) - h for d in range(45))
    log_pzs = sum(-0.5 * z[d] * z[d] - h for d in range(27))
    cc, W, bcls = c.tolist(), p["cls.w"].tolist(), p["cls.b"].tolist()
    logits = [bcls[j] + sum(z[27 + i] * cc[i][j] * W[i][j] for i in range(18)) for j in range(18)]
    if y is None:
        yk = [1 if u[j] < 1.0 / (1.0 + math.exp(-logits[j])) else 0 for j in range(18)]
    else:
        yk = [int(v != 0) for v in y.tolist()]
    softplus = lambda v: max(v, 0.0) + math.log1p(math.exp(-abs(v)))
    log_qy = sum(-softplus(-logits[j]) if yk[j] else -softplus(logits[j]) for j in range(18))
    lt, lf, st, sf = (p[k].tolist() for k in ("prior.loc_true", "prior.loc_false", "prior.scale_true", "prior.scale_false"))
    log_pzc = 0.0
    for i in range(18):
        loc = sum(cc[i][j] * (lt[j][i] if yk[j] else lf[j][i]) for j in range(18))
        s_pre = sum(cc[i][j] * (st[j][i] if yk[j] else sf[j][i]) for j in range(18))
        s = min(max(softplus(s_pre), 1e-3), 1e3)
        log_pzc += -0.5 * ((z[27 + i] - loc) / s) ** 2 - math.log(s) - h
    xhat = O.decoder(p, torch.tensor([z], dtype=torch.float64))[0].reshape(-1).tolist()
    xs = x.reshape(-1).tolist()
    log_pxz = sum(-abs(xs[t] - xhat[t]) - math.log(2.0) for t in range(len(xs)))
    log_w = log_pxz + log_pzs + log_pzc + 18 * math.log(0.5) - log_q
    return log_w - (log_qy if y is None else 0.0)


@pytest.mark.parametrize("labelled", [True, False])
def test_log_weight_matches_a_scalar_loop(labelled):
    p, x, y, eps, U_y, c, _ = _setup(2, 2)
    lw = LO.log_weight_terms(p, x, c, eps, y if labelled else None, U_y)["log_w"]
    for k in range(2):
        for b in range(2):
            want = _scalar_log_w(p, x[b], c, eps[k, b], y[b] if labelled else None, U_y[k, b].tolist())
            assert abs(float(lw[k, b]) - want) <= 1e-9 * abs(want), (k, b, float(lw[k, b]), want)


def test_relation_to_the_elbo_of_unsup_loss():
    """Same eps / U_y as unsup_loss at K = 1: log p(x|z) and log q(y|z_c) are its terms, and
    log w_1 - elbo = KL_closed - KL_MC, with KL_MC = log q(z|x) - log p(z|y) of that draw."""
    B = 6
    p, x, y, eps, U_y, c, (mu, U1, U2) = _setup(B, 1)
    cfg = dict(gate_type="fixed", gate_subtype="inferred", gating_reg=0.0)
    out = O.unsup_loss(p, mu, x, dict(eps=eps[0], U_y=U_y[0], U1=U1, U2=U2), cfg, 0.3)
    assert torch.equal(out["c"], c)
    t = LO.log_weight_terms(p, x, c, eps, None, U_y)
    assert float((t["log_pxz"][0] - out["log_pxz"]).abs().max()) <= 1e-9 * float(out["log_pxz"].abs().max())
    assert float((t["log_qy"][0] - out["log_qy_zc"]).abs().max()) <= 1e-12 * float(out["log_qy_zc"].abs().max())
    assert torch.equal(t["y"][0], out["y"].to(torch.int64))
    kl_mc = t["log_q"][0] - t["log_pzs"][0] - t["log_pzc"][0]
    lhs = t["log_w"][0] - out["elbo"]
    rhs = out["kl"] - kl_mc
    assert float((lhs - rhs).abs().max()) <= 1e-9 * float(out["elbo"].abs().max()), (lhs, rhs)


@pytest.mark.parametrize("labelled", [True, False])
def test_mean_estimate_does_not_decrease_with_k(labelled):
    """An expectation property (E log p_hat_K grows with K), asserted on seeded inputs.  Means over 64 images,
    trained-like parameters, fresh draws per K (K = 1, 4, 16, 64), as recorded:
      labelled (log p(x, y)): -11623.48, -11620.68, -11619.48, -11617.85  (margins 2.80, 1.21, 1.63)
      unlabelled (log p(x)):  -11611.69, -11608.78, -11607.40, -11605.73  (margins 2.91, 1.39, 1.67)"""
    B = 64
    p, x, y, _, _, c, _ = _setup(B, 1)
    g = torch.Generator().manual_seed(17)
    means = []
    for K in (1, 4, 16, 64):
        eps = torch.randn(K, B, 45, generator=g, dtype=torch.float64)
        U_y = torch.rand(K, B, 18, generator=g, dtype=torch.float64)
        est, _, _ = LO.log_likelihood(p, x, c, eps, y if labelled else None, U_y)
        means.append(float(est.mean()))
    margins = [b - a for a, b in zip(means, means[1:])]
    print("labelled={}: mean log p_hat over K = 1, 4, 16, 64: {} (margins {})".format(
        labelled, ["{:.4f}".format(m) for m in means], ["{:.4f}".format(m) for m in margins]))
    assert all(m >= 0.0 for m in margins), (means, margins)
