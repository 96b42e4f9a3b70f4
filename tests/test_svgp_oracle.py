"""The SVGP-baseline oracle (tests/svgp_oracle.py: gpytorch's VariationalStrategy with ScaleKernel(RBFKernel()), what
traditional_vi.py trains, built from oracle/dsvgp_oracle.py's pieces with p = 0) against an independent plain-torch SVGP written from the textbook whitened form, with no
directional code: closed-form RBF, torch.linalg.cholesky, solve_triangular and autograd.  fp64, gate 1e-12 (max-norm
relative per tensor).  CPU only."""
import math

import pytest
import torch
from torch.nn.functional import softplus

from oracle import dsvgp_oracle as O
import svgp_oracle as S

F64 = torch.float64


def rel(a, b):
    a, b = a.detach().reshape(-1), b.detach().reshape(-1)
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-300))


def _rbf(a, b, ell, osc):
    r2 = ((a[:, None, :] - b[None, :, :]) ** 2).sum(-1)
    return osc * torch.exp(-0.5 * r2 / ell ** 2)


def _svgp(Z, m, Ls_raw, c, raw_os, raw_ell, raw_noise, x):
    """whitened SVGP q(f(x)): mean A^T m + c, covariance K_xx + 1e-4 I + A^T (S - I) A with A = L^-1 K_zx,
    L = chol(K_zz + 1e-3 I), S = L_s L_s^T, L_s = tril(Ls_raw)"""
    ell, osc = softplus(raw_ell).reshape(()), softplus(raw_os).reshape(())
    Kzz = _rbf(Z, Z, ell, osc) + 1e-3 * torch.eye(Z.shape[0], dtype=F64)
    L = torch.linalg.cholesky(Kzz)
    A = torch.linalg.solve_triangular(L, _rbf(Z, x, ell, osc), upper=False)
    Ls = Ls_raw.tril()
    mean = A.T @ m + c
    cov = _rbf(x, x, ell, osc) + 1e-4 * torch.eye(x.shape[0], dtype=F64) + A.T @ (Ls @ (Ls.T @ A) - A)
    s2 = softplus(raw_noise).reshape(()) + 1e-4
    kl = 0.5 * ((Ls * Ls).sum() + (m * m).sum() - m.numel() - Ls.diagonal().pow(2).log().sum())
    return mean, cov, s2, kl


def _elbo(args, x, y, num_data):
    mean, cov, s2, kl = _svgp(*args, x)
    var = (cov.diagonal() + s2).clamp_min(1e-10)           # likelihood(model(x)) goes to the ELBO (quirk Q3)
    terms = -0.5 * (((y - mean) ** 2 + var) / s2 + torch.log(s2) + math.log(2 * math.pi))
    return terms.mean() - kl / num_data


def _pll(args, x, y, num_data):
    mean, cov, s2, kl = _svgp(*args, x)
    var = (cov.diagonal() + 2 * s2).clamp_min(1e-10)
    return (-0.5 * ((y - mean) ** 2 / var + var.log() + math.log(2 * math.pi))).mean() - kl / num_data


NAMES = ("Z", "m", "Ls_raw", "c", "raw_os", "raw_ell", "raw_noise")


def _value_and_grads(fn, P, x, y, num_data):
    args = [getattr(P, k).detach().clone().requires_grad_(True) for k in NAMES]
    val = fn(args, x, y, num_data)
    return val.detach(), dict(zip(NAMES, torch.autograd.grad(val, args)))


PROBLEMS = [("plain", 200, 2, 20), ("plain", 97, 5, 33), ("optimal", 120, 3, 24)]


def _problem(kind, n, d, M):
    if kind == "plain":
        return S.make_problem(n, d, M, 0, F64, seed=n + d, variant="svgp", N=10 * n)
    return S.make_trained_problem(n, d, M, 0, F64, seed=n + d, variant="svgp", ell=0.15, kind="optimal", N=10 * n)


@pytest.mark.parametrize("kind,n,d,M", PROBLEMS)
def test_svgp_problem_has_no_directions(kind, n, d, M):
    P, x, Vx, y, num_data = _problem(kind, n, d, M)
    assert P.Vz is None and Vx is None
    assert y.shape == (n,) and torch.equal(y, O.testfun(x)[:, 0])
    assert P.m.shape == (M,) and P.Ls_raw.shape == (M, M) and num_data == 10 * n
    assert P.clone(torch.float32).Vz is None


@pytest.mark.parametrize("kind,n,d,M", PROBLEMS)
def test_svgp_predictive_matches_plain_torch(kind, n, d, M):
    P, x, Vx, y, _ = _problem(kind, n, d, M)
    mean, cov, s2, _ = _svgp(*[getattr(P, k) for k in NAMES], x)
    m_o, v_o = S.predictive(P, x, Vx, variant="svgp")
    assert rel(m_o, mean) < 1e-12 and rel(v_o, cov.diagonal()) < 1e-12
    m_f, c_f = S.predictive_full(P, x, Vx, variant="svgp")
    assert rel(m_f, mean) < 1e-12 and rel(c_f, cov) < 1e-12
    _, c_n = S.predictive_full(P, x, Vx, variant="svgp", add_noise=True)
    assert rel(c_n, cov + s2 * torch.eye(n, dtype=F64)) < 1e-12
    m_p, v_p = S.predict(P, x, Vx, variant="svgp")
    assert rel(v_p, (cov.diagonal() + s2).clamp_min(1e-10)) < 1e-12


@pytest.mark.parametrize("kind,n,d,M", PROBLEMS)
def test_svgp_elbo_and_pll_gradients_match_plain_torch(kind, n, d, M):
    P, x, Vx, y, num_data = _problem(kind, n, d, M)
    for fn, oracle in ((_elbo, S.elbo_and_grads), (_pll, S.pll_and_grads)):
        val, grads = _value_and_grads(fn, P, x, y, num_data)
        o_val, o_grads = oracle(P, x, Vx, y, num_data, variant="svgp")
        assert abs(float(o_val) - float(val)) <= 1e-12 * abs(float(val))
        assert set(o_grads) == set(NAMES)
        for k in NAMES:
            assert rel(o_grads[k], grads[k]) < 1e-12, (fn.__name__, k)


def test_svgp_ngd_gradients_match_plain_torch():
    P, x, Vx, y, num_data = _problem("plain", 150, 3, 25)
    g = torch.Generator().manual_seed(4)
    B = torch.eye(25, dtype=F64) + 0.1 * torch.randn(25, 25, generator=g, dtype=F64).tril()
    Sq = B @ B.T
    nat_mat, nat_vec = -0.5 * torch.linalg.inv(Sq), torch.linalg.solve(Sq, 0.2 * torch.randn(25, generator=g, dtype=F64))
    val, grads = S.ngd_elbo_and_grads(P, nat_vec, nat_mat, x, Vx, y, num_data, variant="svgp")
    # independent: the ELBO as a function of (m, S) with m = S theta1, S = (-2 theta2)^-1; the natural gradient is the
    # ordinary gradient with respect to the expectation parameters (eta1, eta2) = (m, S + m m^T)
    eta1 = (Sq @ nat_vec).clone().requires_grad_(True)
    eta2 = (Sq + torch.outer(Sq @ nat_vec, Sq @ nat_vec)).clone().requires_grad_(True)
    Sx = eta2 - torch.outer(eta1, eta1)
    args = [P.Z, eta1, torch.linalg.cholesky(0.5 * (Sx + Sx.T)), P.c, P.raw_os, P.raw_ell, P.raw_noise]
    ref = _elbo(args, x, y, num_data)
    g1, g2 = torch.autograd.grad(ref, [eta1, eta2])
    assert abs(float(val) - float(ref.detach())) <= 1e-12 * abs(float(ref.detach()))
    assert rel(grads["natural_vec"], g1) < 1e-10
    assert rel(grads["natural_mat"], 0.5 * (g2 + g2.T)) < 1e-10
    assert "Vz" not in grads


def test_svgp_variant_refuses_directions():
    with pytest.raises(AssertionError):
        S.make_problem(50, 3, 10, 1, F64, variant="svgp")
