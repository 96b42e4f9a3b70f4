"""CPU oracle of the plain SVGP baseline -- TEST INFRASTRUCTURE ONLY (imported by tests/test_svgp_*.py).

gpytorch's VariationalStrategy with ScaleKernel(RBFKernel()) as traditional_vi.py uses it: whitened, over the M function
values at the inducing points, no directions on either side, targets y = f(x).  This is the p = 0 case of
oracle/dsvgp_oracle.py's lean structure, built from that module's pieces (closed-form kernel, psd_safe_cholesky, KL,
softplus transforms, the gpytorch 1.4 constants) and restated here with the same function names and signatures, so that the
directional oracle stays as it is.  Every function only takes the SVGP case: direction arguments must be None, p must be 0.
tests/test_svgp_oracle.py checks it against an independent plain-torch SVGP.
"""
import math
from dataclasses import dataclass, fields

import torch

from oracle import dsvgp_oracle as O

F64 = torch.float64
testfun = O.testfun


@dataclass
class Params(O.Params):
    """O.Params with Vz = None (no inducing directions)"""

    def clone(self, dtype=None):
        return Params(**{f.name: (None if getattr(self, f.name) is None else
                                  getattr(self, f.name).detach().clone().to(dtype or getattr(self, f.name).dtype))
                         for f in fields(self)})


def _svgp_only(Vx=None, variant="svgp"):
    assert variant == "svgp" and Vx is None, "the SVGP baseline has no directions"


def _eye(n, like):
    return torch.eye(n, dtype=like.dtype, device=like.device)


def _factor(P, x):
    """A = L^-1 K_zx (model dtype) with L = chol(K_zz + 1e-3 I) in fp64 (DGVS.py:72-75,144 restated for p = 0)"""
    ell, osc = O.lengthscale(P), O.outputscale(P)
    Kzx = osc * O.kernel_closed_form(P.Z, x, None, None, ell)
    Kzz = osc * O.kernel_closed_form(P.Z, P.Z, None, None, ell) + O.KZZ_JITTER * _eye(P.Z.shape[0], P.Z)
    L = O.psd_safe_cholesky(Kzz.double())
    return torch.linalg.solve_triangular(L, Kzx.double(), upper=False).to(x.dtype), ell, osc


def predictive(P, x, Vx=None, variant="svgp"):
    """q(f) at the minibatch: (mean, variance) of length n; variance with the +1e-4 jitter, without likelihood noise"""
    _svgp_only(Vx, variant)
    A, ell, osc = _factor(P, x)
    Ls = O.chol_factor_of_q(P)
    mean = A.transpose(-1, -2) @ P.m + P.c.expand(A.shape[1])
    var = osc * torch.ones(x.shape[0], dtype=x.dtype) + O.PRED_JITTER + (A * (Ls @ (Ls.transpose(-1, -2) @ A) - A)).sum(0)
    return mean, var


def predictive_full(P, x, Vx=None, variant="svgp", add_noise=False):
    """(mean, dense n x n covariance K_xx + 1e-4 I + A^T (S - I) A) [+ sigma^2 I]"""
    _svgp_only(Vx, variant)
    A, ell, osc = _factor(P, x)
    Ls = O.chol_factor_of_q(P)
    mean = A.transpose(-1, -2) @ P.m + P.c.expand(A.shape[1])
    Kxx = osc * O.kernel_closed_form(x, x, None, None, ell)
    cov = Kxx + O.PRED_JITTER * _eye(x.shape[0], Kxx) + A.transpose(-1, -2) @ (Ls @ (Ls.transpose(-1, -2) @ A) - A)
    if add_noise:
        cov = cov + O.noise(P) * _eye(cov.shape[0], cov)
    return mean, cov


def predict(P, x, Vx=None, variant="svgp"):
    """eval_gp's per-batch result: likelihood(model(x)) mean and (clamped) variance including the noise"""
    mean, var = predictive(P, x, Vx, variant)
    return mean, O.clamp_variance(var + O.noise(P))


def elbo(P, x, Vx, y, num_data, variant="svgp", through_likelihood=True):
    """VariationalELBO on likelihood(model(x)) (quirk Q3: the data term sees var + sigma^2)"""
    mean, var = predictive(P, x, Vx, variant)
    s2 = O.noise(P)
    if through_likelihood:
        var = var + s2
    var = O.clamp_variance(var)
    terms = -0.5 * (((y - mean) ** 2 + var) / s2 + torch.log(s2) + math.log(2 * math.pi))
    return terms.sum() / mean.numel() - O.kl_divergence(P) / num_data


def pll(P, x, Vx, y, num_data, variant="svgp", noise_mult=2):
    """PredictiveLogLikelihood on likelihood(model(x)): v = var_f + noise_mult * sigma^2"""
    mean, var = predictive(P, x, Vx, variant)
    var = O.clamp_variance(var + noise_mult * O.noise(P))
    ll = -0.5 * ((y - mean) ** 2 / var + var.log() + math.log(2 * math.pi))
    return ll.sum() / mean.numel() - O.kl_divergence(P) / num_data


def _value_and_grads(fn, P, *args, **kw):
    Q = Params(**P.tensors()).clone().requires_grad_(True)
    val = fn(Q, *args, **kw)
    names = [k for k, t in Q.tensors().items() if t is not None]
    grads = torch.autograd.grad(val, [getattr(Q, k) for k in names], allow_unused=True)
    return val.detach(), {k: (g if g is not None else torch.zeros_like(getattr(Q, k))) for k, g in zip(names, grads)}


def elbo_and_grads(P, x, Vx, y, num_data, variant="svgp", through_likelihood=True):
    """the ELBO and dELBO / dparam of one training step"""
    return _value_and_grads(elbo, P, x, Vx, y, num_data, variant, through_likelihood)


def pll_and_grads(P, x, Vx, y, num_data, variant="svgp", noise_mult=2):
    return _value_and_grads(pll, P, x, Vx, y, num_data, variant, noise_mult)


def ngd_elbo_and_grads(P, nat_vec, nat_mat, x, Vx, y, num_data, variant="svgp"):
    """ELBO of the model whose q(u) is given in natural parameters, and the natural gradients (gpytorch 1.4
    _NaturalToMuVarSqrt semantics, oracle/dsvgp_oracle.py) plus the ordinary gradients of the other parameters"""
    Q = Params(**P.tensors()).clone().requires_grad_(True)
    nv, nm = nat_vec.detach().clone().requires_grad_(True), nat_mat.detach().clone().requires_grad_(True)
    Q.m, Q.Ls_raw = O.natural_to_mean_chol(nv, nm)
    val = elbo(Q, x, Vx, y, num_data, variant)
    names = ["Z", "c", "raw_os", "raw_ell", "raw_noise"]
    grads = torch.autograd.grad(val, [nv, nm] + [getattr(Q, k) for k in names], allow_unused=True)
    out = {"natural_vec": grads[0], "natural_mat": grads[1]}
    out.update({k: g for k, g in zip(names, grads[2:])})
    return val.detach(), out


def elbo_and_grads_chunked(P, x, Vx, y, num_data, variant="svgp", chunk=2048, through_likelihood=True):
    """elbo_and_grads for minibatches too large to differentiate in one piece on the host: the data term chunk by chunk,
    the KL once.  Also returns the predictive (mean, variance + noise, clamped) of every point."""
    _svgp_only(Vx, variant)
    n, nq = x.shape[0], x.shape[0]
    names = [k for k, t in P.tensors().items() if t is not None]
    total = {k: torch.zeros_like(getattr(P, k)) for k in names}
    val, means, variances = 0.0, [], []
    for lo in range(0, n, chunk):
        hi = min(n, lo + chunk)
        Q = Params(**P.tensors()).clone().requires_grad_(True)
        mean, var = predictive(Q, x[lo:hi])
        s2 = O.noise(Q)
        if through_likelihood:
            var = var + s2
        var = O.clamp_variance(var)
        part = (-0.5 * (((y[lo:hi] - mean) ** 2 + var) / s2 + torch.log(s2) + math.log(2 * math.pi))).sum() / nq
        for k, g in zip(names, torch.autograd.grad(part, [getattr(Q, k) for k in names], allow_unused=True)):
            if g is not None:
                total[k] += g
        val += float(part.detach())
        means.append(mean.detach())
        variances.append(var.detach())
    Q = Params(**P.tensors()).clone().requires_grad_(True)
    kl = O.kl_divergence(Q) / num_data
    gk = torch.autograd.grad(kl, [Q.m, Q.Ls_raw])
    total["m"] -= gk[0]
    total["Ls_raw"] -= gk[1]
    return torch.tensor(val - float(kl.detach()), dtype=F64), total, torch.cat(means), torch.cat(variances)


def make_problem(n, d, M, p=0, dtype=F64, seed=0, variant="svgp", N=None):
    """Seeded inputs as oracle/dsvgp_oracle.make_problem draws them (same generator order for x, Z, m, L_s), with no
    directions: V_z = V_x = None, y = f(x) of tests/testfun.py, num_data = N (or n)."""
    assert p == 0 and variant == "svgp", "the SVGP baseline has no directions: p = 0"
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(n, d, generator=g, dtype=F64)
    Z = torch.rand(M, d, generator=g, dtype=F64)
    m = 1e-3 * torch.randn(M, generator=g, dtype=F64)
    Ls = torch.eye(M, dtype=F64) + 0.01 * torch.randn(M, M, generator=g, dtype=F64).tril()
    Ls = Ls + 0.5 * torch.randn(M, M, generator=g, dtype=F64).triu(1)     # arbitrary, must be ignored
    y = testfun(x)[:, 0].clone()
    P = Params(Z=Z, Vz=None, m=m, Ls_raw=Ls, c=torch.full((1,), 0.05, dtype=F64), raw_os=torch.tensor(0.1, dtype=F64),
               raw_ell=torch.full((1, 1), -0.2, dtype=F64), raw_noise=torch.full((1,), -1.0, dtype=F64))
    return P.clone(dtype), x.to(dtype), None, y.to(dtype), (N or n)


def make_trained_problem(n, d, M, p=0, dtype=F64, seed=0, variant="svgp", ell=0.7, kind="optimal", N=None, weight=20.0):
    """Inputs in a TRAINED state as oracle/dsvgp_oracle.make_trained_problem makes them: lengthscale `ell`, two pairs of
    near-duplicate inducing points, and kind="optimal": (m, S) at the ELBO optimum of a fit set of 2n points weighted
    `weight` times, with a 2 % perturbation; kind="rough": unstructured L_s and m."""
    P, x, _, y, num_data = make_problem(n, d, M, p, F64, seed, variant, N=N)
    g = torch.Generator().manual_seed(seed + 7919)
    P.raw_ell = O._inv_softplus(ell).reshape(1, 1)
    P.Z[1] = P.Z[0] + 1e-4 * torch.randn(d, generator=g, dtype=F64)
    P.Z[M - 1] = P.Z[M // 2] + 1e-3 * torch.randn(d, generator=g, dtype=F64)
    upper = P.Ls_raw.triu(1)
    if kind == "rough":
        Ls = torch.diag(0.05 + 0.45 * torch.rand(M, generator=g, dtype=F64)) + 0.3 * torch.randn(M, M, generator=g, dtype=F64).tril(-1)
        P.m = torch.randn(M, generator=g, dtype=F64)
    else:
        xf = torch.rand(2 * n, d, generator=g, dtype=F64)
        yf = testfun(xf)[:, 0]
        A, _, _ = _factor(P, xf)
        s2 = O.noise(P)
        Li = torch.linalg.cholesky(torch.eye(M, dtype=F64) + (weight / s2) * (A @ A.T))
        Wi = torch.linalg.solve_triangular(Li, torch.eye(M, dtype=F64), upper=False)
        S = Wi.T @ Wi
        Ls = torch.linalg.cholesky(0.5 * (S + S.T))
        P.m = (weight / s2) * (S @ (A @ (yf - P.c)))
        Ls = Ls * (1.0 + 0.02 * torch.randn(M, M, generator=g, dtype=F64)).tril()
        P.m = P.m * (1.0 + 0.02 * torch.randn(M, generator=g, dtype=F64))
    P.Ls_raw = Ls.tril() + upper
    return P.clone(dtype), x.to(dtype), None, y.to(dtype), num_data
