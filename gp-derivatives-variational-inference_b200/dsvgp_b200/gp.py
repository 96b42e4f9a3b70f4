"""Host-side mirror of the reference's Python API for the DSVGP hot path (no gpytorch import).

The reference's boundary IS its Python class API (SURVEY.md section 8b): GPModel(gpytorch.models.ApproximateGP),
ScaleKernel(RBFKernelDirectionalGrad()), ConstantMean, CholeskyVariationalDistribution, the three variational
strategies, GaussianLikelihood and VariationalELBO.  This module provides those names with the same constructor
arguments, attributes, state-dict keys and error behaviour, backed by the CUDA engine (engine.py) instead of
eager gpytorch/ATen ops.  What a strategy call returns is a lazy `PredictiveDistribution`; handing it to
VariationalELBO runs ONE fused forward+backward on the GPU and hooks the result into autograd, so
`loss = -mll(likelihood(model(x, **kw)), y); loss.backward()` works unchanged (directional_vi.py:245-249).
"""
import math
import types
import warnings

import torch
from torch.nn import Parameter
from torch.nn.functional import softplus

from . import ops
from .engine import ENGINE, NanError, NotPSDError  # noqa: F401  (re-exported)


class OldVersionWarning(UserWarning):
    pass


def _inv_softplus(v):
    return v + torch.log(-torch.expm1(-v))


# ------------------------------------------------------------------------------------------------- modules
class Module(torch.nn.Module):
    """gpytorch.Module subset: hyperparameters() / variational_parameters() split used by the two optimisers
    (directional_vi.py:186-199)."""

    def named_hyperparameters(self):
        for prefix, mod in self.named_modules():
            if not isinstance(mod, _VariationalDistribution):
                yield from mod.named_parameters(prefix=prefix, recurse=False)

    def named_variational_parameters(self):
        for prefix, mod in self.named_modules():
            if isinstance(mod, _VariationalDistribution):
                yield from mod.named_parameters(prefix=prefix, recurse=False)

    def hyperparameters(self):
        for _, p in self.named_hyperparameters():
            yield p

    def variational_parameters(self):
        for _, p in self.named_variational_parameters():
            yield p


class ConstantMean(Module):
    """gpytorch.means.ConstantMean: state-dict key `constant`, shape (1,)."""

    def __init__(self):
        super().__init__()
        self.register_parameter("constant", Parameter(torch.zeros(1)))

    def forward(self, x):
        return self.constant.expand(x.shape[:-1])


class MultivariateNormal:
    """Dense (mean, covariance) pair -- what model.forward(x) returns on the prior path."""

    def __init__(self, mean, covariance_matrix):
        self.loc = mean
        self.covariance_matrix = covariance_matrix

    @property
    def mean(self):
        return self.loc

    @property
    def lazy_covariance_matrix(self):
        return self.covariance_matrix

    @property
    def variance(self):
        var = self.covariance_matrix.diagonal(dim1=-2, dim2=-1)
        return var.clamp_min(1e-10 if var.dtype == torch.float64 else 1e-6)

    @property
    def stddev(self):
        return self.variance.sqrt()

    @property
    def event_shape(self):
        return self.loc.shape[-1:]


class _LazyNormal(MultivariateNormal):
    """MultivariateNormal whose dense covariance is only built when somebody looks at it (prior / variational q(u))."""

    def __init__(self, mean, make_cov):
        self.loc = mean
        self._make_cov, self._cov = make_cov, None

    @property
    def covariance_matrix(self):
        if self._cov is None:
            self._cov = self._make_cov()
        return self._cov

    @property
    def lazy_covariance_matrix(self):
        return self.covariance_matrix


# --------------------------------------------------------------------------------------------- kernel modules
class _KDir(torch.autograd.Function):
    """K = RBFKernelDirectionalGrad(x1, x2; v1, v2, lengthscale) with the fused backward."""

    @staticmethod
    def forward(ctx, x1, x2, v1, v2, raw_ell, p1, p2):
        x1c, x2c = x1.contiguous(), x2.contiguous()
        hyp = ops.hyp_from_raw(raw_ell.reshape(-1))
        u1, inv1 = ops.normalize_dirs(v1) if p1 else (None, None)
        w2, inv2 = ops.normalize_dirs(v2) if p2 else (None, None)
        K = torch.empty(x1.shape[0] * (p1 + 1), x2.shape[0] * (p2 + 1), dtype=x1.dtype, device=x1.device)
        ops.kdir_fwd(x1c, u1, p1, x2c, w2, p2, hyp, K, use_os=False)
        ctx.save_for_backward(x1c, x2c, u1, inv1, w2, inv2, hyp)
        ctx.p = (p1, p2)
        ctx.raw_shape = raw_ell.shape
        return K

    @staticmethod
    def backward(ctx, dK):
        x1, x2, u1, inv1, w2, inv2, hyp = ctx.saved_tensors
        p1, p2 = ctx.p
        dK = dK.contiguous()
        T, dev = x1.dtype, x1.device
        need = ctx.needs_input_grad
        z = lambda *s: torch.zeros(*s, dtype=torch.float64, device=dev)
        gsc = z(2)
        gx1 = gv1 = gx2 = gv2 = None
        if need[0] or need[2] or need[4]:
            gx1, gv1 = z(*x1.shape), (z(x1.shape[0] * p1, x1.shape[1]) if p1 else None)
            ops.kdir_bwd(x1, u1, inv1, p1, x2, w2, p2, hyp, dK, gx1, gv1, gsc, use_os=False)
        if need[1] or need[3]:
            gx2, gv2 = z(*x2.shape), (z(x2.shape[0] * p2, x2.shape[1]) if p2 else None)
            ops.kdir_bwd(x2, w2, inv2, p2, x1, u1, p1, hyp, dK, gx2, gv2, None, use_os=False, dk_trans=True)
        cast = lambda g, ok: g.to(T) if (g is not None and ok) else None
        g_raw = (gsc[0] * hyp[4]).to(T).reshape(ctx.raw_shape) if need[4] else None
        return cast(gx1, need[0]), cast(gx2, need[1]), cast(gv1, need[2]), cast(gv2, need[3]), g_raw, None, None


class RBFKernelDirectionalGrad(Module):
    """Drop-in for the reference class of the same name (RBFKernelDirectionalGrad.py:8-125).

    forward(x1, x2, diag=False, v1=..., v2=...) returns the dense interleaved
    (n1(p+1), n2(p+1)) block covariance of (value, p directional derivatives); directions are point-major and
    are normalised inside the call; isotropic lengthscale of shape (1,1) under softplus."""

    def __init__(self, **kwargs):
        super().__init__()
        self.register_parameter("raw_lengthscale", Parameter(torch.zeros(1, 1)))
        self.n_dir1 = 0

    @property
    def lengthscale(self):
        return softplus(self.raw_lengthscale)

    @lengthscale.setter
    def lengthscale(self, value):
        value = torch.as_tensor(value, dtype=self.raw_lengthscale.dtype, device=self.raw_lengthscale.device)
        self.raw_lengthscale.data.copy_(_inv_softplus(value).expand(1, 1))

    def set_num_directions(self, num_directions):
        self.n_dir1 = num_directions

    def num_outputs_per_input(self, x1, x2):
        return self.n_dir1 + 1

    def forward(self, x1, x2, diag=False, **params):
        n1, n2 = x1.shape[-2], x2.shape[-2]
        v1, v2 = params["v1"], params["v2"]
        n_dir1, n_dir2 = int(v1.shape[-2] / n1), int(v2.shape[-2] / n2)
        assert n_dir1 == n_dir2, "v1 and v2 must contain same number of directions"
        self.set_num_directions(n_dir1)
        if diag:
            if not (n1 == n2 and torch.eq(x1, x2).all() and torch.eq(v1, v2).all()):
                raise RuntimeError("diag=True only works when x1 == x2 and v1 == v2")
            hyp = ops.hyp_from_raw(self.raw_lengthscale.reshape(-1))
            return ops.kdir_diag(n2, n_dir2, hyp, x1.dtype, use_os=False)
        return _KDir.apply(x1, x2, v1.to(x1.device), v2.to(x1.device), self.raw_lengthscale, n_dir1, n_dir2)

    def __call__(self, x1, x2=None, diag=False, **params):
        return self.forward(x1, x1 if x2 is None else x2, diag=diag, **params)


class RBFKernelGrad(RBFKernelDirectionalGrad):
    """gpytorch.kernels.RBFKernelGrad as used by grad_svgp.py:34: the same kernel with the d canonical
    directions at every point (RBFKernelDirectionalGrad.py:156-161 states the equivalence)."""

    def forward(self, x1, x2, diag=False, **params):
        d = x1.shape[-1]
        eye = torch.eye(d, dtype=x1.dtype, device=x1.device)
        return super().forward(x1, x2, diag=diag, v1=eye.repeat(x1.shape[-2], 1), v2=eye.repeat(x2.shape[-2], 1))

    def num_outputs_per_input(self, x1, x2):
        return x1.size(-1) + 1


class RBFKernel(RBFKernelDirectionalGrad):
    """gpytorch.kernels.RBFKernel as the plain SVGP baseline uses it (traditional_vi.py): isotropic, key `raw_lengthscale`
    (1, 1) under softplus.  forward(x1, x2) is the plain (n1, n2) RBF matrix -- the directional kernel with p = 0 on both
    sides, on the same assembly kernels; diag=True (x1 == x2) is a vector of ones."""

    def num_outputs_per_input(self, x1, x2):
        return 1

    def forward(self, x1, x2, diag=False, **params):
        if diag:
            if not (x1.shape == x2.shape and torch.equal(x1, x2)):
                raise RuntimeError("diag=True only works when x1 == x2")
            return torch.ones(x1.shape[-2], dtype=x1.dtype, device=x1.device)
        return _KDir.apply(x1, x2, None, None, self.raw_lengthscale, 0, 0)


class ScaleKernel(Module):
    """gpytorch.kernels.ScaleKernel: keys `raw_outputscale` (0-dim) and `base_kernel.*`."""

    def __init__(self, base_kernel):
        super().__init__()
        self.base_kernel = base_kernel
        self.register_parameter("raw_outputscale", Parameter(torch.tensor(0.0)))

    @property
    def outputscale(self):
        return softplus(self.raw_outputscale)

    @outputscale.setter
    def outputscale(self, value):
        value = torch.as_tensor(value, dtype=self.raw_outputscale.dtype, device=self.raw_outputscale.device)
        self.raw_outputscale.data.copy_(_inv_softplus(value).reshape(()))

    def num_outputs_per_input(self, x1, x2):
        return self.base_kernel.num_outputs_per_input(x1, x2)

    def forward(self, x1, x2, diag=False, **params):
        return self.base_kernel.forward(x1, x2, diag=diag, **params) * self.outputscale

    def __call__(self, x1, x2=None, diag=False, **params):
        return self.forward(x1, x1 if x2 is None else x2, diag=diag, **params)


# ------------------------------------------------------------------------------------- variational distribution
class _VariationalDistribution(Module):
    pass


class CholeskyVariationalDistribution(_VariationalDistribution):
    """gpytorch.variational.CholeskyVariationalDistribution: keys `variational_mean` (M') and
    `chol_variational_covar` (M', M'); q(u) = N(m, L L^T) with L = tril(param) (no positivity transform)."""

    def __init__(self, num_inducing_points, batch_shape=torch.Size([]), mean_init_std=1e-3, **kwargs):
        super().__init__()
        self.num_inducing_points = num_inducing_points
        self.mean_init_std = mean_init_std
        self.register_parameter("variational_mean", Parameter(torch.zeros(num_inducing_points)))
        self.register_parameter("chol_variational_covar", Parameter(torch.eye(num_inducing_points)))

    def shape(self):
        return torch.Size([self.num_inducing_points])

    def initialize_from_prior(self):
        """First-call initialisation against the whitened prior N(0, I): m <- 1e-3 * randn, L <- I."""
        with torch.no_grad():
            self.variational_mean.zero_().add_(torch.randn_like(self.variational_mean), alpha=self.mean_init_std)
            self.chol_variational_covar.copy_(torch.eye(self.num_inducing_points, dtype=self.chol_variational_covar.dtype,
                                                        device=self.chol_variational_covar.device))

    def mean_and_chol(self):
        return self.variational_mean, self.chol_variational_covar


class _NaturalToMeanChol(torch.autograd.Function):
    """gpytorch 1.4.0 `_NaturalToMuVarSqrt`: (natural_vec, natural_mat) = (S^-1 m, -1/2 S^-1) -> (m, chol(S)), with the
    backward returning the gradient w.r.t. the EXPECTATION parameters, i.e. the natural gradient `gpytorch.optim.NGD`
    applies (directional_vi.py:38-40,187,251).  Everything is M'^3 work on the library's own fp64 kernels: two blocked
    Cholesky + inverse, three triangular products forward; the Cholesky-backward chain W^T Phi(L^T dL) W backward."""

    @staticmethod
    def _chol_inv(A64, n, what):
        """(L, L^-1) of the n x n SPD matrix A64 (fp64, on the device) with the psd_safe_cholesky jitter ladder"""
        dev = A64.device
        Mp, nb0, nlev = ops.chol_plan(n)
        work, L, W = (torch.empty(Mp, Mp, dtype=torch.float64, device=dev) for _ in range(3))
        info = torch.zeros(1, dtype=torch.int32, device=dev)
        for extra in (0.0, 1e-8, 1e-6, 1e-5, 1e-4):
            if Mp > n:
                ops.pad_identity(work, n)
            work[:n, :n] = A64
            if extra:
                work.diagonal()[:n].add_(extra)
            ops.cholesky_inverse(work, L, W, nb0, nlev, info)
            if int(info.item()) == 0:
                return L, W
        if not bool(torch.isfinite(A64).all()):
            raise NanError(f"NaN/inf in {what}")
        raise NotPSDError(f"{what} is not positive definite after adding jitter up to 1e-4")

    @staticmethod
    def forward(ctx, nat_vec, nat_mat):
        T, n = nat_vec.dtype, nat_vec.numel()
        F64 = torch.float64
        _, Lm = _NaturalToMeanChol._chol_inv(-2.0 * nat_mat.detach().to(F64), n, "-2 * natural_mat")     # Lm = chol(S^-1)^-1
        S = torch.empty(n, n, dtype=F64, device=nat_vec.device)
        ops.gemm(Lm, Lm, S, ta=True, a_tri=ops.TRI_UPPER, b_tri=ops.TRI_LOWER, M=n, N=n, K=n)              # S = Lm^T Lm
        mu = torch.empty(n, 1, dtype=F64, device=nat_vec.device)
        ops.gemm(S, nat_vec.detach().to(F64).reshape(n, 1).contiguous(), mu, M=n, N=1, K=n)                 # m = S theta1
        Ls, Ws = _NaturalToMeanChol._chol_inv(S, n, "the variational covariance")
        ctx.save_for_backward(mu, Ls, Ws)
        ctx.n, ctx.T = n, T
        return mu.reshape(n).to(T), Ls[:n, :n].tril().to(T)

    @staticmethod
    def backward(ctx, dmu, dLs):
        mu, Ls, Ws = ctx.saved_tensors
        n, T, F64 = ctx.n, ctx.T, torch.float64
        dev = mu.device
        e = lambda: torch.empty(n, n, dtype=F64, device=dev)
        dL64 = dLs.to(F64).contiguous()
        Y, Phi, T1, G = e(), e(), e(), e()
        ops.gemm(Ls, dL64, Y, ta=True, a_tri=ops.TRI_UPPER, b_tri=ops.TRI_LOWER, c_tri=1, M=n, N=n, K=n)   # tril(L^T dL)
        ops.phi_lower(Y, Phi, n)
        ops.gemm(Phi, Ws, T1, a_tri=ops.TRI_LOWER, b_tri=ops.TRI_LOWER, c_tri=1, M=n, N=n, K=n)             # Phi W (lower)
        ops.gemm(Ws, T1, G, ta=True, a_tri=ops.TRI_UPPER, b_tri=ops.TRI_LOWER, M=n, N=n, K=n)               # W^T Phi W
        ops.symmetrize(G, n)                                                                                # dS
        d1 = torch.empty(n, 1, dtype=F64, device=dev)
        ops.gemm(G, mu, d1, alpha=-2.0, beta=1.0, D=dmu.to(F64).reshape(n, 1).contiguous(), M=n, N=1, K=n)  # dmu - 2 dS m
        return d1.reshape(n).to(T), G.to(T)


class NaturalVariationalDistribution(_VariationalDistribution):
    """gpytorch.variational.NaturalVariationalDistribution: keys `natural_vec` (M') and `natural_mat` (M', M');
    q(u) = N(m, S) with natural_vec = S^-1 m, natural_mat = -1/2 S^-1; trained with `NGD` (use_ngd=True)."""

    def __init__(self, num_inducing_points, batch_shape=torch.Size([]), mean_init_std=1e-3, **kwargs):
        super().__init__()
        self.num_inducing_points = num_inducing_points
        self.mean_init_std = mean_init_std
        self.register_parameter("natural_vec", Parameter(torch.zeros(num_inducing_points)))
        self.register_parameter("natural_mat", Parameter(torch.eye(num_inducing_points).mul(-0.5)))

    def shape(self):
        return torch.Size([self.num_inducing_points])

    def initialize_from_prior(self):
        """Against the whitened prior N(0, I): natural_vec <- 1e-3 * randn, natural_mat <- -1/2 I."""
        with torch.no_grad():
            self.natural_vec.zero_().add_(torch.randn_like(self.natural_vec), alpha=self.mean_init_std)
            self.natural_mat.copy_(-0.5 * torch.eye(self.num_inducing_points, dtype=self.natural_mat.dtype,
                                                    device=self.natural_mat.device))

    def mean_and_chol(self):
        """(m, chol(S)) as differentiable functions of the natural parameters.  Without autograd (eval loops) the
        M'^3 conversion is memoised on the parameters' identity and in-place version."""
        if torch.is_grad_enabled() and (self.natural_vec.requires_grad or self.natural_mat.requires_grad):
            return _NaturalToMeanChol.apply(self.natural_vec, self.natural_mat)
        key = (self.natural_vec.data_ptr(), self.natural_vec._version, self.natural_mat.data_ptr(), self.natural_mat._version)
        if getattr(self, "_memo", None) is None or self._memo[0] != key:
            with torch.no_grad():
                self._memo = (key, _NaturalToMeanChol.apply(self.natural_vec, self.natural_mat))
        return self._memo[1]


class NGD(torch.optim.Optimizer):
    """gpytorch.optim.NGD: p <- p - lr * num_data * p.grad on the natural parameters (whose .grad is already the natural
    gradient of the per-datum objective, see _NaturalToMeanChol)."""

    def __init__(self, params, num_data, lr=0.1):
        self.num_data = num_data
        super().__init__(params, defaults=dict(lr=lr))

    @torch.no_grad()
    def step(self, closure=None):
        for group in self.param_groups:
            for p in group["params"]:
                if p.grad is not None:
                    p.add_(p.grad, alpha=-group["lr"] * self.num_data)
        return None


# ------------------------------------------------------------------------------------------------- likelihood
class _HomoskedasticNoise(Module):
    def __init__(self):
        super().__init__()
        self.register_parameter("raw_noise", Parameter(torch.zeros(1)))

    @property
    def noise(self):
        return softplus(self.raw_noise) + 1e-4          # GreaterThan(1e-4)


class GaussianLikelihood(Module):
    """gpytorch.likelihoods.GaussianLikelihood: key `noise_covar.raw_noise`; likelihood(dist) adds the noise."""

    def __init__(self):
        super().__init__()
        self.noise_covar = _HomoskedasticNoise()

    @property
    def noise(self):
        return self.noise_covar.noise

    @property
    def raw_noise(self):
        return self.noise_covar.raw_noise

    def __call__(self, dist, *args, **kwargs):
        if isinstance(dist, PredictiveDistribution):
            return dist._with_likelihood(self)
        if isinstance(dist, MultivariateNormal):
            n = dist.mean.shape[-1]
            eye = torch.eye(n, dtype=dist.mean.dtype, device=dist.mean.device)
            return MultivariateNormal(dist.mean, dist.covariance_matrix + self.noise * eye)
        raise TypeError("GaussianLikelihood expects the distribution returned by the model")


# ------------------------------------------------------------------------------------- autograd entry points
_PARAM_ORDER = ("Z", "Vz", "m", "Ls_raw", "c", "raw_os", "raw_ell", "raw_noise")


_INPUT_ORDER = ("x", "Vx", "y")


def _inputs_wanted(needs):
    """names of the inputs (x, Vx[, y]) whose entries of ctx.needs_input_grad are set, from position 1 on"""
    return tuple(name for name, need in zip(_INPUT_ORDER, needs[1:]) if need)


def _scaled_input_grads(grads, names, shapes, g_out):
    """the input gradients of a backward pass scaled by the incoming gradient, shaped like the inputs (None where not wanted)"""
    return [grads[name].reshape(shp) * g_out.to(grads[name].dtype) if name in names else None
            for name, shp in zip(_INPUT_ORDER, shapes)]


class _ElboStep(torch.autograd.Function):
    """value = ELBO; the gradients w.r.t. every parameter -- and w.r.t. x, Vx, y when they require it -- are computed by the
    same fused GPU pass and handed to autograd in backward (scaled by the incoming gradient)."""

    @staticmethod
    def forward(ctx, cfg, x, Vx, y, *params):
        P = types.SimpleNamespace(**dict(zip(_PARAM_ORDER, params)))
        want = any(ctx.needs_input_grad[4:])      # (grad mode is off inside forward; this is the reliable signal)
        inputs = _inputs_wanted(ctx.needs_input_grad[:4])
        elbo, grads, mean, var = ENGINE.elbo_step(P, x, Vx, y, cfg["num_data"], cfg["p"], cfg["p2"],
                                                  cfg["through_likelihood"], cfg.get("n_global"), want_grads=want,
                                                  objective=cfg.get("objective", "elbo"), include_kl=cfg.get("include_kl", True),
                                                  reducer=cfg.get("reducer"), input_grads=inputs)
        ctx.grads, ctx.inputs = grads, inputs
        ctx.input_shapes = tuple(None if t is None else t.shape for t in (x, Vx, y))
        ctx.mark_non_differentiable(mean, var)
        return elbo.to(x.dtype), mean, var

    @staticmethod
    def backward(ctx, g_elbo, _gm, _gv):
        grads = ctx.grads
        if grads is None:
            raise RuntimeError("the ELBO was evaluated without gradients (torch.no_grad / no parameter requires grad)")
        wanted = [(k, grads[name]) for k, (name, need) in enumerate(zip(_PARAM_ORDER, ctx.needs_input_grad[4:]))
                  if need and grads.get(name) is not None]
        out = [None] * len(_PARAM_ORDER)
        if wanted:          # one fused multi-tensor launch per dtype instead of one multiply per parameter
            scaled = torch._foreach_mul([g for _, g in wanted], g_elbo.to(wanted[0][1].dtype))
            for (k, _), g in zip(wanted, scaled):
                out[k] = g
        ins = _scaled_input_grads(grads, ctx.inputs, ctx.input_shapes, g_elbo) if ctx.inputs else [None] * 3
        return (None, *ins, *out)


class _Predictive(torch.autograd.Function):
    """(mean, variance) of q(f) [+ noise] as differentiable tensors -- the generic path behind
    PredictiveDistribution.mean / .variance when they are used outside VariationalELBO."""

    @staticmethod
    def forward(ctx, cfg, x, Vx, *params):
        P = types.SimpleNamespace(**dict(zip(_PARAM_ORDER, params)))
        ectx, mean, var = ENGINE.predictive_forward(P, x, Vx, cfg["p"], cfg["p2"], cfg["add_noise"])
        ctx.ectx, ctx.P, ctx.x, ctx.Vx, ctx.cfg = ectx, P, x, Vx, cfg
        ctx.generation = (ectx[0].generation, ectx[1].generation)     # bumped by EVERY later user of the workspace / factor
        return mean, var

    @staticmethod
    def backward(ctx, gmu, gvar):
        if (ctx.ectx[0].generation, ctx.ectx[1].generation) != ctx.generation:
            raise RuntimeError("dsvgp_b200: the predictive workspace was overwritten by a later forward pass before "
                               "backward ran; call backward before evaluating the model again on the same shape")
        inputs = _inputs_wanted(ctx.needs_input_grad[:3])
        grads = ENGINE.predictive_backward(ctx.ectx, ctx.P, ctx.x, gmu, gvar, ctx.cfg["add_noise"], Vx=ctx.Vx,
                                           input_grads=inputs)
        out = []
        for name, need in zip(_PARAM_ORDER, ctx.needs_input_grad[3:]):
            g = grads.get(name)
            out.append(g if (need and g is not None) else None)
        ins = [grads[name] if name in inputs else None for name in _INPUT_ORDER[:2]]
        return (None, *ins, *out)


class _FullPredictive(torch.autograd.Function):
    """(mean, dense covariance) of q(f(X)) [+ noise] as differentiable tensors: what gpytorch's lazy predictive covariance gives the
    reference (DirectionalGradVariationalStrategy.py:192-208).  Used by PredictiveDistribution.covariance_matrix / .rsample when
    gradients are enabled and a parameter requires them."""

    @staticmethod
    def forward(ctx, cfg, x, Vx, *params):
        P = types.SimpleNamespace(**dict(zip(_PARAM_ORDER, params)))
        ectx, mean, cov = ENGINE.full_forward(P, x, Vx, cfg["p"], cfg["p2"], cfg["add_noise"])
        ctx.ectx, ctx.P, ctx.x, ctx.Vx, ctx.cfg = ectx, P, x, Vx, cfg
        ctx.generation = (ectx[0].generation, ectx[1].generation)
        return mean, cov

    @staticmethod
    def backward(ctx, gmean, gcov):
        if (ctx.ectx[0].generation, ctx.ectx[1].generation) != ctx.generation:
            raise RuntimeError("dsvgp_b200: the predictive workspace was overwritten by a later forward pass before "
                               "backward ran; call backward before evaluating the model again on the same shape")
        inputs = _inputs_wanted(ctx.needs_input_grad[:3])
        grads = ENGINE.full_backward(ctx.ectx, ctx.P, ctx.x, gmean, gcov, ctx.cfg["add_noise"], Vx=ctx.Vx, input_grads=inputs)
        out = []
        for name, need in zip(_PARAM_ORDER, ctx.needs_input_grad[3:]):
            g = grads.get(name)
            out.append(g if (need and g is not None) else None)
        ins = [grads[name] if name in inputs else None for name in _INPUT_ORDER[:2]]
        return (None, *ins, *out)


class PredictiveDistribution:
    """Lazy q(f(X)) returned by a variational strategy (stands in for gpytorch's MultivariateNormal with a lazy
    covariance).  Only what the reference's callers consume is offered: .mean / .loc, .variance, .stddev
    (directional_vi.py:256-257, :297-298), plus the full predictive covariance (.covariance_matrix, differentiable) and
    .sample / .rsample (SURVEY.md section 8f rank 4; the draw itself is not reparameterised)."""

    def __init__(self, strategy, x, Vx, likelihood=None, noise_mult=0):
        self._strategy, self._x, self._Vx, self._likelihood = strategy, x, Vx, likelihood
        self._noise_mult = noise_mult       # how many times likelihood() has been applied: each adds sigma^2 I (Q3)
        self._cache = None
        self._full = None

    def _with_likelihood(self, likelihood):
        return PredictiveDistribution(self._strategy, self._x, self._Vx, likelihood, self._noise_mult + 1)

    @property
    def event_shape(self):
        return torch.Size([self._x.shape[0] * (self._strategy._p2() + 1)])

    def _params(self):
        return self._strategy._param_list(self._likelihood)

    def _differentiable(self, params):
        """autograd path: gradients are enabled and a parameter or an input (x, derivative_directions) requires them"""
        return torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in (self._x, self._Vx, *params))

    def _evaluate(self):
        if self._cache is None:
            st = self._strategy
            cfg = dict(p=st._p(), p2=st._p2(), add_noise=self._noise_mult)
            params = self._params()
            if self._differentiable(params):
                self._cache = _Predictive.apply(cfg, self._x, self._Vx, *params)
            else:
                P = types.SimpleNamespace(**dict(zip(_PARAM_ORDER, params)))
                self._cache = ENGINE.predict(P, self._x, self._Vx, cfg["p"], cfg["p2"], cfg["add_noise"],
                                             reuse_factor=not st.training)
        return self._cache

    @property
    def mean(self):
        if self._cache is None and self._full is not None:      # the dense evaluation already has it (and owns the workspace:
            return self._full[0]                                 #  a second, diagonal pass would invalidate its pending backward)
        return self._evaluate()[0]

    loc = mean

    @property
    def variance(self):
        if self._cache is None and self._full is not None:
            min_var = 1e-10 if self._full[1].dtype == torch.float64 else 1e-6      # gpytorch settings.min_variance
            return self._full[1].diagonal().clamp_min(min_var)
        return self._evaluate()[1]

    @property
    def stddev(self):
        return self.variance.sqrt()

    def _evaluate_full(self):
        """(mean, dense covariance): differentiable w.r.t. the parameters when gradients are enabled (the reference's lazy
        covariance is, DGVS.py:192-208); the BO callers sample under eval / no_grad and take the plain evaluation."""
        if self._full is None:
            st = self._strategy
            params = self._params()
            if self._differentiable(params):
                cfg = dict(p=st._p(), p2=st._p2(), add_noise=self._noise_mult)
                self._full = _FullPredictive.apply(cfg, self._x, self._Vx, *params)
            else:
                P = types.SimpleNamespace(**dict(zip(_PARAM_ORDER, (t.detach() if t is not None else None for t in params))))
                with torch.no_grad():
                    self._full = ENGINE.predict_full(P, self._x, self._Vx, st._p(), st._p2(), self._noise_mult,
                                                     reuse_factor=not st.training)
        return self._full

    @property
    def covariance_matrix(self):
        """Dense n' x n' predictive covariance K_xx + 1e-4 I + A^T (S - I) A (+ noise), DGVS.py:192-205."""
        return self._evaluate_full()[1]

    lazy_covariance_matrix = covariance_matrix

    def rsample(self, sample_shape=torch.Size(), base_samples=None):
        mean, cov = (t.detach() for t in self._evaluate_full())      # (the draw is not reparameterised: no gradient through it)
        shape = torch.Size(sample_shape)
        num = int(math.prod(shape)) if len(shape) else 1
        out = ENGINE.sample_mvn(mean, cov, num)
        return out.reshape(*shape, mean.shape[0])

    def sample(self, sample_shape=torch.Size(), base_samples=None):
        """preds.sample(torch.Size([n_samples])) -> (n_samples, n') as gpytorch's MultivariateNormal.sample
        (experiments/rover/test_turbo.py:138)."""
        with torch.no_grad():
            return self.rsample(sample_shape)


# ------------------------------------------------------------------------------------------------ objectives
def _target_like(target, x):
    """The labels in the model's dtype (torch would promote `y - mean` silently in the reference; the kernels read raw
    memory, so the cast is explicit).  A device mismatch is an error, as it is in the reference."""
    if target.device != x.device:
        raise RuntimeError(f"the target is on {target.device}, the model output on {x.device}")
    return target.to(x.dtype).contiguous()


class VariationalELBO(Module):
    """gpytorch.mlls.VariationalELBO(likelihood, model, num_data): (dist, target) -> scalar
    (1/n') sum_j E_q[log p(y_j | f_j)] - KL(q(u) || p(u)) / num_data."""

    def __init__(self, likelihood, model, num_data, beta=1.0, combine_terms=True):
        super().__init__()
        self.likelihood, self.model, self.num_data, self.beta = likelihood, model, num_data, beta
        if not combine_terms:
            raise NotImplementedError("combine_terms=False is not used on the hot path")

    def forward(self, dist, target, **kwargs):
        if not isinstance(dist, PredictiveDistribution):
            raise TypeError("VariationalELBO expects the distribution returned by model(x, ...) or likelihood(model(x, ...))")
        st = dist._strategy
        cfg = dict(p=st._p(), p2=st._p2(), num_data=float(self.num_data) / float(self.beta),
                   through_likelihood=dist._noise_mult, n_global=st._n_global, include_kl=not st._external_kl,
                   reducer=st._reducer)
        params = st._param_list(self.likelihood)
        elbo, mean, var = _ElboStep.apply(cfg, dist._x, dist._Vx, _target_like(target, dist._x), *params)
        dist._cache = (mean, var)      # train loops print output.mean / output.variance (directional_vi.py:256-257)
        if st._external_kl:            # q(u) is not over the M(p+1) inducing values the step saw: KL by autograd, M'^2 work
            elbo = elbo - st.kl_divergence().to(elbo.dtype) / cfg["num_data"]
        return elbo


class PredictiveLogLikelihood(Module):
    """gpytorch.mlls.PredictiveLogLikelihood (mll_type="PLL", directional_vi.py:218-219; SURVEY.md 8f rank 1):
    (1/n') sum_j log N(y_j; mu_j, v_j) - KL/num_data, where v is the variance of likelihood(dist) -- log_marginal
    applies the likelihood itself, so in the reference loop (which already passes likelihood(model(x)), :245) the
    noise is counted twice (quirk Q3).  Runs as ONE fused forward+backward pass like VariationalELBO."""

    def __init__(self, likelihood, model, num_data, beta=1.0):
        super().__init__()
        self.likelihood, self.model, self.num_data, self.beta = likelihood, model, num_data, beta

    def forward(self, dist, target, **kwargs):
        if not isinstance(dist, PredictiveDistribution):
            raise TypeError("PredictiveLogLikelihood expects the distribution returned by model(x, ...) or likelihood(model(x, ...))")
        st = dist._strategy
        cfg = dict(p=st._p(), p2=st._p2(), num_data=float(self.num_data) / float(self.beta), objective="pll",
                   through_likelihood=dist._noise_mult + 1, n_global=st._n_global, include_kl=not st._external_kl,
                   reducer=st._reducer)
        params = st._param_list(self.likelihood)
        val, mean, var = _ElboStep.apply(cfg, dist._x, dist._Vx, _target_like(target, dist._x), *params)
        if st._external_kl:
            val = val - st.kl_divergence().to(val.dtype) / cfg["num_data"]
        # the step's variance carries log_marginal's extra noise; `dist` itself (what the loop prints, :256-257) does not
        dist._cache = (mean, (var - self.likelihood.noise.detach().to(var.dtype)).clamp_min(
            1e-10 if var.dtype == torch.float64 else 1e-6))
        return val


# ---------------------------------------------------------------------------------------------------- models
class ApproximateGP(Module):
    """gpytorch.models.ApproximateGP: model(x, **kwargs) -> variational_strategy(x, **kwargs)."""

    def __init__(self, variational_strategy):
        super().__init__()
        self.variational_strategy = variational_strategy

    def forward(self, x, **kwargs):
        raise NotImplementedError

    def __call__(self, inputs, prior=False, **kwargs):
        if inputs.dim() == 1:
            inputs = inputs.unsqueeze(-1)
        return self.variational_strategy(inputs, prior=prior, **kwargs)


def _ensure_updated_strategy_flag_set(module, state_dict, prefix, *args):
    """load_state_dict pre-hook of the reference strategies (DGVS.py:17-29): checkpoints from before the whitened
    parameterisation lack `updated_strategy`; they get False, which triggers the one-off re-whitening."""
    module._flags_checked = False
    if prefix + "updated_strategy" not in state_dict:
        device = state_dict[list(state_dict.keys())[0]].device
        state_dict[prefix + "updated_strategy"] = torch.tensor(False, device=device)
        warnings.warn("You have loaded a variational GP model from a version that used un-whitened parameters; "
                      "they are converted on the first call. Re-save the model.", OldVersionWarning)


class _DirectionalStrategyBase(Module):
    """Shared machinery of the three strategies (gpytorch _VariationalStrategy + DGVS.py:65-69)."""

    def __init__(self, model, inducing_points, variational_distribution, learn_inducing_locations=True):
        super().__init__()
        object.__setattr__(self, "model", model)
        inducing_points = inducing_points.clone()
        if inducing_points.dim() == 1:
            inducing_points = inducing_points.unsqueeze(-1)
        if learn_inducing_locations:
            self.register_parameter("inducing_points", Parameter(inducing_points))
        else:
            self.register_buffer("inducing_points", inducing_points)
        self._variational_distribution = variational_distribution
        self.register_buffer("variational_params_initialized", torch.tensor(0))
        self.register_buffer("updated_strategy", torch.tensor(True))
        self._register_load_state_dict_pre_hook(_ensure_updated_strategy_flag_set, with_module=True)
        self._n_global = None          # set by distributed.enable(): global minibatch size of a sharded step ...
        self._reducer = None           # ... and the object that sums its payload over ranks (per model, not per process)
        self._flags_checked = False    # host-side memo of the two flag buffers (reset by load_state_dict)
        self._external_kl = False      # True: the fused step leaves the KL term to autograd (shared-direction strategy)

    @property
    def variational_distribution(self):
        """q(u) = N(m, L_s L_s^T) (gpytorch _VariationalStrategy.variational_distribution, used by DGVS.py:222)."""
        m, Ls = self._variational_distribution.mean_and_chol()
        return _LazyNormal(m, lambda: Ls.tril() @ Ls.tril().transpose(-1, -2))

    @property
    def prior_distribution(self):
        """p(u) = N(0, I) of the whitened parameterisation (DGVS.py:77-87)."""
        vd = self._variational_distribution
        ref = next(vd.parameters())
        zeros = torch.zeros(vd.shape(), dtype=ref.dtype, device=ref.device)
        return _LazyNormal(zeros, lambda: torch.eye(zeros.numel(), dtype=ref.dtype, device=ref.device))

    # ---- shape helpers
    def _p(self):
        raise NotImplementedError

    def _p2(self):
        return self._p()

    def _directions(self):
        raise NotImplementedError

    def _param_list(self, likelihood):
        vd, model = self._variational_distribution, self.model
        raw_noise = likelihood.noise_covar.raw_noise if likelihood is not None else None
        m, Ls = vd.mean_and_chol()      # the parameters themselves, or (natural parameterisation) differentiable functions of them
        return (self.inducing_points, self._directions(), m, Ls,
                model.mean_module.constant, model.covar_module.raw_outputscale,
                model.covar_module.base_kernel.raw_lengthscale, raw_noise)

    def train(self, mode=True):
        ENGINE.invalidate()                 # eval-mode memoisation of the Cholesky factor ends here (DGVS.py:72)
        return super().train(mode)

    def kl_divergence(self):
        """KL(q(u) || N(0, I)) of the whitened parameterisation (differentiable, small: plain torch on device)."""
        m, Ls = self._variational_distribution.mean_and_chol()
        Ls = Ls.tril()
        return 0.5 * ((Ls * Ls).sum() + (m * m).sum() - m.numel() - Ls.diagonal().pow(2).log().sum())

    def _data_directions(self, x, kwargs):
        raise NotImplementedError

    def forward(self, x, inducing_points, inducing_values, variational_inducing_covar=None, **kwargs):
        """Same signature as the reference forward (DGVS.py:89).  The fused step reads the inducing points / values from
        the module's own parameters, so anything else in those arguments is refused rather than silently ignored."""
        Vx = self._data_directions(x, kwargs)
        own_m = getattr(self._variational_distribution, "variational_mean", None)
        if (inducing_points is not None and inducing_points is not self.inducing_points) or \
                variational_inducing_covar is not None or (inducing_values is not None and inducing_values is not own_m):
            raise NotImplementedError("dsvgp_b200 strategies evaluate q(f) with the module's own inducing points and variational "
                                      "parameters; foreign inducing_points / inducing_values / variational_inducing_covar "
                                      "arguments are not supported -- load them into the module instead")
        return PredictiveDistribution(self, x.contiguous(), Vx)

    def _rewhiten_legacy_parameters(self):
        """One-off conversion of un-whitened variational parameters (reference __call__, DGVS.py:211-238):
        m <- L^-1 (m - c),  L_s <- L^-1 L_s  with L = chol(K_zz + 1e-3 I)."""
        vd = self._variational_distribution
        params = self._param_list(None)
        P = types.SimpleNamespace(**dict(zip(_PARAM_ORDER, params)))
        T, dev = P.Z.dtype, P.Z.device
        f = ENGINE.factor(dev, T, P.Z.shape[1], P.Z.shape[0], self._p())
        ENGINE._factorise(f, P, T, 0.0)
        if not ENGINE._check(f, P):
            raise NotPSDError("K_zz is not positive definite")
        with torch.no_grad():
            Mq = f.Mq
            rhs = torch.empty(Mq, Mq + 8, dtype=T, device=dev)
            rhs[:, :Mq] = vd.chol_variational_covar.tril()
            rhs[:, Mq] = vd.variational_mean - self.model.mean_module.constant
            out = torch.empty_like(rhs)
            ops.gemm(ENGINE._wt(f), rhs, out, a_tri=ops.TRI_LOWER, M=Mq, N=Mq + 1, K=Mq)
            root = out[:, :Mq].tril()
            sign = torch.where(root.diagonal() < 0, -1.0, 1.0).to(T)
            vd.chol_variational_covar.copy_(root * sign)
            vd.variational_mean.copy_(out[:, Mq])
        ENGINE.invalidate()
        self.updated_strategy.fill_(True)

    def __call__(self, x, prior=False, **kwargs):
        if prior:
            return self.model.forward(x, **kwargs)
        if not self._flags_checked:
            # the two flag buffers are read from the device ONCE (and again after load_state_dict), not on every
            # call as in the reference (DGVS.py:211,:229): each .item() is a host synchronisation per minibatch
            if not self.updated_strategy.item():
                self._rewhiten_legacy_parameters()
            if not self.variational_params_initialized.item():
                self._variational_distribution.initialize_from_prior()
                self.variational_params_initialized.fill_(1)
            self._flags_checked = True
        vd = self._variational_distribution
        return self.forward(x, self.inducing_points, getattr(vd, "variational_mean", None), None, **kwargs)


class DirectionalGradVariationalStrategy(_DirectionalStrategyBase):
    """Drop-in for directionalvi/DirectionalGradVariationalStrategy.py:32-240: whitened SVGP over function values
    and p learned directional derivatives per inducing point.  `kwargs['derivative_directions']` (n*p, d) gives the
    data-side directions."""

    def __init__(self, model, inducing_points, inducing_directions, variational_distribution,
                 learn_inducing_locations=True):
        super().__init__(model, inducing_points, variational_distribution, learn_inducing_locations)
        self.register_parameter(name="inducing_directions", param=Parameter(inducing_directions.clone()))

    def _p(self):
        return int(self.inducing_directions.size(-2) / self.inducing_points.size(-2))

    def _directions(self):
        return self.inducing_directions

    def _data_directions(self, x, kwargs):
        derivative_directions = kwargs["derivative_directions"]
        num_derivative_directions = int(derivative_directions.size(-2) / x.size(-2))
        assert num_derivative_directions == self._p(), "Need minibatch dim to be same as number of directions for kernel"
        self.model.covar_module.base_kernel.set_num_directions(self._p())
        return derivative_directions.to(device=x.device, dtype=x.dtype).contiguous()


class SharedDirectionalGradVariationalStrategy(DirectionalGradVariationalStrategy):
    """Drop-in for directionalvi/SharedDirectionalGradVariationalStrategy.py:32-259 (exported there under the name
    DirectionalGradVariationalStrategy, shared_directional_vi.py:13): ONE set of p inducing directions shared by all
    inducing points (`inducing_directions` is (p, d), repeated per point :95-98), a variational distribution over
    M + p values -- M function values and p shared directional-derivative values, expanded to the M(p+1) inducing values
    [m_i, g_1..g_p] (:99-105) -- and, as shipped, a middle term overwritten with zeros (:209-211): the predictive
    covariance is the prior's K_xx + 1e-4 I, so L_s only enters the objective through the KL term.

    Runs on the same fused step: the expansion of (V, m) is differentiable torch glue (M' numbers), the step is given
    L_s = I (so (S - I) A vanishes identically, which IS the zeroed middle term) and leaves the KL of the (M + p)-variate
    q(u) to autograd."""

    def __init__(self, model, inducing_points, inducing_directions, variational_distribution,
                 learn_inducing_locations=True):
        super().__init__(model, inducing_points, inducing_directions, variational_distribution, learn_inducing_locations)
        self._external_kl = True
        self._eye = None

    def _p(self):
        return int(self.inducing_directions.size(-2))

    def _param_list(self, likelihood):
        vd, model = self._variational_distribution, self.model
        raw_noise = likelihood.noise_covar.raw_noise if likelihood is not None else None
        m, _ = vd.mean_and_chol()
        Z, V = self.inducing_points, self.inducing_directions
        M, p = Z.shape[0], V.shape[0]
        if m.numel() != M + p:
            raise ValueError(f"the shared-direction strategy needs a variational distribution over M + p = {M + p} values, "
                             f"got {m.numel()}")
        m_full = torch.cat([m[:M, None], m[M:].expand(M, p)], 1).reshape(-1)                  # :99-105
        Mq = M * (p + 1)
        if self._eye is None or self._eye.shape[0] != Mq or self._eye.device != Z.device or self._eye.dtype != Z.dtype:
            self._eye = torch.eye(Mq, dtype=Z.dtype, device=Z.device)
        return (Z, V.repeat(M, 1), m_full, self._eye, model.mean_module.constant, model.covar_module.raw_outputscale,
                model.covar_module.base_kernel.raw_lengthscale, raw_noise)

    def _rewhiten_legacy_parameters(self):
        raise NotImplementedError("un-whitened legacy checkpoints are not supported by the shared-direction strategy")


class DFreeDirectionalGradVariationalStrategy(DirectionalGradVariationalStrategy):
    """Drop-in for directionalvi/DFreeDirectionalGradVariationalStrategy.py:32-227: same inducing structure, but the
    data carry no derivative labels -- only the function-value rows/columns of the data side are kept
    (:112,:118,:123,:136), so outputs have length n and the data-side directions influence nothing."""

    def _p2(self):
        return 0


class GradVariationalStrategy(_DirectionalStrategyBase):
    """Drop-in for directionalvi/GradVariationalStrategy.py:32-169: full-gradient inducing variables, i.e. the
    directional strategy with the d canonical directions at every inducing and data point (gpytorch RBFKernelGrad)."""

    def __init__(self, model, inducing_points, variational_distribution, learn_inducing_locations=True):
        super().__init__(model, inducing_points, variational_distribution, learn_inducing_locations)
        self._canon = None

    def _p(self):
        return self.inducing_points.size(-1)

    def _canonical(self, n, like):
        d = like.shape[-1]
        return torch.eye(d, dtype=like.dtype, device=like.device).repeat(n, 1)

    def _directions(self):
        Z = self.inducing_points
        if self._canon is None or self._canon.shape[0] != Z.shape[0] * Z.shape[1] or self._canon.device != Z.device \
                or self._canon.dtype != Z.dtype:
            self._canon = self._canonical(Z.shape[0], Z)
        return self._canon

    def _data_directions(self, x, kwargs):
        return self._canonical(x.shape[0], x)


class VariationalStrategy(_DirectionalStrategyBase):
    """gpytorch.variational.VariationalStrategy as the plain SVGP baseline uses it (traditional_vi.py): whitened, over the
    M function values at the inducing points, labels are function values only.  This is the directional strategy with p = 0
    on both sides, on the same fused step; the gpytorch 1.4 constants are the same as there (K_zz jitter 1e-3, predictive
    jitter 1e-4, the 1e-6 / 1e-5 / 1e-4 Cholesky ladder, the 1e-6 / 1e-10 variance floor)."""

    def _p(self):
        return 0

    def _directions(self):
        return None

    def _data_directions(self, x, kwargs):
        if kwargs.get("derivative_directions") is not None:
            raise TypeError("VariationalStrategy models function values only: it takes no derivative_directions "
                            "(use DirectionalGradVariationalStrategy for derivative information)")
        return None
