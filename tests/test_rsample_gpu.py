"""Reparameterised draws of the predictive distribution: `rsample` = mean + L z with L the fp64 Cholesky factor of the
covariance, differentiable w.r.t. everything the mean and covariance depend on and w.r.t. `base_samples`, as gpytorch's
MultivariateNormal.rsample is.

  * the Cholesky backward dsvgp_chol_bwd_f64 against CPU fp64 autograd of torch.linalg.cholesky (NaN upper triangles, NaN
    sentinels in the output and workspace padding, every refusal);
  * the draws with given base samples against mean + L z of the oracle covariance, sample == rsample, shapes, seeded draws;
  * gradients of every parameter, x, Vx and base_samples against fp64 autograd of oracle -> cholesky -> mean + L z, for every
    strategy in train and eval mode, with and without the likelihood; an MC-acquisition-shaped loss; a full-size fp64
    finite difference; the jitter ladder, accumulation and the workspace guard."""
import ctypes

import pytest
import torch

import svgp_oracle as S
from oracle import dsvgp_oracle as O
from test_input_grads_gpu import PRED_CASES, _model, _problem
from test_step_gpu import F32, F64, KEYMAP, grads_of, rel

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def lib():
    from dsvgp_b200 import _lib, ops
    return _lib, ops


def _cond(A):
    e = torch.linalg.eigvalsh(A.detach().double().cpu())
    return float(e[-1] / e[0])


def _spd(n, seed):
    """B B^T / n + 1e-3 I: eigenvalues in [1e-3, ~4], cond <= 1e4"""
    g = torch.Generator().manual_seed(seed)
    B = torch.randn(n, n, generator=g, dtype=F64)
    return B @ B.T / n + 1e-3 * torch.eye(n, dtype=F64)


def _device_factor(ops, A):
    """L, W = L^-1 of A on the library's padded Mp x Mp layout (identity padding)"""
    n = A.shape[0]
    Mp, nb0, nlev = ops.chol_plan(n)
    work, L, W = (torch.empty(Mp, Mp, dtype=F64, device="cuda") for _ in range(3))
    if Mp > n:
        ops.pad_identity(work, n)
    work[:n, :n] = A.cuda()
    info = torch.zeros(1, dtype=torch.int32, device="cuda")
    ops.cholesky_inverse(work, L, W, nb0, nlev, info)
    assert int(info.item()) == 0
    return L, W


def _nan_upper(M, n, pad=3):
    """the lower triangle of M[:n, :n] in a NaN buffer with `pad` extra rows and columns: NaN above the diagonal"""
    b = torch.full((n + pad, n + pad), float("nan"), dtype=F64, device="cuda")
    b[:n, :n] = torch.where(torch.ones(n, n, dtype=torch.bool, device="cuda").tril(), M[:n, :n], float("nan"))
    return b


# ------------------------------------------------------------------------------------------------ the kernel
@pytest.mark.parametrize("n", [1, 2, 63, 112, 113, 1000, 3072])
def test_chol_bwd_matches_torch_autograd(lib, n):
    _lib, ops = lib
    A = _spd(n, n)
    c = _cond(A)
    assert c <= 1e4, c
    g = torch.Generator().manual_seed(7 * n)
    Lbar = torch.randn(n, n, generator=g, dtype=F64)
    Ar = A.clone().requires_grad_(True)
    (torch.linalg.cholesky(Ar) * Lbar.tril()).sum().backward()
    L, W = _device_factor(ops, A)
    Lb, Wb, Lbb = _nan_upper(L, n), _nan_upper(W, n), _nan_upper(Lbar.cuda(), n)
    out = torch.full((n + 2, n + 5), float("nan"), dtype=F64, device="cuda")
    need = _lib.call_raw("dsvgp_chol_bwd_workspace_f64", n)
    ws = torch.full((need // 8 + 64,), float("nan"), dtype=F64, device="cuda")
    rc = _lib.call("dsvgp_chol_bwd_f64", Lb, n + 3, Wb, n + 3, Lbb, n + 3, out, n + 5, n, ws, need)
    assert rc == 0
    torch.cuda.synchronize()
    got = out[:n, :n]
    assert bool(out[:, n:].isnan().all()) and bool(out[n:].isnan().all())       # output padding untouched
    assert bool(ws[need // 8:].isnan().all())                                     # nothing past the workspace size
    assert not bool(got.isnan().any())
    assert torch.equal(got, got.T)
    r = rel(got, Ar.grad)
    assert r < 1e-10, (r, c)


def test_chol_bwd_refusals(lib):
    """every refusal returns its code and enqueues nothing"""
    _lib, ops = lib
    n = 64
    L, W = _device_factor(ops, _spd(n, 1))
    L, W = L[:n, :n].contiguous(), W[:n, :n].contiguous()
    Lbar = torch.randn(n, n, dtype=F64, device="cuda")
    out = torch.empty(n, n, dtype=F64, device="cuda")
    need = _lib.call_raw("dsvgp_chol_bwd_workspace_f64", n)
    ws = torch.empty(need // 8 + 8, dtype=F64, device="cuda")
    fn = _lib._lib.dsvgp_chol_bwd_f64
    p = lambda t, off=0: ctypes.c_void_p(t.data_ptr() + off)

    def run(Lp=None, ldl=n, Wp=None, ldw=n, Bp=None, ldb=n, Op=None, ldo=n, nn=n, wsp=None, wsb=need):
        before = _lib.launch_count()
        rc = fn(p(L) if Lp is None else Lp, ldl, p(W) if Wp is None else Wp, ldw, p(Lbar) if Bp is None else Bp, ldb,
                p(out) if Op is None else Op, ldo, nn, p(ws) if wsp is None else wsp, wsb, _lib.stream())
        assert _lib.launch_count() == before or rc == 0
        return rc

    assert run() == 0
    null = ctypes.c_void_p(0)
    for kw in (dict(Lp=null), dict(Wp=null), dict(Bp=null), dict(Op=null), dict(wsp=null)):
        assert run(**kw) == -1, kw
    assert run(nn=0) == -1 and run(nn=-3) == -1
    for kw in (dict(ldl=n - 1), dict(ldw=n - 1), dict(ldb=n - 1), dict(ldo=n - 1)):
        assert run(**kw) == -1, kw
    assert run(wsb=need - 1) == -3
    # output or workspace overlapping an input
    assert run(Op=p(Lbar)) == -1 and run(Op=p(L, 8 * n)) == -1 and run(Op=p(W)) == -1
    assert run(wsp=p(L)) == -1 and run(wsp=p(Lbar, 8)) == -1 and run(wsp=p(out)) == -1
    # the products' 8-byte cp.async loads: every pointer 8-byte aligned
    for kw in (dict(Lp=p(L, 4)), dict(Wp=p(W, 4)), dict(Bp=p(Lbar, 4)), dict(Op=p(out, 4)), dict(wsp=p(ws, 4))):
        assert run(**kw) == -1, kw
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------ draws
def _oracle_full(variant, P, X, V, noisy):
    if variant == "svgp":
        return S.predictive_full(P, X, None, add_noise=noisy)
    return O.predictive_full(P, X, V, variant, add_noise=noisy)


def _kw(variant, V):
    return {} if variant in ("grad", "svgp") else {"derivative_directions": V}


DRAW_CASES = [("dsvgp", 200, 4, 40, 2, F64), ("dsvgp", 300, 10, 64, 2, F32), ("svgp", 200, 3, 40, 0, F64),
              ("dfree", 300, 6, 50, 2, F32)]


@pytest.mark.parametrize("variant,n,d,M,p,dtype", DRAW_CASES)
@pytest.mark.parametrize("noisy", [False, True])
def test_draws_with_base_samples_match_oracle(variant, n, d, M, p, dtype, noisy):
    P, x, Vx, _, _ = _problem(variant, n, d, M, p, dtype, seed=3 * n + d)
    model, lik = _model(variant, P, d, dtype)
    model.eval(), lik.eval()
    X, V = x.to(dtype).cuda(), (None if Vx is None else Vx.to(dtype).cuda())
    dist = model(X, **_kw(variant, V))
    dist = lik(dist) if noisy else dist
    nq = dist.event_shape[0]
    g = torch.Generator().manual_seed(n)
    base = torch.randn(3, 2, nq, generator=g, dtype=F64).to(dtype).double()
    draws = dist.rsample(base_samples=base.cuda())
    assert draws.shape == (3, 2, nq) and draws.dtype == dtype
    mean, cov = _oracle_full(variant, P.clone(F64), x.double(), None if Vx is None else Vx.double(), noisy)
    c = _cond(cov)
    assert c <= 1e7, c
    ref = mean + base @ torch.linalg.cholesky(cov).T
    t = 1e-10 if dtype == F64 else 1e-4
    assert rel(draws, ref) < t, (rel(draws, ref), c)
    # sample() is the same draw under no_grad, bit for bit; so is rsample under no_grad
    assert torch.equal(dist.sample(base_samples=base.cuda()), draws)
    with torch.no_grad():
        assert torch.equal(dist.rsample(base_samples=base.to(dtype).cuda()), draws)


def test_base_samples_shapes_and_seeded_draws():
    variant, n, d, M, p, dtype = "dsvgp", 20, 3, 16, 2, F32
    P, x, Vx, _, _ = _problem(variant, n, d, M, p, dtype, seed=2)
    model, lik = _model(variant, P, d, dtype)
    dist = model(x.cuda(), derivative_directions=Vx.cuda())
    nq = dist.event_shape[0]
    with pytest.raises(RuntimeError):
        dist.rsample(base_samples=torch.randn(4, nq + 1, device="cuda"))
    with pytest.raises(RuntimeError):
        dist.sample(base_samples=torch.randn(nq - 1, device="cuda"))
    for shape in ((), (4,), (2, 3)):
        assert dist.rsample(torch.Size(shape)).shape == (*shape, nq)
        assert dist.sample(torch.Size(shape)).shape == (*shape, nq)
        b = torch.randn(*shape, nq, dtype=F64, device="cuda")
        assert dist.rsample(torch.Size([7]), base_samples=b).shape == (*shape, nq)    # sample_shape from base_samples
    # without base samples, the draw takes torch.randn's next (num, n') fp64 normals: the same as passing them in
    torch.manual_seed(123)
    s = dist.rsample(torch.Size([5]))
    torch.manual_seed(123)
    z = torch.randn(5, nq, dtype=F64, device="cuda")
    assert torch.equal(s, dist.rsample(base_samples=z))


# ------------------------------------------------------------------------------------------------ gradients
def _ref_grads(variant, P, x, Vx, noisy, base, wts, cov_value, loss=None):
    """fp64 autograd of oracle -> cholesky -> mean + L z.  The factor is taken of the covariance VALUE the model computed
    (same value, the oracle's gradient path): fp32 rounding of the covariance, amplified by cond in L, is then not charged to
    the draw's backward."""
    Q = P.clone(F64).requires_grad_(True)
    Xr = x.double().clone().requires_grad_(True)
    Vr = None if Vx is None else Vx.double().clone().requires_grad_(True)
    zb = base.clone().requires_grad_(True)
    mean, cov = _oracle_full(variant, Q, Xr, Vr, noisy)
    cov = cov + (cov_value - cov).detach()
    draws = mean + zb @ torch.linalg.cholesky(cov).T
    val = (draws * wts).sum() if loss is None else loss(draws)
    names = [k for k, t in Q.tensors().items() if t is not None and (k in KEYMAP or (k == "raw_noise" and noisy))]
    leaves = [getattr(Q, k) for k in names] + [Xr, zb, mean, cov] + ([Vr] if Vr is not None else [])
    gs = torch.autograd.grad(val, leaves, allow_unused=True)
    gs = [torch.zeros_like(t) if g is None else g for t, g in zip(leaves, gs)]
    out = dict(zip(names, gs[:len(names)]))
    out["x"], out["base"], out["gmean"], out["gcov"] = gs[len(names): len(names) + 4]
    if Vr is not None:
        out["Vx"] = gs[-1]
    return out, _cond(cov)


def _check(got, ref, t, c, skip=()):
    for k, g in ref.items():
        if k in skip:
            continue
        if float(g.abs().max()) == 0.0:
            assert got.get(k) is None or float(got[k].abs().max()) == 0.0, k
            continue
        assert got.get(k) is not None, k
        r = rel(got[k], g)
        assert r < t, (k, r, c)


@pytest.mark.parametrize("variant,n,d,M,p,dtype", PRED_CASES)
@pytest.mark.parametrize("mode", ["train", "eval"])
@pytest.mark.parametrize("noisy", [False, True])
def test_rsample_gradients_match_oracle(variant, n, d, M, p, dtype, mode, noisy):
    P, x, Vx, _, _ = _problem(variant, n, d, M, p, dtype, seed=3 * n + d)
    if variant == "grad":
        Vx = None
    elif Vx is not None:
        g = torch.Generator().manual_seed(d)
        Vx = (Vx.double() + 0.3 * torch.randn(Vx.shape, generator=g, dtype=F64)).to(dtype)
    model, lik = _model(variant, P, d, dtype)
    getattr(model, mode)(), getattr(lik, mode)()
    if mode == "eval":
        with torch.no_grad():            # memoises the factor
            model(x.to(dtype).cuda(), **_kw(variant, None if Vx is None else Vx.to(dtype).cuda())).mean
    X = x.to(dtype).cuda().requires_grad_(True)
    V = None if Vx is None else Vx.to(dtype).cuda().requires_grad_(True)
    dist = model(X, **_kw(variant, V))
    dist = lik(dist) if noisy else dist
    nq = dist.event_shape[0]
    g = torch.Generator().manual_seed(n + 1)
    base = torch.randn(3, nq, generator=g, dtype=F64).to(dtype).double()
    wts = torch.randn(3, nq, generator=g, dtype=F64).to(dtype).double()
    B = base.to(dtype).cuda().requires_grad_(True)
    draws = dist.rsample(base_samples=B)
    assert draws.requires_grad and draws.dtype == dtype
    up = {}                                              # what the draw hands to autograd for (mean, covariance)
    for name, t_ in zip(("gmean", "gcov"), dist._full):
        t_.register_hook(lambda g, name=name: up.__setitem__(name, g))
    (draws * wts.to(dtype).cuda()).sum().backward()
    torch.cuda.synchronize()
    ref, c = _ref_grads(variant, P, x, Vx, noisy, base, wts, dist.covariance_matrix.detach().double().cpu())
    assert c <= 1e7, c
    got = grads_of(model, lik)
    got.update(x=X.grad, base=B.grad, **up)
    if V is not None:
        got["Vx"] = V.grad
    if variant == "dfree":
        assert bool((V.grad == 0).all())
    t = 1e-10 if dtype == F64 else 1e-4
    own = ("gmean", "gcov", "base")
    _check({k: got[k] for k in own}, {k: ref[k] for k in own}, t, c)
    # fp32: the covariance backward that (d mean, d cov) feed runs in fp32, and d cov = sym(W^T Phi W) has entries of order
    # 1/lambda_min(cov) that cancel in its contraction with d cov / d theta: measured on a B200 up to 6.9e-3 (raw_ell, shared
    # strategy, cond 1.4e6) and 2.8e-3 (raw_os, n' = 1800 through the likelihood, cond 4e2); every other fp32 case within 1e-4
    _check(got, {k: v for k, v in ref.items() if k not in own}, 1e-10 if dtype == F64 else 1e-2, c,
           skip=("Vx",) if variant == "dfree" else ())


def test_mc_acquisition_gradient_wrt_candidates():
    """qEI-shaped: relu(max over the value columns of each draw - best).mean() over 512 fixed draws at 8 candidates"""
    variant, n, d, M, p, dtype = "dsvgp", 8, 4, 40, 2, F64
    P, x, Vx, _, _ = _problem(variant, n, d, M, p, dtype, seed=17)
    model, lik = _model(variant, P, d, dtype)
    model.eval(), lik.eval()
    X = x.cuda().requires_grad_(True)
    dist = lik(model(X, derivative_directions=Vx.cuda()))
    nq = dist.event_shape[0]
    base = torch.randn(512, nq, generator=torch.Generator().manual_seed(3), dtype=F64)
    best = float(dist.mean.detach()[:: p + 1].max())
    acq = lambda s: torch.relu(s[:, :: p + 1].max(-1).values - best).mean()
    val = acq(dist.rsample(base_samples=base.cuda()))
    val.backward()
    assert float(val.detach()) > 0
    ref, c = _ref_grads(variant, P, x, Vx, True, base, None, dist.covariance_matrix.detach().cpu(), loss=acq)
    assert c <= 1e7, c
    assert rel(X.grad, ref["x"]) < 1e-10, (rel(X.grad, ref["x"]), c)


def test_rsample_finite_difference_fp64():
    """fp64 central difference at full size (M' = 3072, n = 512, eval mode) through a weighted sum of fixed-base draws,
    along a random direction in (x, Vx, raw lengthscale, raw outputscale)"""
    n, d, M, p = 512, 10, 1024, 2
    P, x, Vx, _, _ = _problem("dsvgp", n, d, M, p, F64, seed=5)
    model, lik = _model("dsvgp", P, d, F64)
    model.eval(), lik.eval()
    g = torch.Generator().manual_seed(9)
    nq = n * (p + 1)
    base = torch.randn(4, nq, generator=g, dtype=F64).cuda()
    wts = torch.randn(4, nq, generator=g, dtype=F64).cuda()
    x0, V0 = x.cuda(), (Vx.double() + 0.2 * torch.randn(Vx.shape, generator=g, dtype=F64)).cuda()
    hx, hV = torch.randn(x.shape, generator=g, dtype=F64).cuda(), torch.randn(Vx.shape, generator=g, dtype=F64).cuda()
    kern = model.covar_module
    raws = [kern.base_kernel.raw_lengthscale, kern.raw_outputscale]
    hr = [torch.randn(r.shape, generator=g, dtype=F64).cuda() for r in raws]

    def L(X, V):
        return (model(X, derivative_directions=V).rsample(base_samples=base) * wts).sum()

    X, V = x0.clone().requires_grad_(True), V0.clone().requires_grad_(True)
    L(X, V).backward()
    ana = float((X.grad * hx).sum() + (V.grad * hV).sum() + sum((r.grad * h).sum() for r, h in zip(raws, hr)))
    eps = 1e-5
    vals = []
    with torch.no_grad():
        for s in (1.0, -1.0):
            for r, h in zip(raws, hr):
                r.add_(s * eps * h)
            vals.append(float(L(x0 + s * eps * hx, V0 + s * eps * hV)))
            for r, h in zip(raws, hr):
                r.sub_(s * eps * h)
    fd = (vals[0] - vals[1]) / (2 * eps)
    assert abs(fd - ana) < 1e-6 * abs(ana), (fd, ana)


# ------------------------------------------------------------------------------------------------ robustness
def test_jitter_ladder_gradient():
    """a rank-deficient PSD covariance (rank 25 of 40, one zero row: an exactly zero pivot) takes the jitter ladder; the
    gradient is autograd of cholesky(cov + jitter_used I)"""
    from dsvgp_b200 import engine, gp
    n, r = 40, 25
    g = torch.Generator().manual_seed(4)
    B = torch.randn(n, r, generator=g, dtype=F64)
    B[5] = 0
    cov = B @ B.T / r
    mean = torch.randn(n, generator=g, dtype=F64)
    base = torch.randn(6, n, generator=g, dtype=F64)
    wts = torch.randn(6, n, generator=g, dtype=F64)
    _, (_, _, _, jitter) = engine.ENGINE.sample_mvn(mean.cuda(), cov.cuda(), 6, base=base.cuda(), keep=True)
    assert jitter > 0
    m, C, Z = (t.cuda().requires_grad_(True) for t in (mean, cov, base))
    (gp._MVNSample.apply(m, C, Z, 6) * wts.cuda()).sum().backward()
    mr, Cr, Zr = (t.clone().requires_grad_(True) for t in (mean, cov, base))
    Cj = Cr + jitter * torch.eye(n, dtype=F64)
    c = _cond(Cj)
    assert c <= 1e10, c                                  # eigenvalues O(1) over the jitter (1e-8 first): cond ~ 5e8
    ((mr + Zr @ torch.linalg.cholesky(Cj).T) * wts).sum().backward()
    t = 100 * 2.2e-16 * c                                # the factor's and the backward's errors grow with cond(cov + jitter I)
    assert rel(m.grad, mr.grad) < 1e-14
    assert rel(C.grad, Cr.grad) < t, (rel(C.grad, Cr.grad), c)
    assert rel(Z.grad, Zr.grad) < t, (rel(Z.grad, Zr.grad), c)


def test_two_draws_and_covariance_accumulate():
    variant, n, d, M, p, dtype = "dsvgp", 60, 4, 30, 2, F64
    P, x, Vx, _, _ = _problem(variant, n, d, M, p, dtype, seed=8)
    model, lik = _model(variant, P, d, dtype)
    g = torch.Generator().manual_seed(1)
    nq = n * (p + 1)
    b1, b2 = (torch.randn(2, nq, generator=g, dtype=F64) for _ in range(2))
    wc = torch.randn(nq, nq, generator=g, dtype=F64)

    def run(parts):
        model.zero_grad(), lik.zero_grad()
        X = x.cuda().requires_grad_(True)
        dist = model(X, derivative_directions=Vx.cuda())
        terms = {"a": lambda: dist.rsample(base_samples=b1.cuda()).sum(), "b": lambda: (dist.rsample(base_samples=b2.cuda()) ** 2).sum(),
                 "c": lambda: (dist.covariance_matrix * wc.cuda()).sum()}
        sum(terms[k]() for k in parts).backward()
        out = {k: v.clone() for k, v in grads_of(model, lik).items() if v is not None}
        out["x"] = X.grad.clone()
        return out

    both = run("abc")
    sep = [run(k) for k in "abc"]
    for k in both:
        s = sum(o[k] for o in sep if k in o)
        assert rel(both[k], s) < 1e-12, k


def test_later_forward_before_backward_raises():
    variant, n, d, M, p, dtype = "dsvgp", 60, 4, 30, 2, F32
    P, x, Vx, _, _ = _problem(variant, n, d, M, p, dtype, seed=8)
    model, lik = _model(variant, P, d, dtype)
    s1 = model(x.cuda(), derivative_directions=Vx.cuda()).rsample(torch.Size([2]))
    _ = model(x.cuda(), derivative_directions=Vx.cuda()).rsample(torch.Size([2]))
    with pytest.raises(RuntimeError):
        s1.sum().backward()


def test_no_grad_draw_is_todays_path(monkeypatch):
    """nothing requires grad: the draw has no graph and takes the plain (non-differentiable) evaluation"""
    from dsvgp_b200 import gp
    variant, n, d, M, p, dtype = "dsvgp", 30, 4, 20, 2, F32
    P, x, Vx, _, _ = _problem(variant, n, d, M, p, dtype, seed=6)
    model, lik = _model(variant, P, d, dtype)
    for t in list(model.parameters()) + list(lik.parameters()):
        t.requires_grad_(False)
    calls = []
    orig = gp._MVNSample.apply
    monkeypatch.setattr(gp._MVNSample, "apply", lambda *a: calls.append(1) or orig(*a))
    dist = model(x.cuda(), derivative_directions=Vx.cuda())
    s = dist.rsample(torch.Size([3]))
    assert not calls and s.grad_fn is None and not dist._full[1].requires_grad
