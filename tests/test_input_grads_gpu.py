"""Gradients w.r.t. the inputs x, the data-side directions Vx and the targets y (what plain autograd over the reference's
torch ops gives `x.grad`, `derivative_directions.grad`, `y.grad`) through the ELBO, the PLL and the predictive
mean / variance / covariance, against fp64 autograd of the CPU oracle with those tensors as leaves.

  * the data-side assembly backward (ops.kdir_bwd_cols): its own kernel for fp32 d <= 20 (every (p1, p2) the row-side
    vectorised backward takes), against fp64 autograd of the closed-form kernel and against the blocked kernel that reads
    dK transposed; NaN-sentinel output padding and NaN unread inputs;
  * the step: every strategy, fp32 / fp64, 1e-4 / 1e-10 max-norm relative per tensor, and every parameter gradient
    bit-identical to the same step run without the inputs requiring grad;
  * predictions in train and eval mode (memoised factor), a full-size fp64 finite difference, no silent None, two forwards
    before one backward, and the sharded step (two GPUs)."""
import os
import socket

import pytest
import torch

import svgp_oracle as S
from oracle import dsvgp_oracle as O
from test_shared_gpu import build_shared
from test_step_gpu import F32, F64, build, rel
from test_svgp_gpu import build_svgp

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    from dsvgp_b200 import ops
    return ops


# ------------------------------------------------------------------------------------------------ the kernel
def _dirs(n, p, d, canonical, g):
    if not p:
        return None
    if canonical:
        v = torch.zeros(n * p, d, dtype=F64)
        v[torch.arange(n * p), torch.randint(0, d, (n * p,), generator=g)] = torch.where(
            torch.rand(n * p, generator=g) < 0.5, -1.0, 1.0).double() * (0.5 + torch.rand(n * p, generator=g, dtype=F64))
        return v
    return torch.randn(n * p, d, generator=g, dtype=F64)


def _check_cols(ops, n1, n2, d, p1, p2, canonical, seed=0):
    g = torch.Generator().manual_seed(1000 * seed + n1 + 7 * n2 + d)
    x1, x2 = torch.rand(n1, d, generator=g, dtype=F64), torch.rand(n2, d, generator=g, dtype=F64)
    v1, v2 = _dirs(n1, p1, d, False, g), _dirs(n2, p2, d, canonical, g)
    x1, x2 = x1.float().double(), x2.float().double()
    v1 = None if v1 is None else v1.float().double()
    v2 = None if v2 is None else v2.float().double()
    dK = torch.randn(n1 * (p1 + 1), n2 * (p2 + 1), generator=g, dtype=F64).float().double()
    raw_ell, raw_os = torch.tensor([[0.3]], dtype=F64), torch.tensor([-0.4], dtype=F64)
    X2 = x2.clone().requires_grad_(True)
    V2 = None if v2 is None else v2.clone().requires_grad_(True)
    ell, osc = torch.nn.functional.softplus(raw_ell).reshape(()), torch.nn.functional.softplus(raw_os)
    (osc * O.kernel_closed_form(x1, X2, v1, V2, ell) * dK).sum().backward()

    dev, nan = "cuda", float("nan")
    hyp = ops.hyp_from_raw(raw_ell.float().reshape(-1).to(dev), raw_os.float().to(dev))
    def nan_tail(t, extra):               # t followed by `extra` rows of NaN: a view of the first rows
        b = torch.full((t.shape[0] + extra, t.shape[1]), nan, dtype=t.dtype, device=dev)
        b[: t.shape[0]] = t
        return b[: t.shape[0]]

    # unread inputs are NaN: rows past n1 of x1 and past n1 p1 of u1, rows past n2 of x2 and past n2 p2 of w2 (and of 1/|v2|),
    # columns past n2(p2+1) of dK (padded leading dimension), rows past n1(p1+1)
    u1 = nan_tail(ops.normalize_dirs(v1.float().to(dev))[0], 4) if p1 else None
    w2, inv2 = ops.normalize_dirs(v2.float().to(dev)) if p2 else (None, None)
    if p2:
        w2 = nan_tail(w2, 6)
        inv2 = nan_tail(inv2.reshape(-1, 1), 6).reshape(-1)
    x1d = nan_tail(x1.float().to(dev), 3)
    x2b = torch.full((n2 + 5, d), nan, device=dev)
    x2b[:n2] = x2.float()
    ld = n2 * (p2 + 1) + 13
    dKb = torch.full((n1 * (p1 + 1) + 2, ld), nan, device=dev)
    dKb[: n1 * (p1 + 1), : n2 * (p2 + 1)] = dK.float()
    dKd = dKb[: n1 * (p1 + 1), : n2 * (p2 + 1)]
    # output padding holds NaN sentinels
    gxb = torch.full((n2 + 3, d), nan, dtype=F64, device=dev)
    gxb[:n2] = 0
    gvb = torch.full((n2 * p2 + 3, d), nan, dtype=F64, device=dev) if p2 else None
    if p2:
        gvb[: n2 * p2] = 0
    took = ops.kdir_bwd_cols(x1d, u1, p1, x2b[:n2], w2, inv2, p2, hyp, dKd, gxb[:n2],
                             gvb[: n2 * p2] if p2 else None)
    assert took, "the dedicated data-side kernel did not take the shape"
    torch.cuda.synchronize()
    assert bool(gxb[n2:].isnan().all()) and (not p2 or bool(gvb[n2 * p2:].isnan().all()))
    gx, gv = gxb[:n2], (gvb[: n2 * p2] if p2 else None)
    assert rel(gx, X2.grad) < 1e-5, rel(gx, X2.grad)
    if p2:
        assert rel(gv, V2.grad) < 1e-5, rel(gv, V2.grad)
    # the blocked kernel on the swapped problem (dK read transposed) gives the same gradients
    z = lambda *s: torch.zeros(*s, dtype=F64, device=dev)
    bx, bv = z(n2, d), (z(n2 * p2, d) if p2 else None)
    ops.kdir_bwd(x2b[:n2], w2, inv2, p2, x1d, u1, p1, hyp, dKd, bx, bv, None, dk_trans=True)
    assert rel(gx, bx) < 1e-5
    if p2:
        assert rel(gv, bv) < 1e-5


PAIRS = [(0, 0), (1, 1), (2, 2), (1, 0), (2, 0)]


@pytest.mark.parametrize("p1,p2", PAIRS)
@pytest.mark.parametrize("d", [2, 3, 10, 18, 20])
@pytest.mark.parametrize("n2", [512, 999])
def test_cols_kernel_matches_fp64_autograd(ops, p1, p2, d, n2):
    _check_cols(ops, 63, n2, d, p1, p2, canonical=False)


@pytest.mark.parametrize("p1,p2", [(1, 1), (2, 2)])
@pytest.mark.parametrize("d", [3, 10, 20])
def test_cols_kernel_canonical_directions(ops, p1, p2, d):
    _check_cols(ops, 63, 999, d, p1, p2, canonical=True)


@pytest.mark.parametrize("p1,p2", PAIRS)
@pytest.mark.parametrize("n1,n2", [(1, 4096), (1024, 512), (63, 4096)])
def test_cols_kernel_row_and_column_extents(ops, p1, p2, n1, n2):
    _check_cols(ops, n1, n2, 10, p1, p2, canonical=(p2 > 0 and n1 == 1))


def test_cols_kernel_other_shapes_take_the_blocked_kernel(ops):
    """n2 < 512, d > 20, p = 3 and fp64 take the blocked kernel (the call reports it) and agree with fp64 autograd"""
    dev = "cuda"
    for n1, n2, d, p, dtype in ((20, 300, 5, 2, F32), (8, 600, 60, 2, F32), (10, 700, 4, 3, F32), (15, 600, 4, 2, F64)):
        g = torch.Generator().manual_seed(n2)
        x1, x2 = torch.rand(n1, d, generator=g, dtype=F64), torch.rand(n2, d, generator=g, dtype=F64)
        v1, v2 = torch.randn(n1 * p, d, generator=g, dtype=F64), torch.randn(n2 * p, d, generator=g, dtype=F64)
        c = lambda t: t.to(dtype).double()
        x1, x2, v1, v2 = c(x1), c(x2), c(v1), c(v2)
        dK = c(torch.randn(n1 * (p + 1), n2 * (p + 1), generator=g, dtype=F64))
        X2, V2 = x2.clone().requires_grad_(True), v2.clone().requires_grad_(True)
        (O.kernel_closed_form(x1, X2, v1, V2, torch.tensor(0.7, dtype=F64)) * dK).sum().backward()
        hyp = ops.hyp_from_raw(torch.tensor([0.7], dtype=F64).expm1().log().to(dtype).to(dev))
        u1 = ops.normalize_dirs(v1.to(dtype).to(dev))[0]
        w2, inv2 = ops.normalize_dirs(v2.to(dtype).to(dev))
        gx, gv = torch.zeros(n2, d, dtype=F64, device=dev), torch.zeros(n2 * p, d, dtype=F64, device=dev)
        took = ops.kdir_bwd_cols(x1.to(dtype).to(dev), u1, p, x2.to(dtype).to(dev), w2, inv2, p, hyp, dK.to(dtype).to(dev), gx, gv,
                                 use_os=False)
        assert not took
        t = 1e-10 if dtype == F64 else 1e-5
        assert rel(gx, X2.grad) < t and rel(gv, V2.grad) < t


# -------------------------------------------------------------------------------------------------- the step
def _model(variant, P, d, dtype):
    if variant == "shared":
        return build_shared(P, d, dtype)
    if variant == "svgp":
        return build_svgp(P, dtype)
    return build(variant, P, d, dtype)


def _problem(variant, n, d, M, p, dtype, seed):
    if variant == "shared":
        return O.make_shared_problem(n, d, M, p, dtype, seed=seed, N=50 * n)
    if variant == "svgp":
        return S.make_problem(n, d, M, dtype=dtype, seed=seed, N=50 * n)
    return O.make_problem(n, d, M, p, dtype, seed=seed, variant=variant, N=50 * n)


def _oracle_objective(variant, objective):
    if variant == "svgp":
        return S.pll if objective == "pll" else S.elbo
    return (lambda *a: O.pll(*a, variant)) if objective == "pll" else (lambda *a: O.elbo(*a, variant))


def _oracle_input_grads(variant, objective, P, x, Vx, y, num_data, chunk=None):
    """fp64 autograd of the oracle objective w.r.t. x, Vx, y.  The data term is a mean over the minibatch and the KL does not
    depend on the data, so the gradients can be taken over chunks of points (scaled by the chunk's share of n')."""
    P64, n = P.clone(F64), x.shape[0]
    chunk = chunk or n
    q = y.numel() // n
    p2 = 0 if Vx is None else Vx.shape[0] // n
    fn = _oracle_objective(variant, objective)
    gx, gV, gy = [], [], []
    for lo in range(0, n, chunk):
        hi = min(n, lo + chunk)
        X = x[lo:hi].double().clone().requires_grad_(True)
        V = None if Vx is None else Vx[lo * p2: hi * p2].double().clone().requires_grad_(True)
        Y = y[lo * q: hi * q].double().clone().requires_grad_(True)
        val = fn(P64, X, V, Y, num_data)
        leaves = [t for t in (X, V, Y) if t is not None]
        gs = torch.autograd.grad(val, leaves, allow_unused=True)
        gs = [torch.zeros_like(t) if gg is None else gg for t, gg in zip(leaves, gs)]
        w = (hi - lo) / n
        gx.append(gs[0] * w)
        if V is not None:
            gV.append(gs[1] * w)
        gy.append(gs[-1] * w)
    return torch.cat(gx), (torch.cat(gV) if gV else None), torch.cat(gy)


def _gpu_step(variant, P, x, Vx, y, num_data, d, dtype, objective, inputs):
    from dsvgp_b200 import gp
    model, lik = _model(variant, P, d, dtype)
    model.train(), lik.train()
    mll = (gp.PredictiveLogLikelihood if objective == "pll" else gp.VariationalELBO)(lik, model, num_data=num_data)
    X = x.to(dtype).cuda().requires_grad_("x" in inputs)
    V = None if Vx is None else Vx.to(dtype).cuda().requires_grad_("Vx" in inputs)
    Y = y.to(dtype).cuda().requires_grad_("y" in inputs)
    kw = {} if variant in ("grad", "svgp") else {"derivative_directions": V}
    val = mll(lik(model(X, **kw)), Y)
    val.backward()
    torch.cuda.synchronize()
    pg = {name: t.grad.clone() for name, t in list(model.named_parameters()) + list(lik.named_parameters()) if t.grad is not None}
    return val.detach(), pg, X.grad, (None if V is None else V.grad), Y.grad


STEP_CASES = [
    # variant, n, d, M, p, dtype, objective, oracle chunk
    ("dsvgp", 200, 2, 20, 2, F32, "elbo", None),           # C1 (tests/test_dsvgp.py as shipped)
    ("dsvgp", 200, 2, 20, 2, F32, "pll", None),
    ("dsvgp", 256, 10, 64, 2, F32, "elbo", None),
    ("dsvgp", 600, 3, 512, 1, F64, "elbo", None),          # C2 (bunny-shaped, fp64)
    ("dsvgp", 600, 3, 512, 1, F64, "pll", None),
    ("dsvgp", 285, 3, 50, 1, F32, "elbo", None),           # ragged n' (n' < 512: blocked data-side kernel)
    ("dsvgp", 999, 10, 64, 2, F32, "elbo", None),          # ragged n' on the dedicated kernel
    ("dsvgp", 257, 10, 96, 2, F64, "elbo", None),          # fp64 at p = 2 (blocked data-side kernel)
    ("dsvgp", 512, 10, 1024, 2, F32, "elbo", None),        # C3-shaped, M' = 3072
    ("dsvgp", 4096, 10, 1024, 2, F32, "elbo", 512),
    ("dsvgp", 300, 60, 40, 3, F32, "elbo", None),          # rover-shaped: d = 60, p = 3 (blocked data-side kernel)
    ("dfree", 1024, 18, 256, 2, F32, "elbo", None),        # derivative-free: the Vx gradient is exactly zero
    ("dfree", 300, 6, 50, 2, F64, "pll", None),
    ("grad", 300, 3, 40, 3, F32, "elbo", None),            # full gradient: x only
    ("grad", 200, 2, 30, 2, F64, "pll", None),
    ("shared", 600, 10, 96, 2, F32, "elbo", None),
    ("shared", 257, 5, 40, 1, F64, "pll", None),
    ("svgp", 1024, 10, 256, 0, F32, "elbo", None),         # plain SVGP: x only
    ("svgp", 999, 18, 128, 0, F32, "pll", None),
    ("svgp", 300, 4, 50, 0, F64, "elbo", None),
]


@pytest.mark.parametrize("variant,n,d,M,p,dtype,objective,chunk", STEP_CASES)
def test_step_input_grads_match_oracle(variant, n, d, M, p, dtype, objective, chunk):
    P, x, Vx, y, num_data = _problem(variant, n, d, M, p, dtype, seed=n + M + d)
    if variant in ("dsvgp", "shared") and Vx is not None:
        # general data-side directions as well as canonical ones
        g = torch.Generator().manual_seed(n)
        Vx = (Vx.double() + 0.3 * torch.randn(Vx.shape, generator=g, dtype=F64)).to(dtype)
    if variant == "grad":
        Vx = None
    rx, rV, ry = _oracle_input_grads(variant, objective, P, x, Vx, y, num_data, chunk)
    inputs = ("x", "y") + (("Vx",) if Vx is not None else ())
    _, pg0, *none = _gpu_step(variant, P, x, Vx, y, num_data, d, dtype, objective, ())
    assert all(t is None for t in none)
    _, pg, gx, gV, gy = _gpu_step(variant, P, x, Vx, y, num_data, d, dtype, objective, inputs)
    t = 1e-10 if dtype == F64 else 1e-4
    assert rel(gx, rx) < t, rel(gx, rx)
    assert rel(gy, ry) < t, rel(gy, ry)
    if variant == "dfree":
        assert gV is not None and bool((gV == 0).all())
    elif Vx is not None:
        assert rel(gV, rV) < t, rel(gV, rV)
    assert pg.keys() == pg0.keys()
    for k in pg:
        assert torch.equal(pg[k], pg0[k]), k


# ---------------------------------------------------------------------------------------------------- predictions
PRED_CASES = [("dsvgp", 300, 10, 64, 2, F32), ("dsvgp", 200, 4, 40, 2, F64), ("dsvgp", 600, 10, 64, 2, F32),
              ("dfree", 300, 6, 50, 2, F32), ("grad", 150, 3, 30, 3, F64), ("shared", 300, 5, 40, 1, F32),
              ("svgp", 600, 10, 128, 0, F32), ("svgp", 200, 3, 40, 0, F64)]


def _oracle_pred(variant, P, X, V, what):
    if variant == "svgp":
        return S.predictive_full(P, X, None)[1] if what == "cov" else S.predictive(P, X, None)
    if what == "cov":
        return O.predictive_full(P, X, V, variant)[1]
    return O.predictive(P, X, V, variant)


@pytest.mark.parametrize("variant,n,d,M,p,dtype", PRED_CASES)
@pytest.mark.parametrize("mode", ["train", "eval"])
def test_prediction_input_grads_match_oracle(variant, n, d, M, p, dtype, mode):
    P, x, Vx, _, _ = _problem(variant, n, d, M, p, dtype, seed=3 * n + d)
    if variant == "grad":
        Vx = None
    elif Vx is not None:
        g = torch.Generator().manual_seed(d)
        Vx = (Vx.double() + 0.3 * torch.randn(Vx.shape, generator=g, dtype=F64)).to(dtype)
    model, lik = _model(variant, P, d, dtype)
    getattr(model, mode)(), getattr(lik, mode)()
    kw = lambda V: {} if variant in ("grad", "svgp") else {"derivative_directions": V}
    if mode == "eval":
        with torch.no_grad():            # memoises the factor
            model(x.to(dtype).cuda(), **kw(None if Vx is None else Vx.to(dtype).cuda())).mean
    P64 = P.clone(F64)
    g = torch.Generator().manual_seed(n)
    t = 1e-10 if dtype == F64 else 1e-4
    for what in ("mean_var", "cov"):
        X = x.to(dtype).cuda().requires_grad_(True)
        V = None if Vx is None else Vx.to(dtype).cuda().requires_grad_(True)
        dist = model(X, **kw(V))
        Xr = x.double().clone().requires_grad_(True)
        Vr = None if Vx is None else Vx.double().clone().requires_grad_(True)
        if what == "cov":
            w = torch.randn(dist.event_shape[0], dist.event_shape[0], generator=g, dtype=F64)
            (dist.covariance_matrix * w.to(dtype).cuda()).sum().backward()
            (_oracle_pred(variant, P64, Xr, Vr, "cov") * w.to(dtype).double()).sum().backward()
        else:
            w1, w2 = (torch.randn(dist.event_shape[0], generator=g, dtype=F64) for _ in range(2))
            ((dist.mean * w1.to(dtype).cuda()).sum() + (dist.variance * w2.to(dtype).cuda()).sum()).backward()
            mean, var = _oracle_pred(variant, P64, Xr, Vr, "mean_var")
            ((mean * w1.to(dtype).double()).sum() + (O.clamp_variance(var) * w2.to(dtype).double()).sum()).backward()
        assert rel(X.grad, Xr.grad) < t, (what, rel(X.grad, Xr.grad))
        if V is not None:
            if variant == "dfree":
                assert bool((V.grad == 0).all())
            else:
                assert rel(V.grad, Vr.grad) < t, (what, rel(V.grad, Vr.grad))


@pytest.mark.parametrize("what", ["mean_var", "cov"])
def test_prediction_input_grads_finite_difference_fp64(what):
    """fp64 directional finite difference at full size (M' = 3072, n = 512) through .mean and .variance, and through
    .covariance_matrix (K_zx and the dense K_xx); fp64 runs the blocked data-side kernel"""
    n, d, M, p = 512, 10, 1024, 2
    P, x, Vx, _, _ = _problem("dsvgp", n, d, M, p, F64, seed=5)
    model, lik = _model("dsvgp", P, d, F64)
    model.eval(), lik.eval()
    g = torch.Generator().manual_seed(9)
    nq = n * (p + 1)
    w1, w2 = (torch.randn(nq, generator=g, dtype=F64).cuda() for _ in range(2))
    wc = torch.randn(nq, nq, generator=g, dtype=F64).cuda()
    hx, hV = torch.randn(x.shape, generator=g, dtype=F64).cuda(), torch.randn(Vx.shape, generator=g, dtype=F64).cuda()
    x0, V0 = x.cuda(), (Vx.double() + 0.2 * torch.randn(Vx.shape, generator=g, dtype=F64)).cuda()

    def L(X, V):
        dist = model(X, derivative_directions=V)
        if what == "cov":
            return (dist.covariance_matrix * wc).sum()
        return (dist.mean * w1).sum() + (dist.variance * w2).sum()

    X, V = x0.clone().requires_grad_(True), V0.clone().requires_grad_(True)
    L(X, V).backward()
    ana = float((X.grad * hx).sum() + (V.grad * hV).sum())
    eps = 1e-5
    with torch.no_grad():
        fd = (float(L(x0 + eps * hx, V0 + eps * hV)) - float(L(x0 - eps * hx, V0 - eps * hV))) / (2 * eps)
    assert abs(fd - ana) < 1e-6 * abs(ana), (fd, ana)


# --------------------------------------------------------------------------------------------- no silent None etc.
@pytest.mark.parametrize("variant", ["dsvgp", "dfree", "grad", "shared", "svgp"])
@pytest.mark.parametrize("dtype", [F32, F64])
def test_every_entry_point_gives_input_grads(variant, dtype):
    from dsvgp_b200 import gp
    d, M, p, n = 3, 12, (3 if variant == "grad" else 0 if variant == "svgp" else 2), 40
    P, x, Vx, y, num_data = _problem(variant, n, d, M, p, dtype, seed=1)
    model, lik = _model(variant, P, d, dtype)
    has_v = variant not in ("grad", "svgp")
    for entry in ("elbo", "pll", "mean", "variance", "cov"):
        model.train(), lik.train()
        X = x.to(dtype).cuda().requires_grad_(True)
        V = Vx.to(dtype).cuda().requires_grad_(True) if has_v else None
        Y = y.to(dtype).cuda().requires_grad_(True)
        dist = model(X, **({"derivative_directions": V} if has_v else {}))
        if entry in ("elbo", "pll"):
            mll = (gp.PredictiveLogLikelihood if entry == "pll" else gp.VariationalELBO)(lik, model, num_data=num_data)
            mll(lik(dist), Y).backward()
            assert Y.grad is not None, entry
        else:
            out = {"mean": lambda: dist.mean, "variance": lambda: dist.variance, "cov": lambda: dist.covariance_matrix}[entry]()
            out.sum().backward()
        assert X.grad is not None and X.grad.shape == X.shape, entry
        if has_v:
            assert V.grad is not None and V.grad.shape == V.shape, entry


def test_two_forwards_before_one_backward():
    from dsvgp_b200 import gp
    n, d, M, p = 300, 10, 64, 2
    P, x, Vx, y, num_data = _problem("dsvgp", n, d, M, p, F32, seed=4)
    model, lik = _model("dsvgp", P, d, F32)
    mll = gp.VariationalELBO(lik, model, num_data=num_data)
    xs = [x.cuda(), (x + 0.01).cuda()]

    def one(xi):
        X, V, Y = xi.clone().requires_grad_(True), Vx.cuda().requires_grad_(True), y.cuda().requires_grad_(True)
        return X, V, Y, mll(lik(model(X, derivative_directions=V)), Y)

    sep = []
    for xi in xs:
        X, V, Y, val = one(xi)
        val.backward()
        sep.append((X.grad, V.grad, Y.grad))
    a, b = one(xs[0]), one(xs[1])
    (a[3] + b[3]).backward()
    for got, want in zip((a, b), sep):
        for t, w in zip(got[:3], want):
            assert torch.equal(t.grad, w)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        import bench
        from dsvgp_b200 import distributed, gp
        wl = dict(bench.WORKLOADS["C3"], M=256, n=1024)
        dev = torch.device("cuda", rank)
        n, d, p = wl["n"], wl["d"], wl["p"]
        x, V, y = bench.synth_batch(n, d, p, "dsvgp", torch.float32, "cpu", 5)

        def grads(xs, Vs, sharded):
            model, lik = bench.build_model(wl, torch.float32, dev)
            if sharded:
                distributed.enable(model, n)
            mll = gp.VariationalELBO(lik, model, num_data=(d + 1) * wl["N"])
            X, Vd = xs.to(dev).requires_grad_(True), Vs.to(dev).requires_grad_(True)
            lo_, hi_ = (lo, hi) if sharded else (0, n)
            loss = -mll(lik(model(X, derivative_directions=Vd)), y[lo_ * (p + 1): hi_ * (p + 1)].to(dev))
            loss.backward()
            distributed.disable(model)
            return X.grad.double(), Vd.grad.double()

        lo, hi = distributed.shard_bounds(n, rank, world)
        gx_s, gv_s = grads(x[lo:hi], V[lo * p: hi * p], True)
        gx_f, gv_f = grads(x, V, False)
        assert float((gx_s - gx_f[lo:hi]).abs().max() / gx_f[lo:hi].abs().max()) < 1e-4
        assert float((gv_s - gv_f[lo * p: hi * p]).abs().max() / gv_f[lo * p: hi * p].abs().max()) < 1e-4
        out[rank] = "ok"
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_sharded_step_input_grads_two_gpus():
    """each rank's x / Vx gradient is its slice of the unsharded one (it never enters the all-reduced buffers)"""
    import torch.multiprocessing as mp
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    assert dict(out) == {0: "ok", 1: "ok"}
