"""The plain SVGP baseline (traditional_vi.py: VariationalStrategy + ScaleKernel(RBFKernel()), the p = 0 case of the fused
step) on the GPU.

  * the value-only assembly kernels of csrc/kdir.cu (kdir_fwd_v4<0, 0, OUT>, kdir_bwd_v4<0, 0, DP, VPL>): every output
    against an fp64 closed form, the half split bit for bit against split_half of the fp32 kernel's K, NaN sentinels in
    every output's padding and NaN in every input row / column the kernels must not read;
  * the whole step against the fp64 SVGP oracle (tests/svgp_oracle.py): 1e-4 (fp32) / 1e-10 (fp64), max-norm relative per tensor, on
    the ELBO / PLL value, every parameter gradient, the mean and the variance;
  * everything around the step: full covariance and its gradients, samples, NGD, graph replay, two forwards before one
    backward, the sharded tail, the state dict, and traditional_vi.train_gp / eval_gp."""
import math

import pytest
import torch

from oracle import dsvgp_oracle as O
import svgp_oracle as S
from test_half_operands_gpu import _buf, _pad_kept, _same_bits, _engine, _last_ws
from test_step_gpu import check_against, grads_of, rel
from test_trained_state_gpu import GATES_3XFP16

pytestmark = pytest.mark.gpu
F16, F32, F64 = torch.float16, torch.float32, torch.float64
KEYMAP = {"Z": "variational_strategy.inducing_points",
          "m": "variational_strategy._variational_distribution.variational_mean",
          "Ls_raw": "variational_strategy._variational_distribution.chol_variational_covar",
          "c": "mean_module.constant", "raw_os": "covar_module.raw_outputscale",
          "raw_ell": "covar_module.base_kernel.raw_lengthscale"}


@pytest.fixture(scope="module")
def ops():
    from dsvgp_b200 import ops
    return ops


def _round_up(a, b):
    return (a + b - 1) // b * b


# ------------------------------------------------------------------------------------------------ assembly kernels
def _points(n, d, seed):
    """(n, d) fp32 points in [0, 1)^d, as the leading rows of a NaN buffer: rows past n must never be read"""
    g = torch.Generator().manual_seed(seed)
    full = torch.full((n + 7, d), float("nan"), dtype=F32, device="cuda")
    full[:n] = torch.rand(n, d, generator=g).cuda()
    return full[:n]


def _hyp(ops):
    return ops.hyp_from_raw(torch.tensor([0.3], dtype=F32, device="cuda"), torch.tensor([-0.4], dtype=F32, device="cuda"))


def _rbf64(x1, x2, hyp):
    """os * exp(-|x1_i - x2_j|^2 / 2 ell^2) in fp64 on the device (difference form: no cancellation)"""
    ell, osc = float(hyp[0]), float(hyp[1])
    a, b = x1.double(), x2.double()
    out = torch.empty(a.shape[0], b.shape[0], dtype=F64, device="cuda")
    for i in range(0, a.shape[0], 128):
        out[i:i + 128] = ((a[i:i + 128, None, :] - b[None, :, :]) ** 2).sum(-1)
    return osc * torch.exp(-0.5 * out / ell ** 2)


def _tf32_lo_ref(K):
    """rn_tf32(x - trunc_tf32(x)) of every element (the kernel's tf32_lo_part), exactly"""
    bits = K.contiguous().view(torch.int32)
    r = (K - (bits & -8192).view(F32)).contiguous()          # 0xFFFFE000: keep sign, exponent, 10 mantissa bits
    rb = r.view(torch.int32)
    mag = ((rb & 0x7FFFFFFF) + 0x1000) & 0x7FFFE000           # round half away from zero on the magnitude
    return (mag | (rb & -0x80000000)).view(F32)


FWD_D, FWD_N2, FWD_N1 = [2, 3, 10, 18, 60], [512, 999, 4096], [1, 63, 1024]


@pytest.mark.parametrize("n1", FWD_N1)
@pytest.mark.parametrize("n2", FWD_N2)
@pytest.mark.parametrize("d", FWD_D)
def test_value_only_forward_all_outputs(ops, d, n2, n1):
    """kdir_fwd_v4<0, 0, OUT> for OUT = K, K + TF32 lo, two-half split only: within 2e-6 of the fp64 closed form, lo exact,
    the split bit-identical to split_half of the fp32 K; padding untouched in every output"""
    hyp = _hyp(ops)
    x1, x2 = _points(n1, d, 3 * d + n1), _points(n2, d, 5 * d + n2)
    Kref = _rbf64(x1, x2, hyp)
    ld = _round_up(n2, 64) + 4
    Kf, K = _buf(n1, n2, ld, F32)
    assert not ops.kdir_fwd(x1, None, 0, x2, None, 0, hyp, K, out_lo=None)
    torch.cuda.synchronize()
    assert rel(K, Kref) < 2e-6 and _pad_kept(Kf, n2)
    # K and its lo companion (operands of the 3xTF32 product)
    K2f, K2 = _buf(n1, n2, ld, F32)
    Lf, Lo = _buf(n1, n2, ld, F32)
    assert ops.kdir_fwd(x1, None, 0, x2, None, 0, hyp, K2, out_lo=Lo)
    torch.cuda.synchronize()
    assert _same_bits(K2, K) and _pad_kept(K2f, n2) and _pad_kept(Lf, n2)
    assert _same_bits(Lo, _tf32_lo_ref(K))
    # only the two-half split of K * s (operands of the 3xFP16 product)
    maxbits = torch.zeros(8, dtype=torch.int32, device="cuda")
    sc = torch.ones(16, dtype=F32, device="cuda")
    ops.tc_scales(hyp, 1e-3, maxbits, n1, sc, 0)
    sK = float(sc[1])
    for hld in (_round_up(n2, 64), _round_up(n2, 4) + 2):     # vector stores / element stores
        (hf, Kh), (lf, Kl) = _buf(n1, n2, hld, F16), _buf(n1, n2, hld, F16)
        Kdf, Kd = _buf(n1, n2, n2, F32)
        assert ops.kdir_fwd_half(x1, None, 0, x2, None, 0, hyp, Kd, Kh, Kl, sc[1:2])
        torch.cuda.synchronize()
        assert bool(torch.isnan(Kdf).all())                    # no fp32 matrix at all
        assert _pad_kept(hf, n2) and _pad_kept(lf, n2)
        assert rel((Kh.double() + Kl.double()) / sK, Kref) < 2e-6
        (rhf, rh), (rlf, rl) = _buf(n1, n2, hld, F16), _buf(n1, n2, hld, F16)
        ops.split_half(K, sc[1:2], rh, rl, rows=n1, cols=n2)
        assert _same_bits(Kh, rh) and _same_bits(Kl, rl), hld


def test_value_only_forward_declines_narrow_tiles(ops):
    """n2 < 512 stays on the blocked kernel: kdir_fwd_half says False and writes fp32 K"""
    hyp = _hyp(ops)
    x1, x2 = _points(40, 3, 1), _points(511, 3, 2)
    (hf, Kh), (lf, Kl) = _buf(40, 511, 512, F16), _buf(40, 511, 512, F16)
    Kf, K = _buf(40, 511, 515, F32)
    assert not ops.kdir_fwd_half(x1, None, 0, x2, None, 0, hyp, K, Kh, Kl, torch.ones(1, dtype=F32, device="cuda"))
    torch.cuda.synchronize()
    assert rel(K, _rbf64(x1, x2, hyp)) < 2e-6 and _pad_kept(Kf, 511)
    assert _pad_kept(hf, 0) and _pad_kept(lf, 0)


BWD = [(n1, n2, d) for d in FWD_D for n2 in FWD_N2 for n1 in (63, 1024)]


@pytest.mark.parametrize("vpl", [4, 2])
@pytest.mark.parametrize("n1,n2,d", BWD)
def test_value_only_backward_matches_fp64_autograd(ops, n1, n2, d, vpl):
    """kdir_bwd_v4<0, 0, DP, VPL> (d <= 20): d/dx1, d ell, d os within 1e-5 relative of fp64 autograd, with NaN in the
    upstream padding and behind the last input rows, and untouched accumulator padding.  d = 60 runs on the blocked kernel
    (the DP = 60 variant spills); there the two scalars, sums over n1 n2 terms of both signs, are gated at 1e-5 of the sum of
    the terms' magnitudes (measured: 5e-6 of |d ell| at n1 = 1024, n2 = 512)"""
    hyp = _hyp(ops)
    x1, x2 = _points(n1, d, 7 * d + n1), _points(n2, d, 11 * d + n2)
    g = torch.Generator().manual_seed(n1 + n2 + d)
    dK64 = torch.randn(n1, n2, generator=g, dtype=F64).cuda()
    ld = _round_up(n2, 64)                                    # the step's layout: staged whole tiles, direct ragged tile
    dKf, dK = _buf(n1, n2, ld, F32)
    dK.copy_(dK64.float())
    X1 = x1.double().clone().requires_grad_(True)
    ell = hyp[0].clone().requires_grad_(True)
    osc = hyp[1].clone().requires_grad_(True)
    r2 = ((X1[:, None, :] - x2.double()[None, :, :]) ** 2).sum(-1)
    (osc * torch.exp(-0.5 * r2 / ell ** 2) * dK.double()).sum().backward()
    with torch.no_grad():
        G = (torch.exp(-0.5 * r2 / ell ** 2) * dK.double()).abs()
        scale = (float(osc * (G * r2).sum() / ell ** 3), float(G.sum())) if d > 20 else (float(ell.grad), float(osc.grad))
    gxf = torch.full((n1 + 3, d), 7.0, dtype=F64, device="cuda")
    gx, gsc = gxf[:n1], torch.zeros(2, dtype=F64, device="cuda")
    gx.zero_()
    ops.set_kdir_bwd_vpl(vpl)
    try:
        ops.kdir_bwd(x1, None, None, 0, x2, None, 0, hyp, dK, gx, None, gsc)
    finally:
        ops.set_kdir_bwd_vpl(4)
    torch.cuda.synchronize()
    assert bool((gxf[n1:] == 7.0).all())
    assert rel(gx, X1.grad) < 1e-5
    assert abs(float(gsc[0]) - float(ell.grad)) < 1e-5 * abs(scale[0])
    assert abs(float(gsc[1]) - float(osc.grad)) < 1e-5 * abs(scale[1])


# ---------------------------------------------------------------------------------------------------------- the step
def build_svgp(P, dtype, ngd=False):
    import traditional_vi
    from dsvgp_b200 import gp
    model = traditional_vi.GPModel(P.Z.detach().to(dtype).cpu(), **({"variational_distribution": "NGD"} if ngd else {}))
    lik = gp.GaussianLikelihood()
    model, lik = model.to("cuda", dtype), lik.to("cuda", dtype)
    sd = model.state_dict()
    for k, name in KEYMAP.items():
        if name in sd:
            sd[name] = getattr(P, k).detach().to(dtype).reshape(sd[name].shape).cuda()
    sd["variational_strategy.variational_params_initialized"] = torch.tensor(1)
    model.load_state_dict(sd)
    lik.load_state_dict({"noise_covar.raw_noise": P.raw_noise.detach().to(dtype).cuda()})
    return model, lik


def svgp_step(P, x, y, num_data, dtype, objective="elbo"):
    from dsvgp_b200 import gp
    model, lik = build_svgp(P, dtype)
    model.train(), lik.train()
    mll = (gp.PredictiveLogLikelihood if objective == "pll" else gp.VariationalELBO)(lik, model, num_data=num_data)
    out = lik(model(x.to(dtype).cuda()))
    loss = -mll(out, y.to(dtype).cuda())
    loss.backward()
    return model, lik, -loss.detach(), {k: -g for k, g in grads_of(model, lik).items()}, out


def _up(t):
    return None if t is None else t.double()


def _check_step(P, x, y, num_data, dtype, objective="elbo", gates=None):
    """one step through traditional_vi.GPModel against the oracle: value, every gradient, train-mode mean / variance and the
    eval-mode prediction; gates None = 1e-4 / 1e-10 on everything"""
    model, lik, val, grads, out = svgp_step(P, x, y, num_data, dtype, objective)
    P64 = P.clone(F64)
    if x.shape[0] > 4096:
        assert objective == "elbo"
        ref_val, ref_grads, mean, var = S.elbo_and_grads_chunked(P64, _up(x), None, _up(y), num_data, "svgp", chunk=2048)
    else:
        fn = S.pll_and_grads if objective == "pll" else S.elbo_and_grads
        ref_val, ref_grads = fn(P64, _up(x), None, _up(y), num_data, variant="svgp")
        mean, var = S.predict(P64, _up(x), None, variant="svgp")
    t = 1e-10 if dtype == F64 else 1e-4
    gates = gates or {}
    err = {"value": abs(float(val) - float(ref_val)) / abs(float(ref_val))}
    err.update({k: rel(grads[k], g) for k, g in ref_grads.items()})
    assert set(ref_grads) == set(KEYMAP) | {"raw_noise"}
    if objective == "elbo":                                   # (PLL: the loop's printout carries one noise, checked below)
        err.update(mean=rel(out.mean, mean), var=rel(out.variance, var))
    model.eval(), lik.eval()
    with torch.no_grad():
        preds = lik(model(x.to(dtype).cuda()))
        err.update(pred_mean=rel(preds.mean, mean), pred_var=rel(preds.variance, var))
    bad = {k: v for k, v in err.items() if not v <= gates.get(k, t)}
    assert not bad, bad
    return model, lik


STEP = [  # n, d, M, dtype, whitening (engine.WHITEN_FP64)
    (200, 2, 20, F32, "auto"),          # config-1-like
    (200, 2, 20, F64, "auto"),
    (285, 5, 150, F32, "auto"),         # ragged n, default (fp64) whitening
    (999, 5, 150, F32, "auto"),
    (999, 5, 150, F32, False),          # ... and on 3xFP16 whitening
    (2048, 10, 256, F32, "auto"),       # n' = 2048: fp64 whitening
    (2049, 10, 256, F32, "auto"),       # n' = 2049: 3xFP16 whitening
    (2048, 60, 800, F32, "auto"),       # rover-shaped (C4), p = 0
    (4096, 3, 1024, F64, "auto"),       # bunny-shaped fp64
    (4096, 10, 3072, F32, "auto"),      # C3-shaped, p = 0, 3xFP16
    (16384, 10, 3072, F32, "auto"),
]


@pytest.mark.parametrize("n,d,M,dtype,whiten", STEP)
def test_svgp_step_matches_oracle(n, d, M, dtype, whiten):
    P, x, _, y, num_data = S.make_problem(n, d, M, 0, dtype, seed=n + d + M, variant="svgp", N=10 * n)
    with _engine(WHITEN_FP64=whiten) as engine:
        _check_step(P, x, y, num_data, dtype)
        if dtype == F32 and M >= 128:                        # the path this case is about was taken
            ws = [w for w in engine.ENGINE._ws.values() if w.n == n][0]
            assert ws.tch and (ws.A64 is not None) == (whiten == "auto" and n <= 2048)


@pytest.mark.parametrize("n,d,M,dtype,whiten", [STEP[0], STEP[1], STEP[4], STEP[6]])
def test_svgp_pll_step_matches_oracle(n, d, M, dtype, whiten):
    P, x, _, y, num_data = S.make_problem(n, d, M, 0, dtype, seed=n + d + M, variant="svgp", N=10 * n)
    with _engine(WHITEN_FP64=whiten):
        _check_step(P, x, y, num_data, dtype, objective="pll")


@pytest.mark.parametrize("dtype", [F64, F32])
@pytest.mark.parametrize("ell", [0.15, 2.0])
def test_svgp_trained_state_matches_oracle(ell, dtype):
    """q(u) at the ELBO optimum of a fit set (kind="optimal"): fp64 at 1e-10; fp32 (fp64 whitening, n' <= 2048) at 1e-4 on the
    value, mean, variance and hyper-parameters and at the converged-state gates of test_trained_state_gpu on (Z, m, L_s, c),
    whose gradients are small differences of large terms that no fp32 evaluation gets to 1e-4 (DESIGN.md section 4.2)"""
    P, x, _, y, num_data = S.make_trained_problem(300, 5, 128, 0, dtype, seed=2, variant="svgp", ell=ell, kind="optimal",
                                                  N=3000)
    gates = None if dtype == F64 else {k: GATES_3XFP16[k] for k in ("Z", "m", "c", "Ls_raw")}
    with _engine(WHITEN_FP64="auto"):
        _check_step(P, x, y, num_data, dtype, gates=gates)


def test_svgp_operands_use_the_fp16_range(monkeypatch):
    """3xFP16 operand scales at p = 0 (tc_scales' a-priori bound of K was derived for p > 0): every hi half of a real
    step finite and within [2^5, 2^15]"""
    from dsvgp_b200 import ops
    P, x, _, y, nd = S.make_problem(3000, 10, 384, 0, F32, seed=5, variant="svgp", N=100000)
    seen = {}
    real = ops.gemm_tch

    def spy(*args, **kw):
        if kw.get("Ch") is not None and kw.get("a_tri") == ops.TRI_LOWER:
            seen["K_zx"] = args[1][0].clone()
        return real(*args, **kw)
    monkeypatch.setattr(ops, "gemm_tch", spy)
    with _engine(WHITEN_FP64=False) as engine:
        svgp_step(P, x, y, nd, F32)
        ws, f = _last_ws(engine), list(engine.ENGINE._fac.values())[-1]
        hi = {"W": f.Wh, "K_zx": seen["K_zx"], "A": ws.Ah, "D": ws.Dh, "dA": ws.Kh, "A_g": ws.Agh}
        stats = {k: (bool(torch.isfinite(t).all()), float(t.float().abs().max())) for k, t in hi.items()}
    print("\nlog2 max|hi| (svgp):", {k: round(math.log2(mx), 2) for k, (_, mx) in stats.items()})
    assert all(ok and 2.0 ** 5 <= mx <= 2.0 ** 15 for ok, mx in stats.values()), stats


# ------------------------------------------------------------------------------------------------ around the step
@pytest.mark.parametrize("n,dtype,noisy", [(600, F32, False), (600, F64, True), (150, F64, False)])
def test_svgp_full_covariance_and_its_gradients(n, dtype, noisy):
    """dense predictive covariance (K_xx on the new forward kernel at n >= 512 in fp32) and its gradients against oracle
    autograd"""
    d, M = 4, 60
    P, x, _, y, _ = S.make_problem(n, d, M, 0, dtype, seed=n, variant="svgp", N=10 * n)
    model, lik = build_svgp(P, dtype)
    model.train(), lik.train()
    g = torch.Generator().manual_seed(1)
    W = torch.randn(n, n, generator=g, dtype=F64)
    wm = torch.randn(n, generator=g, dtype=F64)
    dist = model(x.cuda())
    if noisy:
        dist = lik(dist)
    cov, mean = dist.covariance_matrix, dist.mean
    ((cov * W.to(dtype).cuda()).sum() + (mean * wm.to(dtype).cuda()).sum()).backward()
    Q = P.clone(F64).requires_grad_(True)
    m_o, c_o = S.predictive_full(Q, _up(x), None, variant="svgp", add_noise=noisy)
    t = 1e-10 if dtype == F64 else 1e-4
    assert rel(mean, m_o) < t and rel(cov, c_o) < t
    ((c_o * W).sum() + (m_o * wm).sum()).backward()
    got = grads_of(model, lik)
    for k in KEYMAP:
        assert rel(got[k], getattr(Q, k).grad) < t, k
    if noisy:
        assert rel(got["raw_noise"], Q.raw_noise.grad) < t


def test_svgp_samples_follow_the_predictive_distribution():
    P, x, _, y, _ = S.make_problem(40, 3, 30, 0, F64, seed=3, variant="svgp")
    model, lik = build_svgp(P, F64)
    model.eval(), lik.eval()
    torch.manual_seed(0)
    with torch.no_grad():
        preds = lik(model(x.cuda()))
        s = preds.sample(torch.Size([200000]))
    assert s.shape == (200000, 40)
    m_o, c_o = S.predictive_full(P, x, None, variant="svgp", add_noise=True)
    assert float((s.mean(0).cpu() - m_o).abs().max()) < 5 * float(c_o.diagonal().max().sqrt()) / math.sqrt(200000)
    emp = torch.cov(s.T).cpu()
    assert float((emp - c_o).abs().max()) < 0.02 * float(c_o.abs().max())


def test_svgp_ngd_step_matches_oracle():
    """NaturalVariationalDistribution + NGD: the natural gradients and the hyper-parameter gradients of one step"""
    from dsvgp_b200 import gp
    n, d, M = 300, 3, 40
    P, x, _, y, num_data = S.make_problem(n, d, M, 0, F64, seed=8, variant="svgp", N=10 * n)
    g = torch.Generator().manual_seed(8)
    B = torch.eye(M, dtype=F64) + 0.1 * torch.randn(M, M, generator=g, dtype=F64).tril()
    Sq = B @ B.T
    nat_mat, nat_vec = -0.5 * torch.linalg.inv(Sq), torch.linalg.solve(Sq, 0.2 * torch.randn(M, generator=g, dtype=F64))
    model, lik = build_svgp(P, F64, ngd=True)
    vd = model.variational_strategy._variational_distribution
    with torch.no_grad():
        vd.natural_vec.copy_(nat_vec), vd.natural_mat.copy_(nat_mat)
    model.train(), lik.train()
    mll = gp.VariationalELBO(lik, model, num_data=num_data)
    loss = -mll(lik(model(x.cuda())), y.cuda())
    loss.backward()
    ref_val, ref = S.ngd_elbo_and_grads(P, nat_vec, nat_mat, x, None, y, num_data, variant="svgp")
    assert abs(float(-loss) - float(ref_val)) < 1e-10 * abs(float(ref_val))
    assert rel(-vd.natural_vec.grad, ref["natural_vec"]) < 1e-10
    assert rel(-vd.natural_mat.grad, ref["natural_mat"]) < 1e-10
    got = grads_of(model, lik)
    for k in ("Z", "c", "raw_os", "raw_ell", "raw_noise"):
        assert rel(-got[k], ref[k]) < 1e-10, k
    opt = gp.NGD(model.variational_parameters(), num_data=num_data, lr=0.1)
    before = vd.natural_vec.detach().clone()
    opt.step()
    assert rel(vd.natural_vec.detach() - before, -0.1 * num_data * vd.natural_vec.grad) < 1e-12


@pytest.mark.parametrize("M,n,dtype", [(128, 512, F32), (64, 256, F64)])
def test_svgp_graph_replay_equals_eager(M, n, dtype):
    from dsvgp_b200 import gp
    from dsvgp_b200.graphs import GraphedStep
    P, x, _, y, nd = S.make_problem(n, 5, M, 0, dtype, seed=M, variant="svgp", N=10 * n)
    model, lik = build_svgp(P, dtype)
    model.train(), lik.train()
    mll = gp.VariationalELBO(lik, model, num_data=nd)
    params = [q for q in list(model.parameters()) + list(lik.parameters())]
    _, x2, _, y2, _ = S.make_problem(n, 5, M, 0, dtype, seed=M + 1, variant="svgp", N=10 * n)
    x2, y2 = x2.cuda(), y2.cuda()

    def eager():
        for q in params:
            q.grad = None
        loss = -mll(lik(model(x2)), y2)
        loss.backward()
        return loss.detach().clone(), [q.grad.clone() for q in params]
    loss_e, g_e = eager()
    step = GraphedStep(model, lik, mll, x.cuda(), None, y.cuda())
    for _ in range(2):
        loss_g = step(x2, None, y2)
        assert torch.equal(loss_g, loss_e)
        for q, ge in zip(params, g_e):
            assert torch.equal(q.grad, ge)
    assert step.fallbacks == 0


@pytest.mark.parametrize("dtype", [F64, F32])
def test_svgp_two_forwards_then_one_backward(dtype):
    from dsvgp_b200 import gp
    n, d, M = 96, 3, 24
    P, x, _, y, nd = S.make_problem(2 * n, d, M, 0, dtype, seed=9, variant="svgp", N=5000)
    model, lik = build_svgp(P, dtype)
    model.train(), lik.train()
    mll = gp.VariationalELBO(lik, model, num_data=nd)
    l1 = mll(lik(model(x[:n].cuda())), y[:n].cuda())
    l2 = mll(lik(model(x[n:].cuda())), y[n:].cuda())
    (l1 + l2).backward()
    got = grads_of(model, lik)
    tot = None
    for sl in (slice(0, n), slice(n, 2 * n)):
        _, g = S.elbo_and_grads(P.clone(F64), _up(x[sl]), None, _up(y[sl]), nd, variant="svgp")
        tot = g if tot is None else {a: tot[a] + g[a] for a in g}
    for k, g in tot.items():
        assert rel(got[k], g) < (1e-9 if dtype == F64 else 1e-4), k


@pytest.mark.parametrize("dtype,M,n", [(F64, 96, 300), (F32, 512, 1024)])
def test_svgp_sharded_tail_equals_replicated_tail(dtype, M, n):
    """the N > 1 form of the Cholesky-backward tail (column panels of dK_zz, q = 1 column per inducing point) for both ranks
    of a world of two in one process"""
    from dsvgp_b200 import engine, gp
    P, x, _, y, nd = S.make_problem(n, 10, M, 0, dtype, seed=11, variant="svgp", N=50000)
    model, lik = build_svgp(P, dtype)
    mll = gp.VariationalELBO(lik, model, num_data=nd)
    params = list(model.parameters()) + list(lik.parameters())
    xc, yc = x.cuda(), y.cuda()

    def grads():
        for q in params:
            q.grad = None
        loss = -mll(lik(model(xc)), yc)
        loss.backward()
        return float(loss), torch.cat([q.grad.reshape(-1).double() for q in params])
    l0, g0 = grads()
    engine.ENGINE.tail_shards_debug = 2
    try:
        l1, g1 = grads()
    finally:
        engine.ENGINE.tail_shards_debug = None
    assert l0 == l1
    assert float((g1 - g0).abs().max() / g0.abs().max()) < (1e-11 if dtype == F64 else 2e-6)


def _sharded_worker(rank, world, port, out):
    import os
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from dsvgp_b200 import distributed, gp
        n = 1024
        P, x, _, y, nd = S.make_problem(n, 10, 256, 0, F32, seed=5, variant="svgp", N=50000)

        def grads(xs, ys, sharded):
            model, lik = build_svgp(P, F32)
            if sharded:
                distributed.enable(model, n)
            mll = gp.VariationalELBO(lik, model, num_data=nd)
            loss = -mll(lik(model(xs.cuda())), ys.cuda())
            loss.backward()
            distributed.disable(model)
            return float(loss), torch.cat([q.grad.reshape(-1).double() for q in list(model.parameters()) + list(lik.parameters())])
        lo, hi = distributed.shard_bounds(n, rank, world)
        l_s, g_s = grads(x[lo:hi], y[lo:hi], True)
        l_f, g_f = grads(x, y, False)
        assert abs(l_s - l_f) < 1e-5 * abs(l_f), (l_s, l_f)
        assert float((g_s - g_f).abs().max() / g_f.abs().max()) < 1e-4
        out[rank] = "ok"
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_svgp_sharded_step_two_gpus():
    import torch.multiprocessing as mp
    from test_multigpu import _free_port
    out = mp.Manager().dict()
    mp.spawn(_sharded_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    assert dict(out) == {0: "ok", 1: "ok"}


def test_svgp_state_dict_and_strategy_interface():
    import traditional_vi
    from dsvgp_b200 import gp
    P, x, _, y, nd = S.make_problem(64, 3, 16, 0, F32, seed=1, variant="svgp")
    model, lik = build_svgp(P, F32)
    keys = set(model.state_dict())
    assert keys == {"variational_strategy.inducing_points", "variational_strategy.variational_params_initialized",
                    "variational_strategy.updated_strategy", "variational_strategy._variational_distribution.variational_mean",
                    "variational_strategy._variational_distribution.chol_variational_covar", "mean_module.constant",
                    "covar_module.raw_outputscale", "covar_module.base_kernel.raw_lengthscale"}
    assert model.covar_module.base_kernel.raw_lengthscale.shape == (1, 1)
    vs = model.variational_strategy
    assert vs._p() == 0 and vs._directions() is None
    with pytest.raises(TypeError):
        model(x.cuda(), derivative_directions=torch.eye(3).repeat(64, 1))
    model.eval(), lik.eval()
    with torch.no_grad():
        p1 = lik(model(x.cuda()))
        m1, v1 = p1.mean.clone(), p1.variance.clone()
    fresh, _ = build_svgp(S.make_problem(64, 3, 16, 0, F32, seed=2, variant="svgp")[0], F32)
    fresh.load_state_dict(model.state_dict())
    fresh.eval()
    with torch.no_grad():
        p2 = lik(fresh(x.cuda()))
        assert torch.equal(p2.mean, m1) and torch.equal(p2.variance, v1)
    # prior path and the kernel module itself
    prior = model(x.cuda(), prior=True)
    ell, osc = float(softplus_(P.raw_ell)), float(softplus_(P.raw_os))
    Kref = osc * O.kernel_closed_form(x.double(), x.double(), None, None, torch.tensor(ell, dtype=F64))
    assert rel(prior.covariance_matrix, Kref) < 2e-6
    k = gp.RBFKernel().cuda()
    assert torch.equal(k(x.cuda(), diag=True), torch.ones(64, device="cuda"))
    # legacy checkpoint (before the whitened parameterisation): re-whitened once on the first call
    sd = model.state_dict()
    del sd["variational_strategy.updated_strategy"]
    legacy = traditional_vi.GPModel(P.Z.clone()).cuda()
    with pytest.warns(gp.OldVersionWarning):
        legacy.load_state_dict(sd)
    legacy.eval()
    with torch.no_grad():
        legacy(x.cuda()).mean
    assert bool(legacy.variational_strategy.updated_strategy)


def softplus_(t):
    return torch.nn.functional.softplus(t.double()).reshape(())


def test_traditional_vi_train_gp_first_step_and_eval_gp(monkeypatch):
    """train_gp for 20 steps on testfun data: its first step equals the oracle's step on the same parameters and minibatch;
    eval_gp returns (N,) means and variances"""
    import directional_vi
    import traditional_vi
    from dsvgp_b200 import gp
    from torch.utils.data import TensorDataset
    N, d = 400, 3
    g = torch.Generator().manual_seed(0)
    X = torch.rand(N, d, generator=g)
    ds = TensorDataset(X, O.testfun(X.double())[:, 0].float())
    seen = {}
    real_opt, real_batches, real_fwd = directional_vi._optimizers, directional_vi._batches, gp.VariationalELBO.forward

    def batches(*a, **k):
        for xb, yb in real_batches(*a, **k):
            seen.setdefault("batch", (xb.clone(), yb.clone()))
            yield xb, yb

    def fwd(self, dist, target, **kw):
        val = real_fwd(self, dist, target, **kw)
        seen.setdefault("elbo", float(val))
        seen.setdefault("num_data", self.num_data)
        return val

    def optimizers(model, likelihood, *a, **k):
        vopt, hopt, vs, hs = real_opt(model, likelihood, *a, **k)
        step = vopt.step

        def first_step(*sa, **sk):
            if "params" not in seen:
                sd = {k2: v.detach().clone() for k2, v in model.named_parameters()}
                gr = {k2: v.grad.detach().clone() for k2, v in model.named_parameters()}
                seen["params"] = (sd, gr, likelihood.noise_covar.raw_noise.detach().clone(),
                                  likelihood.noise_covar.raw_noise.grad.detach().clone())
            return step(*sa, **sk)
        vopt.step = first_step
        return vopt, hopt, vs, hs
    monkeypatch.setattr(directional_vi, "_optimizers", optimizers)
    monkeypatch.setattr(directional_vi, "_batches", batches)
    monkeypatch.setattr(gp.VariationalELBO, "forward", fwd)
    torch.manual_seed(0)
    model, lik = traditional_vi.train_gp(ds, d, num_inducing=32, minibatch_size=20, num_epochs=1, verbose=False)
    assert seen["num_data"] == N
    sd, gr, raw_noise, g_noise = seen["params"]
    P = S.Params(Z=sd[KEYMAP["Z"]], Vz=None, m=sd[KEYMAP["m"]], Ls_raw=sd[KEYMAP["Ls_raw"]], c=sd[KEYMAP["c"]],
                 raw_os=sd[KEYMAP["raw_os"]], raw_ell=sd[KEYMAP["raw_ell"]], raw_noise=raw_noise).clone(F64)
    xb, yb = seen["batch"]
    ref_val, ref_grads = S.elbo_and_grads(_cpu(P), _up(xb).cpu(), None, _up(yb).cpu(), N, variant="svgp")
    grads = {k: -gr[name] for k, name in KEYMAP.items()}
    grads["raw_noise"] = -g_noise
    check_against(seen["elbo"], grads, ref_val, ref_grads, 1e-4, 1e-4)
    with pytest.raises(ValueError):
        traditional_vi.train_gp(TensorDataset(X, O.testfun(X.double()).float()), d, num_inducing=8, verbose=False)
    with pytest.raises(NotImplementedError):
        traditional_vi.train_gp(ds, d, use_ciq=True)
    means, variances = traditional_vi.eval_gp(ds, model, lik, minibatch_size=64)
    assert means.shape == (N,) and variances.shape == (N,)
    assert bool(torch.isfinite(means).all()) and bool((variances > 0).all())


def _cpu(P):
    return S.Params(**{k: (None if t is None else t.cpu()) for k, t in P.tensors().items()})
