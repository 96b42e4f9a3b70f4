"""GPU parity of the whole hot path through the reference-facing API (GPModel / likelihood / VariationalELBO, i.e.
through the C ABI), against (a) golden vectors produced by the unmodified reference files, (b) the CPU oracle on
seeded inputs, and (c) size-independent properties at BASELINE.json's full shapes.

Tolerances are north_star's: relative 1e-10 in fp64 and 1e-4 in fp32 on the ELBO, every parameter gradient
(max-norm relative per tensor) and the predictive mean / variance.  fp32 results are compared with the fp64
oracle on the same (fp32-representable) inputs, as SURVEY.md Q8 prescribes."""
import os
import types

import pytest
import torch

from oracle import dsvgp_oracle as O

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
F32, F64 = torch.float32, torch.float64
KEYMAP = {"Z": "variational_strategy.inducing_points", "Vz": "variational_strategy.inducing_directions",
          "m": "variational_strategy._variational_distribution.variational_mean",
          "Ls_raw": "variational_strategy._variational_distribution.chol_variational_covar",
          "c": "mean_module.constant", "raw_os": "covar_module.raw_outputscale",
          "raw_ell": "covar_module.base_kernel.raw_lengthscale"}


def rel(a, b):
    a, b = a.detach().double().cpu().reshape(-1), b.detach().double().cpu().reshape(-1)
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-300))


def build(variant, P, d, dtype):
    """The reference-facing objects, loaded with the parameters of an oracle Params."""
    import dfree_directional_vi
    import directional_vi
    import grad_svgp
    from dsvgp_b200 import gp
    cpu = lambda t: t.detach().to(dtype).cpu()
    if variant == "dsvgp":
        model = directional_vi.GPModel(cpu(P.Z), cpu(P.Vz), d)
    elif variant == "dfree":
        model = dfree_directional_vi.GPModel(cpu(P.Z), cpu(P.Vz), d)
    else:
        model = grad_svgp.GPModel(cpu(P.Z))
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


def grads_of(model, lik):
    sd = dict(model.named_parameters())
    out = {k: sd[name].grad for k, name in KEYMAP.items() if name in sd}
    out["raw_noise"] = lik.noise_covar.raw_noise.grad
    return out


def run_step(variant, P, x, Vx, y, num_data, d, dtype):
    from dsvgp_b200 import gp
    model, lik = build(variant, P, d, dtype)
    model.train(), lik.train()
    mll = gp.VariationalELBO(lik, model, num_data=num_data)
    kw = {} if variant == "grad" else {"derivative_directions": Vx.to(dtype)}     # CPU tensor, as eval_gp passes it
    out = lik(model(x.to(dtype).cuda(), **kw))
    loss = -mll(out, y.to(dtype).cuda())
    loss.backward()
    return model, lik, -loss.detach(), {k: -g for k, g in grads_of(model, lik).items()}, out


def check_against(val, grads, ref_val, ref_grads, t_val, t_grad):
    assert abs(float(val) - float(ref_val)) <= t_val * abs(float(ref_val)), (float(val), float(ref_val))
    for k, g in ref_grads.items():
        assert k in grads and grads[k] is not None, k
        r = rel(grads[k], g)
        assert r < t_grad, (k, r)


@pytest.mark.parametrize("name", ["dsvgp_c1_f64", "dsvgp_c1_f32", "dsvgp_c1_canonical_f64", "dsvgp_d3_p1_f64",
                                  "dsvgp_d6_p3_f64", "dfree_d4_p2_f64", "dfree_d4_p2_f32", "grad_d2_f64", "grad_d3_f32"])
def test_step_matches_unmodified_reference_golden(name):
    c = torch.load(os.path.join(GOLD, "step_cases.pt"))[name]
    dtype = c["x"].dtype
    P = O.Params(**c["params"])
    model, lik, val, grads, out = run_step(c["variant"], P, c["x"], c["Vx"], c["y"], c["num_data"], c["d"], dtype)
    f64 = dtype == F64
    check_against(val, grads, c["elbo"], c["grads"], 1e-10 if f64 else 1e-4, 1e-10 if f64 else 1e-4)
    assert rel(out.mean, c["train_mean"]) < (1e-10 if f64 else 1e-4)
    assert rel(out.variance, c["train_variance"]) < (1e-10 if f64 else 1e-4)
    model.eval(), lik.eval()
    with torch.no_grad():
        kw = {} if c["variant"] == "grad" else {"derivative_directions": c["Vx"]}
        for _ in range(2):          # second call reuses the memoised factor
            preds = lik(model(c["x"].cuda(), **kw))
            assert rel(preds.mean, c["pred_mean"]) < (1e-10 if f64 else 1e-4)
            assert rel(preds.variance, c["pred_variance"]) < (1e-10 if f64 else 1e-4)
        assert rel(preds.covariance_matrix, c["pred_covariance"]) < (1e-10 if f64 else 1e-4)


@pytest.mark.parametrize("name", ["dsvgp_c1_f64", "dsvgp_c1_f32", "dsvgp_d6_p3_f64", "dfree_d4_p2_f64", "dfree_d4_p2_f32",
                                  "grad_d2_f64", "grad_d3_f32"])
def test_pll_step_matches_unmodified_reference_golden(name):
    """mll_type="PLL" exactly as the reference loop drives it: PredictiveLogLikelihood on likelihood(model(x))."""
    from dsvgp_b200 import gp
    c = torch.load(os.path.join(GOLD, "step_cases.pt"))[name]
    dtype, f64 = c["x"].dtype, c["x"].dtype == F64
    model, lik = build(c["variant"], O.Params(**c["params"]), c["d"], dtype)
    model.train(), lik.train()
    mll = gp.PredictiveLogLikelihood(lik, model, num_data=c["num_data"])
    kw = {} if c["variant"] == "grad" else {"derivative_directions": c["Vx"]}
    out = lik(model(c["x"].cuda(), **kw))
    loss = -mll(out, c["y"].cuda())
    loss.backward()
    grads = {k: -g for k, g in grads_of(model, lik).items()}
    # fp32 fixtures hold the reference's OWN fp32 arithmetic, itself only good to a few 1e-5 (tests/test_oracle.py), so
    # two independent fp32 evaluations are compared at 2e-4 here and the fp32 kernels at 1e-4 against the fp64 oracle
    check_against(-loss.detach(), grads, c["pll"], c["pll_grads"], 1e-10 if f64 else 1e-4, 1e-10 if f64 else 2e-4)
    if not f64:
        up = lambda t: None if t is None else t.double()
        ref_val, ref_grads = O.pll_and_grads(O.Params(**c["params"]).clone(F64), up(c["x"]), up(c["Vx"]), up(c["y"]),
                                             c["num_data"], c["variant"], noise_mult=2)
        check_against(-loss.detach(), grads, ref_val, ref_grads, 1e-4, 1e-4)
    assert rel(out.mean, c["train_mean"]) < (1e-10 if f64 else 1e-4)          # what the loop prints (:256-257):
    assert rel(out.variance, c["train_variance"]) < (1e-10 if f64 else 1e-4)  # ONE noise, not log_marginal's two


CASES = [  # variant, n, d, M, p, dtype
    ("dsvgp", 200, 2, 20, 2, F32),          # C1 as shipped (tests/test_dsvgp.py:21-29)
    ("dsvgp", 200, 2, 20, 2, F64),
    ("dsvgp", 500, 3, 128, 1, F64),         # C2-shaped, reduced M
    ("dsvgp", 333, 10, 96, 2, F32),         # C3-shaped, reduced M
    ("dsvgp", 333, 10, 96, 2, F64),
    ("dsvgp", 130, 60, 40, 3, F32),         # C4-shaped, reduced M
    ("dsvgp", 130, 60, 40, 3, F64),
    ("dfree", 257, 18, 64, 2, F32),         # C5-shaped, reduced M
    ("dfree", 257, 18, 64, 2, F64),
    ("grad", 90, 3, 33, 3, F64),
    ("grad", 40, 5, 12, 5, F64),            # p = d > 3: runtime-p kernels
    ("dsvgp", 1, 2, 3, 1, F64),             # single point
    ("dsvgp", 65, 4, 29, 1, F32),           # M' = 58: padded Cholesky block
    ("dsvgp", 95, 5, 43, 2, F32),           # tcgen05 path at ragged sizes: M' = 129, n' = 285
    ("dsvgp", 300, 3, 65, 1, F32),          # M' = 130, n' = 600
    ("dfree", 270, 7, 50, 2, F32),          # M' = 150, n' = 270 (values only)
]


@pytest.mark.parametrize("variant,n,d,M,p,dtype", CASES)
def test_step_matches_oracle(variant, n, d, M, p, dtype):
    P, x, Vx, y, num_data = O.make_problem(n, d, M, p, dtype, seed=n + d + M, variant=variant, N=10 * n)
    up = lambda t: None if t is None else t.double()
    P64 = P.clone(F64)
    ref_val, ref_grads = O.elbo_and_grads(P64, up(x), up(Vx), up(y), num_data, variant)
    model, lik, val, grads, out = run_step(variant, P, x, Vx, y, num_data, d, dtype)
    f64 = dtype == F64
    check_against(val, grads, ref_val, ref_grads, 1e-10 if f64 else 1e-4, 1e-10 if f64 else 1e-4)
    mean, var = O.predict(P64, up(x), up(Vx), variant)
    assert rel(out.mean, mean) < (1e-10 if f64 else 1e-4)
    assert rel(out.variance, var) < (1e-10 if f64 else 1e-4)
    model.eval(), lik.eval()
    with torch.no_grad():
        kw = {} if variant == "grad" else {"derivative_directions": Vx}
        preds = lik(model(x.cuda(), **kw))
    assert rel(preds.mean, mean) < (1e-10 if f64 else 1e-4)
    assert rel(preds.variance, var) < (1e-10 if f64 else 1e-4)


def test_elbo_on_model_output_is_textbook_value():
    """Q3: ELBO(likelihood(model(x))) = ELBO(model(x)) - 0.5 exactly; gradients identical."""
    from dsvgp_b200 import gp
    P, x, Vx, y, nd = O.make_problem(64, 3, 16, 2, F64, 3)
    model, lik = build("dsvgp", P, 3, F64)
    mll = gp.VariationalELBO(lik, model, num_data=nd)
    a = mll(lik(model(x.cuda(), derivative_directions=Vx)), y.cuda())
    a.backward()
    ga = {k: g.clone() for k, g in grads_of(model, lik).items()}
    model.zero_grad(), lik.zero_grad()
    out = model(x.cuda(), derivative_directions=Vx)
    b = mll(out, y.cuda())
    b.backward()
    assert abs(float(a) - (float(b) - 0.5)) < 1e-12
    for k, g in grads_of(model, lik).items():
        assert rel(g, ga[k]) < 1e-11, k
    assert rel(out.variance, O.predictive(P, x, Vx)[1]) < 1e-10          # no noise on model(x)


def test_differentiable_mean_variance_and_pll():
    """Generic autograd path: PredictiveLogLikelihood (mll_type='PLL') against oracle autograd."""
    from dsvgp_b200 import gp
    P, x, Vx, y, nd = O.make_problem(80, 4, 24, 2, F64, 5)
    model, lik = build("dsvgp", P, 4, F64)
    mll = gp.PredictiveLogLikelihood(lik, model, num_data=nd)
    val = mll(model(x.cuda(), derivative_directions=Vx), y.cuda())
    val.backward()
    Q = P.clone().requires_grad_(True)
    mean, var = O.predictive(Q, x, Vx)
    var = var + O.noise(Q)
    ref = (-0.5 * ((y - mean) ** 2 / var + var.log() + torch.log(torch.tensor(2 * torch.pi, dtype=F64)))).sum() / mean.numel() \
        - O.kl_divergence(Q) / nd
    ref.backward()
    assert abs(float(val) - float(ref)) < 1e-10 * abs(float(ref))
    for k, g in grads_of(model, lik).items():
        assert rel(g, getattr(Q, k).grad) < 1e-9, k


def test_training_reduces_loss_and_checkpoint_roundtrip(tmp_path):
    """A few Adam steps through train_gp on the shipped test function (tests/test_dsvgp.py shapes), then
    state_dict save / load / identical predictions."""
    import directional_vi
    from dsvgp_b200 import gp
    torch.manual_seed(0)
    x = torch.rand(600, 2)
    ds = torch.utils.data.TensorDataset(x, O.testfun(x.double()).float())
    model, lik = directional_vi.train_gp(ds, num_inducing=20, num_directions=2, minibatch_size=200, minibatch_dim=2,
                                         num_epochs=40, inducing_data_initialization=False, verbose=False)
    xt = torch.rand(1000, 2)
    yt = O.testfun(xt.double()).float()
    means, variances = directional_vi.eval_gp(torch.utils.data.TensorDataset(xt, yt), model, lik, num_directions=2,
                                              minibatch_size=1000, minibatch_dim=2)
    assert means.shape == (3000,) and variances.shape == (3000,) and bool((variances > 0).all())
    mse0 = float(((yt[:, 0] - yt[:, 0].mean()) ** 2).mean())
    mse = float(((yt[:, 0] - means[::3]) ** 2).mean())
    assert mse < 0.9 * mse0, (mse, mse0)          # 120 steps already beat the constant predictor
    torch.save({"m": model.state_dict(), "l": lik.state_dict()}, tmp_path / "ck.pt")
    ck = torch.load(tmp_path / "ck.pt")
    m2 = directional_vi.GPModel(torch.rand(20, 2), torch.eye(2).repeat(20, 1), 2).cuda()
    l2 = gp.GaussianLikelihood().cuda()
    m2.load_state_dict(ck["m"]), l2.load_state_dict(ck["l"])
    means2, variances2 = directional_vi.eval_gp(torch.utils.data.TensorDataset(xt, yt), m2, l2, num_directions=2,
                                                minibatch_size=400, minibatch_dim=2)      # ragged last batch
    assert rel(means2, means) < 1e-5 and rel(variances2, variances) < 1e-5


def test_eval_factor_cache_is_per_model_and_follows_parameters():
    """Eval-mode memoisation of the Cholesky factor (DGVS.py:72) must not leak between two models of the same shape,
    and must be dropped when parameters change in place or train() is called."""
    P1, x, Vx, y, nd = O.make_problem(40, 3, 12, 2, F64, 21)
    P2, _, _, _, _ = O.make_problem(40, 3, 12, 2, F64, 22)
    m1, l1 = build("dsvgp", P1, 3, F64)
    m2, l2 = build("dsvgp", P2, 3, F64)
    for m, l in ((m1, l1), (m2, l2)):
        m.eval(), l.eval()
    with torch.no_grad():
        a1 = l1(m1(x.cuda(), derivative_directions=Vx)).mean
        a2 = l2(m2(x.cuda(), derivative_directions=Vx)).mean
        b1 = l1(m1(x.cuda(), derivative_directions=Vx)).mean
    assert rel(a1, O.predict(P1, x, Vx)[0]) < 1e-10 and rel(a2, O.predict(P2, x, Vx)[0]) < 1e-10 and rel(b1, a1) < 1e-14
    with torch.no_grad():
        m1.variational_strategy.inducing_points.add_(0.01)
        P1.Z = P1.Z + 0.01
        c1 = l1(m1(x.cuda(), derivative_directions=Vx)).mean
    assert rel(c1, O.predict(P1, x, Vx)[0]) < 1e-10


def test_cholesky_jitter_ladder_and_errors():
    """psd_safe_cholesky semantics: duplicate inducing points + tiny outputscale still factorise thanks to the 1e-3
    jitter; NaN parameters raise NanError; an indefinite matrix raises NotPSDError."""
    from dsvgp_b200 import engine, gp
    P, x, Vx, y, nd = O.make_problem(30, 2, 8, 1, F64, 2)
    P.Z[1] = P.Z[0]
    P.Vz[1] = P.Vz[0]
    model, lik = build("dsvgp", P, 2, F64)
    mll = gp.VariationalELBO(lik, model, num_data=nd)
    v = mll(lik(model(x.cuda(), derivative_directions=Vx)), y.cuda())
    ref = O.elbo(P, x, Vx, y, nd)
    assert abs(float(v) - float(ref)) < 1e-8 * abs(float(ref))
    with torch.no_grad():
        model.variational_strategy.inducing_points[0, 0] = float("nan")
    with pytest.raises(engine.NanError):
        mll(lik(model(x.cuda(), derivative_directions=Vx)), y.cuda())


@pytest.mark.parametrize("variant,n,d,M,p,dtype", [
    ("dsvgp", 500, 3, 512, 1, F64),         # C2 bunny-shaped: full M, the reference's minibatch (bunny.sub:22), fp64
    ("dsvgp", 512, 10, 1024, 2, F32),       # C3 synthetic1-shaped: full M, the reference's minibatch, tcgen05 path
    ("dsvgp", 1024, 10, 1024, 2, F32),
    ("dsvgp", 512, 60, 800, 3, F32),        # C4 rover-shaped, full M
    ("dfree", 512, 18, 1024, 2, F32),       # C5 uci_dfree-shaped, full M
])
def test_full_size_matches_oracle(variant, n, d, M, p, dtype):
    """BASELINE.json's full inducing sizes at the reference's own minibatch sizes against the fp64 CPU oracle
    (1-2 s of oracle time each on the GPU box's host cores)."""
    P, x, Vx, y, num_data = O.make_problem(n, d, M, p, dtype, seed=1, variant=variant, N=100 * n)
    up = lambda t: None if t is None else t.double()
    P64 = P.clone(F64)
    ref_val, ref_grads = O.elbo_and_grads(P64, up(x), up(Vx), up(y), num_data, variant)
    model, lik, val, grads, out = run_step(variant, P, x, Vx, y, num_data, d, dtype)
    f64 = dtype == F64
    check_against(val, grads, ref_val, ref_grads, 1e-10 if f64 else 1e-4, 1e-10 if f64 else 1e-4)
    mean, var = O.predict(P64, up(x), up(Vx), variant)
    assert rel(out.mean, mean) < (1e-10 if f64 else 1e-4)
    assert rel(out.variance, var) < (1e-10 if f64 else 1e-4)


@pytest.mark.parametrize("variant,n,d,M,p,dtype", [
    ("dsvgp", 2048, 3, 512, 1, F64),        # C2 bunny-shaped, full M
    ("dsvgp", 2048, 10, 1024, 2, F32),      # C3 synthetic1-shaped, full M
    ("dsvgp", 1024, 60, 800, 3, F32),       # C4 rover-shaped, full M
    ("dfree", 2048, 18, 1024, 2, F32),      # C5 uci_dfree-shaped, full M
])
def test_full_size_properties(variant, n, d, M, p, dtype):
    """At BASELINE.json's full inducing sizes the oracle is too slow for CI, so check size-independent properties:
    (1) the gradient agrees with a central finite difference of the ELBO along a random direction,
    (2) the data term is additive over a split of the minibatch (what multi-GPU sharding relies on),
    (3) eval-mode prediction equals the train-mode mean / variance."""
    from dsvgp_b200 import gp
    from dsvgp_b200.engine import ENGINE
    P, x, Vx, y, nd = O.make_problem(n, d, M, p, dtype, seed=1, variant=variant, N=100 * n)
    model, lik, val, grads, out = run_step(variant, P, x, Vx, y, nd, d, dtype)
    assert torch.isfinite(val) and all(torch.isfinite(g).all() for g in grads.values())
    # (1) directional finite difference in fp64 arithmetic of the same model (fp32 model: loose)
    names = ["Z", "Vz", "m", "c", "raw_os", "raw_ell", "raw_noise"]
    g = torch.Generator().manual_seed(0)
    delta = {k: torch.randn(getattr(P, k).shape, generator=g, dtype=F64) for k in names}
    h = 1e-5 if dtype == F64 else 2e-3
    vals = []
    for s in (+1, -1):
        Q = P.clone(F64)
        for k in names:
            setattr(Q, k, (getattr(Q, k) + s * h * delta[k]).to(dtype))
        _, _, v, _, _ = run_step(variant, Q, x, Vx, y, nd, d, dtype)
        vals.append(float(v))
    fd = (vals[0] - vals[1]) / (2 * h)
    an = sum(float((grads[k].double().cpu().reshape(-1) * delta[k].reshape(-1)).sum()) for k in names)
    assert abs(fd - an) < (1e-6 if dtype == F64 else 3e-2) * max(1.0, abs(an)), (fd, an)
    # (2) additivity of the data term over a split (KL counted once)
    mll = gp.VariationalELBO(lik, model, num_data=nd)
    h1 = n // 2
    q = p + 1 if variant != "dfree" else 1
    kw = lambda sl: {} if variant == "grad" else {"derivative_directions": Vx[sl.start * p: sl.stop * p].to(dtype)}
    with torch.no_grad():
        parts = []
        for sl in (slice(0, h1), slice(h1, n)):
            parts.append(float(mll(lik(model(x[sl].to(dtype).cuda(), **kw(sl))), y[sl.start * q: sl.stop * q].to(dtype).cuda())))
        kl = float(model.variational_strategy.kl_divergence()) / nd
    whole = float(val)
    combined = (parts[0] + kl) * h1 / n + (parts[1] + kl) * (n - h1) / n - kl
    assert abs(whole - combined) < (1e-11 if dtype == F64 else 2e-5) * abs(whole), (whole, combined)
    # (3) eval path (B^2 - A^2 reduction, memoised factor) equals the train path
    model.eval(), lik.eval()
    with torch.no_grad():
        preds = lik(model(x.to(dtype).cuda(), **({} if variant == "grad" else {"derivative_directions": Vx.to(dtype)})))
    assert rel(preds.mean, out.mean) < (1e-12 if dtype == F64 else 1e-5)
    assert rel(preds.variance, out.variance) < (1e-11 if dtype == F64 else 1e-4)


# -------------------------------------------------------- full predictive covariance + sampling (section 8f rank 4)
@pytest.mark.parametrize("variant,n,d,M,p,dtype", [
    ("dsvgp", 120, 3, 40, 1, F64), ("dsvgp", 150, 10, 64, 2, F32), ("dsvgp", 300, 10, 128, 2, F32),
    ("dfree", 100, 6, 32, 2, F64), ("grad", 40, 3, 20, 3, F64), ("dsvgp", 96, 60, 50, 3, F32)])
def test_full_predictive_covariance_matches_oracle(variant, n, d, M, p, dtype):
    P, x, Vx, y, num_data = O.make_problem(n, d, M, p, dtype, seed=7 + n, variant=variant, N=10 * n)
    up = lambda t: None if t is None else t.double()
    model, lik = build(variant, P, d, dtype)
    model.eval(), lik.eval()
    kw = {} if variant == "grad" else {"derivative_directions": Vx}
    t = 1e-10 if dtype == F64 else 1e-4
    with torch.no_grad():
        for noisy in (False, True):
            dist = model(x.cuda(), **kw)
            dist = lik(dist) if noisy else dist
            mean, cov = O.predictive_full(P.clone(F64), up(x), up(Vx), variant, add_noise=noisy)
            assert rel(dist.mean, mean) < t
            assert rel(dist.covariance_matrix, cov) < t
            assert rel(dist.covariance_matrix.diagonal(), dist.variance) < 10 * t     # same thing two ways
            assert dist.lazy_covariance_matrix.shape == (mean.numel(), mean.numel())


@pytest.mark.parametrize("variant,n,d,M,p,dtype,noisy", [
    ("dsvgp", 60, 3, 40, 1, F64, False), ("dsvgp", 90, 10, 64, 2, F32, True), ("dfree", 80, 6, 32, 2, F64, True),
    ("grad", 30, 3, 20, 3, F64, False), ("dsvgp", 700, 10, 192, 2, F32, False)])
def test_gradients_through_the_full_predictive_covariance(variant, n, d, M, p, dtype, noisy):
    """The reference's predictive covariance is a differentiable lazy tensor (DGVS.py:192-208): a scalar of (mean, dense
    covariance) -- random, NON-symmetric weights on the covariance -- must give the oracle's parameter gradients."""
    P, x, Vx, y, num_data = O.make_problem(n, d, M, p, dtype, seed=11 + n, variant=variant, N=10 * n)
    up = lambda t: None if t is None else t.double()
    model, lik = build(variant, P, d, dtype)
    model.train(), lik.train()                  # (training mode: a fresh factorisation, as an acquisition optimiser would run it)
    kw = {} if variant == "grad" else {"derivative_directions": Vx}
    dist = model(x.cuda(), **kw)
    dist = lik(dist) if noisy else dist
    cov, mean = dist.covariance_matrix, dist.mean
    assert cov.requires_grad and mean.requires_grad
    nq = mean.numel()
    g = torch.Generator().manual_seed(5)
    Wc = torch.randn(nq, nq, generator=g, dtype=torch.float64) / nq
    wm = torch.randn(nq, generator=g, dtype=torch.float64)
    val = (cov * Wc.to(dtype).cuda()).sum() + (mean * wm.to(dtype).cuda()).sum()
    val.backward()
    Q = P.clone(F64).requires_grad_(True)
    rmean, rcov = O.predictive_full(Q, up(x), up(Vx), variant, add_noise=noisy)
    rval = (rcov * Wc).sum() + (rmean * wm).sum()
    names = [k for k, t_ in Q.tensors().items() if not (variant == "grad" and k == "Vz")]
    rg = torch.autograd.grad(rval, [getattr(Q, k) for k in names], allow_unused=True)
    ref = {k: (gk if gk is not None else torch.zeros_like(getattr(Q, k))) for k, gk in zip(names, rg)}
    t = 1e-9 if dtype == F64 else 1e-4
    assert abs(float(val.detach()) - float(rval.detach())) <= t * abs(float(rval.detach()))
    got = grads_of(model, lik)
    for k, gk in ref.items():
        if k == "raw_noise" and not noisy:
            continue
        if float(gk.abs().max()) == 0.0:
            assert got.get(k) is None or float(got[k].abs().max()) == 0.0, k
            continue
        assert got.get(k) is not None, k
        r = rel(got[k], gk)
        assert r < t, (k, r)
    # a second evaluation on the same shape invalidates a pending backward instead of corrupting it
    d1 = model(x.cuda(), **kw)
    c1 = d1.covariance_matrix
    d2 = model(x.cuda(), **kw)
    _ = d2.covariance_matrix
    with pytest.raises(RuntimeError):
        c1.sum().backward()


def test_samples_follow_the_predictive_distribution():
    """preds.sample(torch.Size([n_samples])) (experiments/rover/test_turbo.py:138): shape, and first two moments of
    many draws against the oracle's mean / covariance (statistical tolerance)."""
    variant, n, d, M, p, dtype = "dsvgp", 12, 4, 30, 2, F32
    P, x, Vx, y, num_data = O.make_problem(n, d, M, p, dtype, seed=3, variant=variant, N=10 * n)
    model, lik = build(variant, P, d, dtype)
    model.eval(), lik.eval()
    torch.manual_seed(0)
    with torch.no_grad():
        preds = lik(model(x.cuda(), derivative_directions=Vx))
        s = preds.sample(torch.Size([200000]))
        one = preds.sample()
    assert s.shape == (200000, n * (p + 1)) and one.shape == (n * (p + 1),) and s.dtype == dtype
    mean, cov = O.predictive_full(P.clone(F64), x.double(), Vx.double(), variant, add_noise=True)
    sd = cov.diagonal().sqrt()
    emp_mean = s.double().mean(0).cpu()
    assert float(((emp_mean - mean) / sd).abs().max()) < 0.02            # 200k draws: standard error 0.0022 sd
    emp_cov = torch.cov(s.double().T).cpu()
    assert float(((emp_cov - cov) / (sd[:, None] * sd[None, :])).abs().max()) < 0.03
    y_cand = s[:, ::p + 1].t()                                           # the caller's slicing (test_turbo.py:139)
    assert y_cand.shape == (n, 200000)


def test_memoised_factor_refreshes_noise_and_mean_constant():
    """eval mode: model(x) and likelihood(model(x)) share the memoised Cholesky factor, but the noise (and the mean
    constant) are read fresh on every call -- a stale hyp buffer once dropped the noise from the second call."""
    variant, n, d, M, p, dtype = "dsvgp", 50, 3, 16, 1, F64
    P, x, Vx, y, num_data = O.make_problem(n, d, M, p, dtype, seed=11, variant=variant, N=10 * n)
    model, lik = build(variant, P, d, dtype)
    model.eval(), lik.eval()
    with torch.no_grad():
        latent = model(x.cuda(), derivative_directions=Vx)
        v0, m0 = latent.variance.clone(), latent.mean.clone()
        noisy = lik(model(x.cuda(), derivative_directions=Vx))
        assert rel(noisy.variance - v0, O.noise(P).expand(v0.numel())) < 1e-9
        model.mean_module.constant.add_(0.5)
        assert rel(model(x.cuda(), derivative_directions=Vx).mean - m0, torch.full((m0.numel(),), 0.5, dtype=F64)) < 1e-9


# ------------------------------------------------------------------ natural-gradient variant (section 8f rank 2, NGD)
def _ngd_model(c, dtype):
    import directional_vi
    from dsvgp_b200 import gp
    p = c["params"]
    model = directional_vi.GPModel(p["Z"], p["Vz"], c["d"], variational_distribution="NGD").to("cuda", dtype)
    lik = gp.GaussianLikelihood().to("cuda", dtype)
    vs, vd = model.variational_strategy, model.variational_strategy._variational_distribution
    assert isinstance(vd, gp.NaturalVariationalDistribution)
    assert {"variational_strategy._variational_distribution.natural_vec",
            "variational_strategy._variational_distribution.natural_mat"} <= set(model.state_dict())
    with torch.no_grad():
        vd.natural_vec.copy_(c["natural_vec"])
        vd.natural_mat.copy_(c["natural_mat"])
        vs.variational_params_initialized.fill_(1)
        model.mean_module.constant.copy_(p["c"])
        model.covar_module.raw_outputscale.copy_(p["raw_os"])
        model.covar_module.base_kernel.raw_lengthscale.copy_(p["raw_ell"])
        lik.noise_covar.raw_noise.copy_(p["raw_noise"])
    return model, lik


@pytest.mark.parametrize("name", ["ngd_d3_p1_f64", "ngd_c1_f32"])
def test_ngd_step_matches_unmodified_reference_golden(name):
    """GPModel(variational_distribution="NGD") + gp.NGD: ELBO, natural gradients and the NGD update against the
    unmodified reference model (fixture from oracle/make_golden.py)."""
    from dsvgp_b200 import gp
    c = torch.load(os.path.join(GOLD, "ngd_cases.pt"))[name]
    dtype, f64 = c["x"].dtype, c["x"].dtype == F64
    model, lik = _ngd_model(c, dtype)
    model.train(), lik.train()
    vd = model.variational_strategy._variational_distribution
    mll = gp.VariationalELBO(lik, model, num_data=c["num_data"])
    opt = gp.NGD(model.variational_parameters(), num_data=c["num_data"], lr=0.1)
    loss = -mll(lik(model(c["x"].cuda(), derivative_directions=c["Vx"])), c["y"].cuda())
    loss.backward()
    tv, tg = (1e-10, 1e-9) if f64 else (1e-4, 2e-4)
    assert abs(float(-loss) - float(c["elbo"])) < tv * abs(float(c["elbo"]))
    assert rel(-vd.natural_vec.grad, c["grad_natural_vec"]) < tg
    assert rel(-vd.natural_mat.grad, c["grad_natural_mat"]) < tg
    assert rel(-model.variational_strategy.inducing_points.grad, c["grad_Z"]) < tg
    assert rel(-lik.noise_covar.raw_noise.grad, c["grad_raw_noise"]) < tg
    if not f64:      # the fp32 fixture is the reference's own fp32 arithmetic; the kernels are gated against the fp64 oracle
        z = torch.zeros(1, dtype=F64)
        P = O.Params(m=z, Ls_raw=z, **{k: v.double() for k, v in c["params"].items()})
        val, g = O.ngd_elbo_and_grads(P, c["natural_vec"].double(), c["natural_mat"].double(), c["x"].double(),
                                      c["Vx"].double(), c["y"].double(), c["num_data"])
        assert abs(float(-loss) - float(val)) < 1e-4 * abs(float(val))
        assert rel(-vd.natural_vec.grad, g["natural_vec"]) < 1e-4 and rel(-vd.natural_mat.grad, g["natural_mat"]) < 1e-4
    opt.step()
    assert rel(vd.natural_vec, c["natural_vec_after"]) < (1e-9 if f64 else 2e-4)
    assert rel(vd.natural_mat, c["natural_mat_after"]) < (1e-9 if f64 else 2e-4)
    model.eval(), lik.eval()
    with torch.no_grad():        # eval: the memoised natural -> (m, chol S) conversion follows the updated parameters
        a = lik(model(c["x"].cuda(), derivative_directions=c["Vx"])).mean.clone()
        b = lik(model(c["x"].cuda(), derivative_directions=c["Vx"])).mean
        assert torch.equal(a, b) and bool(torch.isfinite(a).all())


def test_train_gp_with_ngd_reduces_loss():
    import math
    import random
    import directional_vi
    torch.manual_seed(1), random.seed(1)
    n, d = 400, 2
    x = torch.rand(n, d)
    f = torch.sin(2 * math.pi * (x ** 2).sum(1, keepdim=True))
    df = 4 * math.pi * x * torch.cos(2 * math.pi * (x ** 2).sum(1, keepdim=True))
    ds = torch.utils.data.TensorDataset(x, torch.cat([f, df], 1))
    import builtins
    losses, real_print = [], builtins.print

    def spy(*a, **k):
        s = " ".join(str(t) for t in a)
        if "loss:" in s and "total_step" in s:
            losses.append(float(s.split("loss:")[1].split(",")[0]))
    builtins.print = spy
    try:
        model, lik = directional_vi.train_gp(ds, num_inducing=16, num_directions=2, minibatch_size=200, minibatch_dim=2,
                                             num_epochs=60, learning_rate_hypers=0.01, learning_rate_ngd=0.1, use_ngd=True)
    finally:
        builtins.print = real_print
    assert len(losses) >= 3 and losses[-1] < losses[0] - 0.1 and all(math.isfinite(v) for v in losses), losses


def test_training_trajectory_agrees_across_tensor_core_paths():
    """40 Adam steps with a large learning rate at a size that takes the tcgen05 path (M' = 192, n' = 1536): the
    3xFP16 products (scales recomputed from the moving parameters every step), the 3xTF32 products and the mma.sync
    kernels with fp64 master sums give the same loss trajectory; nothing overflows fp16 as L_s, the lengthscale and
    the inducing points move."""
    import math
    import bench
    from dsvgp_b200 import engine, gp
    from dsvgp_b200.optim import FusedAdam

    def run(use_tc, use_fp16, dense_d=True):
        old = (engine.USE_TC, engine.USE_FP16, engine.DENSE_D, engine.WHITEN_FP64)
        # (3xFP16 whitening pinned: "auto" would run A = W K_zx and dK_zx = W^T dA in fp64 at this n' = 1536)
        engine.USE_TC, engine.USE_FP16, engine.DENSE_D, engine.WHITEN_FP64 = use_tc, use_fp16, dense_d, False
        engine.ENGINE._ws.clear(), engine.ENGINE._fac.clear()
        try:
            wl = dict(bench.WORKLOADS["C3"], M=64, n=512, N=5000)
            dev = torch.device("cuda", 0)
            model, lik = bench.build_model(wl, F32, dev)
            d, p = wl["d"], wl["p"]
            mll = gp.VariationalELBO(lik, model, num_data=(d + 1) * wl["N"])
            vd = model.variational_strategy._variational_distribution
            opt = FusedAdam([{"params": list(model.parameters()) + list(lik.parameters())}], lr=0.05,
                            lower_triangular=[vd.chol_variational_covar])
            losses = []
            for it in range(40):
                x, V, y = (t.to(dev) for t in bench.synth_batch(wl["n"], d, p, "dsvgp", F32, "cpu", 100 + it))
                opt.zero_grad()
                loss = -mll(lik(model(x, derivative_directions=V)), y)
                loss.backward()
                opt.step()
                losses.append(float(loss.detach()))
            ws = next(iter(engine.ENGINE._ws.values()))
            assert ws.tc == use_tc and ws.tch == (use_tc and use_fp16)
            return losses, float(model.covar_module.base_kernel.lengthscale), float(vd.chol_variational_covar.abs().max())
        finally:
            engine.USE_TC, engine.USE_FP16, engine.DENSE_D, engine.WHITEN_FP64 = old
            engine.ENGINE._ws.clear(), engine.ENGINE._fac.clear()

    ref, ell_ref, _ = run(False, False)            # mma.sync 3xTF32 with fp64 master sums
    assert all(math.isfinite(v) for v in ref) and ref[-1] < ref[0] - 1.0
    # 3xFP16 with one dense (S - I) A product (default), 3xFP16 with the two triangular products, 3xTF32
    for mode in ((True, True, True), (True, True, False), (True, False, True)):
        got, ell, lmax = run(*mode)
        assert all(math.isfinite(v) for v in got), mode
        dev_rel = max(abs(a - b) / max(1.0, abs(b)) for a, b in zip(got, ref))
        assert dev_rel < 2e-3, (mode, dev_rel)
        assert abs(ell - ell_ref) < 2e-3 * ell_ref


def test_step_is_bitwise_deterministic():
    """The step has no float atomics and a fixed reduction order, so identical inputs give bit-identical losses and
    gradients -- which also makes this a race detector for the engine's and the Cholesky's side streams
    (scratch/soak_determinism.py runs the long version at the bench sizes)."""
    import bench
    from dsvgp_b200 import gp
    wl = dict(bench.WORKLOADS["C3"], M=128, n=1024, N=20000)            # M' = 384, n' = 3072: tcgen05 path, 4 Cholesky blocks
    dev = torch.device("cuda", 0)
    model, lik = bench.build_model(wl, F32, dev)
    mll = gp.VariationalELBO(lik, model, num_data=(wl["d"] + 1) * wl["N"])
    x, V, y = (t.to(dev) for t in bench.synth_batch(wl["n"], wl["d"], wl["p"], "dsvgp", F32, "cpu", 3))
    params = list(model.parameters()) + list(lik.parameters())

    def step():
        for q in params:
            q.grad = None
        loss = -mll(lik(model(x, derivative_directions=V)), y)
        loss.backward()
        return torch.cat([loss.detach().reshape(1).double()] + [q.grad.reshape(-1).double() for q in params])
    ref = step()
    assert bool(torch.isfinite(ref).all())
    for _ in range(12):
        assert torch.equal(step(), ref)


def test_deferred_side_work_is_bit_identical():
    """engine.DEFER_SIDE_WORK only moves the overlapped assembly / L_s operand products behind a mid-chain diagonal block of the
    factorisation (ops.chol_wait_mid): results must not change, for any release point, and the wait must be a no-op for
    factorisations with too few blocks."""
    import bench
    from dsvgp_b200 import engine, gp, ops
    dev = torch.device("cuda", 0)
    for M in (32, 512):                                                  # M' = 96 (one block: no mid event), 1536 (16 blocks)
        wl = dict(bench.WORKLOADS["C3"], M=M, n=640, N=20000)
        model, lik = bench.build_model(wl, F32, dev)
        mll = gp.VariationalELBO(lik, model, num_data=(wl["d"] + 1) * wl["N"])
        x, V, y = (t.to(dev) for t in bench.synth_batch(wl["n"], wl["d"], wl["p"], "dsvgp", F32, "cpu", 5))
        params = list(model.parameters()) + list(lik.parameters())

        def step():
            for q in params:
                q.grad = None
            loss = -mll(lik(model(x, derivative_directions=V)), y)
            loss.backward()
            return torch.cat([loss.detach().reshape(1).double()] + [q.grad.reshape(-1).double() for q in params])
        try:
            engine.DEFER_SIDE_WORK = False
            ref = step()
            for ws in engine.ENGINE._ws.values():            # the tail writes / reads the LOWER triangle of Psi only (ops.phi_outer)
                ws.Psi.fill_(float("nan"))
            assert torch.equal(step(), ref)
            engine.DEFER_SIDE_WORK = True
            for mid in (20, 2, 0, -1, 9):
                ops.set_chol_mid_link(mid)
                assert torch.equal(step(), ref), (M, mid)
        finally:
            engine.DEFER_SIDE_WORK = True
            ops.set_chol_mid_link(20)
