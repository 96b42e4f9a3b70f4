"""Plain SVGP baseline drivers (reference directionalvi/traditional_vi.py, the model the experiment drivers compare DSVGP
against): gpytorch's whitened VariationalStrategy with ScaleKernel(RBFKernel()) over function values only, no derivative
information on either side.  Same names as the reference; the signatures follow this repository's grad_svgp.py, the
closest sibling, minus everything about derivatives.

It runs on the same fused B200 step as the directional models, with p = 0 inducing directions and p = 0 data-side
directions (dsvgp_b200.gp.VariationalStrategy).  The gpytorch 1.4 semantics are restated, not pinned to the reference
file: K_zz jitter 1e-3, predictive jitter 1e-4, the 1e-6 / 1e-5 / 1e-4 psd_safe_cholesky ladder and the 1e-6 (fp32) /
1e-10 (fp64) variance floor, exactly as for the other strategies.  num_data = N, and the training loop hands
likelihood(model(x)) to the mll as every other driver here does (quirk Q3).
"""
import sys

import torch

from dsvgp_b200 import gp

import directional_vi as _dvi
from utils.count_params import count_params


class GPModel(gp.ApproximateGP):
    """SVGP over function values: M inducing points, q(u) over their M values."""

    def __init__(self, inducing_points, **kwargs):
        if kwargs.get("variational_strategy") == "CIQ":
            raise NotImplementedError("the CIQ strategy is outside the B200 hot path")
        vd_class = gp.NaturalVariationalDistribution if kwargs.get("variational_distribution") == "NGD" \
            else gp.CholeskyVariationalDistribution
        variational_distribution = vd_class(inducing_points.size(0))
        variational_strategy = gp.VariationalStrategy(self, inducing_points, variational_distribution,
                                                      learn_inducing_locations=kwargs.get("learn_inducing_locations", True))
        super().__init__(variational_strategy)
        self.mean_module = gp.ConstantMean()
        self.covar_module = gp.ScaleKernel(gp.RBFKernel())

    def forward(self, x):
        return gp.MultivariateNormal(self.mean_module(x), self.covar_module(x))


def _values(y_batch):
    """the function-value labels of a minibatch as a vector; derivative columns are refused, not silently dropped"""
    if y_batch.dim() > 1 and y_batch.shape[-1] != 1:
        raise ValueError(f"traditional_vi fits function values only: the targets have {y_batch.shape[-1]} columns; pass y = f(x) "
                         "(use directional_vi / grad_svgp for derivative labels)")
    return y_batch.reshape(-1)


def train_gp(train_dataset, dim, num_inducing=128, minibatch_size=1, num_epochs=1, use_ngd=False, use_ciq=False,
             learning_rate_hypers=0.01, learning_rate_ngd=0.1, lr_sched=None, mll_type="ELBO",
             num_contour_quadrature=15, watch_model=False, gamma=0.1, verbose=True, **args):
    """Train the SVGP baseline.  Returns (model, likelihood)."""
    if use_ciq:
        raise NotImplementedError("use_ciq (contour-integral-quadrature whitening) is outside the B200 hot path")
    device = _dvi._require_cuda()
    n_samples = len(train_dataset)
    dtype = train_dataset[0][0].dtype
    _values(train_dataset[0][1].reshape(1, -1))
    model = GPModel(torch.rand(num_inducing, dim).to(dtype),
                    **({"variational_distribution": "NGD"} if use_ngd else {})).to(device=device, dtype=dtype)
    likelihood = gp.GaussianLikelihood().to(device=device, dtype=dtype)
    model.train()
    likelihood.train()
    if verbose:
        count_params(model, likelihood)
    vopt, hopt, vsched, hsched = _dvi._optimizers(model, likelihood, learning_rate_hypers, lr_sched, n_samples,
                                                  minibatch_size, num_epochs, gamma,
                                                  ngd=dict(num_data=n_samples, lr=learning_rate_ngd) if use_ngd else None)
    mll_cls = {"ELBO": gp.VariationalELBO, "PLL": gp.PredictiveLogLikelihood}[mll_type]
    mll = mll_cls(likelihood, model, num_data=n_samples)
    total_step, loss = 0, None
    for i in range(num_epochs):
        for x_batch, y_batch in _dvi._batches(train_dataset, minibatch_size, True, device):
            y_batch = _values(y_batch)
            vopt.zero_grad()
            hopt.zero_grad()
            output = likelihood(model(x_batch))
            loss = -mll(output, y_batch)
            loss.backward()
            vopt.step()
            vsched.step()
            hopt.step()
            hsched.step()
            if total_step % 50 == 0 and verbose:
                nll = -torch.distributions.Normal(output.mean, output.variance.sqrt()).log_prob(y_batch).mean()
                print(f"Epoch: {i}; total_step: {total_step}, loss: {loss.item()}, nll: {nll}")
                sys.stdout.flush()
            total_step += 1
    if verbose and loss is not None:
        print(f"Done! loss: {loss.item()}")
        print("\nDone Training!")
    return model, likelihood


def eval_gp(test_dataset, model, likelihood, mll_type="ELBO", num_inducing=128, minibatch_size=1):
    """Predictive means and variances (incl. likelihood noise) of every test point, concatenated on the CPU: (N,) each."""
    device = _dvi._require_cuda()
    model.eval()
    likelihood.eval()
    means, variances = [], []
    with torch.no_grad():
        for x_batch, _ in _dvi._batches(test_dataset, minibatch_size, False, device):
            preds = likelihood(model(x_batch))
            means.append(preds.mean.cpu())
            variances.append(preds.variance.cpu())
    return torch.cat(means), torch.cat(variances)
