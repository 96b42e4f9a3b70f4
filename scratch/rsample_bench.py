"""Time the reparameterised draw and its backward on the C3 model (d = 10, M' = 3072, p = 2, fp32), and the fp64 Cholesky
backward dsvgp_chol_bwd_f64 alone.

  python scratch/rsample_bench.py [--out DIR]

For n' in {24, 1536, 6144} (8, 512, 2048 candidates): CUDA-event times of
  * cov:     model(x) -> (covariance_matrix * w).sum().backward()      (what the predictive covariance already cost)
  * rsample: model(x) -> (rsample(base_samples=z) * w).sum().backward()  with 16 fixed draws
and of dsvgp_chol_bwd_f64 at n' alone.  The Cholesky backward's flops are counted from the triangles of its three products:
P = tril(L^T Lbar) n^3/3, Phi(P) W n^3/3, W^T Y 2n^3/3 (4n^3/3 in all), and given as a rate against the dense fp64 product
(the "dense NN" case of scratch/gemm64_bench.py) measured in the same run.  Prints one JSON line (also DIR/rsample_bench.json)
with the card's name, power limit and maximum SM clock."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "gp-derivatives-variational-inference_b200")):
    sys.path.insert(0, p)

import bench  # noqa: E402
from dsvgp_b200 import ops  # noqa: E402

F32, F64 = torch.float32, torch.float64


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this measurement needs the GPU"
    dev = torch.device("cuda")
    wl = dict(bench.WORKLOADS["C3"])
    model, lik = bench.build_model(wl, F32, dev)
    model.eval(), lik.eval()
    d, p = wl["d"], wl["p"]
    res = {"card": card(), "draws": 16}
    g = torch.Generator().manual_seed(0)
    for n in (8, 512, 2048):
        nq = n * (p + 1)
        x, V, _ = bench.synth_batch(n, d, p, "dsvgp", F32, "cpu", 1)
        x, V = x.to(dev), V.to(dev)
        z = torch.randn(16, nq, generator=g, dtype=F64).to(dev)
        w = torch.randn(16, nq, generator=g).to(dev)
        wc = torch.randn(nq, nq, generator=g).to(dev)

        def cov():
            X = x.clone().requires_grad_(True)
            (model(X, derivative_directions=V).covariance_matrix * wc).sum().backward()

        def draw():
            X = x.clone().requires_grad_(True)
            (model(X, derivative_directions=V).rsample(base_samples=z) * w).sum().backward()

        reps = 20 if nq <= 1536 else 5
        t_cov, t_draw = [], []
        for _ in range(3):                     # alternated
            t_cov.append(timed(cov, reps))
            t_draw.append(timed(draw, reps))
        res[f"n'={nq}"] = {"cov_backward_ms": [round(t, 3) for t in t_cov], "rsample_backward_ms": [round(t, 3) for t in t_draw]}

    for nq in (24, 1536, 6144):
        A = torch.randn(nq, nq, dtype=F64, device=dev)
        S = A @ A.T / nq + torch.eye(nq, dtype=F64, device=dev)
        Mp, nb0, nlev = ops.chol_plan(nq)
        work, L, W = (torch.empty(Mp, Mp, dtype=F64, device=dev) for _ in range(3))
        if Mp > nq:
            ops.pad_identity(work, nq)
        work[:nq, :nq] = S
        info = torch.zeros(1, dtype=torch.int32, device=dev)
        ops.cholesky_inverse(work, L, W, nb0, nlev, info)
        assert int(info.item()) == 0
        Lbar = torch.randn(nq, nq, dtype=F64, device=dev)
        out = torch.empty(nq, nq, dtype=F64, device=dev)
        reps = 200 if nq <= 1536 else 20
        ms = timed(lambda: ops.chol_backward(L[:nq, :nq], W[:nq, :nq], Lbar, out, nq), reps)
        B, C = torch.randn(nq, nq, dtype=F64, device=dev), torch.empty(nq, nq, dtype=F64, device=dev)
        ms_dense = timed(lambda: ops.gemm(A, B, C), reps)
        flops = 4.0 * nq ** 3 / 3
        rate, rate_dense = flops / ms / 1e9, 2.0 * nq ** 3 / ms_dense / 1e9
        res[f"chol_bwd n'={nq}"] = {"ms": round(ms, 4), "TFLOP/s": round(rate, 2), "dense_fp64_TFLOP/s": round(rate_dense, 2),
                                    "share_of_dense": round(rate / rate_dense, 3)}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "rsample_bench.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
