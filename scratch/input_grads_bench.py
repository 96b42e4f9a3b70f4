"""Time the data-side assembly backward (ops.kdir_bwd_cols) at the C3 shape and the C3 training step with x requiring grad.

  python scratch/input_grads_bench.py [--n 16384] [--out DIR]

Prints one JSON line (also written to DIR/input_grads_bench.json): the card's name and power limit, the kernel time of the
data-side kernel and of its fp64 chunk reduction (torch.profiler, CUDA activities), the same call timed with CUDA events,
the blocked kernel reading dK transposed (what the call falls back to outside its shapes) and the row-side kdir_bwd on the
same dK, the rate against the bytes of dK_zx, and the C3 step time with and without x / Vx requiring grad (alternated)."""
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
from dsvgp_b200 import gp, ops  # noqa: E402

F32, F64 = torch.float32, torch.float64


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def timed(fn, reps=20, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def kernels(n):
    wl = bench.WORKLOADS["C3"]
    d, M, p = wl["d"], wl["M"], wl["p"]
    g = torch.Generator().manual_seed(0)
    Z, x = torch.rand(M, d, generator=g).cuda(), torch.rand(n, d, generator=g).cuda()
    Vz = (torch.eye(d)[:p].repeat(M, 1) + 0.1 * torch.randn(M * p, d, generator=g)).cuda()
    Vx = torch.eye(d)[:p].repeat(n, 1).cuda()
    hyp = ops.hyp_from_raw(torch.full((1,), -0.2).cuda(), torch.full((1,), 0.1).cuda())
    uz, invz = ops.normalize_dirs(Vz)
    wx, invx = ops.normalize_dirs(Vx)
    Mq, nq = M * (p + 1), n * (p + 1)
    dK = torch.randn(Mq, (nq + 63) // 64 * 64, generator=g).cuda()[:, :nq]     # the step's layout; 604 MB at n = 16384
    z = lambda *s: torch.zeros(*s, dtype=F64, device="cuda")
    gx, gv, gZ, gVz, gsc = z(n, d), z(n * p, d), z(M, d), z(M * p, d), z(2)
    cols = lambda: ops.kdir_bwd_cols(Z, uz, p, x, wx, invx, p, hyp, dK, gx, gv)
    rows = lambda: ops.kdir_bwd(Z, uz, invz, p, x, wx, p, hyp, dK, gZ, gVz, gsc)
    blocked = lambda: ops.kdir_bwd(x, wx, invx, p, Z, uz, p, hyp, dK, gx, gv, None, dk_trans=True)
    assert cols()
    out = {"dK_bytes": Mq * nq * 4, "cols_call_ms": timed(cols), "rows_call_ms": timed(rows), "blocked_call_ms": timed(blocked, 5, 1)}
    cols()
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(10):
            cols()
        torch.cuda.synchronize()
    per = {}
    for e in prof.key_averages():
        if "kdir_bwd_cols_v4" in e.key or "kdir_bwd_reduce_rows" in e.key:
            name = "cols_kernel" if "kdir_bwd_cols_v4" in e.key else "reduce"
            per[name + "_ms"] = e.device_time_total / 1e3 / max(1, e.count)
    out.update(per)
    out["cols_kernel_TBps"] = out["dK_bytes"] / (out["cols_kernel_ms"] * 1e-3) / 1e12
    return out


def step_times(n, rounds=3, steps=20):
    wl = dict(bench.WORKLOADS["C3"], n=n)
    d, p = wl["d"], wl["p"]
    dev = torch.device("cuda", 0)
    model, lik = bench.build_model(wl, F32, dev)
    mll = gp.VariationalELBO(lik, model, num_data=(d + 1) * wl["N"])
    x, V, y = (t.to(dev) for t in bench.synth_batch(n, d, p, "dsvgp", F32, "cpu", 5))
    params = list(model.parameters()) + list(lik.parameters())

    def step(inputs):
        for q in params:
            q.grad = None
        X, Vd = x.detach().requires_grad_(inputs), V.detach().requires_grad_(inputs)
        loss = -mll(lik(model(X, derivative_directions=Vd)), y)
        loss.backward()

    res = {"params_only_ms": [], "with_x_Vx_ms": []}
    for _ in range(rounds):
        res["params_only_ms"].append(timed(lambda: step(False), steps, 3))
        res["with_x_Vx_ms"].append(timed(lambda: step(True), steps, 3))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=16384)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    torch.cuda.set_device(0)
    res = {"card": card(), "n": a.n, **kernels(a.n), "step": step_times(a.n)}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "input_grads_bench.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
