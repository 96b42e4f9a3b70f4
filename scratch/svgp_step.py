"""SVGP baseline (p = 0) on one GPU: the value-only assembly kernels and the fp32 step at M = 3072, n = 16384, d = 10.

    python scratch/svgp_step.py [--root TREE] [--tag NAME] [--out DIR]

--root selects the source tree whose library is loaded (default: this checkout).  Run it once on this tree and once on
a checkout of the parent commit in the same session: there the p = 0 calls take the blocked kernels, which is the
before / after comparison (there is no runtime switch between the two).  Prints and writes one JSON line:

  * the card name and power limit (nvidia-smi);
  * per kernel (torch.profiler, CUDA activity only, 20 launches each after a warm-up): K_zx forward as fp32 K, as K + TF32
    lo and as the two-half split, and the K_zx backward; achieved bandwidth against the algorithmic bytes
    4 (M n + (M + n) d) (one fp32 read or write of the M x n matrix plus the two point sets);
  * the fp32 ELBO step (forward + backward, default 3xFP16 path) through the engine with no directions, timed with CUDA
    events over 10 steps after 3 warm-up steps.
"""
import argparse
import json
import os
import subprocess
import sys


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    ap.add_argument("--tag", default="new")
    ap.add_argument("--out", default=None)
    ap.add_argument("--M", type=int, default=3072)
    ap.add_argument("--n", type=int, default=16384)
    ap.add_argument("--d", type=int, default=10)
    args = ap.parse_args()
    root = os.path.abspath(args.root)
    for p in (root, os.path.join(root, "gp-derivatives-variational-inference_b200")):
        sys.path.insert(0, p)
    import torch
    import types
    from torch.profiler import ProfilerActivity, profile
    from dsvgp_b200 import ops
    from dsvgp_b200.engine import ENGINE
    assert torch.cuda.is_available(), "needs a CUDA device"
    M, n, d = args.M, args.n, args.d
    dev = torch.device("cuda", 0)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    g = torch.Generator(device=dev).manual_seed(0)
    Z, x = torch.rand(M, d, device=dev, generator=g), torch.rand(n, d, device=dev, generator=g)
    hyp = ops.hyp_from_raw(torch.tensor([0.3], device=dev), torch.tensor([-0.4], device=dev))
    ld = (n + 63) // 64 * 64
    K, Klo = torch.empty(M, ld, device=dev)[:, :n], torch.empty(M, ld, device=dev)[:, :n]
    Kh, Kl = (torch.empty(M, ld, dtype=torch.float16, device=dev)[:, :n] for _ in range(2))
    sK = torch.tensor([2.0 ** 14], device=dev)
    dK = torch.randn(M, ld, device=dev, generator=g)[:, :n]
    gZ, gsc = torch.zeros(M, d, dtype=torch.float64, device=dev), torch.zeros(2, dtype=torch.float64, device=dev)
    calls = {
        "fwd_K": lambda: ops.kdir_fwd(Z, None, 0, x, None, 0, hyp, K),
        "fwd_K_lo": lambda: ops.kdir_fwd(Z, None, 0, x, None, 0, hyp, K, out_lo=Klo),
        "fwd_half": lambda: ops.kdir_fwd_half(Z, None, 0, x, None, 0, hyp, K, Kh, Kl, sK),
        "bwd": lambda: ops.kdir_bwd(Z, None, None, 0, x, None, 0, hyp, dK, gZ, None, gsc),
    }
    alg_bytes = 4 * (M * n + (M + n) * d)
    res = dict(tag=args.tag, card=smi, M=M, n=n, d=d, alg_bytes=alg_bytes, kernels={})
    for name, fn in calls.items():
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(20):
                fn()
            torch.cuda.synchronize()
        per = {}
        for ev in prof.key_averages():
            if ev.device_type.name == "CUDA" and ev.count >= 20 and "kdir" in ev.key:
                per[ev.key[:120]] = ev.device_time_total / ev.count / 1000.0     # ms per launch
        main_ms = max(per.values()) if per else float("nan")
        res["kernels"][name] = dict(per_kernel_ms=per, main_ms=main_ms, GBps=alg_bytes / (main_ms * 1e-3) / 1e9)
    # the fp32 ELBO step through the engine, p = 0 on both sides
    gq = torch.Generator(device=dev).manual_seed(1)
    P = types.SimpleNamespace(Z=Z.clone(), Vz=None, m=1e-3 * torch.randn(M, device=dev, generator=gq),
                              Ls_raw=torch.eye(M, device=dev) + 0.01 * torch.randn(M, M, device=dev, generator=gq).tril(),
                              c=torch.full((1,), 0.05, device=dev), raw_os=torch.tensor(0.1, device=dev),
                              raw_ell=torch.full((1, 1), -0.2, device=dev), raw_noise=torch.full((1,), -1.0, device=dev))
    y = torch.sin(x.sum(1))

    def step():
        return ENGINE.elbo_step(P, x, None, y, 10 * n, 0, 0, 1)
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        out = step()
    e1.record()
    torch.cuda.synchronize()
    res["step_ms"] = e0.elapsed_time(e1) / 10
    res["elbo"] = float(out[0])
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, f"svgp_step_{args.tag}.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
