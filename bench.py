#!/usr/bin/env python
"""Benchmark of the DSVGP minibatch hot path (BASELINE.json metric: DSVGP train points/s, ELBO fwd+bwd).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload C3|C2|C4|C5|C1] [--impl b200|reference]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
           bench.py --gpus N --steps K --warmup W

A step is ONE ELBO forward+backward over one minibatch through the reference-facing API
(`loss = -mll(likelihood(model(x, derivative_directions=V)), y); loss.backward()`), including the gradient
all-reduce when N > 1, excluding the optimiser step and data loading (SURVEY.md section 8d).  Weak scaling: every
rank owns `n_per_gpu` minibatch points; the data term is normalised by the global minibatch.

One JSON line is printed by rank 0:
  value / ms_per_step   inputs already resident in HBM (CUDA events, barrier + synchronize on both sides, max over ranks)
  e2e                   the same step with x, y, V copied from pinned host memory and the loss read back every step
  sweep                 the same step at per-GPU minibatches 512 / 4096 / 16384 (512 is what every reference driver ships:
                        experiments/synthetic1/run_exp.py:25), eager and -- where the step is launch-bound -- replayed from a
                        CUDA graph; vs_cpu_same_n = GPU points/s over CPU points/s at the SAME n = 512 (like for like)
  strong_scaling        global batch 131072 (SURVEY.md section 8d's headline point) split over the N ranks, next to the same
                        batch on ONE GPU measured by rank 0 alone in the same run: efficiency = T_1 / (N T_N)
  dist_parity           (N > 1) sharded ELBO / gradients = unsharded, and gradients bit-identical on every rank, asserted
  roofline              dominant kernel (whitening product A = L^-1 K_zx) timed ALONE with CUDA events: algorithmic flops
                        M'^2 n' (triangular) over the BURST tensor peak / 3 (3xFP16 passes); fp64 models: over the fp64 DMMA
                        peak measured in this process (dsvgp_dmma_peak_f64)
  roofline_assembly     the fused kernel-assembly kernel against measured HBM copy bandwidth
  extra                 (N = 1, workload C3) short runs of the other BASELINE.json workloads C2 / C4 / C5
  cpu_baseline          (N = 1) the oracle's reference-structured step on the host cores, >= 5 timed after 2 warm-ups
`--impl reference` times only that CPU arm (rank 0), on the same `config`; every step is a bounded sample of the workload
(the reference's shipped minibatch of 512 points: a 16384-point step would materialise a 49152^2 K_xx on the host).

`--dump-outputs DIR` (rank 0) writes what the last timed step returned to its caller, in the model dtype: DIR/loss.npy and
DIR/grad.<parameter name>.npy for every model and likelihood parameter.  Inputs and parameters are seeded, so two builds
run with the same arguments can be compared output for output.
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "gp-derivatives-variational-inference_b200")
for _p in (ROOT, PKG):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import torch  # noqa: E402

WORKLOADS = {  # name: variant, d, M, p, dtype, N (dataset size), default per-GPU minibatch, reference minibatch
    "C1": dict(variant="dsvgp", d=2, M=20, p=2, dtype="f32", N=600, n=200, n_ref=200,
               desc="tests/test_dsvgp.py as shipped"),
    "C2": dict(variant="dsvgp", d=3, M=512, p=1, dtype="f64", N=35000, n=4096, n_ref=500, desc="bunny-shaped"),
    "C3": dict(variant="dsvgp", d=10, M=1024, p=2, dtype="f32", N=1000000, n=16384, n_ref=512,
               desc="synthetic1-shaped, 1M points"),
    "C4": dict(variant="dsvgp", d=60, M=800, p=3, dtype="f32", N=2048, n=2048, n_ref=512, desc="rover-shaped"),
    "C5": dict(variant="dfree", d=18, M=1024, p=2, dtype="f32", N=500000, n=16384, n_ref=512, desc="uci_dfree-shaped"),
}
METRIC = "DSVGP train points/s (ELBO fwd+bwd)"
DUMP_LIMIT_BYTES = 64 << 20           # --dump-outputs: larger outputs are cut to a seeded sample of their elements
STRONG_GLOBAL_BATCH = 131072          # SURVEY.md section 8d: the headline strong-scaling point of C3
SWEEP_N = (512, 4096, 16384)          # SURVEY.md section 8d / BASELINE.md section 2: per-GPU minibatches of the C3 sweep


def synth_batch(n, d, p, variant, dtype, device, seed):
    """x ~ U[0,1]^d, canonical data directions, y = [f, df/dx_1..p] of f = sum_k sin(2 pi x_k^2) (O(1) values)."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    x = torch.rand(n, d, generator=g, dtype=torch.float64)
    f = torch.sin(2 * math.pi * x * x).sum(1, keepdim=True)
    grad = 4 * math.pi * x * torch.cos(2 * math.pi * x * x)
    if variant == "dfree":
        y = f.reshape(-1)
    elif variant == "grad":
        y = torch.cat([f, grad], 1).reshape(-1)
    else:
        y = torch.cat([f, grad[:, :p]], 1).reshape(-1)
    V = torch.eye(d, dtype=torch.float64)[:p].repeat(n, 1)
    return x.to(dtype), V.to(dtype), y.to(dtype)


def synth_params(d, M, p, dtype, seed=0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    Z = torch.rand(M, d, generator=g, dtype=torch.float64)
    Vz = torch.eye(d, dtype=torch.float64)[:p].repeat(M, 1) + 0.1 * torch.randn(M * p, d, generator=g, dtype=torch.float64)
    Mq = M * (p + 1)
    m = 1e-3 * torch.randn(Mq, generator=g, dtype=torch.float64)
    Ls = torch.eye(Mq, dtype=torch.float64) + 0.01 * torch.randn(Mq, Mq, generator=g, dtype=torch.float64).tril()
    return dict(Z=Z.to(dtype), Vz=Vz.to(dtype), m=m.to(dtype), Ls_raw=Ls.to(dtype))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.path = gpu_index, None, f"/tmp/dsvgp_clocks_{os.getpid()}.csv"

    def __enter__(self):
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.gpu)], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            self.proc.wait()
            self.f.close()

    def summary(self):
        rows = []
        try:
            for line in open(self.path):
                c = [t.strip() for t in line.split(",")]
                if len(c) >= 9:
                    rows.append(c)
            os.remove(self.path)
        except OSError:
            pass
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = [float(r[1]) for r in rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [nm for k, nm in enumerate(names) if any(r[5 + k].lower().startswith("active") for r in rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": float(rows[0][2]), "reasons": reasons,
                "samples": len(rows)}


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(hbm=float(p["hbm_gbs"]), bf16_burst=float(p["bf16_tflops"]),
                    bf16_sustained=float(p.get("bf16_tflops_sustained", p["bf16_tflops"])), src="measured")
    except (OSError, KeyError, ValueError):
        return dict(hbm=6650.0, bf16_burst=1590.0, bf16_sustained=1400.0, src="fallback")


def ncu_traffic(kernel_key):
    """dram bytes per launch of the named kernel from the committed ncu summary (profiles/traffic.json names the capture)."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f).get(kernel_key)
    except (OSError, ValueError):
        return None


def make_config(name, wl, world):
    """Identical for both arms (the driver compares them): names the workload, not the implementation."""
    return {"workload": f"{name} {wl['desc']}: d={wl['d']} M={wl['M']} p={wl['p']} M'={wl['M'] * (wl['p'] + 1)} "
                        f"{wl['dtype']} N={wl['N']}", "n_per_gpu": wl["n"], "global_batch": wl["n"] * world,
            "variant": wl["variant"], "parallelism": f"dp{world}", "l2_policy": "inputs_exceed_l2"}


# ----------------------------------------------------------------------------------------------------- CPU arm
def cpu_reference_arm(wl, steps, warmup):
    """The reference's algorithm on the host cores: oracle, reference op structure, fwd + autograd bwd."""
    from oracle import dsvgp_oracle as O            # the one place bench.py executes oracle/
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    dtype = torch.float64 if wl["dtype"] == "f64" else torch.float32
    n = wl["n_ref"]
    x, V, y = synth_batch(n, wl["d"], wl["p"], wl["variant"], dtype, "cpu", 123)
    sp = synth_params(wl["d"], wl["M"], wl["p"], dtype)
    z = lambda *s: torch.zeros(*s, dtype=dtype)
    P = O.Params(Z=sp["Z"], Vz=sp["Vz"], m=sp["m"], Ls_raw=sp["Ls_raw"], c=z(1), raw_os=z(()), raw_ell=z(1, 1), raw_noise=z(1))
    num_data = (wl["d"] + 1) * wl["N"]
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        O.elbo_and_grads(P, x, V, y, num_data, wl["variant"], structure="reference")
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    t = statistics.median(times)
    return dict(value=n / t, unit="points/s", cores=cores, kind="port", ms_per_step=1e3 * t, sample_n=n,
                sample=f"reference-structured oracle step (4 kernel evaluations incl. full K_xx, fp64 Cholesky + 2 triangular "
                       f"solves, autograd backward) on a {n}-point sample of the minibatch = the reference's own shipped minibatch "
                       f"(a {wl['n']}-point step would materialise a {wl['n'] * (wl['p'] + 1)}^2 K_xx on the host; per-point cost "
                       f"of the reference structure only grows with n), same d/M/p/dtype; median of {steps} after {warmup} "
                       f"warm-up; torch {torch.__version__} CPU, {cores} threads")


# ----------------------------------------------------------------------------------------------------- GPU arm
def build_model(wl, dtype, device):
    import dfree_directional_vi
    import directional_vi
    from dsvgp_b200 import gp
    sp = synth_params(wl["d"], wl["M"], wl["p"], dtype)
    cls = dfree_directional_vi.GPModel if wl["variant"] == "dfree" else directional_vi.GPModel
    model = cls(sp["Z"], sp["Vz"], wl["d"]).to(device=device, dtype=dtype)
    lik = gp.GaussianLikelihood().to(device=device, dtype=dtype)
    vs = model.variational_strategy
    with torch.no_grad():
        vs._variational_distribution.variational_mean.copy_(sp["m"])
        vs._variational_distribution.chol_variational_covar.copy_(sp["Ls_raw"])
        vs.variational_params_initialized.fill_(1)
    model.train(), lik.train()
    return model, lik


def _emit(line):
    """The ONE JSON line goes to the real stdout; everything else a library prints there (NCCL's version banner, ...)
    has been diverted to stderr by _guard_stdout()."""
    os.write(_REAL_STDOUT, (line + "\n").encode())


_REAL_STDOUT = 1


def _guard_stdout():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


class Arm:
    """One model + likelihood + objective on this rank's GPU, and the timing helpers every measurement shares."""

    def __init__(self, wl, device, rank, world):
        from dsvgp_b200 import distributed, gp
        self.wl, self.device, self.rank, self.world = wl, device, rank, world
        self.dtype = torch.float64 if wl["dtype"] == "f64" else torch.float32
        self.model, self.lik = build_model(wl, self.dtype, device)
        if world > 1:
            distributed.broadcast_parameters(self.model, self.lik)
        self.mll = gp.VariationalELBO(self.lik, self.model, num_data=(wl["d"] + 1) * wl["N"])
        self.params = list(self.model.parameters()) + list(self.lik.parameters())

    def shard(self, n_global):
        from dsvgp_b200 import distributed
        if n_global is None:
            distributed.disable(self.model)
        else:
            distributed.enable(self.model, n_global)

    def batch(self, n, seed):
        wl = self.wl
        return tuple(t.pin_memory() for t in synth_batch(n, wl["d"], wl["p"], wl["variant"], self.dtype, "cpu", seed))

    def step(self, xb, Vb, yb):
        for q in self.params:
            q.grad = None
        loss = -self.mll(self.lik(self.model(xb, derivative_directions=Vb)), yb)
        loss.backward()
        return loss

    def flat_grads(self):
        return torch.cat([q.grad.reshape(-1).double() for q in self.params])

    def barrier(self, collective=True):
        if self.world > 1 and collective:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def timed(self, fn, k, collective=True):
        """ms per call of fn over exactly k calls, CUDA events, barrier + synchronize on both sides, max over ranks."""
        self.barrier(collective)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        self.barrier(collective)
        ms = torch.tensor([e0.elapsed_time(e1)], device=self.device, dtype=torch.float64)
        if self.world > 1 and collective:
            import torch.distributed as dist
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms) / k

    def time_steps(self, n, seed, warmup, steps, collective=True):
        x, V, y = (t.to(self.device) for t in self.batch(n, seed))
        for _ in range(warmup):
            self.step(x, V, y)
        return self.timed(lambda: self.step(x, V, y), steps, collective)

    def release(self):
        from dsvgp_b200.engine import ENGINE
        ENGINE._ws.clear()
        torch.cuda.empty_cache()


def dist_parity(arm, n_each=512):
    """Asserted during warm-up at N > 1: the sharded step (payload summed over ranks, replicated tail) reproduces the
    unsharded step on the same global minibatch, and every rank ends with bit-identical gradients."""
    import torch.distributed as dist
    from dsvgp_b200 import distributed
    wl, world, rank = arm.wl, arm.world, arm.rank
    n, p = n_each * world, wl["p"]
    q = 1 if wl["variant"] == "dfree" else p + 1
    x, V, y = (t.to(arm.device) for t in arm.batch(n, 4242))           # the same global minibatch on every rank
    lo, hi = distributed.shard_bounds(n, rank, world)
    arm.shard(n)
    l_s = float(arm.step(x[lo:hi], V[lo * p: hi * p], y[lo * q: hi * q]).detach())
    g_s = arm.flat_grads()
    arm.shard(None)
    l_f = float(arm.step(x, V, y).detach())
    g_f = arm.flat_grads()
    err_l = abs(l_s - l_f) / abs(l_f)
    err_g = float((g_s - g_f).abs().max() / g_f.abs().max())
    both = [torch.zeros_like(g_s) for _ in range(world)]
    dist.all_gather(both, g_s)
    identical = all(torch.equal(both[0], b) for b in both[1:])
    ok = err_l < 1e-5 and err_g < 1e-4 and identical
    flag = torch.tensor([1.0 if ok else 0.0], device=arm.device)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if float(flag) != 1.0:
        raise SystemExit(f"dist_parity FAILED on rank {rank}: loss err {err_l:.2e}, gradient err {err_g:.2e}, "
                         f"rank-identical gradients: {identical}")
    arm.release()
    return {"ok": True, "n_global": n, "loss_rel_err": err_l, "grad_rel_err_vs_unsharded": err_g, "rank_identical_gradients": identical}


def step_outputs(arm, loss):
    """What a caller of the training step receives: the loss and the gradient of every model and likelihood parameter."""
    out = {"loss": loss.detach()}
    for owner, module in (("model", arm.model), ("likelihood", arm.lik)):
        for name, q in module.named_parameters():
            if q.grad is not None:
                out[f"grad.{owner}.{name}"] = q.grad.detach()
    return out


def dump_outputs(path, arrays, seed=0):
    """Writes {name: tensor} as path/<name>.npy, DUMP_LIMIT_BYTES in all.  The budget is shared out smallest array first, so
    small outputs are always whole; an array larger than its share is replaced by its flattened elements at sorted indices
    drawn from a generator seeded with `seed` (the same indices for the same shape, so dumps of two builds stay comparable)."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    budget = DUMP_LIMIT_BYTES - 1024 * len(arrays)                          # 1 KiB per file for the .npy header
    order = sorted(arrays, key=lambda k: arrays[k].numel())
    for i, name in enumerate(order):
        t = arrays[name].cpu()
        keep = min(t.numel(), budget // (len(order) - i) // t.element_size())
        if keep < t.numel():
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(seed))[:keep].sort().values
            t = t.reshape(-1)[idx]
        budget -= t.numel() * t.element_size()
        np.save(os.path.join(path, name + ".npy"), t.numpy())


def main():
    _guard_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C3", choices=sorted(WORKLOADS))
    ap.add_argument("--n-per-gpu", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip sweep / strong scaling / other workloads (headline only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the loss and parameter gradients of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU step (--impl b200)")
    wl = dict(WORKLOADS[args.workload])
    if args.n_per_gpu:
        wl["n"] = args.n_per_gpu
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    config = make_config(args.workload, wl, world if args.impl == "b200" else max(args.gpus, 1))

    if args.impl == "reference":
        if rank != 0:
            return
        cb = cpu_reference_arm(wl, args.steps, args.warmup)
        _emit(json.dumps({"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "points/s", "n_gpus": args.gpus,
                          "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["ms_per_step"],
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": wl["dtype"],
                          "data": "synthetic", "config": config,
                          "arithmetic": "torch CPU ops in the model dtype, fp64 Cholesky and triangular solves (as the reference, "
                                        "DGVS.py:74,181,183)",
                          "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "sample_n")},
                          "e2e": {"value": cb["value"], "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                          "gpu_launches": 0}))
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device: the hot path has no CPU implementation")
    import torch.distributed as dist
    from dsvgp_b200 import _lib, ops
    from dsvgp_b200 import engine as _eng
    from dsvgp_b200.engine import ENGINE
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    n, d, M, p = wl["n"], wl["d"], wl["M"], wl["p"]
    p2 = 0 if wl["variant"] == "dfree" else p
    arm = Arm(wl, device, rank, world)
    dtype = arm.dtype
    parity = dist_parity(arm) if world > 1 else None
    if world > 1:
        arm.shard(n * world)
    xh, Vh, yh = arm.batch(n, 1000 + rank)
    x, V, y = xh.to(device), Vh.to(device), yh.to(device)

    for _ in range(warmup):
        arm.step(x, V, y)
    launches0 = _lib.launch_count()
    last = [None]

    def timed_step():
        # detached: a live loss keeps its autograd graph, and the AccumulateGrad nodes of that graph (bound to this stream)
        # would be inherited by the side-stream warm-up of the CUDA-graph capture in the sweep below and break the capture
        last[0] = arm.step(x, V, y).detach()
    with ClockSampler(local_rank) as clk:
        ms_step = arm.timed(timed_step, args.steps)
    launches = _lib.launch_count() - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, step_outputs(arm, last[0]))

    def e2e_step():
        xb, Vb, yb = xh.to(device, non_blocking=True), Vh.to(device, non_blocking=True), yh.to(device, non_blocking=True)
        return float(arm.step(xb, Vb, yb).item())            # device -> host read of the step's loss
    for _ in range(2):
        e2e_step()
    ms_e2e = arm.timed(e2e_step, args.steps)
    h2d = sum(t.numel() * t.element_size() for t in (xh, Vh, yh))

    # ---- sweep over the per-GPU minibatch and the strong-scaling point (every rank takes part: the step has a collective)
    sweep, strong = [], None
    if not args.no_extras and args.workload == "C3":
        from dsvgp_b200 import graphs
        for ns in SWEEP_N:
            if world > 1:
                arm.shard(ns * world)
            ms = ms_step if ns == n else arm.time_steps(ns, 2000 + rank, 3, 5)
            row = {"n_per_gpu": ns, "global_batch": ns * world, "ms_per_step": ms, "points_per_s": ns * world / (ms * 1e-3)}
            p2s = 0 if wl["variant"] == "dfree" else wl["p"]
            row["whitening"] = ("fp64 DMMA (engine.WHITEN_FP64 = 'auto': the two products with W = L^-1 as the reference's fp64 "
                                "triangular solves)") if (_eng.WHITEN_FP64 == "auto" and ns * (p2s + 1) <= _eng.WHITEN_FP64_MAX_NQ) \
                else "3xFP16 tcgen05"
            if ns <= graphs.MAX_GRAPH_N and world == 1:
                row["ms_per_step_cuda_graph"] = graphs.time_graphed_step(arm, ns, 2000 + rank, 3, 10)
                row["points_per_s_cuda_graph"] = ns / (row["ms_per_step_cuda_graph"] * 1e-3)
            if row["whitening"].startswith("fp64") and world == 1:
                old = _eng.WHITEN_FP64                      # the same minibatch with the 3xFP16 products forced, for comparison
                _eng.WHITEN_FP64 = False
                arm.release()
                row["ms_per_step_3xfp16_whitening"] = arm.time_steps(ns, 2000 + rank, 3, 5)
                _eng.WHITEN_FP64 = old
            sweep.append(row)
            if ns != n:
                arm.release()
        ng = STRONG_GLOBAL_BATCH // world
        arm.shard(STRONG_GLOBAL_BATCH if world > 1 else None)
        ms_n = ms_step if (ng == n) else arm.time_steps(ng, 3000 + rank, 3, 5)
        arm.release()
        strong = {"global_batch": STRONG_GLOBAL_BATCH, "n_per_gpu": ng, "n_gpus": world, "ms_per_step": ms_n,
                  "points_per_s": STRONG_GLOBAL_BATCH / (ms_n * 1e-3)}
        if world > 1:
            arm.shard(None)
            ms_1 = arm.time_steps(STRONG_GLOBAL_BATCH, 3000, 2, 3, collective=False) if rank == 0 else None
            arm.barrier()
            arm.release()
            strong.update({"ms_per_step_1gpu_same_run": ms_1, "efficiency": (ms_1 / (world * ms_n)) if ms_1 else None,
                           "note": "T_1 measured by rank 0 alone (unsharded, other ranks idle at a barrier) in this same run"})
        else:
            strong.update({"ms_per_step_1gpu_same_run": ms_n, "efficiency": 1.0})
        if world > 1:
            arm.shard(n * world)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    arm.shard(None)
    pk = peaks()
    Mq, nq = M * (p + 1), n * (p2 + 1)
    ws = ENGINE.workspace(device, dtype, n, d, M, p, p2)
    fac = ENGINE.factor(device, dtype, d, M, p)
    reps = 5

    def timed_local(fn, k):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / k

    # ---- fp64 tensor (DMMA) peak of this device, measured here: register-resident mma.sync m8n8k4 chains
    sink = torch.zeros(1, dtype=torch.float64, device=device)
    import ctypes
    fl = ctypes.c_double(0.0)
    dm = lambda: _lib._lib.dsvgp_dmma_peak_f64(20000, 148 * 4, ctypes.c_void_p(sink.data_ptr()), ctypes.byref(fl), _lib.stream())
    dm()
    fp64_peak = max(fl.value / (timed_local(dm, 1) * 1e-3) / 1e12 for _ in range(3))
    # ---- replicated fp64 spine, alone: K_zz assembly + blocked Cholesky + inverse
    P_Z = arm.model.variational_strategy.inducing_points.detach()

    def chol_inv():
        ops.kdir_fwd(P_Z, fac.uz64, p, P_Z, fac.uz64, p, fac.hyp, fac.Kzz, diag_add=1e-3)
        ops.cholesky_inverse(fac.Kzz, fac.L, fac.W, fac.nb0, fac.nlev, fac.info)
    chol_inv()
    ms_chol = timed_local(chol_inv, reps)
    chol_flops = 2.0 * float(fac.Mp) ** 3 / 3.0

    # ---- dominant kernel alone: A = W K_zx (lower-triangular W), algorithmic flops M'^2 n'
    wx = ENGINE._data_dirs(ws, V, dtype)          # normalised data directions + on-device canonical detection (sets ws.canon)
    ops.kdir_fwd(P_Z, fac.uzT, p, x, wx, p2, fac.hyp, ws.Kzx)
    use_tc = bool(getattr(ws, "tc", False) and getattr(fac, "tc", False))
    use_tch = bool(getattr(ws, "tch", False) and getattr(fac, "tch", False))
    if use_tch:
        ops.kdir_fwd_half(P_Z, fac.uzT, p, x, wx, p2, fac.hyp, ws.Kzx, ws.Kh, ws.Kl, fac.scales[1:2], canon=ws.canon)
        whiten = lambda: ops.gemm_tch((fac.Wh, fac.Wl), (ws.Kh, ws.Kl), ws.A, Mq, nq, Mq, fac.scales[8:9], a_tri=ops.TRI_LOWER,
                                      chunk=_eng.TCH_CHUNK, Ch=(ws.Ah, ws.Al), c_scale=fac.scales[3:4])
        kname = ("gemm_tch2p_kernel (A = L^-1 K_zx: tcgen05.mma kind::f16 x3 (3xFP16 on power-of-two-scaled two-half operands, "
                 f"22 significand bits), TMA-fed, PERSISTENT CTA pairs walking a host-balanced work list, TMEM accumulators restarted "
                 f"every {_eng.TCH_CHUNK} k-block(s) of 64, fp32 master sums in registers moved to the epilogue warps with setmaxnreg; "
                 "epilogue also writes the split of A for the next product)")
    elif use_tc:
        ops.split_lo(ws.Kzx, ws.lo1, Mq, nq)
        whiten = lambda: ops.gemm_tc(fac.Wt, fac.Wt_lo, ws.Kzx, ws.lo1, ws.A, Mq, nq, Mq, a_tri=ops.TRI_LOWER,
                                     chunk=_eng.TC_CHUNK, C_lo=ws.lo2)
        kname = ("gemm_tc_kernel (A = L^-1 K_zx: tcgen05.mma kind::tf32 x3 (3xTF32), TMA-fed, TMEM accumulators restarted every "
                 f"{_eng.TC_CHUNK} k-blocks, fp32 master sums)")
    else:
        Wm = ENGINE._wt(fac)
        whiten = lambda: ops.gemm(Wm, ws.Kzx, ws.A, a_tri=ops.TRI_LOWER, M=Mq, N=nq, K=Mq)
        kname = ("gemm_kernel (A = L^-1 K_zx, fp64 DMMA mma.sync)" if dtype == torch.float64
                 else "gemm_kernel (A = L^-1 K_zx, 3xTF32 mma.sync, fp64 master accumulation)")
    whiten()
    ms_gemm = timed_local(whiten, reps)
    # kernel assembly as the step runs it (K_zx as the two-half split on the 3xFP16 path) and K only
    if use_tch:
        ms_asm = timed_local(lambda: ops.kdir_fwd_half(P_Z, fac.uzT, p, x, wx, p2, fac.hyp, ws.Kzx, ws.Kh, ws.Kl, fac.scales[1:2],
                                                       canon=ws.canon), reps)
    else:
        asm_lo = ws.lo1 if use_tc else None
        ms_asm = timed_local(lambda: ops.kdir_fwd(P_Z, fac.uzT, p, x, wx, p2, fac.hyp, ws.Kzx, canon=ws.canon, out_lo=asm_lo), reps)
    ms_asm_k = timed_local(lambda: ops.kdir_fwd(P_Z, fac.uzT, p, x, wx, p2, fac.hyp, ws.Kzx, canon=ws.canon), reps)
    ms_asm_general = timed_local(lambda: ops.kdir_fwd(P_Z, fac.uzT, p, x, wx, p2, fac.hyp, ws.Kzx), reps)
    s = 8 if dtype == torch.float64 else 4
    gemm_flops = float(Mq) * Mq * nq
    if dtype == torch.float64:
        tensor_peak = fp64_peak
        peak_note = f"fp64 DMMA peak measured in this process ({fp64_peak:.1f} TFLOP/s, dsvgp_dmma_peak_f64: register-resident m8n8k4 chains)"
    elif use_tch:
        tensor_peak = pk["bf16_burst"] / 3
        peak_note = (f"{pk['src']} bf16 dense BURST {pk['bf16_burst']} TFLOP/s (the kernel is timed alone, {reps} reps; fp16 runs at "
                     f"the bf16 rate) / 3 (3xFP16 passes)")
    else:
        tensor_peak = pk["bf16_burst"] / 2 / 3
        peak_note = f"{pk['src']} bf16 dense BURST {pk['bf16_burst']} TFLOP/s / 2 (TF32 rate) / 3 (3xTF32 passes)"
    asm_bytes = s * (float(Mq) * nq + (M + n) * d + (M * p + n * p2) * d)
    arith = ("fp64 throughout (DMMA)" if wl["dtype"] == "f64" else
             "fp32 model; K_zz / Cholesky / Cholesky-backward in fp64; whitening products on tensor cores as 3xFP16 (two-half "
             "operands = 22 significand bits, scales from measured maxima, fp32 accumulation in chains of K=64, fp32 master sums): "
             "fp32-grade, parity-tested at 1e-4 against the fp64 oracle incl. trained-state q(u) and the bench size")
    out = {
        "metric": METRIC, "value": n * world / (ms_step * 1e-3), "unit": "points/s", "n_gpus": world, "steps": args.steps,
        "warmup": warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": wl["dtype"], "data": "synthetic", "config": config, "impl": "b200", "arithmetic": arith,
        "e2e": {"value": n * world / (ms_e2e * 1e-3), "unit": "points/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": 4 + (8 if dtype == torch.float64 else 4)},
        "gpu_launches": launches, "launches_per_step": launches / args.steps,
        "clocks": clk.summary(),
        "roofline": {"kernel": kname, "bound": "tensor",
                     "achieved": gemm_flops / (ms_gemm * 1e-3) / 1e12, "peak": tensor_peak, "unit": "TFLOP/s",
                     "frac": gemm_flops / (ms_gemm * 1e-3) / 1e12 / tensor_peak, "traffic": ncu_traffic("gemm_whiten"),
                     "ms": ms_gemm, "flops_per_launch": gemm_flops, "peak_note": peak_note,
                     "traffic_source": ncu_traffic("_source")},
        "roofline_assembly": {"kernel": "kdir_fwd_v4 / kdir_fwd_blocked (K_zx), K only -- what RBFKernelDirectionalGrad.forward returns",
                              "bound": "hbm", "achieved": asm_bytes / (ms_asm_k * 1e-3) / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                              "frac": asm_bytes / (ms_asm_k * 1e-3) / 1e9 / pk["hbm"], "traffic": ncu_traffic("kdir_fwd_k_only"),
                              "ms": ms_asm_k, "bytes_per_launch": asm_bytes,
                              "path": "canonical data-side directions (detected on device)" if ws.canon is not None else "general directions",
                              "general_directions_ms": ms_asm_general,
                              "general_directions_frac": asm_bytes / (ms_asm_general * 1e-3) / 1e9 / pk["hbm"],
                              "in_step": {"note": ("inside the training step the same kernel writes only the two-half (fp16 hi, lo) split of "
                                                   "K_zx * scale, the operand of the 3xFP16 product: the same bytes as K alone") if use_tch
                                                  else ("inside the training step the same launch also writes the TF32 lo companion of "
                                                        "K_zx (fused, replaces a separate split pass): twice the bytes"),
                                          "ms": ms_asm, "bytes_written": asm_bytes * (2 if (use_tc and not use_tch) else 1),
                                          "hbm_frac": asm_bytes * (2 if (use_tc and not use_tch) else 1) / (ms_asm * 1e-3) / 1e9 / pk["hbm"],
                                          "traffic": ncu_traffic("kdir_fwd")},
                              "peak_note": f"{pk['src']} copy bandwidth"},
        "fp64_spine": {"dmma_peak_tflops_measured": fp64_peak, "chol_plus_inverse_ms": ms_chol,
                       "chol_plus_inverse_tflops": chol_flops / (ms_chol * 1e-3) / 1e12, "Mp": fac.Mp,
                       "note": "K_zz assembly + blocked fp64 Cholesky + explicit inverse W = L^-1 (2 M'^3 / 3 flop), replicated on every "
                               "rank; timed alone"},
    }
    if sweep:
        out["sweep"] = sweep
    if strong:
        out["strong_scaling"] = strong
    if parity:
        out["dist_parity"] = True
        out["dist_parity_detail"] = parity
    if world == 1 and not args.no_cpu_baseline:
        ENGINE._ws.clear()
        cb = cpu_reference_arm(wl, 5, 2)
        out["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "sample_n")}
        same = [r for r in sweep if r["n_per_gpu"] == cb["sample_n"]]
        if same:
            out["vs_cpu_same_n"] = {"n": cb["sample_n"], "gpu_points_per_s": same[0]["points_per_s"], "cpu_points_per_s": cb["value"],
                                    "ratio": same[0]["points_per_s"] / cb["value"],
                                    "gpu_points_per_s_cuda_graph": same[0].get("points_per_s_cuda_graph"),
                                    "ratio_cuda_graph": (same[0]["points_per_s_cuda_graph"] / cb["value"])
                                    if same[0].get("points_per_s_cuda_graph") else None,
                                    "note": "both arms at the reference's shipped minibatch; the headline `value` is at n_per_gpu"}
    if world == 1 and not args.no_extras and args.workload == "C3":
        # the other BASELINE.json workloads, short runs (3 warm-up + 5 timed), so that the driver's record carries them
        extra = {}
        del ws, fac
        ENGINE._ws.clear(), ENGINE._fac.clear()
        torch.cuda.empty_cache()
        for name in ("C2", "C4", "C5"):
            w2 = dict(WORKLOADS[name])
            a2 = Arm(w2, device, 0, 1)
            ms = a2.time_steps(w2["n"], 77, 3, 5)
            ms_ref_n = a2.time_steps(w2["n_ref"], 78, 3, 5)
            # kernel assembly of this workload alone (K_zx, K only), against HBM and -- where the dot products dominate
            # (d = 60) -- against the fp32 FMA pipe: per point pair 2 d (1 + p1)(1 + p2) flops for Delta.Delta, Delta.u,
            # Delta.w, u.w, nominal fp32 peak 148 SMs x 128 FMA x 2 x sm_max_mhz
            dt2 = a2.dtype
            x2, V2, _ = (t.to(device) for t in a2.batch(w2["n"], 77))
            pp2 = 0 if w2["variant"] == "dfree" else w2["p"]
            ws2 = ENGINE.workspace(device, dt2, w2["n"], w2["d"], w2["M"], w2["p"], pp2)
            f2 = ENGINE.factor(device, dt2, w2["d"], w2["M"], w2["p"])
            wx2 = ENGINE._data_dirs(ws2, V2, dt2)
            Z2 = a2.model.variational_strategy.inducing_points.detach()
            asm = lambda: ops.kdir_fwd(Z2, f2.uzT, w2["p"], x2, wx2, pp2, f2.hyp, ws2.Kzx, canon=ws2.canon)
            asm()
            ms_a = timed_local(asm, 10)
            sz = 8 if dt2 == torch.float64 else 4
            Mq2, nq2 = w2["M"] * (w2["p"] + 1), w2["n"] * (pp2 + 1)
            by2 = sz * (float(Mq2) * nq2 + (w2["M"] + w2["n"]) * w2["d"] + (w2["M"] * w2["p"] + w2["n"] * pp2) * w2["d"])
            fl2 = 2.0 * w2["d"] * (1 + w2["p"]) * (1 + pp2) * w2["M"] * w2["n"]
            fp32_peak = 148 * 128 * 2 * 1.965e9
            extra[name] = {"workload": make_config(name, w2, 1)["workload"], "n": w2["n"], "ms_per_step": ms,
                           "points_per_s": w2["n"] / (ms * 1e-3), "n_ref": w2["n_ref"], "ms_per_step_at_n_ref": ms_ref_n,
                           "dtype": w2["dtype"],
                           "assembly": {"ms": ms_a, "bytes": by2, "gbs": by2 / (ms_a * 1e-3) / 1e9, "hbm_frac": by2 / (ms_a * 1e-3) / 1e9 / pk["hbm"],
                                        "dot_product_flops": fl2,
                                        "fp32_pipe_frac": (fl2 / (ms_a * 1e-3) / fp32_peak) if dt2 == torch.float32 else None,
                                        "bound": "fp32 FMA pipe" if (dt2 == torch.float32 and fl2 / fp32_peak > by2 / (pk["hbm"] * 1e9)) else "hbm"}}
            del ws2, f2
            ENGINE._ws.clear(), ENGINE._fac.clear()
            del a2
            torch.cuda.empty_cache()
        out["extra"] = extra
    if world > 1:
        dist.destroy_process_group()
    _emit(json.dumps(out))


if __name__ == "__main__":
    main()
