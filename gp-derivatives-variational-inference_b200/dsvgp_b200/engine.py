"""The DSVGP minibatch step on one GPU: kernel launches in the order the data flows, no host synchronisation
except the single Cholesky-status read at the end of a step.

What the reference does per step (DirectionalGradVariationalStrategy.forward, DGVS.py:89-208, plus the gpytorch
likelihood / ELBO / KL and their autograd backward) and what happens here instead:

  reference                                         here (all on torch's current stream)
  ------------------------------------------------  ---------------------------------------------------------
  K_zx, K_xz, K_zz, full K_xx (4 kernel calls)      K_zz (fp64) and K_zx only; K_xx diagonal in closed form
  psd_safe_cholesky(K_zz.double())                  blocked fp64 Cholesky + explicit W = L^-1
  two fp64 triangular solves                        one triangular product A = W K_zx (tensor cores)
  (S - I) A through two dense L_s products          B = L_s^T A, C = L_s B - A (triangular products)
  mean, diag via MatmulLazyTensor.diag              column reductions of A.m and A*C
  likelihood + ELBO + KL elementwise ops            one fused kernel each
  autograd through everything (fp64 Cholesky bwd)   hand-derived backward: dA in place, dK_zx = W^T dA,
                                                    G = A diag(g) A^T, and a replicated M'^3 fp64 tail
                                                    (dL, Phi, W^T Psi W) feeding the assembly backward

Multi-GPU (distributed.py): everything up to and including G is local to a minibatch shard; a per-model `Reducer`
sums the two buffers that have to be summed over ranks before the replicated tail runs ([G | t] underneath the
dK_zx product and the K_zx assembly backward).
"""
import os

import torch

from . import ops
from .ops import F32, F64, TRI_LOWER, TRI_UPPER

KZZ_JITTER = 1e-3          # add_jitter() default            DGVS.py:144
PRED_JITTER = 1e-4         # data_data_covar.add_jitter(1e-4) DGVS.py:198,203
CHOL_RETRY = (1e-6, 1e-5, 1e-4)   # psd_safe_cholesky(jitter=1e-6): 1e-6 * 10**i, i < 3   DGVS.py:74
USE_TC = True      # fp32 model: run the big whitening products on tcgen05 (set False to force the mma.sync kernels)
USE_FP16 = True    # ... as 3xFP16 (kind::f16, scaled two-half operands) instead of 3xTF32: same 22 significand bits, 1.6x faster
DENSE_D = True     # 3xFP16 training path: (S - I) A as ONE dense product with D = E + E^T + E E^T (False: B' = E^T A, C = E B + B')
WHITEN_FP64 = "auto"  # fp32 model: run the two products that multiply by W = L^-1 (A = W K_zx, dK_zx = W^T dA) in fp64 on DMMA, the
                      # way the reference does its triangular solves (DGVS.py:181,183), instead of as 3xFP16.  |W||K_zx| / |A| is the
                      # conditioning of K_zz + 1e-3 I (~4e2 at the BASELINE inputs, 1e3-1e4 for long lengthscales / converged q(u)):
                      # a 22-bit operand split and fp32 accumulation carry that factor into A, fp64 does not.  Costs 2 M'^2 n' DMMA
                      # flops per step (+1.2 ms at C3 with n = 512; 31 ms at n = 16384).  True / False / "auto" = whenever the
                      # minibatch is small enough for that to be cheap (n' <= WHITEN_FP64_MAX_NQ: every minibatch size the
                      # reference's drivers ship).  DESIGN.md section 4.2 has the measured error table of both forms.
WHITEN_FP64_MAX_NQ = 2048
DEFER_SIDE_WORK = True   # elbo_step: the work overlapped with the factorisation (K_zx assembly, L_s operand products, KL) starts after the
                         # chain's throughput-bound first links (ops.chol_wait_mid) instead of competing with their trailing updates
TC_CHUNK = 2       # k-blocks (of 32) per tensor-core accumulation chain before the fp32 master sum
TCH_CHUNK = 1      # the same chain length (K = 64) in k-blocks of 64 halves
WORKSPACE_CACHE = 6    # problem shapes whose buffers are kept (least recently used evicted)
PERSISTENT_UNDER_REDUCE = os.environ.get("DSVGP_PERSISTENT_UNDER_REDUCE", "1") != "0"   # N > 1: dK_zx product under the [G | t] all-reduce
HALF_A = False     # 3xFP16 training step (DENSE_D): True = A = W K_zx leaves the whitening product ONLY as its two-half split (the operand
                   # of C = (S - I) A and of the Gram product) and the column reductions / the dA pass read that split (A_ij = (hi + lo) / s_A,
                   # 22 significand bits).  The product's store phase is bound by the SM's 32 B/clk write port and exposed, so 8 instead of
                   # 16 bytes per element shortens the product (0.98 -> 0.91 ms alone), but the half-reading column pass costs 0.03 ms more
                   # and the whole step does not move (11.34 / 11.42 ms, A/B in one process: the step is power-capped there) -- off.
F16 = torch.float16
_PARAM_NAMES = ("Z", "Vz", "m", "Ls_raw", "c", "raw_os", "raw_ell", "raw_noise")


class NanError(RuntimeError):
    """gpytorch.utils.errors.NanError equivalent."""


class NotPSDError(RuntimeError):
    """gpytorch.utils.errors.NotPSDError equivalent."""


def _round_up(a, b):
    return (a + b - 1) // b * b


class Factor:
    """Everything that depends on the parameters only (not on the minibatch): transformed hyper-parameters,
    normalised inducing directions, the fp64 Cholesky factor L of K_zz + jitter*I and W = L^-1.
    Recomputed every training step, memoised across batches in eval mode (DGVS.py:72 `@cached`)."""

    def __init__(self, device, dtype, d, M, p):
        self.key = (str(device), dtype, d, M, p)
        self.d, self.M, self.p = d, M, p
        self.Mq = M * (p + 1)
        self.Mp, self.nb0, self.nlev = ops.chol_plan(self.Mq)
        e = lambda *s, dt=F64: torch.empty(*s, dtype=dt, device=device)
        self.hyp = e(8)
        self.info = torch.zeros(1, dtype=torch.int32, device=device)
        # the status travels to pinned host memory right after the factorisation; the host waits for THAT event only
        self.info_host = torch.zeros(1, dtype=torch.int32).pin_memory()
        self.info_event = torch.cuda.Event()
        self.Kzz, self.L, self.W = e(self.Mp, self.Mp), e(self.Mp, self.Mp), e(self.Mp, self.Mp)
        self.ldm = _round_up(self.Mq, 8)
        self.Wt = e(self.Mq, self.ldm, dt=dtype)[:, : self.Mq] if dtype == F32 else self.W   # W in the model dtype
        # operands of the tcgen05 products (fp32 model): explicit transposes and "lo" parts (x - trunc_tf32(x))
        self.tc = dtype == F32 and USE_TC
        self.tch = self.tc and USE_FP16
        if self.tc:
            mk = lambda: e(self.Mq, self.ldm, dt=dtype)[:, : self.Mq]
            self.Wt_lo, self.WtT, self.WtT_lo = mk(), mk(), mk()
        if self.tch:
            # two-half splits of W * sW and its transpose; power-of-two scales of every operand (layout: csrc/tc_prep.cu)
            mh = lambda: e(self.Mq, self.ldm, dt=F16)[:, : self.Mq]
            self.Wh, self.Wl, self.WTh, self.WTl = mh(), mh(), mh(), mh()
            self.scales = torch.ones(16, dtype=F32, device=device)
            self.maxbits = torch.zeros(8, dtype=torch.int32, device=device)   # layout: csrc/tc_prep.cu
        self.jitter = KZZ_JITTER
        self.Wt_fresh = False
        self.uzT = self.invzT = self.uz64 = self.invz64 = None
        self.valid = False
        self.generation = 0
        self.owner = None          # (strategy id, parameter versions) the memoised factor belongs to


class Workspace:
    """Every minibatch-sized buffer one (dtype, n, d, M, p, p2) problem needs, allocated once, reused per step."""

    def __init__(self, device, dtype, n, d, M, p, p2):
        T = dtype
        self.n, self.d, self.M, self.p, self.p2 = n, d, M, p, p2
        self.Mq, self.nq = M * (p + 1), n * (p2 + 1)
        Mq, nq = self.Mq, self.nq
        self.ldn = _round_up(max(nq, 1), 64)       # whole 32-float / 64-half column blocks (128 B, TMA) inside every row
        self.ldm = _round_up(Mq, 8)
        self.ldg = _round_up(Mq, 32)
        e = lambda *s, dt=T: torch.empty(*s, dtype=dt, device=device)
        self.tc = T == F32 and USE_TC and Mq >= 128 and nq >= 256
        self.tch = self.tc and USE_FP16
        self.Kzx, self.A, self.Bp, self.C = (e(Mq, self.ldn) for _ in range(4))
        self.B = None if self.tch else e(Mq, self.ldn)
        sq = lambda: e(Mq, self.ldm)[:, :Mq]
        self.E, self.Hp = sq(), sq()
        if self.tch:
            # two-half operands of the 3xFP16 products.  (Kh, Kl) holds K_zx, then dA; (Ah, Al) holds A
            # from the forward pass to the Gram product; (Agh, Agl) holds A diag(g_var).
            hb = lambda: e(Mq, self.ldn, dt=F16)[:, :nq]
            self.Kh, self.Kl, self.Ah, self.Al, self.Agh, self.Agl = (hb() for _ in range(6))
            sh = lambda: e(Mq, self.ldm, dt=F16)[:, :Mq]
            self.Eh, self.El, self.ETh, self.ETl = sh(), sh(), sh(), sh()
            self.Dh, self.Dl = sh(), sh()               # split of D = S - I = E + E^T + E E^T (training: C = D A)
            self.P = e(Mq, self.ldg)[:, :Mq]            # E E^T (lower tiles)
        self.A64 = self.B64 = None                      # fp64 operands of the W products (Engine._w64 allocates them)
        if self.tc:
            if not self.tch:
                self.lo1, self.lo2, self.lo3 = (e(Mq, self.ldn) for _ in range(3))   # "lo" parts of the current big operands
            self.E_lo, self.ET, self.ET_lo = sq(), sq(), sq()
            sg = lambda: e(Mq, self.ldg)[:, :Mq]
            self.G_lo, self.H_lo = sg(), sg()
            # split-K of the Gram product: its lower 128x256 tiles alone (156 at M' = 3072) leave the second wave of a
            # 148-SM part nearly empty; 8 k-slices give 8.4 waves and an fp64 sum over the slices
            self.syrk_split = max(1, min(8, self.nq // 4096))
            self.split_ws = e(self.syrk_split * Mq * _round_up(Mq, 4)) if self.syrk_split > 1 else None
        self.nslab = max(1, ops.reduce_slabs(Mq, nq))
        self.pm, self.pv = e(self.nslab, nq), e(self.nslab, nq)
        self.mu, self.var, self.gmu, self.gvar = e(nq), e(nq), e(nq), e(nq)
        self.tp = e(max(1, min(64, nq // 2048)), Mq)
        # [G | t] (model dtype) and [scalars(8) | gZ | gVz] (double) are the two buffers summed over ranks.
        # scalars: 0 data term, 1 explicit dELBO/dnoise, 4 d ell, 5 d outputscale, 6 d noise via variance, 7 d c
        self.big = torch.zeros(Mq * self.ldg + Mq, dtype=T, device=device)
        self.G, self.t = self.big[: Mq * self.ldg].view(Mq, self.ldg)[:, :Mq], self.big[Mq * self.ldg:]
        self.small = torch.zeros(8 + M * d + M * p * d, dtype=F64, device=device)
        self.sc = self.small[:8]
        self.gZ = self.small[8: 8 + M * d].view(M, d)
        self.gVz = self.small[8 + M * d:].view(M * p, d) if p else None
        self.small2 = torch.zeros_like(self.small)        # sharded tail (N > 1): this rank's panels, summed over ranks separately
        self.gZ2 = self.small2[8: 8 + M * d].view(M, d)
        self.gVz2 = self.small2[8 + M * d:].view(M * p, d) if p else None
        self.kl = torch.zeros(1, dtype=F64, device=device)
        self.scratch = e(max(8192, 2 * ((nq + 255) // 256) + 64), dt=F64)   # elbo_terms / pll_terms: 2 * ceil(nq / 256) partial sums
        self.scratch_kl = e(512, dt=F64)           # (its own partial-sum buffer: the KL runs on the side stream)
        self.H = e(Mq, self.ldg)[:, :Mq] if T == F32 else sq()
        self.X = sq()
        self.Y, self.Psi, self.S = (e(Mq, Mq, dt=F64) for _ in range(3))
        self.gm = self.gLs = None      # allocated fresh by every backward pass (handed to autograd without a copy)
        self.gx = self.gVx = None      # (fp64) d/dx, d/dVx: allocated fresh by a backward pass that wants them
        self.wx = self.invx = None     # normalised data-side directions and 1/|Vx|
        self.generation = 0
        self.canon = None          # (cidx, flag) of the data-side directions when detected canonical on device


class Engine:
    def __init__(self):
        self._ws, self._fac, self._streams, self._events = {}, {}, {}, {}

    def _fork_event(self, device):
        key = str(device)
        ev = self._events.get(key)
        if ev is None:
            ev = self._events[key] = torch.cuda.Event()
        return ev

    def _scales_event(self, device):
        key = "scales:" + str(device)
        ev = self._events.get(key)
        if ev is None:
            ev = self._events[key] = torch.cuda.Event()
        return ev

    def _side_stream(self, device):
        key = str(device)
        st = self._streams.get(key)
        if st is None:
            st = self._streams[key] = torch.cuda.Stream(device=device)
        return st

    def workspace(self, device, dtype, n, d, M, p, p2):
        key = (str(device), dtype, n, d, M, p, p2)
        ws = self._ws.pop(key, None)
        if ws is None:
            # eval batches of many sizes: do not hoard HBM -- but evict the LEAST recently used shape only (a training loop with a
            # ragged last minibatch and an evaluation loop alternate between four or five shapes; clearing everything made each
            # of them re-allocate gigabytes per epoch)
            while len(self._ws) >= WORKSPACE_CACHE:
                self._ws.pop(next(iter(self._ws)))
            ws = Workspace(device, dtype, n, d, M, p, p2)
        self._ws[key] = ws            # (re-inserted last: dict order is the LRU order)
        ws.generation += 1            # every user overwrites it: a saved-for-backward reference can tell (gp._Predictive)
        return ws

    def factor(self, device, dtype, d, M, p):
        key = (str(device), dtype, d, M, p)
        f = self._fac.pop(key, None)
        if f is None:
            while len(self._fac) >= WORKSPACE_CACHE:
                self._fac.pop(next(iter(self._fac)))
            f = Factor(device, dtype, d, M, p)
        self._fac[key] = f
        f.generation += 1
        return f

    @staticmethod
    def _validate(P, x, Vx, p, p2, y=None):
        """Raw pointers cross the C ABI next: everything must be what the kernels will assume it is.  The reference
        (torch / gpytorch) raises a dtype or broadcast error in the same situations; here a mismatch would be
        reinterpreted memory."""
        if x.dim() != 2:
            raise ValueError(f"x must be (n, d); got {tuple(x.shape)}")
        if not x.is_cuda:
            raise TypeError("dsvgp_b200 runs on CUDA tensors only (there is no CPU path)")
        T, dev = x.dtype, x.device
        if T not in (F32, F64):
            raise TypeError(f"unsupported dtype {T}: the hot path is built for float32 and float64")
        n, d = x.shape
        M = P.Z.shape[0]
        Mq = M * (p + 1)
        want = {"Z": (M, d), "Vz": (M * p, d) if p else None, "m": (Mq,), "Ls_raw": (Mq, Mq)}
        for name in _PARAM_NAMES:
            t = getattr(P, name, None)
            if t is None:
                continue
            if t.dtype != T or t.device != dev:
                raise TypeError(f"parameter `{name}` is {t.dtype} on {t.device}, the inputs are {T} on {dev}: move the "
                                "model and the likelihood to the dtype / device of the data (model.to(...))")
            shp = want.get(name)
            if shp is not None and tuple(t.shape) != shp:
                raise ValueError(f"parameter `{name}` has shape {tuple(t.shape)}, expected {shp}")
            if name in ("Z", "Vz", "m", "Ls_raw") and not t.is_contiguous():
                raise ValueError(f"parameter `{name}` must be contiguous")
        if p2:
            if Vx is None or Vx.dtype != T or Vx.device != dev or tuple(Vx.shape) != (n * p2, d):
                got = None if Vx is None else (tuple(Vx.shape), Vx.dtype, str(Vx.device))
                raise ValueError(f"derivative_directions must be ({n * p2}, {d}) {T} on {dev}; got {got}")
        if y is not None:
            if y.dtype != T or y.device != dev:
                raise TypeError(f"the target is {y.dtype} on {y.device}, the model output is {T} on {dev}")
            if y.numel() != n * (p2 + 1):
                raise ValueError(f"the target has {y.numel()} entries, the model output {n * (p2 + 1)} "
                                 f"(n = {n} points x {p2 + 1} outputs per point)")
        if torch.cuda.current_device() != dev.index:
            raise RuntimeError(f"the tensors live on {dev} but the current CUDA device is {torch.cuda.current_device()}: "
                               "wrap the call in torch.cuda.device(...) (streams and kernel attributes are per device)")

    # ------------------------------------------------------------------------------------------ factorisation
    @staticmethod
    def _hyp(f, P):
        ops.hyp_from_raw(P.raw_ell.reshape(-1), P.raw_os.reshape(-1),
                         None if P.raw_noise is None else P.raw_noise.reshape(-1), P.c.reshape(-1), out=f.hyp)

    @staticmethod
    def _prep(f, P, T):
        """hyper-parameter transforms and direction normalisation (everything K_zx and K_zz both need)"""
        Engine._hyp(f, P)
        if f.p:
            f.uzT, f.invzT = ops.normalize_dirs(P.Vz, T)
            f.uz64, f.invz64 = (f.uzT, f.invzT) if T == F64 else ops.normalize_dirs(P.Vz, F64)

    @staticmethod
    def _scales0(f, P, jitter=None):
        """3xFP16 path: power-of-two operand scales of the forward pass from hyp, the jitter and max|tril(L_s) - I|"""
        f.maxbits.zero_()
        ops.absmax(P.Ls_raw, f.maxbits[0:1], mode=2)
        ops.tc_scales(f.hyp, f.jitter if jitter is None else jitter, f.maxbits, f.Mq, f.scales, 0)

    @staticmethod
    def _factorise(f, P, T, extra_jitter, prep=True, wait=None):
        """[hyper-parameter transforms, direction normalisation,] K_zz + (1e-3 + extra) I in fp64 -> L, W = L^-1.
        wait: event after which f.scales is valid (elbo_step computes the scales on its side stream)."""
        if prep:
            Engine._prep(f, P, T)
        Engine._factorise_enqueue(f, P, extra_jitter)
        if f.tch and prep:
            Engine._scales0(f, P)
        Engine._factorise_finish(f, T, wait)

    @staticmethod
    def _factorise_enqueue(f, P, extra_jitter):
        """K_zz assembly + the whole factorisation / inverse chain + the status copy: the critical path of a step, and all it
        needs are hyp and the fp64 inducing directions."""
        if f.Mp > f.Mq:
            ops.pad_identity(f.Kzz, f.Mq)
        ops.kdir_fwd(P.Z, f.uz64, f.p, P.Z, f.uz64, f.p, f.hyp, f.Kzz, diag_add=KZZ_JITTER + extra_jitter)
        ops.cholesky_inverse(f.Kzz, f.L, f.W, f.nb0, f.nlev, f.info)
        if not torch.cuda.is_current_stream_capturing():      # (under CUDA-graph capture the owner of the graph reads f.info
            f.info_host.copy_(f.info, non_blocking=True)      #  after the replay: graphs.GraphedStep)
            f.info_event.record()
        f.jitter = KZZ_JITTER + extra_jitter

    @staticmethod
    def _factorise_finish(f, T, wait=None):
        """W in the forms the products read (after the operand scales exist: `wait`)."""
        if f.tch:
            if wait is not None:
                torch.cuda.current_stream(f.W.device).wait_event(wait)
            ops.split_half(f.W, f.scales[0:1], f.Wh, f.Wl, mode=1, hiT=f.WTh, loT=f.WTl, rows=f.Mq, cols=f.Mq)
        f.Wt_fresh = T != F32
        if T == F32 and not f.tch:                  # (the 3xFP16 path reads W only through its two-half split: see _wt)
            ops.cast2d(f.W, f.Wt, f.Mq, f.Mq, tril=True)
            f.Wt_fresh = True
            if f.tc:
                ops.split_lo(f.Wt, f.Wt_lo)
                ops.transpose(f.Wt, f.WtT)
                ops.split_lo(f.WtT, f.WtT_lo)

    @staticmethod
    def _wt(f):
        """W in the model dtype, made on demand for the consumers outside the 3xFP16 path (small minibatches that take
        the mma.sync kernels, the legacy re-whitening)."""
        if not f.Wt_fresh:
            ops.cast2d(f.W, f.Wt, f.Mq, f.Mq, tril=True)
            f.Wt_fresh = True
        return f.Wt

    @staticmethod
    def _check(f, P):
        # The one host synchronisation of a step -- on the event recorded right after the factorisation, not on the
        # whole step: by the time the host has enqueued the rest of the step the status is usually there already, and
        # the host goes on to prepare the next step while the GPU is still working on this one.
        f.info_event.synchronize()
        info = int(f.info_host[0])
        if info == 0:
            return True
        for name in ("Z", "Vz", "raw_ell", "raw_os"):
            t = getattr(P, name, None)
            if t is not None and not bool(torch.isfinite(t).all()):
                raise NanError(f"NaN/inf in `{name}` reached the Cholesky factorisation of K_zz")
        return False

    @staticmethod
    def _data_dirs(ws, Vx, T):
        """normalised data-side directions (+ on-device detection of canonical rows for the fp32 fast path)"""
        if not ws.p2:
            ws.canon = ws.invx = None
            return None
        if T == F32:
            wx, ws.invx, cidx, flag = ops.normalize_dirs_canon(Vx)
            ws.canon = (cidx, flag)
            return wx
        ws.canon = None
        wx, ws.invx = ops.normalize_dirs(Vx, T)
        return wx

    @staticmethod
    def _w64(ws):
        """fp64 whitening for this workspace?  (allocates its two fp64 M' x n' operands on first use)"""
        on = WHITEN_FP64 is True or (WHITEN_FP64 == "auto" and ws.nq <= WHITEN_FP64_MAX_NQ)
        if on and getattr(ws, "A64", None) is None:
            ws.A64, ws.B64 = (torch.empty(ws.Mq, ws.ldn, dtype=F64, device=ws.A.device) for _ in range(2))
        return on

    # ------------------------------------------------------------------------------------------------ forward
    @staticmethod
    def _assemble(ws, f, P, x, wx, need_C=True):
        """Everything of the forward pass that does not need the Cholesky factor: K_zx (+ its TF32 lo part) and the
        operands made from L_s.  elbo_step runs this on a side stream while K_zz is being factorised."""
        Mq, nq = ws.Mq, ws.nq
        tc = ws.tc and f.tc
        if ws.tch and f.tch:
            if Engine._w64(ws):
                # fp64 whitening: K_zx in the model's fp32 arithmetic (what the reference's kernel returns), widened below
                ops.kdir_fwd(P.Z, f.uzT, ws.p, x, wx, ws.p2, f.hyp, ws.Kzx, canon=ws.canon)
            # 3xFP16 path: K_zx leaves the assembly kernel only as the two-half split of K * sK (no fp32 matrix at all)
            elif not ops.kdir_fwd_half(P.Z, f.uzT, ws.p, x, wx, ws.p2, f.hyp, ws.Kzx, ws.Kh, ws.Kl, f.scales[1:2], canon=ws.canon):
                ops.split_half(ws.Kzx, f.scales[1:2], ws.Kh, ws.Kl, rows=Mq, cols=nq)
            if need_C and DENSE_D:
                # training: D = S - I = E + E^T + E E^T explicitly (every term is small when S ~ I: no cancellation), so
                # that (S - I) A is ONE dense product instead of B' = E^T A, C = E B + B'.  E and E^T (fp32 + lo) are also
                # the operands of the two M'^3 products of the backward tail.
                ops.tril_minus_eye(P.Ls_raw, ws.E)
                ops.split_lo(ws.E, ws.E_lo)
                ops.transpose(ws.E, ws.ET)
                ops.split_lo(ws.ET, ws.ET_lo)
                # (one CTA pair per tile here, not the persistent kernel: this product is a filler under the latency-bound Cholesky,
                # and persistent CTAs hold every SM for its whole 0.1 ms -- the next diagonal block of the factorisation, a 4-CTA
                # cluster, then waits for it: seen as a 45 us + 70 us hole in the chain in the profiler trace)
                ops.set_tc_persistent(False)
                try:
                    ops.gemm_tc(ws.E, ws.E_lo, ws.E, ws.E_lo, ws.P, Mq, Mq, Mq, b_kmajor=True, a_tri=TRI_LOWER, c_lower=True,
                                chunk=TC_CHUNK)                                               # lower tiles of E E^T
                finally:
                    ops.set_tc_persistent(True)
                # the scale of D from its MEASURED maximum (the a-priori bound is loose by ~M' max|E| for a trained q(u))
                ops.build_d_absmax(ws.E, ws.P, f.maxbits[4:5], Mq)
                ops.tc_scales(f.hyp, f.jitter, f.maxbits, Mq, f.scales, 2)
                ops.build_d_split(ws.E, ws.P, f.scales[7:8], ws.Dh, ws.Dl, Mq)
            else:
                ops.split_half(P.Ls_raw, f.scales[2:3], ws.Eh, ws.El, mode=2, hiT=ws.ETh, loT=ws.ETl, rows=Mq, cols=Mq)
                if need_C:                            # (DENSE_D off) fp32 operands of the two M'^3 products of the tail
                    ops.tril_minus_eye(P.Ls_raw, ws.E)
                    ops.split_lo(ws.E, ws.E_lo)
                    ops.transpose(ws.E, ws.ET)
                    ops.split_lo(ws.ET, ws.ET_lo)
            return
        have_lo = ops.kdir_fwd(P.Z, f.uzT, ws.p, x, wx, ws.p2, f.hyp, ws.Kzx, canon=ws.canon, out_lo=ws.lo1 if tc else None)
        # L_s = I + E:  B' = E^T A, B = L_s^T A = A + B', C = (S - I) A = E B + B'   (no cancellation against A)
        ops.tril_minus_eye(P.Ls_raw, ws.E)
        if tc:
            # tcgen05 path: every operand as (raw, lo); A operands are explicit (transposed) triangular matrices
            ops.split_lo(ws.E, ws.E_lo)
            ops.transpose(ws.E, ws.ET)
            ops.split_lo(ws.ET, ws.ET_lo)
            if not have_lo:
                ops.split_lo(ws.Kzx, ws.lo1, Mq, nq)

    @staticmethod
    def _forward(ws, f, P, x, wx, add_noise, need_C, assembled=False):
        Mq, nq = ws.Mq, ws.nq
        Kzx, A, B, C = ws.Kzx, ws.A, ws.B, ws.C
        tc = ws.tc and f.tc
        if not assembled:
            Engine._assemble(ws, f, P, x, wx, need_C)
        if ws.tch and f.tch:
            sc, H = f.scales, TCH_CHUNK
            if Engine._w64(ws):
                # K_zx -> fp64, A = W K_zx on DMMA (W = L^-1 in fp64), back to fp32 + the two-half split the next products read
                ops.cast2d(ws.Kzx, ws.B64, Mq, nq)
                ops.gemm(f.W, ws.B64, ws.A64, a_tri=TRI_LOWER, M=Mq, N=nq, K=Mq)
                ops.cast2d(ws.A64, A, Mq, nq)
                ops.split_half(ws.A64, sc[3:4], ws.Ah, ws.Al, rows=Mq, cols=nq)
                ws.a_half = False
            else:
                ws.a_half = bool(HALF_A and need_C and DENSE_D)
                ops.gemm_tch((f.Wh, f.Wl), (ws.Kh, ws.Kl), None if ws.a_half else A, Mq, nq, Mq, sc[8:9], a_tri=TRI_LOWER, chunk=H,
                             Ch=(ws.Ah, ws.Al), c_scale=sc[3:4])                              # A = L^-1 K_zx (+ its split)
            if need_C and DENSE_D:
                ops.gemm_tch((ws.Dh, ws.Dl), (ws.Ah, ws.Al), C, Mq, nq, Mq, sc[13:14], chunk=H)   # C = (S - I) A, dense
                if ws.a_half:
                    ops.col_dots_half((ws.Ah, ws.Al), sc[3:4], P.m, ws.pm, ws.pv, Mq, nq, C, cmax=f.maxbits[5:6])
                else:
                    ops.col_dots(A, P.m, ws.pm, ws.pv, Mq, nq, C=C, cmax=f.maxbits[5:6])
            elif need_C:
                ops.gemm_tch((ws.ETh, ws.ETl), (ws.Ah, ws.Al), ws.Bp, Mq, nq, Mq, sc[9:10], a_tri=TRI_UPPER, chunk=H,
                             D2=A, C2h=(ws.Kh, ws.Kl), c2_scale=sc[4:5])                      # B' = E^T A ; split of B = A + B'
                ops.gemm_tch((ws.Eh, ws.El), (ws.Kh, ws.Kl), C, Mq, nq, Mq, sc[10:11], a_tri=TRI_LOWER, chunk=H, beta=1.0,
                             D=ws.Bp)                                                          # C = E B + B'
                ops.col_dots(A, P.m, ws.pm, ws.pv, Mq, nq, C=C, cmax=f.maxbits[5:6])
            else:
                ops.gemm_tch((ws.ETh, ws.ETl), (ws.Ah, ws.Al), ws.Bp, Mq, nq, Mq, sc[9:10], a_tri=TRI_UPPER, chunk=H)
                ops.col_dots(A, P.m, ws.pm, ws.pv, Mq, nq, Bp=ws.Bp)
            ops.predict_finish(ws.pm, ws.pv, nq, ws.p2, f.hyp, ws.mu, ws.var, add_noise, PRED_JITTER)
            return
        if tc:
            ops.gemm_tc(f.Wt, f.Wt_lo, Kzx, ws.lo1, A, Mq, nq, Mq, a_tri=TRI_LOWER, chunk=TC_CHUNK,
                        C_lo=ws.lo2)                                                     # A = L^-1 K_zx  (+ A_lo)
            ops.gemm_tc(ws.ET, ws.ET_lo, A, ws.lo2, ws.Bp, Mq, nq, Mq, a_tri=TRI_UPPER, chunk=TC_CHUNK,
                        C2=B if need_C else None, D2=A if need_C else None, C2_lo=ws.lo1 if need_C else None)
            if need_C:
                ops.gemm_tc(ws.E, ws.E_lo, B, ws.lo1, C, Mq, nq, Mq, a_tri=TRI_LOWER, beta=1.0, D=ws.Bp, chunk=TC_CHUNK)
                ops.col_dots(A, P.m, ws.pm, ws.pv, Mq, nq, C=C)
            else:
                ops.col_dots(A, P.m, ws.pm, ws.pv, Mq, nq, Bp=ws.Bp)
            ops.predict_finish(ws.pm, ws.pv, nq, ws.p2, f.hyp, ws.mu, ws.var, add_noise, PRED_JITTER)
            return
        ops.gemm(Engine._wt(f), Kzx, A, a_tri=TRI_LOWER, M=Mq, N=nq, K=Mq)               # A = L^-1 K_zx
        ops.gemm(ws.E, A, ws.Bp, ta=True, a_tri=TRI_UPPER, M=Mq, N=nq, K=Mq, C2=B if need_C else None,
                 D2=A if need_C else None)
        if need_C:
            ops.gemm(ws.E, B, C, a_tri=TRI_LOWER, beta=1.0, D=ws.Bp, M=Mq, N=nq, K=Mq)
            ops.col_dots(A, P.m, ws.pm, ws.pv, Mq, nq, C=C)
        else:
            ops.col_dots(A, P.m, ws.pm, ws.pv, Mq, nq, Bp=ws.Bp)                         # sum_i B^2 - A^2
        ops.predict_finish(ws.pm, ws.pv, nq, ws.p2, f.hyp, ws.mu, ws.var, add_noise, PRED_JITTER)

    # ----------------------------------------------------------------------------------------------- backward
    @staticmethod
    def _input_grads(ws, f, P, x, wx, dKzx):
        """d/dx and d/dVx (fp64, fresh) of the data side of K_zx from dK_zx.  They stay local to a minibatch shard: nothing here
        enters the buffers that are summed over ranks."""
        n, d = x.shape
        ws.gx = torch.zeros(n, d, dtype=F64, device=x.device)
        ws.gVx = torch.zeros(n * ws.p2, d, dtype=F64, device=x.device) if ws.p2 else None
        ops.kdir_bwd_cols(P.Z, f.uzT, ws.p, x, wx, ws.invx, ws.p2, f.hyp, dKzx, ws.gx, ws.gVx)

    @staticmethod
    def _input_grad_dict(ws, x, Vx, gmu, names):
        """{"x", "Vx", "y"} gradients in the model dtype (those in `names`): Vx gets exact zeros when the data side keeps no
        derivative rows (p2 = 0: Vx influences nothing), y gets -d/dmu (the Gaussian data terms depend on y - mu only)."""
        g = {}
        if "x" in names:
            g["x"] = ws.gx.to(x.dtype)
        if "Vx" in names:
            g["Vx"] = ws.gVx.to(x.dtype) if ws.gVx is not None else torch.zeros_like(Vx)
        if "y" in names:
            g["y"] = torch.neg(gmu)
        return g

    def _backward(self, ws, f, P, x, wx, gmu, gvar, add_noise, inv_num_data, reducer=None, want_inputs=False):
        """Gradients of a scalar whose derivatives w.r.t. (mean, variance) are (gmu, gvar), plus the KL gradient
        scaled by -inv_num_data.  Results: ws.gm, ws.gLs (model dtype), ws.small (double); with want_inputs also ws.gx, ws.gVx.

        Order: the Gram product G = A diag(g_var) A^T comes FIRST, because [G | t] is what has to be summed over ranks:
        its all-reduce is started as soon as G exists (reducer.begin) and runs underneath dK_zx = L^-T dA and the K_zx
        assembly backward (1.8 ms at C3, independent of G); the small fp64 buffer those two write into follows
        (reducer.end), and only then does the replicated tail need the sums."""
        T, Mq, nq = x.dtype, ws.Mq, ws.nq
        A, Ag, C, dKzx = ws.A, ws.B, ws.C, ws.Kzx
        ops.pred_bwd_scalars(gmu, gvar, ws.p2, f.hyp, add_noise, ws.sc[4:], ws.scratch)
        ws.gx = ws.gVx = None
        tc = ws.tc and f.tc
        if ws.tch and f.tch:
            # 3xFP16: scales of dA and A_g from max|m|, max|g_mu|, max|g_var|, max|C| (order-independent maxima: deterministic)
            sc = f.scales
            f.maxbits[1:4].zero_()
            ops.absmax(P.m, f.maxbits[1:2])
            ops.absmax(gmu, f.maxbits[2:3])
            ops.absmax(gvar, f.maxbits[3:4])
            ops.tc_scales(f.hyp, f.jitter, f.maxbits, Mq, sc, 1)
            # dA = m g_mu^T + 2 C diag(g_var) and A_g = A diag(g_var) leave only as two-half splits; t = A g_mu
            if getattr(ws, "a_half", False):
                ops.dA_apply_half(None, C, Mq, nq, P.m, gmu, gvar, ws.tp, ws.t, ws.Kh, ws.Kl, ws.Agh, ws.Agl, sc[5:6], sc[6:7],
                                  A_half=(ws.Ah, ws.Al), a_scale=sc[3:4])
            else:
                ops.dA_apply_half(A, C, Mq, nq, P.m, gmu, gvar, ws.tp, ws.t, ws.Kh, ws.Kl, ws.Agh, ws.Agl, sc[5:6], sc[6:7])
            ops.gemm_tch((ws.Agh, ws.Agl), (ws.Ah, ws.Al), ws.G, Mq, Mq, nq, sc[12:13], b_kmajor=True, c_lower=True,
                         chunk=TCH_CHUNK, nsplit=ws.syrk_split, split_ws=ws.split_ws)                                     # G = A_g A^T
            ops.mirror_lower(ws.G, Mq)
            if reducer is not None:
                reducer.begin(ws.big)
            if self._w64(ws):
                # dA = m g_mu^T + 2 C diag(g_var) in fp64 (torch glue on M' x n' numbers), dK_zx = W^T dA on DMMA
                torch.mul(C[:, :nq], gvar, out=ws.B64[:, :nq])
                ws.B64[:, :nq].mul_(2.0).addmm_(P.m.double().unsqueeze(1), gmu.double().unsqueeze(0))
                ops.gemm(f.W, ws.B64, ws.A64, ta=True, a_tri=TRI_UPPER, M=Mq, N=nq, K=Mq)
                ops.cast2d(ws.A64, dKzx, Mq, nq)
            else:
                # (under an overlapping all-reduce the collective's CTAs hold a few SMs when this product starts: the persistent
                # kernel's static work lists assume all pairs start together, one pair per tile absorbs the late SMs)
                under_reduce = reducer is not None and getattr(reducer, "overlap", False) and not PERSISTENT_UNDER_REDUCE
                if under_reduce:
                    ops.set_tc_persistent(False)
                try:
                    ops.gemm_tch((f.WTh, f.WTl), (ws.Kh, ws.Kl), dKzx, Mq, nq, Mq, sc[11:12], a_tri=TRI_UPPER, chunk=TCH_CHUNK)   # dK_zx = L^-T dA
                finally:
                    if under_reduce:
                        ops.set_tc_persistent(True)
            ops.kdir_bwd(P.Z, f.uzT, f.invzT, ws.p, x, wx, ws.p2, f.hyp, dKzx, ws.gZ, ws.gVz, ws.sc[4:6])
            if want_inputs:
                self._input_grads(ws, f, P, x, wx, dKzx)
            # (E, E^T as fp32 + lo for the two M'^3 products of the tail were made by _assemble)
        else:
            ops.dA_apply(A, C, Ag, Mq, nq, P.m, gmu, gvar, ws.tp, ws.t,                  # C <- dA ; Ag ; t = A gmu
                         C_lo=ws.lo1 if tc else None, Ag_lo=ws.lo3 if tc else None)      # (+ their lo parts)
            if tc:                                                                       # G = A diag(gvar) A^T
                # (A_lo is still in ws.lo2 from the forward pass)
                ops.gemm_tc(Ag, ws.lo3, A, ws.lo2, ws.G, Mq, Mq, nq, b_kmajor=True, c_lower=True, chunk=TC_CHUNK,
                            nsplit=ws.syrk_split, split_ws=ws.split_ws)
            else:
                ops.gemm(Ag, A, ws.G, tb=True, c_tri=1, M=Mq, N=Mq, K=nq)
            ops.mirror_lower(ws.G, Mq)
            if reducer is not None:
                reducer.begin(ws.big)
            if tc:
                ops.gemm_tc(f.WtT, f.WtT_lo, C, ws.lo1, dKzx, Mq, nq, Mq, a_tri=TRI_UPPER, chunk=TC_CHUNK)   # dK_zx = L^-T dA
            else:
                ops.gemm(self._wt(f), C, dKzx, ta=True, a_tri=TRI_UPPER, M=Mq, N=nq, K=Mq)
            ops.kdir_bwd(P.Z, f.uzT, f.invzT, ws.p, x, wx, ws.p2, f.hyp, dKzx, ws.gZ, ws.gVz, ws.sc[4:6])
            if want_inputs:
                self._input_grads(ws, f, P, x, wx, dKzx)
        if reducer is not None:
            reducer.end(ws.small)
        self._backward_tail(ws, f, P, T, inv_num_data, reducer)

    def _backward_tail(self, ws, f, P, T, inv_num_data, reducer=None):
        """The O(M'^3) part of the backward pass, identical on every rank: from G (symmetric, with dA A^T = m t^T + 2 (S - I) G),
        t = A g_mu and the K_zx contributions already in ws.small to the gradients of m, L_s, Z, V_z, ell, os."""
        Mq = ws.Mq
        tc = ws.tc and f.tc
        # ---- replicated tail: O(M'^3), identical on every rank
        W = f.W
        if tc:
            ops.split_lo(ws.G, ws.G_lo)
            ops.gemm_tc(ws.ET, ws.ET_lo, ws.G, ws.G_lo, ws.Hp, Mq, Mq, Mq, a_tri=TRI_UPPER, chunk=TC_CHUNK, C2=ws.H,
                        D2=ws.G, C2_lo=ws.H_lo)                                          # H = L_s^T G = G + E^T G
            ops.gemm_tc(ws.E, ws.E_lo, ws.H, ws.H_lo, ws.X, Mq, Mq, Mq, a_tri=TRI_LOWER, alpha=2.0, beta=2.0, D=ws.Hp,
                        chunk=TC_CHUNK)                                                  # 2 (S - I) G
        else:
            ops.gemm(ws.E, ws.G, ws.Hp, ta=True, a_tri=TRI_UPPER, M=Mq, N=Mq, K=Mq, C2=ws.H, D2=ws.G)
            ops.gemm(ws.E, ws.H, ws.X, a_tri=TRI_LOWER, alpha=2.0, beta=2.0, D=ws.Hp, M=Mq, N=Mq, K=Mq)
        # X + m t^T = dA A^T enters only through Phi(.): one pass writes the lower triangle of Psi in fp64 (ops.phi_outer)
        # Cholesky backward composed with the whitening backward.  With U = L^-T X (X = dA A^T), dL = -tril(U) and
        # L^T dL = -L^T (U - su(U)) = -X + L^T su(U), where su = strictly upper part; L^T (upper) times a strictly upper matrix
        # is strictly upper, so  tril(L^T dL) = -tril(X)  EXACTLY and  dK_zz = sym(L^-T Phi(L^T dL) L^-1) = -sym(W^T Phi(X) W):
        # the two M'^3 fp64 products dL = -tril(W^T X) and Y = L^T dL of round 1 are not needed at all (0.78 ms of 2.1 at C3).
        ops.phi_outer(ws.X, P.m, ws.t, ws.Psi, Mq)                        # lower triangle of Phi(X + m t^T): tril, halved diagonal
        shards = self._tail_shards(reducer)
        if shards is None:
            ops.gemm(ws.Psi, W, ws.Y, a_tri=TRI_LOWER, b_tri=TRI_LOWER, c_tri=1, alpha=-1.0, M=Mq, N=Mq, K=Mq)   # Y = -Phi(X) W (lower)
            ops.gemm(W, ws.Y, ws.S, ta=True, a_tri=TRI_UPPER, b_tri=TRI_LOWER, M=Mq, N=Mq, K=Mq)          # W^T (-Phi(X) W)
            ops.symmetrize(ws.S, Mq)
            ops.kdir_bwd(P.Z, f.uz64, f.invz64, ws.p, P.Z, f.uz64, ws.p, f.hyp, ws.S, ws.gZ, ws.gVz, ws.sc[4:6],
                         scale=2.0)
        else:
            # N > 1: the two fp64 products and the K_zz assembly backward are SHARDED over the ranks by column panels of
            # dK_zz (every rank holds X, W; panel J of Y = -Phi(X) W and of S = W^T Y needs nothing from the other panels),
            # and what is summed over ranks is the contraction of S[:, J] with dK_zz/d(Z, V_z, ell, os) -- 250 KB -- instead
            # of the replicated 1.3 ms of DMMA work.  sum_ij S_ij dK_ij needs no symmetrisation (dK/dtheta is symmetric):
            # row side + column side of the unsymmetrised panel.
            ws.small2.zero_()
            for rank, world in shards:
                for c0, c1 in self.tail_panels(Mq, ws.p + 1, rank, world):
                    self._tail_panel(ws, f, P, c0, c1)
            if reducer is not None:
                reducer.reduce_tail(ws.small2)
            ws.small.add_(ws.small2)
        # (fresh outputs every step: they are handed to autograd as they are, see _collect)
        ws.gm, ws.gLs = torch.empty(Mq, dtype=T, device=ws.small.device), torch.empty(Mq, Mq, dtype=T, device=ws.small.device)
        ops.var_grads(ws.H, P.Ls_raw, ws.t, P.m, inv_num_data, ws.gm, ws.gLs)

    tail_shards_debug = None      # tests: a world size whose panels THIS process loops over (single-GPU check of the sharded tail)

    def _tail_shards(self, reducer):
        """[(rank, world), ...] whose column panels of the tail this process computes, or None for the unsharded tail"""
        if self.tail_shards_debug:
            return [(r, self.tail_shards_debug) for r in range(self.tail_shards_debug)]
        if reducer is not None and getattr(reducer, "world", 1) > 1 and getattr(reducer, "shard_tail", True):
            return [(reducer.rank, reducer.world)]
        return None

    @staticmethod
    def tail_panels(Mq, q, rank, world):
        """Column panels [c0, c1) of dK_zz owned by `rank`: 2 * world blocks of whole inducing points (q = p + 1 columns
        each); block b and block 2 * world - 1 - b go to the same rank, because the cost of a panel falls with c0 (only
        rows >= c0 of the lower-triangular factors take part)."""
        M, nb = Mq // q, 2 * world
        bounds = [(M * b) // nb * q for b in range(nb + 1)]
        return [(bounds[b], bounds[b + 1]) for b in (rank, nb - 1 - rank) if bounds[b + 1] > bounds[b]]

    @staticmethod
    def _tail_panel(ws, f, P, c0, c1):
        """contribution of the column panel J = [c0, c1) of dK_zz = -W^T Phi(X) W to d(Z, V_z, ell, os), into ws.small2"""
        Mq, p, q = ws.Mq, ws.p, ws.p + 1
        W, nJ, Kk = f.W, c1 - c0, ws.Mq - c0
        Yp = ws.Y[c0:, c0:c1]                              # only rows >= c0 of Y[:, J] are non-zero (lower x lower)
        ops.gemm(ws.Psi[c0:, c0:], W[c0:Mq, c0:c1], Yp, a_tri=TRI_LOWER, b_tri=TRI_LOWER, c_tri=1, alpha=-1.0, M=Kk, N=nJ, K=Kk)
        if c0 > 0:                                         # S[:c0, J] = W[c0:, :c0]^T Y[c0:, J]   (dense block of W)
            ops.gemm(W[c0:Mq, :c0], Yp, ws.S[:c0, c0:c1], ta=True, b_tri=TRI_LOWER, M=c0, N=nJ, K=Kk)
        ops.gemm(W[c0:Mq, c0:Mq], Yp, ws.S[c0:, c0:c1], ta=True, a_tri=TRI_UPPER, b_tri=TRI_LOWER, M=Kk, N=nJ, K=Kk)
        j0, j1 = c0 // q, c1 // q                          # the inducing points of the panel
        Sp = ws.S[:, c0:c1]
        uz, iz = f.uz64, f.invz64
        sl = slice(j0 * p, j1 * p)
        gZ2, gV2, sc2 = ws.gZ2, ws.gVz2, ws.small2[4:6]
        ops.kdir_bwd(P.Z, uz, iz, p, P.Z[j0:j1], uz[sl] if p else None, p, f.hyp, Sp, gZ2, gV2, sc2)                 # row side
        ops.kdir_bwd(P.Z[j0:j1], uz[sl] if p else None, iz[sl] if p else None, p, P.Z, uz, p, f.hyp, Sp, gZ2[j0:j1],
                     gV2[sl] if p else None, None, dk_trans=True)                                                    # column side

    @staticmethod
    def _collect(ws, f, P, T, noise_mode):
        """dict of gradients shaped like the parameters (device ops only, no sync).  noise_mode 1: d noise = explicit ELBO term +
        the term through the variance (training step), 0: through the variance only (generic predictive backward).
        Every entry is a fresh tensor (ws.small is zeroed by the next step: two forwards before one backward must not read it
        -- VERDICT r01 weak #4): the small ones are views of ONE buffer filled by ONE launch (collect_grads; they used to be
        ~20 one-microsecond torch kernels at the very end of the step, 0.1 ms of launch latency), m / L_s were written into
        fresh tensors by var_grads."""
        M, d, p = ws.M, ws.d, ws.p
        nZ, nV = M * d, M * p * d
        out = torch.empty(nZ + nV + 4, dtype=T, device=ws.small.device)
        ops.collect_grads(ws.small, nZ, nV, f.hyp, noise_mode, out)
        g = {"Z": out[:nZ].view(M, d), "m": ws.gm, "Ls_raw": ws.gLs, "c": out[nZ + nV].reshape(P.c.shape),
             "raw_os": out[nZ + nV + 1].reshape(P.raw_os.shape), "raw_ell": out[nZ + nV + 2].reshape(P.raw_ell.shape)}
        if ws.gVz is not None:
            g["Vz"] = out[nZ:nZ + nV].view(M * p, d)
        if P.raw_noise is not None:
            g["raw_noise"] = out[nZ + nV + 3].reshape(P.raw_noise.shape)
        return g

    # ------------------------------------------------------------------------------------------ public: train
    def elbo_step(self, P, x, Vx, y, num_data, p, p2, through_likelihood=True, n_global=None, want_grads=True,
                  objective="elbo", include_kl=True, reducer=None, input_grads=()):
        """One fused forward(+backward) of VariationalELBO(likelihood, model, num_data)(likelihood(model(x)), y)
        -- or, objective="pll", of PredictiveLogLikelihood (directional_vi.py:218-219).

        Returns (objective value [0-dim float64 tensor], grads dict or None, mean, variance).  `through_likelihood`
        is the number of times likelihood() has been applied to the distribution whose variance the data term sees
        (bool or int): 1 for the ELBO on likelihood(model(x)) (directional_vi.py:245, Q3); for PLL the caller counts
        log_marginal's own application too (2 in the reference loop).  `variance` includes that many noises.
        include_kl=False leaves the KL term (value and gradient) to the caller: the shared-direction strategy's q(u) lives
        on M + p values, not on the M(p+1) inducing values the step sees.
        reducer (distributed.Reducer or None): sums [G | t] and the small fp64 buffer over the ranks of a sharded step.
        input_grads: names among "x", "Vx", "y" whose gradients the grads dict should also carry (this shard's own)."""
        self._validate(P, x, Vx, p, p2, y)
        T, dev = x.dtype, x.device
        n, d = x.shape
        M = P.Z.shape[0]
        ws = self.workspace(dev, T, n, d, M, p, p2)
        f = self.factor(dev, T, d, M, p)
        f.valid = False
        nq_global = (n_global if n_global is not None else n) * (p2 + 1)
        # Host order.  The factorisation is the critical path of a step and, when the caller reads the loss back every step, the
        # GPU is idle until its first diagonal block is launched: everything that block does not need (data-side directions,
        # fp32 inducing directions, operand scales -- 0.2 ms of host time, scratch/host_latency.py) is enqueued AFTER the chain,
        # on the side stream, where the K_zx assembly and the L_s operands (which do not depend on the factor either) run
        # underneath the latency-bound Cholesky (32 sequential diagonal blocks leave most SMs idle).
        self._hyp(f, P)
        if f.p:
            f.uz64, f.invz64 = ops.normalize_dirs(P.Vz, F64)
        cur, side = torch.cuda.current_stream(dev), self._side_stream(dev)
        capturing = torch.cuda.is_current_stream_capturing()
        fork = torch.cuda.Event() if capturing else self._fork_event(dev)
        fork.record(cur)
        wx = None
        for extra in (0.0,) + CHOL_RETRY:
            if extra == 0.0:
                self._factorise_enqueue(f, P, 0.0)
                scales_ready = None
                side.wait_event(fork)
                with torch.cuda.stream(side):
                    if f.p:
                        f.uzT, f.invzT = (f.uz64, f.invz64) if T == F64 else ops.normalize_dirs(P.Vz, T)
                    wx = self._data_dirs(ws, Vx, T)
                    # (allocated while the side stream is current, read by kernels of the caller's stream later in the step:
                    #  tell the caching allocator, so that a freed block is not handed out again before those have run)
                    for t_ in (wx, ws.invx, *((f.uzT, f.invzT) if (f.p and T != F64) else ()), *(ws.canon or ())):
                        if t_ is not None:
                            t_.record_stream(cur)
                    if f.tch:
                        self._scales0(f, P, KZZ_JITTER)
                        scales_ready = torch.cuda.Event() if capturing else self._scales_event(dev)
                        scales_ready.record(side)
                self._factorise_finish(f, T, scales_ready)
                with torch.cuda.stream(side):
                    if DEFER_SIDE_WORK:
                        # the first ~10 links of the chain are bound by their trailing updates (the GPU is full) and only the later
                        # ones leave the SMs idle: the assembly and the L_s operand products start beside THOSE
                        ops.chol_wait_mid()
                    self._assemble(ws, f, P, x, wx)
                    ws.kl.zero_()                      # KL(q(u) || p(u)) needs the parameters only: also under the Cholesky
                    if include_kl:
                        ops.kl_divergence(P.m, P.Ls_raw, ws.kl, ws.scratch_kl)
                cur.wait_stream(side)
            else:
                if f.tch:
                    self._scales0(f, P, KZZ_JITTER + extra)
                self._factorise(f, P, T, extra, prep=False)
            self._forward(ws, f, P, x, wx, through_likelihood, need_C=True, assembled=(extra == 0.0))
            ws.small.zero_()
            if objective == "pll":
                ops.pll_terms(ws.mu, ws.var, y, 1.0 / nq_global, ws.gmu, ws.gvar, ws.sc, ws.scratch)
            else:
                ops.elbo_terms(ws.mu, ws.var, y, f.hyp, 1.0 / nq_global, ws.gmu, ws.gvar, ws.sc, ws.scratch)
            want_inputs = "x" in input_grads or "Vx" in input_grads
            if want_grads or want_inputs:
                self._backward(ws, f, P, x, wx, ws.gmu, ws.gvar, through_likelihood, (1.0 / num_data) if include_kl else 0.0,
                               reducer, want_inputs)
            elif reducer is not None:
                reducer.end(ws.small)
            # everything the caller gets is enqueued BEFORE the one host synchronisation of the step (the Cholesky status
            # read), so the GPU never waits for the host at the end of a step
            elbo = ws.sc[0] - ws.kl[0] / num_data
            grads = self._collect(ws, f, P, T, 1) if (want_grads or want_inputs) else None
            if input_grads:
                grads = {**(grads or {}), **self._input_grad_dict(ws, x, Vx, ws.gmu, input_grads)}
            mean, var = ws.mu.clone(), ws.var.clone()
            if capturing:
                # CUDA-graph capture: no host synchronisation inside the captured region.  The factorisation status stays in
                # f.info (device); whoever replays the graph reads it afterwards and, if the unjittered factorisation failed,
                # re-runs the step eagerly through the psd_safe_cholesky ladder (graphs.GraphedStep).
                break
            if self._check(f, P):
                break
        else:
            raise NotPSDError("K_zz is not positive definite after adding jitter up to 1e-4 (psd_safe_cholesky ladder)")
        return elbo, grads, mean, var

    # --------------------------------------------------------------------------- public: differentiable q(f)
    def predictive_forward(self, P, x, Vx, p, p2, add_noise):
        """mean, variance of q(f) (+ noise), keeping A and C for predictive_backward (generic autograd path)."""
        self._validate(P, x, Vx, p, p2)
        T = x.dtype
        n, d = x.shape
        ws = self.workspace(x.device, T, n, d, P.Z.shape[0], p, p2)
        f = self.factor(x.device, T, d, P.Z.shape[0], p)
        f.valid = False
        ws.wx = self._data_dirs(ws, Vx, T)
        for extra in (0.0,) + CHOL_RETRY:
            self._factorise(f, P, T, extra)
            self._forward(ws, f, P, x, ws.wx, add_noise, need_C=True)
            if self._check(f, P):
                return (ws, f), ws.mu.clone(), ws.var.clone()
        raise NotPSDError("K_zz is not positive definite after adding jitter up to 1e-4 (psd_safe_cholesky ladder)")

    def predictive_backward(self, ctx, P, x, gmu, gvar, add_noise, Vx=None, input_grads=()):
        """input_grads: names among "x", "Vx" whose gradients the returned dict should also carry."""
        ws, f = ctx
        ws.small.zero_()
        min_var = 1e-10 if x.dtype == F64 else 1e-6
        gvar = torch.where(ws.var > min_var, gvar, torch.zeros_like(gvar)).contiguous()
        self._backward(ws, f, P, x, ws.wx, gmu.contiguous(), gvar, add_noise, 0.0, want_inputs=bool(input_grads))
        grads = self._collect(ws, f, P, x.dtype, 0)
        if input_grads:
            grads.update(self._input_grad_dict(ws, x, Vx, None, input_grads))
        return grads

    # ------------------------------------------------------------------------------------------ public: eval
    @staticmethod
    def _owner_token(P):
        """identity + in-place version of every parameter the factor depends on"""
        return tuple((t.data_ptr(), t._version) for t in (P.Z, P.Vz, P.raw_ell, P.raw_os) if t is not None)

    def predict(self, P, x, Vx, p, p2, add_noise, reuse_factor=False):
        """eval_gp's per-batch prediction (directional_vi.py:296-298).  reuse_factor: eval-mode memoisation of
        the Cholesky factor (DGVS.py:72) -- K_zz is factorised once and reused until the strategy invalidates it."""
        self._validate(P, x, Vx, p, p2)
        T = x.dtype
        n, d = x.shape
        M = P.Z.shape[0]
        ws = self.workspace(x.device, T, n, d, M, p, p2)
        f = self.factor(x.device, T, d, M, p)
        token = self._owner_token(P)
        if not (reuse_factor and f.valid and f.owner == token):
            f.valid = False
            for extra in (0.0,) + CHOL_RETRY:
                self._factorise(f, P, T, extra)
                if self._check(f, P):
                    break
            else:
                raise NotPSDError("K_zz is not positive definite after adding jitter up to 1e-4")
            f.valid = reuse_factor
            f.owner = token
        else:
            self._hyp(f, P)        # the memoised factor does not depend on the noise / mean constant; hyp[2:4] do
            if f.tch:
                self._scales0(f, P)
        wx = self._data_dirs(ws, Vx, T)
        self._forward(ws, f, P, x, wx, add_noise, need_C=False)
        return ws.mu.clone(), ws.var.clone()

    # ----------------------------------------------------------- public: full predictive covariance and samples
    def predict_full(self, P, x, Vx, p, p2, add_noise, reuse_factor=False, return_ctx=False):
        """mean (n') and the dense n' x n' covariance of q(f(X)) [+ noise]:
        K_xx + 1e-4 I + A^T (S - I) A  (DGVS.py:192-205; SURVEY section 8f rank 4 -- what `preds.sample` of the BO
        callers consumes, experiments/rover/test_turbo.py:119-150).  The training path never forms this matrix."""
        self._validate(P, x, Vx, p, p2)
        T = x.dtype
        n, d = x.shape
        M = P.Z.shape[0]
        ws = self.workspace(x.device, T, n, d, M, p, p2)
        f = self.factor(x.device, T, d, M, p)
        token = self._owner_token(P)
        if not (reuse_factor and f.valid and f.owner == token):
            f.valid = False
            for extra in (0.0,) + CHOL_RETRY:
                self._factorise(f, P, T, extra)
                if self._check(f, P):
                    break
            else:
                raise NotPSDError("K_zz is not positive definite after adding jitter up to 1e-4")
            f.valid = reuse_factor
            f.owner = token
        else:
            self._hyp(f, P)
            if f.tch:
                self._scales0(f, P)
        wx = self._data_dirs(ws, Vx, T)
        self._forward(ws, f, P, x, wx, add_noise, need_C=True)
        nq, Mq = ws.nq, ws.Mq
        cov = torch.empty(nq, _round_up(nq, 4), dtype=T, device=x.device)[:, :nq]
        ops.kdir_fwd(x, wx, p2, x, wx, p2, f.hyp, cov, diag_add=PRED_JITTER)
        if add_noise:
            cov.diagonal().add_((f.hyp[2] * int(add_noise)).to(T))
        ops.gemm(ws.A, ws.C, cov, ta=True, beta=1.0, M=nq, N=nq, K=Mq)            # += A^T (S - I) A
        if return_ctx:
            ws.wx = wx
            return (ws, f), ws.mu.clone(), cov
        return ws.mu.clone(), cov

    # ----------------------------------------------------------------- public: differentiable FULL predictive covariance
    def full_forward(self, P, x, Vx, p, p2, add_noise):
        """(ctx, mean, dense covariance) with everything full_backward needs kept in the workspace: the differentiable form of
        predict_full (the reference's lazy predictive covariance is differentiable, DGVS.py:192-208)."""
        return self.predict_full(P, x, Vx, p, p2, add_noise, reuse_factor=False, return_ctx=True)

    def full_backward(self, ctx, P, x, gmean, gcov, add_noise, Vx=None, input_grads=()):
        """Gradients of a scalar whose derivatives w.r.t. (mean, covariance) of q(f(X)) are (gmean, gcov).
        Sigma = K_xx + 1e-4 I + A^T D A (+ noise), D = S - I:  with Gs = gcov + gcov^T,
            dA = m gmean^T + D (A Gs),   G = 1/2 (A Gs) A^T  (then dA A^T = m t^T + 2 D G, t = A gmean, dL_s = tril(2 G L_s)),
        i.e. the same (dA, G, t) interface as the diagonal case, after which dK_zx = W^T dA, the assembly backward and the
        O(M'^3) tail are the training step's own (_backward_tail).  K_xx contributes to the lengthscale / outputscale only.
        Evaluation sizes (BO candidates: n' of a few hundred to a few thousand): every product on the generic mma.sync GEMM.
        input_grads: names among "x", "Vx" whose gradients the returned dict should also carry; x and Vx enter through K_zx
        and through the dense K_xx (whose diagonal does not depend on them)."""
        ws, f = ctx
        T, Mq, nq = x.dtype, ws.Mq, ws.nq
        wx = ws.wx
        ws.small.zero_()
        if ws.B is None:                              # (the 3xFP16 training path has no use for this M' x n' buffer)
            ws.B = torch.empty(Mq, ws.ldn, dtype=T, device=x.device)
        A, AG, Bp, B2 = ws.A, ws.B, ws.Bp, ws.Kzx
        gmean = gmean.contiguous()
        Gs = (gcov + gcov.transpose(0, 1)).contiguous()
        ops.pred_bwd_scalars(gmean, gcov.diagonal().contiguous(), ws.p2, f.hyp, add_noise, ws.sc[4:], ws.scratch)   # d noise, d c
        ops.gemm(A, Gs, AG, M=Mq, N=nq, K=nq)                                                   # A Gs
        torch.mv(A[:, :nq], gmean, out=ws.t)                                                    # t = A gmean
        ops.gemm(AG, A, ws.G, tb=True, alpha=0.5, M=Mq, N=Mq, K=nq)                             # G = 1/2 (A Gs) A^T (symmetric)
        # D (A Gs) without forming D:  B' = E^T Y,  D Y = E (Y + B') + B'   (E = tril(L_s) - I; no cancellation against Y)
        ops.gemm(ws.E, AG, Bp, ta=True, a_tri=TRI_UPPER, M=Mq, N=nq, K=Mq, C2=B2, D2=AG)
        ops.gemm(ws.E, B2, Bp, a_tri=TRI_LOWER, beta=1.0, M=Mq, N=nq, K=Mq)
        Bp[:, :nq].addr_(P.m, gmean)                                                            # dA = m gmean^T + D A Gs
        dKzx = ws.Kzx
        ops.gemm(self._wt(f), Bp, dKzx, ta=True, a_tri=TRI_UPPER, M=Mq, N=nq, K=Mq)             # dK_zx = L^-T dA
        ops.kdir_bwd(P.Z, f.uzT, f.invzT, ws.p, x, wx, ws.p2, f.hyp, dKzx, ws.gZ, ws.gVz, ws.sc[4:6])
        ws.gx = ws.gVx = None
        if input_grads:
            self._input_grads(ws, f, P, x, wx, dKzx)
        # K_xx: of the parameters only the kernel hyper-parameters depend on it.  Its DIAGONAL (closed form in ell, os) is already in
        # pred_bwd_scalars' terms above: the assembly backward gets the off-diagonal part.
        goff = gcov.clone()
        goff.diagonal().zero_()
        ops.kdir_bwd(x, wx if ws.p2 else None, None, ws.p2, x, wx if ws.p2 else None, ws.p2, f.hyp, goff, None, None, ws.sc[4:6])
        if input_grads:
            # x (and Vx) are both arguments of K_xx(x, x): the gradient w.r.t. the second equals the row-side gradient of the
            # transposed upstream block, so the two sides are one row-side pass over goff + goff^T
            gsym = goff + goff.transpose(0, 1)
            ops.kdir_bwd(x, wx if ws.p2 else None, ws.invx, ws.p2, x, wx if ws.p2 else None, ws.p2, f.hyp, gsym, ws.gx, ws.gVx, None)
        self._backward_tail(ws, f, P, T, 0.0)
        grads = self._collect(ws, f, P, T, 0)
        if input_grads:
            grads.update(self._input_grad_dict(ws, x, Vx, None, input_grads))
        return grads

    def sample_mvn(self, mean, cov, num_samples, generator=None, base=None, keep=False):
        """num_samples draws of N(mean, cov): fp64 Cholesky of cov on the library's own blocked factorisation (same
        jitter ladder as psd_safe_cholesky), then mean + z L^T as one triangular product.  base: fp64 (num_samples, n')
        standard normals used as z instead of fresh ones.  keep: also return (L, W, z, jitter) for sample_backward, with
        L, W = L^-1 the padded Mp x Mp factors (the identity padding decouples their leading n' x n' block)."""
        nq = mean.shape[0]
        dev = mean.device
        Mp, nb0, nlev = ops.chol_plan(nq)
        work, L, W = (torch.empty(Mp, Mp, dtype=F64, device=dev) for _ in range(3))
        info = torch.zeros(1, dtype=torch.int32, device=dev)
        for extra in (0.0, 1e-8, 1e-6, 1e-5, 1e-4):
            if Mp > nq:
                ops.pad_identity(work, nq)
            work[:nq, :nq] = cov
            if extra:
                work.diagonal()[:nq].add_(extra)
            ops.cholesky_inverse(work, L, W, nb0, nlev, info)
            if int(info.item()) == 0:
                break
        else:
            raise NotPSDError("the predictive covariance is not positive definite after adding jitter up to 1e-4")
        z = torch.randn(num_samples, nq, dtype=F64, device=dev, generator=generator) if base is None else base
        out = torch.empty(num_samples, nq, dtype=F64, device=dev)
        ops.gemm(z, L, out, tb=True, b_tri=TRI_UPPER, M=num_samples, N=nq, K=nq)      # z L^T
        res = (out + mean.to(F64)).to(mean.dtype)
        return (res, (L, W, z, extra)) if keep else res

    def sample_backward(self, L, W, z, gout, want_base=False):
        """Gradients of draws = mean + z L^T (sample_mvn with keep=True) given gout = dloss/d draws (num, n'):
        (d mean, d cov, d z or None).  d L = tril(gout^T z) and d cov = sym(W^T Phi(L^T dL) W) (ops.chol_backward); the
        jitter of the factorisation is a constant, so d cov is the gradient w.r.t. the covariance the caller passed."""
        num, nq = z.shape
        dev = z.device
        gout = gout.to(F64).contiguous()
        gmean = gout.sum(0)
        Lbar = torch.empty(nq, _round_up(nq, 2), dtype=F64, device=dev)[:, :nq]
        ops.gemm(gout, z, Lbar, ta=True, c_tri=1, M=nq, N=nq, K=num)               # lower triangle of gout^T z
        gcov = torch.empty(nq, _round_up(nq, 2), dtype=F64, device=dev)[:, :nq]
        ops.chol_backward(L[:nq, :nq], W[:nq, :nq], Lbar, gcov, nq)
        gz = None
        if want_base:
            gz = torch.empty(num, nq, dtype=F64, device=dev)
            ops.gemm(gout, L, gz, b_tri=TRI_LOWER, M=num, N=nq, K=nq)                # gout L
        return gmean, gcov, gz

    def invalidate(self):
        for f in self._fac.values():
            f.valid = False


ENGINE = Engine()
