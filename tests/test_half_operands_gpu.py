"""The operands of the fp32 model's 3xFP16 training step, kernel by kernel, against fp64 references.

Every tensor-core operand of that step is the two-half split (hi, lo) of x * s, s a power of two per matrix
(csrc/tc_prep.cu).  A wrong lo half, an off-by-one scale exponent or a dropped odd column costs ~2^-12 on a few elements:
far below the step's 1e-4 gate once summed into gradients.  So each kernel is checked here on its own, at the shapes
where kernels go wrong (ragged tiles, odd columns, leading dimensions that rule out vector accesses, misaligned views):

  * output padding holds a sentinel (NaN; fp16 0x7C01) that must survive the call -- out-of-bounds writes;
  * inputs the kernel must not read (upper triangles, padding columns) are NaN -- the result must stay finite;
  * a split of an fp32 value the test can reproduce exactly is compared bit for bit with _split_ref; otherwise
    |hi + lo - v| <= 2^-22 |v| + 2^-25 elementwise (the split gate).

The last part runs whole steps on 3xFP16 whitening (engine.WHITEN_FP64 = False) at ragged shapes, and audits the fp16
range of every operand of a real step."""
import math
from contextlib import contextmanager

import numpy as np
import pytest
import torch

from oracle import dsvgp_oracle as O
from test_kernels_gpu import _split_ref, rel
from test_step_gpu import check_against, run_step

pytestmark = pytest.mark.gpu
F16, F32, F64 = torch.float16, torch.float32, torch.float64
NAN16 = 0x7C01                       # an fp16 NaN: the padding sentinel of half buffers
INT = {F16: torch.int16, F32: torch.int32, F64: torch.int64}


@pytest.fixture(scope="module")
def ops():
    from dsvgp_b200 import ops
    return ops


def _round_up(a, b):
    return (a + b - 1) // b * b


def _buf(rows, cols, ld, dtype):
    """(full, view): a rows x ld buffer filled with the sentinel, and its rows x cols view"""
    if dtype == F16:
        full = torch.full((rows, ld), NAN16, dtype=torch.int16, device="cuda").view(F16)
    else:
        full = torch.full((rows, ld), float("nan"), dtype=dtype, device="cuda")
    return full, full[:, :cols]


def _poisoned(t, ld, dtype=None, upper=False, col0=0):
    """t copied into a NaN buffer of leading dimension ld (from column col0 on: a misaligned view when col0 > 0);
    upper=True also poisons the entries above the diagonal"""
    dtype = dtype or t.dtype
    rows, cols = t.shape
    full, _ = _buf(rows, col0 + cols, ld, dtype)
    v = full[:, col0:col0 + cols]
    v.copy_(t.to(dtype))
    if upper:
        v.masked_fill_(torch.ones(rows, cols, dtype=torch.bool, device="cuda").triu(1), float("nan"))
    return full, v


def _pad_kept(full, cols, col0=0):
    """the columns of `full` outside [col0, cols) still hold the sentinel"""
    for pad in (full[:, cols:], full[:, :col0]):
        if full.dtype == F16 and not bool((pad.view(torch.int16) == NAN16).all()):
            return False
        if full.dtype != F16 and not bool(torch.isnan(pad).all()):
            return False
    return True


def _same_bits(a, b):
    return torch.equal(a.contiguous().view(INT[a.dtype]), b.contiguous().view(INT[b.dtype]))


def _split_gate(hi, lo, v, extra=0.0):
    """max over elements of |hi + lo - v| - (2^-22 |v| + 2^-25 + extra); <= 0 passes"""
    v = v.double()
    err = (hi.double() + lo.double() - v).abs()
    return float((err - (2.0 ** -22 * v.abs() + 2.0 ** -25 + extra)).max())


def _pow2_for(x, top=14):
    """a power of two that maps max|x| to (2^(top-1), 2^top]"""
    return 2.0 ** (top - math.ceil(math.log2(float(x.abs().max()))))


def _scale(s):
    return torch.tensor([s], dtype=F32, device="cuda")


# ----------------------------------------------------------------------------------------------------------- split_half
@pytest.mark.parametrize("rows,cols", [(1, 1), (33, 65), (129, 300), (3072, 3072)])
@pytest.mark.parametrize("trans", [False, True])
@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("sdt", [F32, F64])
def test_split_half_is_bit_exact(ops, sdt, mode, trans, rows, cols):
    """hi, lo (and their transposes) = _split_ref(op(src).float() * s) bit for bit, op = identity / tril / tril - I"""
    g = torch.Generator(device="cuda").manual_seed(rows + 7 * cols + mode)
    X = torch.randn(rows, cols, generator=g, dtype=F64, device="cuda")
    X[:, ::7] *= 1e-4                                       # entries whose lo half is an fp16 subnormal
    if mode == 2:
        X = 0.05 * X + torch.eye(rows, cols, dtype=F64, device="cuda")
    _, src = _poisoned(X, cols + 3, sdt, upper=mode != 0)
    s = 2.0 ** 9
    ld = cols + 3 if rows % 2 else _round_up(cols, 64)      # odd and 64-aligned leading dimensions
    (hf, hi), (lf, lo) = _buf(rows, cols, ld, F16), _buf(rows, cols, ld, F16)
    (hTf, hiT), (lTf, loT) = _buf(cols, rows, rows + 5, F16), _buf(cols, rows, rows + 5, F16)
    ops.split_half(src, _scale(s), hi, lo, mode=mode, hiT=hiT if trans else None, loT=loT if trans else None)
    v = X.to(sdt).float()                                   # the kernel's order: fp32 first, then tril, then - 1
    if mode:
        v = v.tril()
    if mode == 2:
        v = v - torch.eye(rows, cols, dtype=F32, device="cuda")
    rh, rl = _split_ref(v, s)
    assert _same_bits(hi, rh) and _same_bits(lo, rl)
    if mode:
        up = torch.ones(rows, cols, dtype=torch.bool, device="cuda").triu(1)
        assert bool((hi.view(torch.int16)[up] == 0).all()) and bool((lo.view(torch.int16)[up] == 0).all())
    assert _pad_kept(hf, cols) and _pad_kept(lf, cols)
    if trans:
        assert _same_bits(hiT, hi.T) and _same_bits(loT, lo.T)
        assert _pad_kept(hTf, rows) and _pad_kept(lTf, rows)
    else:
        assert _pad_kept(hTf, 0) and _pad_kept(lTf, 0)


# ------------------------------------------------------------------------------------ D = S - I = E + E^T + E E^T
@pytest.mark.parametrize("n", [1, 255, 257, 3072])
def test_build_d_absmax_and_split(ops, n):
    g = torch.Generator(device="cuda").manual_seed(n)
    Ls = torch.eye(n, dtype=F32, device="cuda") + 0.05 * torch.randn(n, n, generator=g, device="cuda")
    E = Ls.tril() - torch.eye(n, dtype=F32, device="cuda")
    P = (E.double() @ E.double().T).float()
    _, Ev = _poisoned(E, n + 3, upper=True)
    _, Pv = _poisoned(P, n + 5, upper=True)
    # D from the lower triangles in the kernel's fp32 order: P + E, plus E once more on the diagonal
    Dl = (P + E).tril()
    Dl.diagonal().add_(E.diagonal())
    D = Dl + Dl.tril(-1).T
    bits = torch.zeros(1, dtype=torch.int32, device="cuda")
    ops.build_d_absmax(Ev, Pv, bits, n)
    assert float(bits.view(F32)) == float(D.abs().max())
    s = _pow2_for(D)
    ld = n + 3 if n % 2 else _round_up(n, 64)
    (hf, hi), (lf, lo) = _buf(n, n, ld, F16), _buf(n, n, ld, F16)
    ops.build_d_split(Ev, Pv, _scale(s), hi, lo, n)
    rh, rl = _split_ref(D, s)
    assert _same_bits(hi, rh) and _same_bits(lo, rl)
    assert _pad_kept(hf, n) and _pad_kept(lf, n)


# ----------------------------------------------------------------------------------------- K_zx as its fp16 split
def _hyp(ops, raw_ell=0.3, raw_os=-0.4):
    return ops.hyp_from_raw(torch.tensor([raw_ell], dtype=F32, device="cuda"), torch.tensor([raw_os], dtype=F32, device="cuda"))


def _kdir_inputs(n1, n2, d, p1, p2, canonical, seed):
    g = torch.Generator().manual_seed(seed)
    x1, x2 = torch.rand(n1, d, generator=g), torch.rand(n2, d, generator=g)
    v1 = torch.randn(n1 * p1, d, generator=g) if p1 else None
    if not p2:
        v2 = None
    elif canonical:                                        # one-hot rows, any sign and length
        v2 = torch.zeros(n2 * p2, d)
        sc = torch.randn(n2 * p2, generator=g)
        sc[sc.abs() < 0.1] = 0.7
        v2[torch.arange(n2 * p2), torch.randint(0, d, (n2 * p2,), generator=g)] = sc
    else:
        v2 = torch.randn(n2 * p2, d, generator=g)
    return x1, x2, v1, v2


@pytest.mark.parametrize("d", [3, 10, 18, 60])
@pytest.mark.parametrize("p1,p2", [(1, 1), (2, 2), (3, 3), (1, 0), (2, 0), (3, 0)])
def test_kdir_fwd_half_matches_fp64_and_fp32_kernel(ops, p1, p2, d):
    n1, n2 = 45, 600                                       # n1: no multiple of 32 / 64; n2 >= 512, no multiple of 128
    rows, cols = n1 * (p1 + 1), n2 * (p2 + 1)
    hyp = _hyp(ops)
    ell, osc = (float(v) for v in hyp[:2].cpu())
    maxbits = torch.zeros(8, dtype=torch.int32, device="cuda")
    sc = torch.ones(16, dtype=F32, device="cuda")
    ops.tc_scales(hyp, 1e-3, maxbits, rows, sc, 0)
    sK = float(sc[1])
    try:
        for canonical in ((True, False) if p2 else (False,)):
            x1, x2, v1, v2 = _kdir_inputs(n1, n2, d, p1, p2, canonical, 10 * d + p1 + p2)
            Kref = osc * O.kernel_closed_form(x1.double(), x2.double(), None if v1 is None else v1.double(),
                                              None if v2 is None else v2.double(), torch.tensor(ell, dtype=F64))
            x1c, x2c = x1.cuda(), x2.cuda()
            u1 = ops.normalize_dirs(v1.cuda())[0] if p1 else None
            if p2:
                w2, _, cidx, flag = ops.normalize_dirs_canon(v2.cuda())
                assert int(flag.item()) == int(canonical)
                canon = (cidx, flag)
            else:
                w2, canon = None, None
            ops.set_kdir_fwd_knobs(0, 2)
            Kf, K32 = _buf(rows, cols, _round_up(cols, 64), F32)
            ops.kdir_fwd(x1c, u1, p1, x2c, w2, p2, hyp, K32, canon=canon if p2 else (None, None))
            assert rel(K32, Kref) < 2e-6
            for ld in (_round_up(cols, 64), _round_up(cols, 4) + 2):   # vector stores / element stores
                for stream_stores in (0, 1):
                    ops.set_kdir_fwd_knobs(32, stream_stores)
                    (hf, Kh), (lf, Kl) = _buf(rows, cols, ld, F16), _buf(rows, cols, ld, F16)
                    Kd_full, Kd = _buf(rows, cols, cols, F32)
                    assert ops.kdir_fwd_half(x1c, u1, p1, x2c, w2, p2, hyp, Kd, Kh, Kl, sc[1:2], canon=canon)
                    torch.cuda.synchronize()
                    assert bool(torch.isnan(Kd_full).all())            # no fp32 matrix at all
                    assert _pad_kept(hf, cols) and _pad_kept(lf, cols)
                    assert rel((Kh.double() + Kl.double()) / sK, Kref) < 2e-6
                    # the same kernel with another store: the split of the fp32 kernel's K, bit for bit
                    rh, rl = _split_ref(K32, sK)
                    where = (canonical, ld, stream_stores)
                    assert _same_bits(Kh, rh), where
                    assert _same_bits(Kl, rl), where
    finally:
        ops.set_kdir_fwd_knobs(0, 2)


@pytest.mark.parametrize("n2,p1,p2", [(300, 2, 2), (511, 1, 0), (600, 4, 4)])
def test_kdir_fwd_half_declines_other_shapes(ops, n2, p1, p2):
    """shapes the vectorised kernel does not take: False, and K is written in fp32 instead"""
    n1, d = 37, 5
    rows, cols = n1 * (p1 + 1), n2 * (p2 + 1)
    hyp = _hyp(ops)
    ell, osc = (float(v) for v in hyp[:2].cpu())
    x1, x2, v1, v2 = _kdir_inputs(n1, n2, d, p1, p2, False, n2)
    u1 = ops.normalize_dirs(v1.cuda())[0] if p1 else None
    w2, canon = (None, None)
    if p2:
        w2, _, cidx, flag = ops.normalize_dirs_canon(v2.cuda())
        canon = (cidx, flag)
    (hf, Kh), (lf, Kl) = _buf(rows, cols, _round_up(cols, 64), F16), _buf(rows, cols, _round_up(cols, 64), F16)
    Kf, K = _buf(rows, cols, cols + 3, F32)
    assert not ops.kdir_fwd_half(x1.cuda(), u1, p1, x2.cuda(), w2, p2, hyp, K, Kh, Kl, _scale(2.0 ** 10), canon=canon)
    Kref = osc * O.kernel_closed_form(x1.double(), x2.double(), None if v1 is None else v1.double(),
                                      None if v2 is None else v2.double(), torch.tensor(ell, dtype=F64))
    assert rel(K, Kref) < 2e-6 and _pad_kept(Kf, cols)
    assert _pad_kept(hf, 0) and _pad_kept(lf, 0)


# ---------------------------------------------------------------------------- dA, A_g and t of the backward pass
@pytest.mark.parametrize("nslab", ["auto", 1])
@pytest.mark.parametrize("layout", ["vector", "scalar", "misaligned"])
@pytest.mark.parametrize("form", ["fp32_A", "half_A"])
def test_dA_apply_half_matches_fp64(ops, form, layout, nslab):
    rows, nq = 300, 999                                   # rows: a partial CTA of 8 rows; nq odd
    g = torch.Generator(device="cuda").manual_seed(rows + nq + len(layout))
    rnd = lambda *s: torch.randn(*s, generator=g, device="cuda", dtype=F64)
    ld, ldh, col0 = {"vector": (_round_up(nq, 64), _round_up(nq, 64), 0), "scalar": (nq + 2, nq + 2, 0),
                     "misaligned": (_round_up(nq, 64), _round_up(nq, 64), 1)}[layout]
    a_scale = 2.0 ** 11
    A64 = rnd(rows, nq)
    if form == "half_A":                                  # A known only as the split of A * a_scale
        Ah0, Al0 = _split_ref(A64, a_scale)
        _, Ah = _poisoned(Ah0, ldh, col0=col0)
        _, Al = _poisoned(Al0, ldh, col0=col0)
        A32 = (Ah0.float() + Al0.float()) * (1.0 / a_scale)
    else:
        A32 = A64.float()
        _, A = _poisoned(A32, ld, col0=col0)
    A64 = A32.double()                                    # exact
    C32 = (0.3 * rnd(rows, nq)).float()
    Cf, C = _poisoned(C32, ld, col0=col0)
    C_before = Cf.clone()
    m, gmu, gvar = (0.5 * rnd(rows)).float(), (0.1 * rnd(nq)).float(), (0.01 * rnd(nq)).float()
    gvar[::5] = 0.0
    m64, gm64, gv64, C64 = m.double(), gmu.double(), gvar.double(), C32.double()
    dA64 = m64[:, None] * gm64[None] + 2 * C64 * gv64[None]
    Ag32 = A32 * gvar                                     # the kernel's fp32 product, reproducible exactly
    s_dA, s_Ag = _pow2_for(dA64), _pow2_for(Ag32)
    ns = ops.reduce_slabs(rows, nq) if nslab == "auto" else 1
    tp = torch.full((ns, rows), float("nan"), dtype=F32, device="cuda")
    t = torch.full((rows,), float("nan"), dtype=F32, device="cuda")
    outs = [_buf(rows, nq + col0, ldh, F16) for _ in range(4)]
    dAh, dAl, Agh, Agl = (o[0][:, col0:col0 + nq] for o in outs)
    if form == "half_A":
        ops.dA_apply_half(None, C, rows, nq, m, gmu, gvar, tp, t, dAh, dAl, Agh, Agl, _scale(s_dA), _scale(s_Ag),
                          A_half=(Ah, Al), a_scale=_scale(a_scale))
    else:
        ops.dA_apply_half(A, C, rows, nq, m, gmu, gvar, tp, t, dAh, dAl, Agh, Agl, _scale(s_dA), _scale(s_Ag))
    assert _same_bits(Cf, C_before)                      # C is read, never written (unlike the fp32 dA_apply)
    assert all(_pad_kept(full, nq + col0, col0) for full, _ in outs)
    assert rel((dAh.double() + dAl.double()) / s_dA, dA64) < 1e-6
    # dA's fp32 value m_i g_j + 2 g_j C_ij (contracted or not) is not reproducible in torch: the split gate on the fp64 value,
    # widened by the one fp32 rounding of each term (which cancellation can make large relative to |dA|)
    fp32_err = 2.0 ** -23 * s_dA * ((m64[:, None] * gm64[None]).abs() + (2 * C64 * gv64[None]).abs())
    assert _split_gate(dAh, dAl, dA64 * s_dA, fp32_err) <= 0
    rh, rl = _split_ref(Ag32, s_Ag)
    assert _same_bits(Agh, rh) and _same_bits(Agl, rl)
    assert rel((Agh.double() + Agl.double()) / s_Ag, A64 * gv64[None]) < 1e-6
    assert rel(t, A64 @ gm64) < 2e-5


# ------------------------------------------------------------------------------- column reductions on the split A
@pytest.mark.parametrize("rows,nq,nslab", [(300, 999, "auto"), (45, 285, 1), (1000, 1001, 7), (129, 64, "auto"), (8, 1, 1)])
def test_col_dots_half_matches_fp64(ops, rows, nq, nslab):
    """pm = A^T m and pv = sum_i A_ij C_ij per row slab, A = (hi + lo) / a_scale; cmax = max|C| bit for bit"""
    g = torch.Generator(device="cuda").manual_seed(rows * nq)
    rnd = lambda *s: torch.randn(*s, generator=g, device="cuda", dtype=F64)
    a_scale = 2.0 ** 11
    ldh, ld = _round_up(nq, 64), _round_up(nq, 2) + 2    # (the kernel needs even leading dimensions)
    Ah0, Al0 = _split_ref(rnd(rows, nq), a_scale)
    _, Ah = _poisoned(Ah0, ldh)
    _, Al = _poisoned(Al0, ldh)
    A32 = (Ah0.float() + Al0.float()) * (1.0 / a_scale)
    A64 = A32.double()
    C32 = rnd(rows, nq).float()
    _, C = _poisoned(C32, ld)
    m = rnd(rows).float()
    ns = ops.reduce_slabs(rows, nq) if nslab == "auto" else nslab
    pm, pv = (torch.full((ns, nq), float("nan"), dtype=F32, device="cuda") for _ in range(2))
    cmax = torch.zeros(1, dtype=torch.int32, device="cuda")
    ops.col_dots_half((Ah, Al), _scale(a_scale), m, pm, pv, rows, nq, C, cmax=cmax)
    assert rel(pm.double().sum(0), A64.T @ m.double()) < 2e-5
    assert rel(pv.double().sum(0), (A64 * C32.double()).sum(0)) < 2e-5
    assert float(cmax.view(F32)) == float(C32.abs().max())
    # the fp32 column reduction on the reconstructed A agrees (same slabs, another summation order)
    _, A = _poisoned(A32, ld)
    pm2, pv2 = (torch.full((ns, nq), float("nan"), dtype=F32, device="cuda") for _ in range(2))
    cmax2 = torch.zeros(1, dtype=torch.int32, device="cuda")
    ops.col_dots(A, m, pm2, pv2, rows, nq, C=C, cmax=cmax2)
    assert rel(pm.sum(0), pm2.sum(0)) < 1e-5 and rel(pv.sum(0), pv2.sum(0)) < 1e-5
    assert int(cmax2) == int(cmax)


# --------------------------------------------------------------------------------------- operand scales and maxima
def _pow2_exp(bound):
    """csrc/tc_prep.cu pow2_scale restated: (exponent, whether log2f may round it to the neighbour)"""
    b = float(bound)
    if not (b > 0) or not (b < 3.0e38):
        return 0, False
    lg = math.log2(b)
    ex = max(-60, min(60, 15 - math.ceil(lg)))
    return ex, abs(b - 2.0 ** round(lg)) <= 1e-6 * b


def _bits(*vals):
    return torch.tensor([float(v) for v in vals], dtype=F32).view(torch.int32).cuda()


SCALE_CASES = [  # ell, os, jitter, M', max|E|, max|m|, max|g_mu|, max|g_var|, max|D|, max|C|
    (0.5, 1.7, 1e-3, 150, 0.3, 1.2, 0.05, 1e-4, 2.5, 7.0),
    (0.15, 0.7, 1e-3, 3072, 0.9, 3.0, 1e-3, 3e-6, 40.0, 0.0),      # max|C| not measured: the a-priori fallback
    (2.0, 30.0, 1.1e-3, 384, 0.5, 1e-3, 2.0, 0.5, 0.25, 0.2),      # bounds that are exact powers of two
    (1.0, 1.0, 1e-3, 288, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0),           # the state at initialisation: every maximum 0
    (0.7, 1.3, 1e-3, 200, math.inf, 0.0, math.inf, 1e-3, math.inf, math.inf),   # NaN maxima (absmax: +inf)
]


@pytest.mark.parametrize("case", range(len(SCALE_CASES)))
def test_tc_scales_follow_the_stated_bounds(ops, case):
    ell, os_, jit, Mq, mE, mm, gm, gv, mD, mC = SCALE_CASES[case]
    hyp = torch.tensor([ell, os_, 0.3, 0.0, 0, 0, 0, 0], dtype=F64, device="cuda")
    maxbits = torch.cat([_bits(mE, mm, gm, gv, mD, mC), torch.zeros(2, dtype=torch.int32, device="cuda")])
    sc = torch.full((16,), 7.0, dtype=F32, device="cuda")          # 7: not written by any stage
    ops.tc_scales(hyp, jit, maxbits, Mq, sc, 0)
    s0 = sc.cpu().clone()
    assert all(float(s0[k]) == 7.0 for k in (5, 6, 11, 12, 14, 15))
    ops.tc_scales(hyp, jit, maxbits, Mq, sc, 2)
    s2 = sc.cpu().clone()
    assert torch.equal(torch.cat([s2[:7], s2[8:13]]), torch.cat([s0[:7], s0[8:13]]))
    ops.tc_scales(hyp, jit, maxbits, Mq, sc, 1)
    s = sc.cpu()
    assert torch.equal(s[[0, 1, 2, 3, 4, 7, 8, 9, 10, 13]], s2[[0, 1, 2, 3, 4, 7, 8, 9, 10, 13]])
    assert bool(torch.isfinite(s).all())
    # the bounds of the comment block at the top of csrc/tc_prep.cu, in float32 (inf / NaN maxima: numpy would warn)
    np_err = np.seterr(invalid="ignore", over="ignore")
    f = np.float32
    el, o = f(ell), f(os_)
    a = f(1.01) * np.sqrt(o * max(f(1), f(1) / (el * el)))
    e = f(Mq) * f(mE)
    cmax = f(mC) if mC != 0 else e * (f(2) + e) * a
    bounds = {0: f(1.01) / np.sqrt(f(jit)), 1: f(1.01) * o * max(f(1), max(f(1) / el, f(2) / (el * el))), 2: f(mE), 3: a,
              4: (f(1) + e) * a, 5: f(1.01) * (f(mm) * f(gm) + f(2) * f(gv) * cmax), 6: f(1.01) * a * f(gv), 7: f(1.01) * f(mD)}
    stage0_7 = f(1.01) * (f(2) * f(mE) + f(Mq) * f(mE) * f(mE))
    np.seterr(**np_err)
    for k, b in list(bounds.items()) + [("7 (stage 0)", stage0_7)]:
        got = float((s0 if k == "7 (stage 0)" else s)[7 if k == "7 (stage 0)" else k])
        lg = math.log2(got)
        assert lg == round(lg), (k, got)                                # an exact power of two
        ex, near = _pow2_exp(b)
        assert round(lg) == ex or (near and abs(round(lg) - ex) == 1), (k, float(b), got, ex)
        if not (float(b) > 0) or not (float(b) < 3.0e38):
            assert got == 1.0, k
    rec = lambda x, y: float(np.float32(1) / (np.float32(x) * np.float32(y)))
    assert float(s0[13]) == rec(s0[7], s0[3])
    for k, (i, j) in {8: (0, 1), 9: (2, 3), 10: (2, 4), 11: (0, 5), 12: (6, 3), 13: (7, 3)}.items():
        assert float(s[k]) == rec(s[i], s[j]), k


def test_absmax_maxima_and_nan_rule(ops):
    g = torch.Generator(device="cuda").manual_seed(1)
    n = 257
    for dt in (F32, F64):
        Ls = torch.eye(n, dtype=dt, device="cuda")
        bits = torch.zeros(3, dtype=torch.int32, device="cuda")
        ops.absmax(Ls, bits[0:1], mode=2)                             # L_s = I: max|tril(L_s) - I| = 0
        ops.absmax(torch.zeros(1000, dtype=dt, device="cuda"), bits[1:2])
        assert int(bits[0]) == 0 and int(bits[1]) == 0
        X = torch.randn(n, n + 3, generator=g, dtype=F64, device="cuda").to(dt)[:, :n]
        X[3, 200] = 1e9                                               # above the diagonal: ignored in mode 2
        ops.absmax(X, bits[2:3], mode=2)
        E = X.float().tril() - torch.eye(n, dtype=F32, device="cuda")     # the kernel's order: fp32 first, then - 1
        assert float(bits[2:3].view(F32)) == float(E.abs().max())
        for mode in (0, 2):
            X[7, 3] = float("nan")
            b = torch.zeros(1, dtype=torch.int32, device="cuda")
            ops.absmax(X, b, mode=mode)
            assert int(b) == 0x7F800000                               # NaN -> +inf: the scale falls back to 1
        v = torch.randn(777, generator=g, dtype=F64, device="cuda").to(dt)
        b = torch.zeros(1, dtype=torch.int32, device="cuda")
        ops.absmax(v, b)
        assert float(b.view(F32)) == float(v.float().abs().max())


# --------------------------------------------------------------------------------------------------- small extras
@pytest.mark.parametrize("dtype", [F32, F64])
def test_pll_terms_match_fp64_autograd(ops, dtype):
    nq = 1000
    g = torch.Generator().manual_seed(4)
    min_var = 1e-10 if dtype == F64 else 1e-6
    mu, y = torch.randn(nq, generator=g, dtype=F64), torch.randn(nq, generator=g, dtype=F64)
    var = torch.rand(nq, generator=g, dtype=F64) + 0.05
    var[::97] = min_var                                    # at and below the floor: g_var must be exactly 0
    var[5], y[5] = 0.5 * min_var, mu[5]
    mu, y, var = (t.to(dtype) for t in (mu, y, var))
    w = 1.0 / 3000
    d = lambda t: t.cuda()
    gmu, gvar = (torch.full((nq,), float("nan"), dtype=dtype, device="cuda") for _ in range(2))
    sc = torch.zeros(8, dtype=F64, device="cuda")
    ws = torch.empty(8192, dtype=F64, device="cuda")
    ops.pll_terms(d(mu), d(var), d(y), w, gmu, gvar, sc, ws)
    MU, VAR = mu.double().requires_grad_(True), var.double().requires_grad_(True)
    Y = y.double()
    val = (-0.5 * ((Y - MU) ** 2 / VAR + VAR.log() + math.log(2 * math.pi)) * w).sum()
    val.backward()
    val = float(val.detach())
    assert abs(float(sc[0]) - val) <= 1e-12 * abs(val) and float(sc[1]) == 0.0
    t = 1e-12 if dtype == F64 else 1e-7
    assert rel(gmu, MU.grad) < t
    floor = var.double() <= min_var
    assert int(floor.sum()) >= 10 and bool((gvar.cpu()[floor] == 0).all())
    assert rel(gvar.cpu()[~floor], VAR.grad[~floor]) < t


@pytest.mark.parametrize("dtype", [F32, F64])
def test_kdir_diag_with_outputscale(ops, dtype):
    hyp = ops.hyp_from_raw(torch.tensor([0.3], dtype=dtype, device="cuda"), torch.tensor([0.8], dtype=dtype, device="cuda"))
    ell, osc = hyp[0].cpu(), hyp[1].cpu()
    for n, p in ((37, 3), (1, 0), (300, 2)):
        got = ops.kdir_diag(n, p, hyp, dtype, use_os=True)
        assert rel(got, osc * O.kernel_diag(n, p, ell)) < (1e-15 if dtype == F64 else 1e-7)


# ------------------------------------------------------------------ epilogues of the tensor-core products: alignment
EPI_CASES = [  # M (None: = N), K, options
    (200, 96, {}),
    (200, 96, dict(alpha=2.0, beta=-1.5)),
    (384, 384, dict(a_tri=1, dual=True)),
    (None, 200, dict(b_kmajor=True, c_lower=True)),
]


def _epi_layout(N, odd):
    return N + 2 if odd else _round_up(N, 64)                     # N is odd: N + 2 is an odd leading dimension


def _check_epilogue(C, Cf, ref, c_lower, N):
    assert (rel(C.tril(), ref.tril()) if c_lower else rel(C, ref)) < 2e-6
    assert _pad_kept(Cf, N)


@pytest.mark.parametrize("case", range(len(EPI_CASES)))
@pytest.mark.parametrize("odd_ld", [False, True])
@pytest.mark.parametrize("N", [285, 1001])
@pytest.mark.parametrize("cg,persistent", [(1, 1), (2, 1), (2, 0)])
def test_gemm_tch_epilogue_edges_and_unaligned_outputs(ops, cg, persistent, N, odd_ld, case):
    """3xFP16 product with N % 4 != 0 (edge pieces past col + 3) and, with odd_ld, outputs / addends on odd leading
    dimensions: the whole epilogue runs element by element"""
    M, K, kw = EPI_CASES[case]
    M = N if M is None else M
    b_kmajor, a_tri, c_lower = kw.get("b_kmajor", False), kw.get("a_tri", 0), kw.get("c_lower", False)
    alpha, beta, dual = kw.get("alpha", 1.0), kw.get("beta", 0.0), kw.get("dual", False)
    prev = ops.set_tc_cta_group(cg)
    ops.set_tc_persistent(persistent)
    try:
        g = torch.Generator(device="cuda").manual_seed(M + N + K + case)
        A = torch.randn(M, K, device="cuda", dtype=F64, generator=g)
        A = A.tril() if a_tri == 1 else A
        B = torch.randn((N, K) if b_kmajor else (K, N), device="cuda", dtype=F64, generator=g)
        sA, sB = 2.0 ** 11, 2.0 ** 12
        lda, ldb = _round_up(K, 8), (_round_up(K, 8) if b_kmajor else _round_up(N, 64))
        zp = lambda t, ld: torch.nn.functional.pad(t, (0, ld - t.shape[1]))[:, :t.shape[1]]   # TMA operands: zero padding
        Ah, Al = (zp(t, lda) for t in _split_ref(A, sA))
        Bh, Bl = (zp(t, ldb) for t in _split_ref(B, sB))
        ldo = _epi_layout(N, odd_ld)
        D, D2 = (_poisoned(torch.randn(M, N, device="cuda", dtype=F32, generator=g), ldo)[1] for _ in range(2))
        (Cf, C), (C2f, C2) = _buf(M, N, ldo, F32), _buf(M, N, ldo, F32)
        hbufs = [_buf(M, N, ldo, F16) for _ in range(4)]
        Ch, C2h = (hbufs[0][1], hbufs[1][1]), (hbufs[2][1], hbufs[3][1])
        inv = torch.tensor([1.0 / (sA * sB)], device="cuda", dtype=F32)
        cs, c2s = _scale(8.0), _scale(4.0)
        Aq, Bq = (Ah.double() + Al.double()) / sA, (Bh.double() + Bl.double()) / sB
        ref = alpha * (Aq @ (Bq.T if b_kmajor else Bq)) + beta * D.double()

        def run(out):
            ops.gemm_tch((Ah, Al), (Bh, Bl), out, M, N, K, inv, b_kmajor=b_kmajor, alpha=alpha, beta=beta, D=D if beta else None,
                         C2=C2 if dual else None, D2=D2 if dual else None, Ch=Ch if dual else None, c_scale=cs,
                         C2h=C2h if dual else None, c2_scale=c2s, a_tri=a_tri, c_lower=c_lower)
        run(C)
        _check_epilogue(C, Cf, ref, c_lower, N)
        if dual:
            assert rel(C2, ref + D2.double()) < 2e-6 and _pad_kept(C2f, N)
            assert rel((Ch[0].double() + Ch[1].double()) / 8.0, ref) < 2e-6
            assert rel((C2h[0].double() + C2h[1].double()) / 4.0, ref + D2.double()) < 2e-6
            assert all(_pad_kept(f, N) for f, _ in hbufs)
        if cg == 2 and persistent:
            # the persistent kernel adds the same chunks in the same order: bit-identical to one pair per tile
            ops.set_tc_persistent(0)
            Cf1, C1 = _buf(M, N, ldo, F32)
            run(C1)
            a_, b_ = (C.tril(), C1.tril()) if c_lower else (C, C1)
            assert _same_bits(a_, b_) and _pad_kept(Cf1, N)
    finally:
        ops.set_tc_cta_group(prev)
        ops.set_tc_persistent(1)


@pytest.mark.parametrize("case", range(len(EPI_CASES)))
@pytest.mark.parametrize("odd_ld", [False, True])
@pytest.mark.parametrize("N", [285, 1001])
@pytest.mark.parametrize("cg,persistent", [(1, 1), (2, 1), (2, 0)])
def test_gemm_tc_3xtf32_epilogue_edges_and_unaligned_outputs(ops, cg, persistent, N, odd_ld, case):
    M, K, kw = EPI_CASES[case]
    M = N if M is None else M
    b_kmajor, a_tri, c_lower = kw.get("b_kmajor", False), kw.get("a_tri", 0), kw.get("c_lower", False)
    alpha, beta, dual = kw.get("alpha", 1.0), kw.get("beta", 0.0), kw.get("dual", False)
    prev = ops.set_tc_cta_group(cg)
    ops.set_tc_persistent(persistent)
    try:
        g = torch.Generator(device="cuda").manual_seed(3 * M + N + K + case)
        A = torch.randn(M, K, device="cuda", dtype=F32, generator=g)
        A = A.tril() if a_tri == 1 else A
        B = torch.randn((N, K) if b_kmajor else (K, N), device="cuda", dtype=F32, generator=g)
        lda, ldb = _round_up(K, 8), (_round_up(K, 8) if b_kmajor else _round_up(N, 32))
        zp = lambda t, ld: torch.nn.functional.pad(t, (0, ld - t.shape[1]))[:, :t.shape[1]]
        Af, Bf = zp(A, lda), zp(B, ldb)
        Alo, Blo = zp(torch.zeros_like(A), lda), zp(torch.zeros_like(B), ldb)
        ops.split_lo(Af, Alo)
        ops.split_lo(Bf, Blo)
        ldo = _epi_layout(N, odd_ld)
        D, D2 = (_poisoned(torch.randn(M, N, device="cuda", dtype=F32, generator=g), ldo)[1] for _ in range(2))
        bufs = [_buf(M, N, ldo, F32) for _ in range(4)]
        (Cf, C), (C2f, C2), (Clof, Clo), (C2lof, C2lo) = bufs
        ref = alpha * (A.double() @ (B.double().T if b_kmajor else B.double())) + beta * D.double()

        def run(out, out_lo):
            ops.gemm_tc(Af, Alo, Bf, Blo, out, M, N, K, b_kmajor=b_kmajor, alpha=alpha, beta=beta, D=D if beta else None,
                        C2=C2 if dual else None, D2=D2 if dual else None, a_tri=a_tri, c_lower=c_lower, chunk=2,
                        C_lo=out_lo if dual else None, C2_lo=C2lo if dual else None)
        run(C, Clo)
        _check_epilogue(C, Cf, ref, c_lower, N)
        if dual:
            assert rel(C2, ref + D2.double()) < 2e-6
            trunc = lambda t: (t.contiguous().view(torch.int32) & ~0x1FFF).view(F32)
            assert float((C - trunc(C) - Clo).abs().max()) <= 2.0 ** -21 * float(C.abs().max())
            assert float((C2 - trunc(C2) - C2lo).abs().max()) <= 2.0 ** -21 * float(C2.abs().max())
            assert all(_pad_kept(f, N) for f, _ in bufs)
        if cg == 2 and persistent:
            ops.set_tc_persistent(0)
            (Cf1, C1), (_, Clo1) = _buf(M, N, ldo, F32), _buf(M, N, ldo, F32)
            run(C1, Clo1)
            a_, b_ = (C.tril(), C1.tril()) if c_lower else (C, C1)
            assert _same_bits(a_, b_) and _pad_kept(Cf1, N)
    finally:
        ops.set_tc_cta_group(prev)
        ops.set_tc_persistent(1)


@pytest.mark.parametrize("cg,persistent", [(1, 1), (2, 1), (2, 0)])
def test_gemm_tch_ignores_the_padding_of_an_mn_major_b(ops, cg, persistent):
    """NaN in the padding columns of B (K x N, leading dimension a multiple of 64) must not reach the valid outputs"""
    M, N, K = 200, 285, 96
    prev = ops.set_tc_cta_group(cg)
    ops.set_tc_persistent(persistent)
    try:
        g = torch.Generator(device="cuda").manual_seed(17)
        A = torch.randn(M, K, device="cuda", dtype=F64, generator=g)
        B = torch.randn(K, N, device="cuda", dtype=F64, generator=g)
        Ah, Al = (torch.nn.functional.pad(t, (0, _round_up(K, 8) - K))[:, :K] for t in _split_ref(A, 2.0 ** 11))
        inv = torch.tensor([2.0 ** -23], device="cuda", dtype=F32)
        outs = []
        for poison in (False, True):
            (Bhf, Bh), (Blf, Bl) = (_poisoned(t, _round_up(N, 64)) for t in _split_ref(B, 2.0 ** 12))
            if not poison:
                Bhf[:, N:].zero_(), Blf[:, N:].zero_()
            Cf, C = _buf(M, N, _round_up(N, 64), F32)
            ops.gemm_tch((Ah, Al), (Bh, Bl), C, M, N, K, inv)
            assert _pad_kept(Cf, N) and bool(torch.isfinite(C).all())
            outs.append(C)
        assert _same_bits(outs[0], outs[1])
    finally:
        ops.set_tc_cta_group(prev)
        ops.set_tc_persistent(1)


# ------------------------------------------------------------------------------- steps on 3xFP16 whitening
@contextmanager
def _engine(**flags):
    """engine module flags set for the block; workspaces and factors dropped before and after"""
    from dsvgp_b200 import engine
    old = {k: getattr(engine, k) for k in flags}
    for k, v in flags.items():
        setattr(engine, k, v)
    engine.ENGINE._ws.clear(), engine.ENGINE._fac.clear()
    try:
        yield engine
    finally:
        for k, v in old.items():
            setattr(engine, k, v)
        engine.ENGINE._ws.clear(), engine.ENGINE._fac.clear()


def _last_ws(engine):
    return list(engine.ENGINE._ws.values())[-1]


RAGGED = [  # the fp32 tcgen05 shapes of test_step_gpu.CASES: M' / n'
    ("dsvgp", 95, 5, 43, 2),      # 129 / 285
    ("dsvgp", 300, 3, 65, 1),     # 130 / 600
    ("dfree", 270, 7, 50, 2),     # 150 / 270, values only
    ("dsvgp", 333, 10, 96, 2),    # 288 / 999
]


def _oracle(variant, P, x, Vx, y, num_data):
    up = lambda t: None if t is None else t.double()
    P64 = P.clone(F64)
    val, grads = O.elbo_and_grads(P64, up(x), up(Vx), up(y), num_data, variant)
    mean, var = O.predict(P64, up(x), up(Vx), variant)
    return val, grads, mean, var


def _step_and_predict(engine, variant, P, x, Vx, y, num_data, d, expect_half_a):
    model, lik, val, grads, out = run_step(variant, P, x, Vx, y, num_data, d, F32)
    ws = _last_ws(engine)
    assert ws.tch and ws.A64 is None and ws.a_half == expect_half_a     # the path this test is about was taken
    model.eval(), lik.eval()
    with torch.no_grad():
        kw = {} if variant == "grad" else {"derivative_directions": Vx}
        preds = lik(model(x.cuda(), **kw))
    return val, grads, out, preds


@pytest.mark.parametrize("half_a", [False, True])
@pytest.mark.parametrize("variant,n,d,M,p", RAGGED)
def test_ragged_step_on_3xfp16_whitening(variant, n, d, M, p, half_a):
    """A = W K_zx and dK_zx = W^T dA as 3xFP16 products (fp64 whitening off) at ragged M' / n'; with half_a, A is kept only
    as its split (engine.HALF_A: the column reductions and the dA pass read hi + lo).  north_star's 1e-4 against the
    fp64 oracle on the ELBO, every gradient, and the train- and eval-mode mean / variance."""
    P, x, Vx, y, num_data = O.make_problem(n, d, M, p, F32, seed=n + d + M, variant=variant, N=10 * n)
    ref_val, ref_grads, mean, var = _oracle(variant, P, x, Vx, y, num_data)
    with _engine(WHITEN_FP64=False, HALF_A=half_a) as engine:
        val, grads, out, preds = _step_and_predict(engine, variant, P, x, Vx, y, num_data, d, half_a)
    check_against(val, grads, ref_val, ref_grads, 1e-4, 1e-4)
    for got, want in ((out.mean, mean), (out.variance, var), (preds.mean, mean), (preds.variance, var)):
        assert rel(got, want) < 1e-4


def test_auto_whitening_takes_3xfp16_above_the_threshold():
    """WHITEN_FP64 = "auto" with n' = 2049, one above engine.WHITEN_FP64_MAX_NQ: 3xFP16 whitening, same gate"""
    variant, n, d, M, p = "dsvgp", 683, 10, 64, 2
    P, x, Vx, y, num_data = O.make_problem(n, d, M, p, F32, seed=6, variant=variant, N=10 * n)
    ref_val, ref_grads, mean, var = _oracle(variant, P, x, Vx, y, num_data)
    with _engine(WHITEN_FP64="auto") as engine:
        assert engine.WHITEN_FP64_MAX_NQ == 2048
        val, grads, out, preds = _step_and_predict(engine, variant, P, x, Vx, y, num_data, d, False)
        assert _last_ws(engine).nq == 2049
    check_against(val, grads, ref_val, ref_grads, 1e-4, 1e-4)
    for got, want in ((out.mean, mean), (out.variance, var), (preds.mean, mean), (preds.variance, var)):
        assert rel(got, want) < 1e-4


def test_operand_scales_are_per_step_state():
    """a step at trained parameters, then one near the prior on the same engine: the second must be bit-identical to the
    same step on a fresh engine (stale maxima -- max|D|, max|C| are only ever raised by atomicMax -- or scales would show)"""
    variant, n, d, M, p = "dsvgp", 300, 10, 96, 2
    Pt, x, Vx, y, nd = O.make_trained_problem(n, d, M, p, F32, seed=3, variant=variant, ell=0.7, kind="rough", N=10 * n)
    Pn, x2, _, _, _ = O.make_problem(n, d, M, p, F32, seed=3, variant=variant, N=10 * n)
    assert torch.equal(x, x2)

    def step(P):
        _, _, val, grads, _ = run_step(variant, P, x, Vx, y, nd, d, F32)
        return torch.cat([val.reshape(1).double().cpu()] + [grads[k].reshape(-1).double().cpu() for k in sorted(grads)])
    with _engine(WHITEN_FP64=False) as engine:
        first = step(Pt)
        second = step(Pn)
        assert not torch.equal(first, second)
        engine.ENGINE._ws.clear(), engine.ENGINE._fac.clear()
        fresh = step(Pn)
    assert torch.equal(second, fresh)


AUDIT = [("near_identity", None, None), ("trained", 0.15, None), ("trained", 0.7, None), ("trained", 2.0, None),
         ("near_identity", None, 30.0)]


@pytest.mark.parametrize("state,ell,outputscale", AUDIT)
def test_3xfp16_operands_use_the_fp16_range(monkeypatch, state, ell, outputscale):
    """Every two-half operand of a real step: hi finite and max|hi| <= 2^15 (65504 is never approached), and max|hi| >= 2^5
    (no scale loose by more than the 2^10 that csrc/tc_prep.cu says starts to cost: round 1's loose bound on |C| pushed
    the scaled dA into fp16 subnormals).  C3-shaped at reduced M: M' = 384, n' = 3000."""
    from dsvgp_b200 import ops
    variant, n, d, M, p = "dsvgp", 1000, 10, 128, 2
    if state == "trained":
        P, x, Vx, y, nd = O.make_trained_problem(n, d, M, p, F32, seed=5, variant=variant, ell=ell, kind="optimal", N=100 * n)
    else:
        P, x, Vx, y, nd = O.make_problem(n, d, M, p, F32, seed=5, variant=variant, N=100 * n)
    if outputscale is not None:
        P.raw_os = O._inv_softplus(outputscale).to(F32).reshape(P.raw_os.shape)
    seen = {}
    real = ops.gemm_tch

    def spy(*args, **kw):
        if kw.get("Ch") is not None and kw.get("a_tri") == ops.TRI_LOWER:   # A = W K_zx: its B operand is K_zx's split
            seen["K_zx"] = args[1][0].clone()
        return real(*args, **kw)
    monkeypatch.setattr(ops, "gemm_tch", spy)
    with _engine(WHITEN_FP64=False) as engine:
        run_step(variant, P, x, Vx, y, nd, d, F32)
        ws, f = _last_ws(engine), list(engine.ENGINE._fac.values())[-1]
        hi = {"W": f.Wh, "K_zx": seen["K_zx"], "A": ws.Ah, "D": ws.Dh, "dA": ws.Kh, "A_g": ws.Agh}
        stats = {k: (bool(torch.isfinite(t).all()), float(t.float().abs().max())) for k, t in hi.items()}
    headroom = {k: round(math.log2(mx), 2) if mx > 0 else -math.inf for k, (_, mx) in stats.items()}
    print(f"\nlog2 max|hi| ({state}, ell={ell}, os={outputscale}):", headroom)
    assert all(ok for ok, _ in stats.values()), stats
    assert all(mx <= 2.0 ** 15 for _, mx in stats.values()), headroom
    assert all(mx >= 2.0 ** 5 for _, mx in stats.values()), headroom
