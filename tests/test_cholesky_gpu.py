"""The fp64 blocked Cholesky and inverse of csrc/chol.cu (dsvgp_chol_f64) against LAPACK.

Every step, the NGD path (gp._chol_inv) and engine.sample_mvn go through this factorisation.  A backward-stable Cholesky
has a residual of a few ulps whatever the conditioning, so the gates compare residuals, not forward errors:

    rL(L)    = max|L L^T - A| / max|A|
    rW(W, L) = max(max|W L - I|, max|L W - I|)

computed for the library's pair (lower triangles of the Mq x Mq corner) and for LAPACK's pair on the same matrix
(torch.linalg.cholesky_ex on the CPU, W = solve_triangular(L, I)); the library must stay within GATE * r_lapack + 16 eps.
The residual products themselves run on the device in fp64 (torch.matmul), the same way for both pairs, after a check
that the device's fp64 product agrees with the CPU's to a few ulps.

Every call writes into NaN-sentinel buffers: Awork, L and W are (Mp, Mp + 8) tensors viewed as Mp x Mp, so an
out-of-bounds write, an unwritten lower entry or a read of an entry the factorisation must not read shows up as NaN."""
import contextlib
import math

import pytest
import torch

pytestmark = pytest.mark.gpu
F64 = torch.float64
EPS = torch.finfo(F64).eps
NAN = float("nan")
GATE = 8.0           # largest ratio measured on a B200 over the passing cases: 3.8 (factor, one block of 100)
DEFAULT_VARIANT = 3


@pytest.fixture(scope="module")
def ops():
    from dsvgp_b200 import ops
    return ops


@contextlib.contextmanager
def chol_variant(ops, v):
    assert ops.set_chol_variant(v) == v
    try:
        yield
    finally:
        ops.set_chol_variant(DEFAULT_VARIANT)


# ----------------------------------------------------------------------------------------------------- matrices
def _sym(A):
    """the symmetric matrix the factorisation sees: the lower triangle mirrored"""
    return A.tril() + A.tril(-1).T


def wishart(Mq, seed):
    """R R^T with R Mq x 2Mq Gaussian / sqrt(2 Mq): eigenvalues within [0.08, 3], on the device"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    R = torch.randn(Mq, 2 * Mq, generator=g, dtype=F64, device="cuda") / math.sqrt(2 * Mq)
    return _sym(R @ R.T)


def near_collinear(Mq, pairs, seed, cos=1.0 - 1e-10):
    """Gram matrix of Gaussian rows in which row b of every pair (a, b) is row a turned by the angle acos(cos):
    the Schur complement of b is (1 - cos^2) |row b|^2, cond ~ 1e10"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    B = torch.randn(Mq, 2 * Mq, generator=g, dtype=F64, device="cuda") / math.sqrt(2 * Mq)
    for a, b in pairs:
        u = B[a] / B[a].norm()
        v = B[b] - (B[b] @ u) * u
        v = v / v.norm()
        B[b] = B[a].norm() * (cos * u + math.sqrt(1.0 - cos * cos) * v)
    return _sym(B @ B.T)


def kzz(ops, M, d, p, ell, outputscale, jitter, seed, duplicate=None):
    """K_zz as the library assembles it (kdir_fwd, fp64) for M inducing points in [0,1]^d with p directions each;
    duplicate = (i, dist): point i + 1 is point i moved by dist, with the same directions"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.rand(M, d, generator=g, dtype=F64, device="cuda")
    v = torch.randn(M * p, d, generator=g, dtype=F64, device="cuda")
    if duplicate is not None:
        i, dist = duplicate
        s = torch.randn(d, generator=g, dtype=F64, device="cuda")
        x[i + 1] = x[i] + dist * s / s.norm()
        v[(i + 1) * p:(i + 2) * p] = v[i * p:(i + 1) * p]
    raw = lambda t: torch.tensor([math.log(math.expm1(t))], dtype=F64, device="cuda")
    hyp = ops.hyp_from_raw(raw(ell), raw(outputscale))
    u = ops.normalize_dirs(v, F64)[0]
    Mq = M * (p + 1)
    K = torch.empty(Mq, Mq, dtype=F64, device="cuda")
    ops.kdir_fwd(x, u, p, x, u, p, hyp, K, diag_add=jitter)
    return _sym(K)


def cond(A):
    ev = torch.linalg.eigvalsh(A.cpu())
    return float(ev[-1] / ev[0])


# ----------------------------------------------------------------------------------------------------- running it
def factor(ops, A, upper_fill=None, lda_pad=8):
    """dsvgp_chol_f64 on A (device, symmetric) in NaN-sentinel buffers.  Checks info == 0, the sentinel columns, finite
    lower triangles and the identity padding; returns (tril L, tril W) of the Mq x Mq corner and the raw Mp x Mp views."""
    Mq = A.shape[0]
    Mp, nb0, nlev = ops.chol_plan(Mq)
    bufs = [torch.full((Mp, Mp + lda_pad), NAN, dtype=F64, device="cuda") for _ in range(3)]
    Aw, L, W = (b[:, :Mp] for b in bufs)
    Aw[:Mq, :Mq] = A if upper_fill is None else A.tril() + torch.full_like(A, upper_fill).triu(1)
    ops.pad_identity(Aw, Mq)
    info = torch.full((1,), 12345, dtype=torch.int32, device="cuda")
    ops.cholesky_inverse(Aw, L, W, nb0, nlev, info)
    assert int(info.item()) == 0
    for b in bufs:
        assert bool(b[:, Mp:].isnan().all()), "write beyond the Mp columns"
    for X in (L, W):
        T = X.tril()
        assert bool(T.isfinite().all()), "lower triangle not fully written"
        if Mp > Mq:
            assert bool((T[Mq:, :Mq] == 0).all())
            pad = T[Mq:, Mq:]
            assert bool((pad.tril(-1) == 0).all())
            assert float((pad.diagonal() - 1).abs().max()) <= 4 * EPS    # (l22 = sqrt(det) / l11 next to a real pivot)
    return L[:Mq, :Mq].tril(), W[:Mq, :Mq].tril(), (Aw, L, W)


_device_products_checked = []


def _check_device_products():
    """The residual products run on the device (an M' = 7200 residual on the CPU takes tens of seconds).  They must be plain
    fp64: a product of the size of the largest block here agrees with the CPU's to 16 ulps of |A| |B|."""
    if _device_products_checked:
        return
    g = torch.Generator().manual_seed(0)
    X, Y = torch.randn(448, 448, generator=g, dtype=F64), torch.randn(448, 448, generator=g, dtype=F64)
    err = float(((X.cuda() @ Y.cuda()).cpu() - X @ Y).abs().max() / (X.abs() @ Y.abs()).max())
    assert err <= 16 * EPS, f"device fp64 product off by {err:.2e} of |A||B|: the residuals cannot be measured there"
    _device_products_checked.append(err)


def residuals(L, W, A):
    """(rL, rW) on the device in fp64"""
    _check_device_products()
    I = torch.eye(A.shape[0], dtype=F64, device=A.device)
    rL = float((L @ L.T - A).abs().max() / A.abs().max())
    rW = max(float((W @ L - I).abs().max()), float((L @ W - I).abs().max()))
    return rL, rW


_lapack_cache = {}


def lapack(A, key=None):
    """LAPACK's (L, W = L^-1) of A on the CPU, returned on the device"""
    if key is not None and key in _lapack_cache:
        return _lapack_cache[key]
    Ac = A.cpu()
    Lr, info = torch.linalg.cholesky_ex(Ac)
    assert int(info) == 0
    Wr = torch.linalg.solve_triangular(Lr, torch.eye(A.shape[0], dtype=F64), upper=False)
    out = (Lr.cuda(), Wr.cuda())
    if key is not None:
        _lapack_cache[key] = out
    return out


def gate(what, L, W, A, ref=None, key=None):
    """the library's residuals against LAPACK's on the same matrix; returns the two ratios"""
    Lr, Wr = ref if ref is not None else lapack(A, key)
    rL, rW = residuals(L, W, A)
    rLr, rWr = residuals(Lr, Wr, A)
    qL, qW = rL / max(rLr, EPS), rW / max(rWr, EPS)
    print(f"[chol-residual] {what}: rL {rL:.3e} lapack {rLr:.3e} ratio {qL:.2f} | rW {rW:.3e} lapack {rWr:.3e} ratio {qW:.2f}")
    assert rL <= GATE * rLr + 16 * EPS, f"{what}: factor residual {rL:.3e} vs LAPACK {rLr:.3e}"
    assert rW <= GATE * rWr + 16 * EPS, f"{what}: inverse residual {rW:.3e} vs LAPACK {rWr:.3e}"
    return qL, qW


# ----------------------------------------------------------------------------------------------------- layouts
@pytest.mark.parametrize("nb0", list(range(60, 113, 4)))
@pytest.mark.parametrize("nblk", [2, 4])
def test_every_block_width(ops, nb0, nblk):
    """Every diagonal-block width the plan produces once there is more than one block (the cluster kernel's tile columns
    per CTA change with nb0), with two blocks exactly and with four blocks and three rows of identity padding."""
    Mq = nblk * nb0 - (3 if nblk == 4 else 0)
    assert ops.chol_plan(Mq)[1:] == (nb0, {2: 1, 4: 2}[nblk])
    A = wishart(Mq, 100 + Mq)
    L, W, _ = factor(ops, A)
    gate(f"nb0={nb0} Mq={Mq}", L, W, A)


@pytest.mark.parametrize("Mq", [3072, 3200])
def test_model_layouts(ops, Mq):
    """The layouts of the flagship configurations: nb0 = 96 and 100 (nbp = 104, not a multiple of 8 tiles of 8), 32 blocks."""
    assert ops.chol_plan(Mq)[2] == 5
    A = wishart(Mq, Mq)
    L, W, _ = factor(ops, A)
    gate(f"Mq={Mq}", L, W, A, key=("wishart", Mq, Mq))


@pytest.mark.parametrize("Mq", [100, 224, 400, 1000, 3200])
def test_every_variant(ops, Mq):
    """dsvgp_set_chol_variant 1 (single-CTA kernel + batched recursive inverse), 2 (multi-CTA update + block kernel) and 3
    (cluster kernel, default) each pass the gate, and their factors agree to 1e-13."""
    A = wishart(Mq, Mq)
    key = ("wishart", Mq, Mq)
    out = {}
    for v in (3, 1, 2):
        with chol_variant(ops, v):
            L, W, _ = factor(ops, A)
        gate(f"variant {v} Mq={Mq}", L, W, A, key=key)
        out[v] = L
    for v in (1, 2):
        assert float((out[v] - out[3]).abs().max() / out[3].abs().max()) < 1e-13


@pytest.mark.parametrize("Mq", [7168, 7200])
def test_more_than_64_blocks(ops, Mq):
    """7168 = 64 blocks of 112, the largest size on the two-chain schedule with the eager inverse; 7200 = 128 blocks of 60:
    everything on the caller's stream and the batched recursive inverse (Awork as its scratch), as sample_mvn and _chol_inv
    take it for any covariance above 7168 rows."""
    Mp, nb0, nlev = ops.chol_plan(Mq)
    assert (Mp, nb0, nlev) == {7168: (7168, 112, 6), 7200: (7680, 60, 7)}[Mq]
    A = wishart(Mq, Mq)
    L, W, _ = factor(ops, A)
    gate(f"Mq={Mq}", L, W, A, key=("wishart", Mq, Mq))


# ----------------------------------------------------------------------------------------------------- numerics
@pytest.mark.parametrize("ell", [0.15, 0.7, 2.0])
@pytest.mark.parametrize("duplicate", [False, True])
def test_kzz_conditioning(ops, ell, duplicate):
    """K_zz as a step assembles it (fp64, jitter 1e-3, outputscale 1.7, d = 10, p = 2, M' = 1500), also with two inducing
    points 1e-6 apart, as trained states have them."""
    A = kzz(ops, 500, 10, 2, ell, 1.7, 1e-3, seed=7, duplicate=(250, 1e-6) if duplicate else None)
    print(f"[chol-cond] kzz ell={ell} duplicate={duplicate}: cond {cond(A):.3e}")
    L, W, _ = factor(ops, A)
    gate(f"kzz ell={ell} dup={duplicate}", L, W, A)


def _pair_rows(nb0, nblk, where, aligned):
    """one near-collinear pair per block: at its start, inside it, at its end (straddling: across the block boundary), or
    at an 8-row tile boundary of the pivot chain"""
    out = []
    for k in range(nblk):
        s, e = k * nb0, (k + 1) * nb0 - 1
        a = {"start": s if aligned else s + 1, "inside": s + 40 if aligned else s + 41,
             "end": e - 1 if aligned else e, "tile": s + 16 if aligned else s + 15}[where]
        if 0 <= a and a + 1 < nblk * nb0:
            out.append((a, a + 1))
    return out


# The panel solves multiply by explicit inverses (L21 = A21 W11^T across blocks, A_panel D^T with D = inv(L11) on the 8x8
# tiles inside a block).  A tiny pivot with more rows of its block after it makes that product lose cond(L11) ~ 1e5 of
# accuracy: measured on a B200, factor residual 2e-13 .. 5e-13 against LAPACK's 6e-16 (ratio 340 - 920), with variant 1
# and 3 alike, for every placement but the block end.  The det form itself is not the cause: straddling pairs, which go
# through sequential pivots, fail the same way.  Known open defect; these cases pass once the panels are solved stably.
_EXPLICIT_INVERSE_PANEL = pytest.mark.xfail(strict=True, reason="panel solves by explicit inverse of an ill-conditioned "
                                            "diagonal block: factor residual ~500x LAPACK's")


@pytest.mark.parametrize("where", [pytest.param("start", marks=_EXPLICIT_INVERSE_PANEL),
                                   pytest.param("inside", marks=_EXPLICIT_INVERSE_PANEL), "end",
                                   pytest.param("tile", marks=_EXPLICIT_INVERSE_PANEL)])
@pytest.mark.parametrize("aligned", [True, False])
@pytest.mark.parametrize("variant", [1, 3])
def test_adjacent_near_collinear_rows(ops, where, aligned, variant):
    """Two adjacent rows at cos = 1 - 1e-10 (cond ~ 1e10), once both in one two-pivot step (rows 2m, 2m+1: the second
    pivot comes from det = a11 a22 - a21^2) and once straddling two steps (2m+1, 2m+2), at block starts, inside blocks,
    at block ends and across the 8x8 tiles of the pivot chain."""
    Mq = 400
    Mp, nb0, nlev = ops.chol_plan(Mq)
    pairs = _pair_rows(nb0, Mq // nb0, where, aligned)
    assert pairs and all((a % 2 == 0) == aligned for a, _ in pairs)
    A = near_collinear(Mq, pairs, seed=2 * ["start", "inside", "end", "tile"].index(where) + int(aligned))
    if variant == 3:
        print(f"[chol-cond] near-collinear {where} aligned={aligned}: cond {cond(A):.3e}")
    with chol_variant(ops, variant):
        L, W, _ = factor(ops, A)
    gate(f"collinear {where} aligned={aligned} v{variant}", L, W, A, key=("collinear", where, aligned))


@pytest.mark.parametrize("scale", ["2^100", "2^-100", "graded"])
@pytest.mark.parametrize("variant", [1, 3])
def test_pivots_outside_the_fp32_range(ops, scale, variant):
    """c^2 A with c = 2^100 and 2^-100 puts every pivot outside (1e-30, 1e30), where the fp32 rsqrt seed cannot go and the
    sqrt / division branch takes over; D A D with D = diag(2^u), u in [-60, 60], has pivots on both sides in one matrix.
    Power-of-two scaling commutes with the factorisation, so it is undone exactly and the gate is against LAPACK on A."""
    Mq = 1000
    A = wishart(Mq, 5)
    if scale == "graded":
        g = torch.Generator().manual_seed(9)
        d = torch.pow(2.0, torch.randint(-60, 61, (Mq,), generator=g).to(F64)).cuda()
    else:
        d = torch.full((Mq,), 2.0 ** (100 if scale == "2^100" else -100), dtype=F64, device="cuda")
    As = d[:, None] * A * d[None, :]
    piv = torch.linalg.cholesky(As.cpu()).diagonal() ** 2
    low, high = piv < 1e-30, piv > 1e30
    if scale == "graded":
        assert bool(low.any()) and bool(high.any()) and not bool((low | high).all())
    else:
        assert bool((low | high).all())
    with chol_variant(ops, variant):
        Ls, Ws, _ = factor(ops, As)
    L, W = Ls / d[:, None], Ws * d[None, :]
    gate(f"scale {scale} v{variant}", L, W, A, key=("wishart", Mq, 5))


@pytest.mark.parametrize("Mq", [224, 1000])
@pytest.mark.parametrize("variant", [1, 2, 3])
def test_upper_triangle_is_never_read(ops, Mq, variant):
    """A NaN upper triangle of Awork gives bit for bit the factor and inverse of a zero one."""
    A = wishart(Mq, 3)
    with chol_variant(ops, variant):
        _, _, (_, L0, W0) = factor(ops, A, upper_fill=0.0)
        _, _, (_, L1, W1) = factor(ops, A, upper_fill=NAN)
    assert torch.equal(L0.tril(), L1.tril()) and torch.equal(W0.tril(), W1.tril())


# ----------------------------------------------------------------------------------------------------- info
def _info_rows(Mq, nb0):
    nblk = -(-Mq // nb0)
    mid = (nblk // 2) * nb0 + 1
    return sorted({0, 1, 6, 7, nb0 - 1, nb0, nb0 + 1, mid, Mq - 1})


_lapack_info = {}


@pytest.mark.parametrize("Mq", [224, 3072, 7200])
@pytest.mark.parametrize("variant", [1, 2, 3])
def test_info_is_the_first_bad_pivot(ops, Mq, variant):
    """*info = 1 + the index of the first pivot that is not a positive finite number, in every block and at both positions
    of a two-pivot step: pivot j made negative (A[j,j] -= 1.5 L[j,j]^2, where LAPACK reports j + 1 too), a NaN on the
    diagonal, a NaN at A[j, i] with i in an earlier block, and +inf on the diagonal."""
    Mp, nb0, nlev = ops.chol_plan(Mq)
    A = wishart(Mq, Mq)
    Lr, _ = lapack(A, key=("wishart", Mq, Mq))
    piv = Lr.diagonal() ** 2
    rows = _info_rows(Mq, nb0)
    assert {j % 2 for j in rows} == {0, 1}
    bufs = [torch.full((Mp, Mp + 8), NAN, dtype=F64, device="cuda") for _ in range(3)]
    Aw, L, W = (b[:, :Mp] for b in bufs)
    info = torch.empty(1, dtype=torch.int32, device="cuda")

    def run(j, i, value):
        Aw[:Mq, :Mq] = A
        ops.pad_identity(Aw, Mq)
        Aw[j, i] = value if value is not None else Aw[j, i] - 1.5 * piv[j]
        info.fill_(-7)
        ops.cholesky_inverse(Aw, L, W, nb0, nlev, info)
        return int(info.item())

    with chol_variant(ops, variant):
        for j in rows:
            key = (Mq, j)
            if key not in _lapack_info:
                Ac = A[:j + 1, :j + 1].cpu()
                Ac[j, j] -= 1.5 * float(piv[j])
                _lapack_info[key] = int(torch.linalg.cholesky_ex(Ac).info)
            assert _lapack_info[key] == j + 1
            assert run(j, j, None) == j + 1, f"negative pivot {j}"
            assert run(j, j, NAN) == j + 1, f"NaN pivot {j}"
            assert run(j, j, math.inf) == j + 1, f"+inf pivot {j}"
            if j >= nb0:
                i = max(0, j - nb0 - 1)
                assert run(j, i, NAN) == j + 1, f"NaN at ({j}, {i})"
        Aw[:Mq, :Mq] = A                        # the same buffers after all those failures: info goes back to 0 and
        ops.pad_identity(Aw, Mq)                # both lower triangles are rewritten in full
        ops.cholesky_inverse(Aw, L, W, nb0, nlev, info)
        assert int(info.item()) == 0
    assert bool(L.tril().isfinite().all()) and bool(W.tril().isfinite().all())
    for b in bufs:
        assert bool(b[:, Mp:].isnan().all()), "write beyond the Mp columns"


# ----------------------------------------------------------------------------------------------------- pieces
@pytest.mark.parametrize("b", [60, 192])
@pytest.mark.parametrize("batch", [2, 5])
def test_batched_gemm_f64(ops, b, batch):
    """dsvgp_gemm_f64 with batch > 1 and the strides and triangle flags of the recursive inverse (chol.cu): pair q of a level
    with blocks of b sits at rows / columns 2bq; T_q = L21_q W11_q goes into the work matrix, W21_q = -W22_q T_q into W.
    b = 60 takes the register-staged kernel, b = 192 (K > 128) the cp.async one.  The triangles the flags exclude hold
    NaN; everything outside the written blocks must keep its NaN."""
    from dsvgp_b200 import _lib
    n = 2 * b * batch
    ld = n + 6
    g = torch.Generator().manual_seed(b + batch)
    Lc = torch.randn(n, n, generator=g, dtype=F64)
    Wc = torch.randn(n, n, generator=g, dtype=F64)
    Lc, Wc = Lc.tril() + torch.full((n, n), NAN, dtype=F64).triu(1), Wc.tril() + torch.full((n, n), NAN, dtype=F64).triu(1)
    L = torch.full((n, ld), NAN, dtype=F64, device="cuda")[:, :n]
    W = torch.full((n, ld), NAN, dtype=F64, device="cuda")[:, :n]
    Aw = torch.full((n, ld), NAN, dtype=F64, device="cuda")[:, :n]
    L.copy_(Lc)
    W.copy_(Wc)
    s = 2 * b * ld + 2 * b
    _lib.call("dsvgp_gemm_f64", 0, 0, b, b, b, 1.0, L[b:], ld, W, ld, 0.0, Aw[b:], ld, 0, 1, 0, batch, s, s, s,
              None, 0, None, 0, None, 0)
    _lib.call("dsvgp_gemm_f64", 0, 0, b, b, b, -1.0, W[b:, b:], ld, Aw[b:], ld, 0.0, W[b:], ld, 1, 0, 0, batch, s, s, s,
              None, 0, None, 0, None, 0)
    Awc, Wg = Aw.cpu(), W.cpu()
    written = torch.zeros(n, n, dtype=torch.bool)
    for q in range(batch):
        o = 2 * b * q
        T = Lc[o + b:o + 2 * b, o:o + b] @ Wc[o:o + b, o:o + b].tril()
        W21 = -Wc[o + b:o + 2 * b, o + b:o + 2 * b].tril() @ T
        for got, want in ((Awc[o + b:o + 2 * b, o:o + b], T), (Wg[o + b:o + 2 * b, o:o + b], W21)):
            assert float((got - want).abs().max() / want.abs().max()) < 1e-13
        written[o + b:o + 2 * b, o:o + b] = True
    assert bool(Awc[~written].isnan().all())
    keep = ~written
    assert torch.equal(Wg[keep].nan_to_num(7.0), Wc[keep].nan_to_num(7.0))


def test_odd_leading_dimension_is_refused(ops):
    """The factorisation loads Awork two doubles at a time from the start of every block column: an odd leading dimension,
    an Awork that is not 16-byte aligned, or an odd block width with more than one block (block column 2 then starts at an
    odd element) is refused before anything is enqueued (info, L and W keep what they held)."""
    from dsvgp_b200._lib import DsvgpError
    Mq = 224
    Mp, nb0, nlev = ops.chol_plan(Mq)
    A = wishart(Mq, 1)
    odd = torch.zeros(Mp, Mp + 1, dtype=F64, device="cuda")[:, :Mp]
    flat = torch.zeros(Mp * (Mp + 8) + 1, dtype=F64, device="cuda")
    shifted = flat[1:].view(Mp, Mp + 8)[:, :Mp]
    assert odd.stride(0) % 2 == 1 and shifted.data_ptr() % 16 == 8
    aligned = torch.zeros(244, 252, dtype=F64, device="cuda")[:, :244]
    # (Aw, nb0, nlev): odd lda; Awork at 8 mod 16 bytes; aligned Awork and even lda, but four blocks of nb0 = 61 (Mp = 244)
    cases = [(odd, nb0, nlev), (shifted, nb0, nlev), (aligned, 61, 2)]
    for Aw, nb, nl in cases:
        n = min(Mq, Aw.shape[0])
        Aw[:n, :n] = A[:n, :n]
        ops.pad_identity(Aw, n)
        m = Aw.shape[0]
        L, W = (torch.full((m, m + 8), NAN, dtype=F64, device="cuda")[:, :m] for _ in range(2))
        info = torch.full((1,), 4321, dtype=torch.int32, device="cuda")
        with pytest.raises(DsvgpError):
            ops.cholesky_inverse(Aw, L, W, nb, nl, info)
        torch.cuda.synchronize()
        assert int(info.item()) == 4321
        assert bool(L.isnan().all()) and bool(W.isnan().all())
