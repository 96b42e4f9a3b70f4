"""Direct tests of the general GEMM (csrc/gemm.cu, dsvgp_gemm_{f32,f64}) on each of its four kernels, and of the triangle
helpers beside it (csrc/misc.cu: symmetrize, mirror_lower, tril_minus_eye, sym_phi).

Kernels, and how a test selects one:
    reg64    register-staged fp64 kernel: K <= 128, or any K with dsvgp_set_gemm64_async(0)
    async64  cp.async fp64 kernel: K > 128 with the default dsvgp_set_gemm64_async(1)
    rank64   fp64 rank-update kernel: set_rank_update(1) and an eligible product (!ta, tb, even 8 <= K <= 128, no flags, ...)
    f32      3xTF32 kernel with the fp64 master sum
test_each_kernel_is_reached checks with torch.profiler that these settings launch the kernel they name.

Exact tests.  Every operand entry is an integer, |a|, |b| <= 2^10 in fp64 and <= 8 in fp32; alpha is a power of two or
-1 and beta * D is a multiple of 1/2.  The true result is then representable and every partial sum is exact: in fp64
because K * 2^20 < 2^53; in 3xTF32 because the integers fit TF32 (lo = 0), a 16-term tile sum stays below 2^23 and the
total below 2^24.  A correct kernel returns the CPU fp64 product bit for bit, so a dropped, duplicated or misplaced term,
a wrong stage buffer, stride or mask fails with no tolerance to hide in.  The triangle a flag excludes and every operand's
padding hold NaN, so a masked element that is loaded at all (even to be multiplied by zero) poisons the result.  Outputs
sit inside NaN-filled buffers with extra rows and columns; everything outside [:M, :N], and with c_tri = 1 every 64 x 64
tile strictly above the diagonal band, must still hold what it held before the call.

Rounding tests.  fp64 is held to a componentwise bound in |op(A)| |op(B)| against cuBLAS fp64 on the device; fp32
(3xTF32) to c * 2^-21 |A| |B| + 2^-24 |C| against an fp64 product of the same fp32 values, with c four times the maximum
measured on an NVIDIA B200 (1000 W power limit) -- see C32 below."""
import contextlib

import pytest
import torch

pytestmark = pytest.mark.gpu
F32, F64 = torch.float32, torch.float64
NAN = float("nan")
BM = 64                                          # output tile of every kernel (gemm.cu: BM = BN = 64)
LAYOUTS = ("even", "odd", "shift")               # double2 epilogue / odd leading dimension / base 8 bytes past 16-byte alignment
TT = ((False, False), (False, True), (True, False), (True, True))
ALPHAS = (1.0, -1.0, 2.0, 0.5)
BETAS = (1.0, -1.0, 2.0, 0.5)

# fp32 (3xTF32) rounding: |C - ref| <= C32 * 2^-21 (|A||B|)_ij + 2^-24 |ref_ij|.  Over the cases of test_f32_rounding_bound
# and test_f32_long_k_uses_the_fp64_master_sum the largest (|C - ref| - 2^-24 |ref|) / (2^-21 |A||B|) measured on an NVIDIA
# B200 (1000 W power limit) was 0.70 (W^T Y, 1000^3); C32 is four times that.
C32 = 2.8


@pytest.fixture(scope="module")
def ops():
    from dsvgp_b200 import ops
    return ops


@pytest.fixture(scope="module")
def lib():
    from dsvgp_b200 import _lib
    return _lib


@contextlib.contextmanager
def _kernel(name):
    """Select the kernel family `name` for the calls inside; restore the defaults (async 1, rank-update 0) after."""
    from dsvgp_b200 import _lib, ops
    _lib.call_raw("dsvgp_set_gemm64_async", 0 if name == "reg64" else 1)
    ops.set_rank_update(1 if name == "rank64" else 0)
    try:
        yield F32 if name == "f32" else F64
    finally:
        _lib.call_raw("dsvgp_set_gemm64_async", 1)
        ops.set_rank_update(0)


# ------------------------------------------------------------------------------------------------ layouts and checks
def _spec(lay, cols):
    """-> (leading dimension, element offset into the buffer) of a `cols`-wide matrix in layout `lay`."""
    if isinstance(lay, tuple):
        return lay
    if lay == "tight":
        return cols, 0
    if lay == "odd":
        return (cols + 2) | 1, 0
    return (cols + 3) // 2 * 2, (1 if lay == "shift" else 0)


def _place(host, lay, dtype, extra_rows=2):
    """host (rows x cols, may hold NaN) in a NaN-filled device buffer -> (view, flat buffer, ld, offset)."""
    rows, cols = host.shape
    ld, off = _spec(lay, cols)
    flat = torch.full((off + (rows + extra_rows) * ld + 3,), NAN, dtype=dtype, device="cuda")
    view = flat.as_strided((rows, cols), (ld, 1), off)
    if rows and cols:
        view.copy_(host.to(dtype))
    return view, flat, ld, off


def _expect(before, off, ld, ref, done):
    """The buffer `before` (CPU) with ref written where `done` (over the [:M, :N] view at off / ld) and nothing else."""
    exp = before.double().clone()
    if ref.numel():
        view = exp.as_strided(tuple(ref.shape), (ld, 1), off)
        view[done] = ref[done]
    return exp


def _assert_same(got, exp, what):
    """Bit-for-bit equality (NaN where NaN is expected, +0 == -0)."""
    got = got.double().cpu()
    gn, en = got.isnan(), exp.isnan()
    bad = (gn != en) | (~en & ~gn & (got != exp))
    if bool(bad.any()):
        i = int(bad.nonzero()[0])
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} elements differ; first at flat index {i}: "
                             f"got {float(got[i])!r}, want {float(exp[i])!r}")


def _done(M, N, c_tri):
    """Which elements of [:M, :N] a product writes: all, or with c_tri = 1 the tiles with n0 < m0 + 64."""
    if not c_tri:
        return torch.ones(M, N, dtype=torch.bool)
    return (torch.arange(N).unsqueeze(0) // BM) <= (torch.arange(M).unsqueeze(1) // BM)


def _keep(rows, cols, tri):
    keep = torch.ones(rows, cols, dtype=torch.bool)
    return keep.tril() if tri == 1 else keep.triu() if tri == 2 else keep


def _ints(g, shape, dtype):
    r = 1024 if dtype == F64 else 8
    return torch.randint(-r, r + 1, shape, generator=g).double()


def _tri_operand(g, rows, cols, tri, dtype):
    """-> (stored values with NaN in the excluded triangle, the operand as the product must see it)."""
    v = _ints(g, (rows, cols), dtype)
    keep = _keep(rows, cols, tri)
    return torch.where(keep, v, NAN), torch.where(keep, v, 0.0)


def _mode(i):
    """Epilogue input i % 4: (beta, explicit D, second output C2)."""
    return ((0.0, False, False), (BETAS[i // 4 % 4], False, False), (BETAS[(i // 4 + 1) % 4], True, False),
            (BETAS[(i // 4 + 2) % 4], True, True))[i % 4]


def _exact(ops, kernel, ta, tb, M, N, K, a_tri=0, b_tri=0, c_tri=0, alpha=1.0, beta=0.0, use_D=False, use_C2=False,
           lay=("even",) * 4, op_lay=("even", "even"), seed=0):
    """One call of ops.gemm on integer operands, checked bit for bit (C and C2 buffers, sentinels included).
    lay: layouts of C, D, C2, D2; op_lay: layouts of the stored A and B (names of _spec or (ld, offset))."""
    with _kernel(kernel) as dt:
        g = torch.Generator().manual_seed(seed * 1000003 + M * 10007 + N * 101 + K)
        Ah, Ar = _tri_operand(g, M, K, a_tri, dt)
        Bh, Br = _tri_operand(g, K, N, b_tri, dt)
        A = _place(Ah.T if ta else Ah, op_lay[0], dt)[0]
        B = _place(Bh.T if tb else Bh, op_lay[1], dt)[0]
        prod = Ar @ Br
        in_place = beta != 0 and not use_D
        Cin = _ints(g, (M, N), dt) if in_place else torch.full((M, N), NAN, dtype=F64)
        C, Cf, ldc, offc = _place(Cin, lay[0], dt)
        D = C2 = D2 = None
        if use_D:
            Dh = _ints(g, (M, N), dt)
            D = _place(Dh, lay[1], dt)[0]
        if use_C2:
            C2, C2f, ldc2, offc2 = _place(torch.full((M, N), NAN, dtype=F64), lay[2], dt)
            D2h = _ints(g, (M, N), dt)
            D2 = _place(D2h, lay[3], dt)[0]
            C2_before = C2f.cpu()
        C_before = Cf.cpu()
        ops.gemm(A, B, C, ta=ta, tb=tb, alpha=alpha, beta=beta, a_tri=a_tri, b_tri=b_tri, c_tri=c_tri, D=D, M=M, N=N, K=K,
                 C2=C2, D2=D2)
        ref = alpha * prod
        if beta != 0:
            ref = ref + beta * (Dh if use_D else Cin)
        done = _done(M, N, c_tri)
        what = (f"{kernel} ta={ta} tb={tb} M={M} N={N} K={K} a_tri={a_tri} b_tri={b_tri} c_tri={c_tri} alpha={alpha} "
                f"beta={beta} D={use_D} C2={use_C2} lay={lay} op_lay={op_lay}")
        _assert_same(Cf, _expect(C_before, offc, ldc, ref, done), "C: " + what)
        if use_C2:
            _assert_same(C2f, _expect(C2_before, offc2, ldc2, ref + D2h, done), "C2: " + what)


# ------------------------------------------------------------------------------------------------ 1. exact tests
SWEEP = ([("reg64", s) for s in [(129, 65, 128), (63, 127, 17), (65, 64, 1), (7, 129, 64), (129, 65, 130), (65, 7, 257)]]
         + [("async64", s) for s in [(129, 65, 130), (63, 127, 129), (7, 129, 200), (130, 7, 257)]]
         + [("f32", s) for s in [(129, 65, 128), (63, 127, 17), (7, 129, 64), (129, 65, 130), (65, 7, 257)]])


@pytest.mark.parametrize("kernel,shape", SWEEP, ids=[f"{k}-{m}x{n}x{kk}" for k, (m, n, kk) in SWEEP])
def test_exact_transpose_triangle_sweep(ops, kernel, shape):
    """All 4 (ta, tb) x a_tri x b_tri x c_tri at shapes with ragged tiles, M > K and K > M; the epilogue input, the
    output layouts and the stored operand layouts rotate with the case."""
    M, N, K = shape
    i = 0
    for ta, tb in TT:
        for a_tri in range(3):
            for b_tri in range(3):
                for c_tri in (0, 1):
                    beta, use_D, use_C2 = _mode(i)
                    _exact(ops, kernel, ta, tb, M, N, K, a_tri, b_tri, c_tri, alpha=ALPHAS[i // 4 % 4], beta=beta,
                           use_D=use_D, use_C2=use_C2, lay=tuple(LAYOUTS[(i + j) % 3] for j in range(4)),
                           op_lay=(LAYOUTS[i % 3], LAYOUTS[(i + 1) % 3]), seed=i)
                    i += 1


EDGES = (1, 7, 63, 64, 65, 127, 129)


@pytest.mark.parametrize("kernel", ["reg64", "async64", "f32"])
def test_exact_tile_edges(ops, kernel):
    """Every (M, N, K) from {1, 7, 63, 64, 65, 127, 129} (async64: K in {129, 130}); transposes and layouts rotate."""
    ks = (129, 130) if kernel == "async64" else EDGES
    i = 0
    for M in EDGES:
        for N in EDGES:
            for K in ks:
                ta, tb = TT[i % 4]
                _exact(ops, kernel, ta, tb, M, N, K, alpha=ALPHAS[i % 4], lay=(LAYOUTS[i % 3],) * 4,
                       op_lay=(LAYOUTS[(i + 1) % 3], LAYOUTS[(i + 2) % 3]), seed=i)
                i += 1


@pytest.mark.parametrize("kernel", ["reg64", "default64", "f32"])
@pytest.mark.parametrize("K", [0, 1, 4, 15, 16, 17, 128, 129, 130])
def test_exact_k_edges(ops, kernel, K):
    """The dispatch (K = 128 / 129) and k-tile edges; K = 0 must give beta * D.  default64: the fp64 dispatch as shipped."""
    kern = "async64" if kernel == "default64" else kernel
    i = 0
    for ta, tb in TT:
        for a_tri, b_tri in ((0, 0), (1, 0), (2, 1), (0, 2), (1, 1)):
            beta, use_D, use_C2 = _mode(i + 1)
            _exact(ops, kern, ta, tb, 65, 63, K, a_tri, b_tri, c_tri=i % 2, alpha=ALPHAS[i % 4], beta=beta, use_D=use_D,
                   use_C2=use_C2, lay=tuple(LAYOUTS[(i + j) % 3] for j in range(4)), seed=i)
            i += 1


@pytest.mark.parametrize("kernel", ["reg64", "async64", "rank64", "f32"])
@pytest.mark.parametrize("N", [66, 67])
def test_exact_epilogue(ops, kernel, N):
    """Every epilogue input (beta = 0 over a NaN C, in place on C, explicit D, C2 = C + D2) with each of C, D, C2 and D2 in
    each layout, every alpha, with c_tri 0 and 1; N = 66 / 67: even and odd right edge.  rank64 runs only the products
    that kernel takes (C2 goes to the general kernel)."""
    M, K = 70, {"reg64": 40, "async64": 150, "rank64": 64, "f32": 40}[kernel]
    cases = []
    for a in range(4):
        for lc in LAYOUTS:
            cases.append((ALPHAS[a], 0.0, False, False, (lc, "even", "even", "even")))
            cases.append((ALPHAS[a], BETAS[a], False, False, (lc, "even", "even", "even")))
    for lc in LAYOUTS:
        for ld_ in LAYOUTS:
            cases.append((-1.0, 0.5, True, False, (lc, ld_, "even", "even")))
            for lc2 in LAYOUTS:
                cases.append((2.0, 1.0, False, True, (lc, "even", lc2, ld_)))
                for ld2 in LAYOUTS:
                    cases.append((0.5, -1.0, True, True, (lc, ld_, lc2, ld2)))
    for i, (alpha, beta, use_D, use_C2, lay) in enumerate(cases):
        ta, tb = (False, True) if kernel == "rank64" else TT[i % 4]
        a_tri = 0 if kernel == "rank64" else (0, 1, 2)[i % 3]
        _exact(ops, kernel, ta, tb, M, N, K, a_tri=a_tri, c_tri=i % 2, alpha=alpha, beta=beta, use_D=use_D, use_C2=use_C2,
               lay=lay, seed=i)


@pytest.mark.parametrize("K", [128, 98, 8, 16, 96, 100])
def test_exact_rank_update(ops, K):
    """The rank-update kernel at the K it takes (K = 98: a 4-wide DMMA step half past K), ragged tiles, c_tri 0 / 1,
    beta = 0 / in place / explicit D, every output layout."""
    i = 0
    for M, N in ((1, 1), (7, 64), (65, 63), (129, 130)):
        for c_tri in (0, 1):
            for m in range(3):
                beta, use_D, _ = _mode(m + 4 * i)
                _exact(ops, "rank64", False, True, M, N, K, c_tri=c_tri, alpha=ALPHAS[i % 4], beta=beta, use_D=use_D,
                       lay=(LAYOUTS[i % 3], LAYOUTS[(i + 1) % 3], "even", "even"), seed=i)
                i += 1


def test_each_kernel_is_reached(ops):
    """The settings the tests above use launch the kernel they name (torch.profiler kernel names)."""
    from torch.profiler import ProfilerActivity, profile
    cases = [("reg64", False, False, 0, 130, "gemm_kernel<double"), ("async64", False, False, 0, 128, "gemm_kernel<double"),
             ("async64", True, False, 1, 129, "gemm64_async_kernel"), ("rank64", False, True, 0, 98, "rank_update64_kernel"),
             ("rank64", False, True, 1, 98, "gemm_kernel<double"), ("f32", True, True, 2, 300, "gemm_kernel<float")]
    for kernel, ta, tb, a_tri, K, name in cases:
        with _kernel(kernel) as dt:
            A = torch.zeros((K, 70) if ta else (70, K), dtype=dt, device="cuda")
            B = torch.zeros((66, K) if tb else (K, 66), dtype=dt, device="cuda")
            C = torch.empty(70, 66, dtype=dt, device="cuda")
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                ops.gemm(A, B, C, ta=ta, tb=tb, a_tri=a_tri)
                torch.cuda.synchronize()
            names = [e.key for e in prof.key_averages() if "gemm" in e.key or "rank_update" in e.key]
            assert len(names) == 1 and name in names[0], (kernel, K, names)


def _batched(ops, lib, kernel, batch, K, ta, tb, a_tri, b_tri, c_tri, mode, seed):
    """dsvgp_gemm with `batch` products at strides that are not multiples of a tile and are odd, so that odd-numbered
    batches sit 8 bytes off 16-byte alignment (the scalar epilogue) and even-numbered ones do not; sA != sB.
    mode 0: beta = 0 over NaN; 1: explicit D, which every batch shares; 2: in place."""
    M, N = 70, 45
    with _kernel(kernel) as dt:
        g = torch.Generator().manual_seed(seed)
        rA, cA = (K, M) if ta else (M, K)
        rB, cB = (N, K) if tb else (K, N)
        lda, ldb, ldc = cA + 3, cB + 2, N + 3 + (N + 3) % 2
        sA, sB, sC = rA * lda + 3, rB * ldb + 5, M * ldc + 1
        Af, Bf, Cf = (torch.full((batch * s + 7,), NAN, dtype=dt, device="cuda") for s in (sA, sB, sC))
        view = lambda f, z, s, r, c, ld: f.as_strided((r, c), (ld, 1), z * s)
        beta = (0.0, -1.0, 2.0)[mode]
        Dh = _ints(g, (M, N), dt)
        D = _place(Dh, "odd", dt)[0] if mode == 1 else None
        refs = []
        for z in range(batch):
            Ah, Ar = _tri_operand(g, M, K, a_tri, dt)
            Bh, Br = _tri_operand(g, K, N, b_tri, dt)
            view(Af, z, sA, rA, cA, lda).copy_((Ah.T if ta else Ah).to(dt))
            view(Bf, z, sB, rB, cB, ldb).copy_((Bh.T if tb else Bh).to(dt))
            ref = 2.0 * (Ar @ Br)
            if mode == 1:
                ref = ref + beta * Dh
            if mode == 2:
                Cin = _ints(g, (M, N), dt)
                view(Cf, z, sC, M, N, ldc).copy_(Cin.to(dt))
                ref = ref + beta * Cin
            refs.append(ref)
        before = Cf.cpu()
        lib.call("dsvgp_gemm_" + lib.suffix(dt), int(ta), int(tb), M, N, K, 2.0, Af, lda, Bf, ldb, beta, Cf, ldc, a_tri, b_tri,
                 c_tri, batch, sA, sB, sC, D, ldc if D is None else D.stride(0), None, 0, None, 0)
        exp = before.double().clone()
        done = _done(M, N, c_tri)
        for z, ref in enumerate(refs):
            exp.as_strided((M, N), (ldc, 1), z * sC)[done] = ref[done]
        _assert_same(Cf, exp, f"batched {kernel} batch={batch} K={K} ta={ta} tb={tb} tri={a_tri},{b_tri},{c_tri} mode={mode}")


@pytest.mark.parametrize("kernel,K", [("reg64", 60), ("async64", 150), ("f32", 60)])
@pytest.mark.parametrize("batch", [2, 5])
def test_exact_batched(ops, lib, kernel, K, batch):
    pats = ((False, False, 1, 0, 0), (True, False, 2, 1, 0), (False, True, 0, 2, 1), (True, True, 1, 1, 1), (False, True, 2, 0, 0))
    for i, (ta, tb, a_tri, b_tri, c_tri) in enumerate(pats):
        for mode in range(3):
            _batched(ops, lib, kernel, batch, K, ta, tb, a_tri, b_tri, c_tri, mode, seed=10 * i + mode)


def _engine_calls(Mq, nq, num):
    """(name, ta, tb, a_tri, b_tri, c_tri, alpha, beta, D, C2, M, N, K, (layouts of C, D, C2, D2), (layouts of A, B)) of the
    products engine.py and gp.py make, on buffers laid out as they lay them out."""
    ev = ("even",) * 4
    c0 = 3 * (Mq // 9)                      # a column panel [c0, c1) of the sharded backward tail (q = p + 1 = 3)
    c1, Kk = 2 * c0, Mq - c0
    nJ = c1 - c0
    diag = (Mq, c0 * Mq + c0)               # a view [c0:, c0:] of an Mq x Mq matrix
    return [
        ("A = W Kzx", False, False, 1, 0, 0, 1.0, 0.0, False, False, Mq, nq, Mq, ev, ("tight", "even")),
        ("B' = E^T A, B = A + B'", True, False, 2, 0, 0, 1.0, 0.0, False, True, Mq, nq, Mq, ev, ("tight", "even")),
        ("C = E B + B'", False, False, 1, 0, 0, 1.0, 1.0, True, False, Mq, nq, Mq, ev, ("tight", "even")),
        ("dKzx = W^T dA", True, False, 2, 0, 0, 1.0, 0.0, False, False, Mq, nq, Mq, ev, ("tight", "even")),
        ("G = Ag A^T (lower tiles)", False, True, 0, 0, 1, 1.0, 0.0, False, False, Mq, Mq, nq, ev, ("even", "even")),
        ("H' = E^T G, H = G + H'", True, False, 2, 0, 0, 1.0, 0.0, False, True, Mq, Mq, Mq, ev, ("tight", "tight")),
        ("X = 2 E H + 2 H'", False, False, 1, 0, 0, 2.0, 2.0, True, False, Mq, Mq, Mq, ev, ("tight", "tight")),
        ("Y = -Phi W (lower)", False, False, 1, 1, 1, -1.0, 0.0, False, False, Mq, Mq, Mq, ev, ("tight", "tight")),
        ("S = W^T Y", True, False, 2, 1, 0, 1.0, 0.0, False, False, Mq, Mq, Mq, ev, ("tight", "tight")),
        ("panel Y[c0:, J] = -Psi[c0:, c0:] W[c0:, J]", False, False, 1, 1, 1, -1.0, 0.0, False, False, Kk, nJ, Kk,
         (diag,) + ("even",) * 3, (diag, diag)),
        ("panel S[:c0, J] = W[c0:, :c0]^T Y[c0:, J]", True, False, 0, 1, 0, 1.0, 0.0, False, False, c0, nJ, Kk,
         ((Mq, c0),) + ("even",) * 3, ((Mq, c0 * Mq), diag)),
        ("panel S[c0:, J] = W[c0:, c0:]^T Y[c0:, J]", True, False, 2, 1, 0, 1.0, 0.0, False, False, Kk, nJ, Kk,
         (diag,) + ("even",) * 3, (diag, diag)),
        ("cov += A^T (S - I) A", True, False, 0, 0, 0, 1.0, 1.0, False, False, nq, nq, Mq, ev, ("even", "even")),
        ("A Gs", False, False, 0, 0, 0, 1.0, 0.0, False, False, Mq, nq, nq, ev, ("even", "tight")),
        ("G = 1/2 (A Gs) A^T", False, True, 0, 0, 0, 0.5, 0.0, False, False, Mq, Mq, nq, ev, ("even", "even")),
        ("draws z L^T", False, True, 0, 2, 0, 1.0, 0.0, False, False, num, nq, nq, ("tight",) * 4, ("tight", (nq + 11, 0))),
        ("Lbar = tril(gout^T z)", True, False, 0, 0, 1, 1.0, 0.0, False, False, nq, nq, num, ev, ("tight", "tight")),
        ("dz = gout L", False, False, 0, 1, 0, 1.0, 0.0, False, False, num, nq, nq, ("tight",) * 4, ("tight", (nq + 11, 0))),
        ("NGD S = Lm^T Lm", True, False, 2, 1, 0, 1.0, 0.0, False, False, Mq, Mq, Mq, ("tight",) * 4, ("tight", "tight")),
        ("NGD m = S theta (N = 1, ld 1)", False, False, 0, 0, 0, 1.0, 0.0, False, False, Mq, 1, Mq, ("tight",) * 4,
         ("tight", "tight")),
        ("NGD tril(L^T dL)", True, False, 2, 1, 1, 1.0, 0.0, False, False, Mq, Mq, Mq, ("tight",) * 4, ("tight", "tight")),
        ("NGD Phi W (lower)", False, False, 1, 1, 1, 1.0, 0.0, False, False, Mq, Mq, Mq, ("tight",) * 4, ("tight", "tight")),
        ("NGD dmu - 2 dS m (N = 1, ld 1)", False, False, 0, 0, 0, -2.0, 1.0, True, False, Mq, 1, Mq, ("tight",) * 4,
         ("tight", "tight")),
    ]


@pytest.mark.parametrize("dtype", [F64, F32])
@pytest.mark.parametrize("Mq", [60, 384])
def test_exact_engine_call_patterns(ops, dtype, Mq):
    """The flags, shapes, views (offset panels, ld = 1 vectors) and epilogues of every ops.gemm call of engine.py and
    gp.py, at a ragged (60: C1) and an aligned (384) M', on the dispatch as shipped."""
    for i, (name, ta, tb, a_tri, b_tri, c_tri, alpha, beta, use_D, use_C2, M, N, K, lay, op_lay) in \
            enumerate(_engine_calls(Mq, 133, 5)):
        _exact(ops, "f32" if dtype == F32 else "async64", ta, tb, M, N, K, a_tri, b_tri, c_tri, alpha=alpha, beta=beta,
               use_D=use_D, use_C2=use_C2, lay=lay, op_lay=op_lay, seed=i)


def test_refusals_and_empty_products(lib):
    """C2 without D2, K < 0, and a NULL operand with K > 0 are refused with DSVGP_ERR_ARG; M = 0, N = 0 and batch = 0 return
    OK and write nothing; K = 0 with NULL operands gives beta * C."""
    for dt in (F64, F32):
        fn = "dsvgp_gemm_" + lib.suffix(dt)
        A, B = torch.ones(8, 8, dtype=dt, device="cuda"), torch.ones(8, 8, dtype=dt, device="cuda")
        C = torch.full((8, 8), NAN, dtype=dt, device="cuda")
        C2 = torch.full((8, 8), NAN, dtype=dt, device="cuda")
        args = lambda M, N, K, batch, c2, d2, a=A, b=B, beta=0.0: (0, 0, M, N, K, 1.0, a, 8, b, 8, beta, C, 8, 0, 0, 0, batch,
                                                                  0, 0, 0, None, 0, c2, 8, d2, 8, None)
        assert lib.call_raw(fn, *args(8, 8, 8, 1, C2, None)) == -1
        assert lib.call_raw(fn, *args(8, 8, -1, 1, None, None)) == -1
        assert lib.call_raw(fn, *args(8, 8, 8, 1, None, None, a=None)) == -1
        assert lib.call_raw(fn, *args(8, 8, 8, 1, None, None, b=None)) == -1
        for M, N, batch in ((0, 8, 1), (8, 0, 1), (8, 8, 0)):
            assert lib.call_raw(fn, *args(M, N, 8, batch, C2, A)) == 0
        torch.cuda.synchronize()
        assert bool(C.isnan().all()) and bool(C2.isnan().all())
        C.fill_(3.0)
        assert lib.call_raw(fn, *args(8, 8, 0, 1, None, None, a=None, b=None, beta=-0.5)) == 0
        torch.cuda.synchronize()
        assert bool((C == -1.5).all())


@pytest.mark.parametrize("K", [130, 3072])
def test_reg_and_async_kernels_are_bit_identical(ops, K):
    """On real fp64 operands the register-staged and cp.async kernels feed the same DMMA fragments in the same k order."""
    g = torch.Generator(device="cuda").manual_seed(K)
    M, N = 200, 190
    for ta, tb, a_tri, b_tri, c_tri in ((False, False, 0, 0, 0), (True, False, 2, 1, 0), (False, True, 0, 0, 1),
                                        (False, False, 1, 1, 1), (True, True, 1, 2, 0)):
        Ms, Ns = (K if a_tri else M), (K if b_tri else N)       # triangular operands square, as the library uses them
        A = torch.randn((K, Ms) if ta else (Ms, K), generator=g, dtype=F64, device="cuda")
        B = torch.randn((Ns, K) if tb else (K, Ns), generator=g, dtype=F64, device="cuda")
        D = torch.randn(Ms, Ns, generator=g, dtype=F64, device="cuda")
        outs = []
        for kernel in ("reg64", "async64"):
            C = torch.full((Ms, Ns), NAN, dtype=F64, device="cuda")
            with _kernel(kernel):
                ops.gemm(A, B, C, ta=ta, tb=tb, alpha=2.0, beta=1.0, D=D, a_tri=a_tri, b_tri=b_tri, c_tri=c_tri)
            outs.append(C.cpu())
        _assert_same(outs[1].reshape(-1), outs[0].reshape(-1),
                     f"async vs register-staged K={K} ta={ta} tb={tb} tri={a_tri},{b_tri},{c_tri}")


@pytest.mark.parametrize("K", [8, 96, 98, 128])
def test_rank_update_and_reg_kernels_are_bit_identical(ops, K):
    g = torch.Generator(device="cuda").manual_seed(K)
    M, N = 300, 200
    A = torch.randn(M, K, generator=g, dtype=F64, device="cuda")
    B = torch.randn(N, K, generator=g, dtype=F64, device="cuda")
    D = torch.randn(M, N, generator=g, dtype=F64, device="cuda")
    for c_tri in (0, 1):
        outs = []
        for kernel in ("rank64", "reg64"):
            C = torch.full((M, N), NAN, dtype=F64, device="cuda")
            with _kernel(kernel):
                ops.gemm(A, B, C, tb=True, alpha=2.0, beta=1.0, D=D, c_tri=c_tri)
            outs.append(C.cpu().reshape(-1))
        _assert_same(outs[0], outs[1], f"rank-update vs register-staged K={K} c_tri={c_tri}")


# ------------------------------------------------------------------------------------------------ 2. rounding
U64 = 2.0 ** -53


def _check_f64_bound(C, ref, absprod, K, alpha, what, done=None):
    """|C - ref| <= 2 (K + 4) u |alpha| (|A||B|)_ij + u |ref|_ij element by element (u = 2^-53); -> max err / (u |alpha| |A||B|)."""
    err = (C - ref).abs()
    lim = (2 * (K + 4) * U64 * abs(alpha)) * absprod + U64 * ref.abs()
    ok = err <= lim
    if done is not None:
        ok |= ~done
        assert bool(C[~done].isnan().all()), what + ": a tile above the diagonal band was written"
    assert bool(ok.all()), f"{what}: {int((~ok).sum())} elements outside the bound"
    ratio = err / (U64 * abs(alpha) * absprod).clamp_min(1e-300)
    if done is not None:
        ratio = torch.where(done, ratio, 0.0)
    r = float(ratio.max())
    print(f"MEASURED fp64 {what}: max |C - ref| / (u |alpha| |A||B|) = {r:.3g} (bound {2 * (K + 4)})")
    return r


def test_f64_rounding_bound(ops):
    """fp64 on random real operands at model shapes, against cuBLAS fp64 (first checked against the CPU at a small shape)."""
    g = torch.Generator(device="cuda").manual_seed(7)
    A = torch.randn(150, 300, generator=g, dtype=F64, device="cuda")
    B = torch.randn(300, 120, generator=g, dtype=F64, device="cuda")
    ref_cpu = A.cpu() @ B.cpu()
    _check_f64_bound((A @ B).cpu(), ref_cpu, A.abs().cpu() @ B.abs().cpu(), 300, 1.0, "cuBLAS vs CPU 150x120x300")
    # C3 whitening product W K_zx: lower op(A), M = K = 3072, N = 16384; the upper triangle of W holds NaN
    M, N = 3072, 16384
    W = torch.randn(M, M, generator=g, dtype=F64, device="cuda").tril()
    Wn = W + torch.full((M, M), NAN, dtype=F64, device="cuda").triu(1)
    Kzx = torch.randn(M, N, generator=g, dtype=F64, device="cuda")
    C = torch.empty(M, N, dtype=F64, device="cuda")
    ops.gemm(Wn, Kzx, C, a_tri=ops.TRI_LOWER)
    _check_f64_bound(C, W @ Kzx, W.abs() @ Kzx.abs(), M, 1.0, "whitening 3072x16384x3072 a_tri=LOWER")
    del W, Wn, Kzx, C
    # Gram product A diag(g) A^T: tb, c_tri = 1, M = N = 3072, K = 16384
    Ag = torch.randn(M, N, generator=g, dtype=F64, device="cuda")
    Ak = torch.randn(M, N, generator=g, dtype=F64, device="cuda")
    G = torch.full((M, M), NAN, dtype=F64, device="cuda")
    ops.gemm(Ag, Ak, G, tb=True, c_tri=1, alpha=0.5)
    done = _done(M, M, 1).cuda()
    _check_f64_bound(G, 0.5 * (Ag @ Ak.T), Ag.abs() @ Ak.abs().T, N, 0.5, "Gram 3072x3072x16384 tb c_tri=1", done)
    del Ag, Ak, G, done
    # M' = 7200: dK_zx = W^T dA (ta, upper op(A)), N = 2048
    M, N = 7200, 2048
    W = torch.randn(M, M, generator=g, dtype=F64, device="cuda").tril()
    Wn = W + torch.full((M, M), NAN, dtype=F64, device="cuda").triu(1)
    dA = torch.randn(M, N, generator=g, dtype=F64, device="cuda")
    C = torch.empty(M, N, dtype=F64, device="cuda")
    ops.gemm(Wn, dA, C, ta=True, a_tri=ops.TRI_UPPER, alpha=-1.0)
    _check_f64_bound(C, -(W.T @ dA), W.abs().T @ dA.abs(), M, -1.0, "M'=7200 7200x2048x7200 ta a_tri=UPPER")


def _f32_ratio(C, A64, B64, what, done=None):
    """-> (max over ij of (|C - ref| - 2^-24 |ref|) / (2^-21 (|A||B|)_ij), the same without the 2^-24 |ref| term),
    ref = A64 @ B64 in fp64 (cuBLAS)."""
    ref = A64 @ B64
    scale = (2.0 ** -21 * (A64.abs() @ B64.abs())).clamp_min(1e-300)
    err = (C.double() - ref).abs()
    excess, raw = (err - 2.0 ** -24 * ref.abs()) / scale, err / scale
    if done is not None:
        assert bool(C[~done].isnan().all()), what + ": a tile above the diagonal band was written"
        excess, raw = torch.where(done, excess, -1.0), torch.where(done, raw, -1.0)
    r, r_raw = max(float(excess.max()), 0.0), float(raw.max())
    print(f"MEASURED fp32 {what}: max (|C - ref| - 2^-24 |ref|) / (2^-21 |A||B|) = {r:.4f}, "
          f"max |C - ref| / (2^-21 |A||B|) = {r_raw:.4f} (C32 = {C32})")
    return r, r_raw


def test_f32_rounding_bound(ops):
    """3xTF32 on random fp32 operands against the fp64 product of the same values, componentwise; includes a cancelling
    product whose result is ~1e-6 of |A||B| and an fp32 C rounded from it."""
    g = torch.Generator(device="cuda").manual_seed(11)
    cases = []
    # whitening shape: lower op(A) with NaN above, M = K = 2048, N = 4096
    M, N = 2048, 4096
    W = torch.randn(M, M, generator=g, device="cuda").tril()
    Wn = W + torch.full((M, M), NAN, device="cuda").triu(1)
    X = torch.randn(M, N, generator=g, device="cuda")
    C = torch.empty(M, N, device="cuda")
    ops.gemm(Wn, X, C, a_tri=ops.TRI_LOWER)
    cases.append(_f32_ratio(C, W.double(), X.double(), "whitening 2048x4096x2048 a_tri=LOWER")[0])
    # Gram product, tb, c_tri = 1, K = 16384
    A = torch.randn(1024, 16384, generator=g, device="cuda")
    B = torch.randn(1024, 16384, generator=g, device="cuda")
    G = torch.full((1024, 1024), NAN, device="cuda")
    ops.gemm(A, B, G, tb=True, c_tri=1)
    cases.append(_f32_ratio(G, A.double(), B.double().T, "Gram 1024x1024x16384 tb c_tri=1", _done(1024, 1024, 1).cuda())[0])
    # ta, upper x lower (W^T Y of the Cholesky backward), square 1000
    L1 = torch.randn(1000, 1000, generator=g, device="cuda").tril()
    L2 = torch.randn(1000, 1000, generator=g, device="cuda").tril()
    C = torch.empty(1000, 1000, device="cuda")
    ops.gemm(L1 + torch.full_like(L1, NAN).triu(1), L2 + torch.full_like(L2, NAN).triu(1), C, ta=True, a_tri=ops.TRI_UPPER,
             b_tri=ops.TRI_LOWER)
    cases.append(_f32_ratio(C, L1.double().T, L2.double(), "W^T Y 1000^3 ta a_tri=UPPER b_tri=LOWER")[0])
    # cancelling: A = [X X], B = [Y; -Y'] with Y' = Y (1 + ~2^-20): C ~ 1e-6 |A||B|
    X = torch.randn(512, 2048, generator=g, device="cuda")
    Y = torch.randn(2048, 512, generator=g, device="cuda")
    Yp = (Y.double() * (1 + 2.0 ** -20 * torch.randn(2048, 512, generator=g, dtype=F64, device="cuda"))).float()
    A, B = torch.cat([X, X], 1), torch.cat([Y, -Yp], 0)
    C = torch.empty(512, 512, device="cuda")
    ops.gemm(A, B, C)
    ref = A.double() @ B.double()
    assert float(ref.abs().max()) < 1e-4 * float((A.double().abs() @ B.double().abs()).min())      # it does cancel
    cases.append(_f32_ratio(C, A.double(), B.double(), "cancelling 512x512x4096")[0])
    assert max(cases) <= C32, cases


def test_f32_long_k_uses_the_fp64_master_sum(ops):
    """On non-negative operands (no cancellation to hide a long fp32 chain's drift) the error ratio to |A||B| must not
    grow with K: each 16-wide k-tile is summed in fp32 and then added to an fp64 master sum.  An fp32 chain over all of
    K would make it grow roughly like K.  The growth is measured on |C - ref| / (2^-21 |A||B|) with the final rounding
    to fp32 (at most 1/8 of that unit here, where |ref| = |A||B|) included, so that it never compares against zero."""
    g = torch.Generator(device="cuda").manual_seed(13)
    excess, raw = {}, {}
    for K in (16, 3072, 16384, 65536):
        A = torch.rand(128, K, generator=g, device="cuda")
        B = torch.rand(K, 128, generator=g, device="cuda")
        C = torch.empty(128, 128, device="cuda")
        ops.gemm(A, B, C)
        excess[K], raw[K] = _f32_ratio(C, A.double(), B.double(), f"non-negative 128x128x{K}")
    assert max(excess.values()) <= C32, excess
    assert raw[65536] <= 2.0 * raw[3072], raw


# ------------------------------------------------------------------------------------------------ 3. triangle helpers
HELPER_N = (1, 31, 32, 33, 150, 3072)


def _square(host, dtype):
    """n x n host matrix in a NaN-filled buffer with an odd leading dimension and extra rows."""
    return _place(host, "odd", dtype)


@pytest.mark.parametrize("n", HELPER_N)
def test_symmetrize(ops, n):
    g = torch.Generator().manual_seed(n)
    X = torch.randn(n, n, generator=g, dtype=F64)
    A, flat, ld, off = _square(X, F64)
    before = flat.cpu()
    ops.symmetrize(A, n)
    _assert_same(flat, _expect(before, off, ld, 0.5 * (X + X.T), _done(n, n, 0)), f"symmetrize n={n}")


@pytest.mark.parametrize("dtype", [F64, F32])
@pytest.mark.parametrize("n", HELPER_N)
def test_mirror_lower(ops, dtype, n):
    g = torch.Generator().manual_seed(n)
    X = torch.randn(n, n, generator=g, dtype=F64).to(dtype).double()
    low = _keep(n, n, 1)
    A, flat, ld, off = _square(torch.where(low, X, NAN), dtype)      # the upper triangle holds NaN, as a c_tri product leaves it
    before = flat.cpu()
    ops.mirror_lower(A, n)
    _assert_same(flat, _expect(before, off, ld, torch.where(low, X, X.T), _done(n, n, 0)), f"mirror_lower n={n}")


@pytest.mark.parametrize("dtype", [F64, F32])
@pytest.mark.parametrize("n", HELPER_N)
def test_tril_minus_eye(ops, dtype, n):
    g = torch.Generator().manual_seed(n)
    X = torch.randn(n, n, generator=g, dtype=F64).to(dtype)
    low = _keep(n, n, 1)
    Ls = _square(torch.where(low, X.double(), NAN), dtype)[0]           # not read above the diagonal
    E, flat, ld, off = _square(torch.full((n, n), NAN, dtype=F64), dtype)
    before = flat.cpu()
    ops.tril_minus_eye(Ls, E)
    ref = (X.tril() - torch.eye(n, dtype=dtype)).double()               # the subtraction rounded in the kernel's dtype
    _assert_same(flat, _expect(before, off, ld, ref, _done(n, n, 0)), f"tril_minus_eye n={n}")


@pytest.mark.parametrize("n", HELPER_N)
def test_sym_phi(ops, n):
    g = torch.Generator().manual_seed(n)
    Y = torch.randn(n, n, generator=g, dtype=F64)
    low = _keep(n, n, 1)
    Yd = _square(torch.where(low, Y, NAN), F64)[0]
    P, flat, ld, off = _square(torch.full((n, n), NAN, dtype=F64), F64)
    before = flat.cpu()
    ops.sym_phi(Yd, P, n)
    _assert_same(flat, _expect(before, off, ld, 0.5 * torch.where(low, Y, Y.T), _done(n, n, 0)), f"sym_phi n={n}")
