"""Tensor-level wrappers over the C ABI (one Python function per kernel family).

Every function takes CUDA tensors, enqueues work on torch's current stream and returns without synchronising.
Matrices are row-major; a 2-D tensor must have unit stride in its last dimension, its first stride is the
leading dimension.  These are the building blocks of engine.py and of the autograd Functions in functions.py.
"""
import torch

from . import _lib
from ._lib import call, call_raw, suffix

TRI_NONE, TRI_LOWER, TRI_UPPER = 0, 1, 2
F32, F64 = torch.float32, torch.float64


def _ld(t):
    assert t.dim() == 2 and t.stride(1) == 1, "matrix operands must be row-major with unit inner stride"
    return t.stride(0)


def _pair_suffix(t_in, t_k):
    if t_in == t_k:
        return suffix(t_in)
    if t_in == F32 and t_k == F64:
        return "f32f64"
    raise _lib.DsvgpError(f"unsupported dtype pair {t_in}/{t_k}")


def hyp_from_raw(raw_ell, raw_os=None, raw_noise=None, c=None, out=None):
    """-> device double[8] {ell, os, noise, c, sigmoid(raw_ell), sigmoid(raw_os), sigmoid(raw_noise), 0}."""
    out = torch.empty(8, dtype=F64, device=raw_ell.device) if out is None else out
    call("dsvgp_hyp_from_raw_" + suffix(raw_ell.dtype), raw_ell, raw_os, raw_noise, c, out)
    return out


def normalize_dirs(v, k_dtype=None):
    """Row-normalised directions and 1/|v| in k_dtype (RBFKernelDirectionalGrad.py:57-58)."""
    k_dtype = k_dtype or v.dtype
    v = v.contiguous()
    vhat = torch.empty(v.shape, dtype=k_dtype, device=v.device)
    inv = torch.empty(v.shape[0], dtype=k_dtype, device=v.device)
    call("dsvgp_normalize_dirs_" + _pair_suffix(v.dtype, k_dtype), v, v.shape[0], v.shape[1], vhat, inv)
    return vhat, inv


def normalize_dirs_canon(v):
    """fp32 normalize_dirs that also detects one-hot (canonical) rows on the device: returns
    (vhat, inv_norm, cidx int32[rows], flag int32[1]); flag stays 1 iff every row is one-hot."""
    v = v.contiguous()
    vhat, inv = torch.empty_like(v), torch.empty(v.shape[0], dtype=v.dtype, device=v.device)
    cidx = torch.empty(v.shape[0], dtype=torch.int32, device=v.device)
    flag = torch.ones(1, dtype=torch.int32, device=v.device)
    call("dsvgp_normalize_dirs_canon_f32", v, v.shape[0], v.shape[1], vhat, inv, cidx, flag)
    return vhat, inv, cidx, flag


def kdir_fwd(x1, u1, p1, x2, w2, p2, hyp, out, use_os=True, diag_add=0.0, canon=None, out_lo=None):
    """out[:n1(p1+1), :n2(p2+1)] = [os*] K(x1, x2; u1, w2) (+ diag_add on the diagonal).
    canon = (cidx, flag) from normalize_dirs_canon(v2) enables the canonical-direction fast path (fp32).
    out_lo (fp32, same leading dimension): TF32 'lo' companion; the return value says whether it was written."""
    n1, d = x1.shape
    n2 = x2.shape[0]
    assert out.shape[0] >= n1 * (p1 + 1) and out.shape[1] >= n2 * (p2 + 1)
    if x1.dtype == F32 and out.dtype == F32 and (canon is not None or out_lo is not None):
        assert out_lo is None or _ld(out_lo) == _ld(out)
        cidx, flag = canon if (canon is not None and p2) else (None, None)
        rc = call("dsvgp_kdir_fwd_canon_f32", x1, u1 if p1 else None, n1, p1, x2, w2 if p2 else None, cidx, flag, n2, p2, d,
                  hyp, int(use_os), float(diag_add), out, _ld(out), out_lo)
        return rc == 1
    call("dsvgp_kdir_fwd_" + _pair_suffix(x1.dtype, out.dtype), x1, u1 if p1 else None, n1, p1, x2,
         w2 if p2 else None, n2, p2, d, hyp, int(use_os), float(diag_add), out, _ld(out))
    return False


def kdir_diag(n, p, hyp, dtype, use_os=True):
    out = torch.empty(n * (p + 1), dtype=dtype, device=hyp.device)
    call("dsvgp_kdir_diag_" + suffix(dtype), n, p, hyp, int(use_os), out)
    return out


_ws_cache = {}


def _workspace(nbytes, device, tag):
    key = (tag, device)
    buf = _ws_cache.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(nbytes, 1 << 16), dtype=torch.uint8, device=device)
        _ws_cache[key] = buf
    return buf


def kdir_bwd(x1, u1, inv1, p1, x2, w2, p2, hyp, dK, gx, gv, gsc, use_os=True, dk_trans=False, scale=1.0):
    """Accumulate scale*dL/dx1 into gx, scale*dL/dv1 into gv and dL/d(ell, os) into gsc[0:2] (all float64)."""
    n1, d = x1.shape
    n2 = x2.shape[0]
    nbytes = call_raw("dsvgp_kdir_bwd_workspace_" + suffix(dK.dtype), n1, p1, n2, p2, d)
    ws = _workspace(nbytes, x1.device, "kdir_bwd")
    call("dsvgp_kdir_bwd_" + _pair_suffix(x1.dtype, dK.dtype), x1, u1 if p1 else None, inv1 if (p1 and gv is not None) else None, n1, p1,
         x2, w2 if p2 else None, n2, p2, d, hyp, int(use_os), dK, _ld(dK), int(dk_trans), float(scale), gx,
         gv if p1 else None, gsc, ws, ws.numel())


def kdir_bwd_cols(x1, u1, p1, x2, w2, inv2, p2, hyp, dK, gx, gv, use_os=True, scale=1.0):
    """Accumulate scale*dL/dx2 into gx and scale*dL/dv2 into gv (float64): the data-side gradient of K(x1, x2) given dK
    (laid out as kdir_fwd writes K).  True when the dedicated fp32 kernel ran, False when the blocked one read dK transposed."""
    n1, d = x1.shape
    n2 = x2.shape[0]
    nbytes = call_raw("dsvgp_kdir_bwd_cols_workspace_" + suffix(dK.dtype), n1, p1, n2, p2, d)
    ws = _workspace(nbytes, x1.device, "kdir_bwd_cols")
    rc = call("dsvgp_kdir_bwd_cols_" + suffix(dK.dtype), x1, u1 if p1 else None, n1, p1, x2, w2 if p2 else None,
              inv2 if (p2 and gv is not None) else None, n2, p2, d, hyp, int(use_os), dK, _ld(dK), float(scale), gx,
              gv if p2 else None, ws, ws.numel())
    return rc == 1


def gemm(A, B, C, ta=False, tb=False, alpha=1.0, beta=0.0, a_tri=TRI_NONE, b_tri=TRI_NONE, c_tri=0, D=None,
         M=None, N=None, K=None, C2=None, D2=None):
    """C[:M,:N] = alpha*op(A)[:M,:K] @ op(B)[:K,:N] + beta*(D or C); optionally also C2 = C + D2.
    Triangle flags: see include/dsvgp_b200.h."""
    if M is None:
        M = A.shape[1] if ta else A.shape[0]
    if K is None:
        K = A.shape[0] if ta else A.shape[1]
    if N is None:
        N = B.shape[0] if tb else B.shape[1]
    call("dsvgp_gemm_" + suffix(C.dtype), int(ta), int(tb), M, N, K, float(alpha), A, _ld(A), B, _ld(B), float(beta),
         C, _ld(C), a_tri, b_tri, c_tri, 1, 0, 0, 0, D, _ld(D) if D is not None else 0,
         C2, _ld(C2) if C2 is not None else 0, D2, _ld(D2) if D2 is not None else 0)
    return C


def split_lo(x, lo=None, rows=None, cols=None):
    """lo = x - trunc_tf32(x) (the part of x the TF32 tensor core does not see)."""
    lo = torch.empty_like(x) if lo is None else lo
    call("dsvgp_split_lo_f32", x, _ld(x), lo, _ld(lo), x.shape[0] if rows is None else rows,
         x.shape[1] if cols is None else cols)
    return lo


def transpose(src, dst, rows=None, cols=None):
    call("dsvgp_transpose_f32", src, _ld(src), dst, _ld(dst), src.shape[0] if rows is None else rows,
         src.shape[1] if cols is None else cols)
    return dst


def set_rank_update(on):
    """fp64 rank-K update kernel (K <= 128) for A B^T products: 0 off, 1 every eligible product, 2 only small (latency-bound) launches."""
    return call_raw("dsvgp_set_rank_update", int(on))


def set_chol_variant(v):
    """Diagonal-block kernel of the factorisation: 3 = 4-CTA cluster kernel (default), 2 = multi-CTA update + block kernel,
    1 = the single-CTA round-1 kernel with the batched recursive inverse.  Returns the value in force."""
    return call_raw("dsvgp_set_chol_variant", int(v))


def set_chol_lookahead(on):
    """Trailing updates of the factorisation split into an urgent thin part and a bulk part on its own stream (default off)."""
    return call_raw("dsvgp_set_chol_lookahead", int(bool(on)))


def set_chol_mid_link(k):
    """Diagonal block of the factorisation whose completion chol_wait_mid waits for (default 20, capped at the last block; negative: never)."""
    return call_raw("dsvgp_set_chol_mid_link", int(k))


def chol_wait_mid():
    """The current stream waits for the mid-chain diagonal block of the factorisation enqueued last (see include/dsvgp_b200.h)."""
    return call("dsvgp_chol_wait_mid")


def set_chol_inv_streams(n):
    """Streams of the eager inverse (3: one per level of the recursive doubling, default; 2: T products on one extra stream; 1: one)."""
    return call_raw("dsvgp_set_chol_inv_streams", int(n))


def set_chol_graph(on):
    """The factorisation as a cached CUDA graph of its own (one cudaGraphLaunch instead of ~650 host calls); default off."""
    return call_raw("dsvgp_set_chol_graph", int(bool(on)))


def set_chol_priority(on):
    """Factorisation chains on the library's high-priority streams, or (default) the diagonal chain on the caller's stream."""
    return call_raw("dsvgp_set_chol_priority", int(bool(on)))


def set_kdir_bwd_vpl(vpl):
    """Column points per lane of the vectorised fp32 assembly backward (2 or 4)."""
    return call_raw("dsvgp_set_kdir_bwd_vpl", int(vpl))


def set_tc_cta_group(cg):
    """1: one CTA per 128x256 tile; 2: CTA pairs (tcgen05 cta_group::2) on 256x256 tiles."""
    return call_raw("dsvgp_set_tc_cta_group", int(cg))


def set_tc_tile_n(n):
    """N extent of a CTA-pair tile of the 3xFP16 product: 256, or 128 = two pairs resident per SM pair."""
    return call_raw("dsvgp_set_tc_tile_n", int(n))


def set_tc_max_pairs(n):
    """Persistent tensor-core products on at most n CTA pairs (0 = all)."""
    return call_raw("dsvgp_set_tc_max_pairs", int(n))


def set_tc_persistent(on):
    """CTA-pair tensor-core products as persistent pairs over a balanced work list (default) or one pair per tile."""
    return call_raw("dsvgp_set_tc_persistent", int(bool(on)))


def gemm_tch(A, B, C, M, N, K, ab_inv, b_kmajor=False, alpha=1.0, beta=0.0, D=None, C2=None, D2=None, Ch=None, c_scale=None,
             C2h=None, c2_scale=None, a_tri=TRI_NONE, c_lower=False, chunk=1, nsplit=1, split_ws=None):
    """tcgen05 3xFP16 product.  A, B, Ch, C2h are (hi, lo) pairs of float16 matrices holding the split of x * scale;
    ab_inv / c_scale / c2_scale are 1-element float32 device tensors.  C (fp32) may be None when only Ch is wanted."""
    ld = lambda t: _ld(t) if t is not None else 0
    call("dsvgp_gemm_tch_f32", A[0], A[1], _ld(A[0]), B[0], B[1], _ld(B[0]), int(b_kmajor), M, N, K, float(alpha), float(beta),
         ab_inv, C, ld(C), D, ld(D), C2, ld(C2), D2, ld(D2), Ch[0] if Ch else None, Ch[1] if Ch else None,
         _ld(Ch[0]) if Ch else 0, c_scale, C2h[0] if C2h else None, C2h[1] if C2h else None, _ld(C2h[0]) if C2h else 0, c2_scale,
         a_tri, int(c_lower), chunk, int(nsplit), split_ws)
    return C


def absmax(x, out_bits, mode=0):
    """out_bits (uint32/int32[1] device tensor, zeroed by the caller) = max(out_bits, bits of max|x|); mode 2: tril(x) - I."""
    x2 = x if x.dim() == 2 else x.reshape(1, -1)
    call("dsvgp_absmax_" + suffix(x.dtype), x2, _ld(x2), x2.shape[0], x2.shape[1], mode, out_bits)


def tc_scales(hyp, jitter, maxbits, Mq, scales, stage):
    call("dsvgp_tc_scales_f32", hyp, float(jitter), maxbits, int(Mq), scales, int(stage))


def split_half(src, scale, hi, lo, mode=0, hiT=None, loT=None, rows=None, cols=None):
    call("dsvgp_split_half_" + suffix(src.dtype), src, _ld(src), src.shape[0] if rows is None else rows,
         src.shape[1] if cols is None else cols, mode, scale, hi, lo, _ld(hi), hiT, loT, _ld(hiT) if hiT is not None else 0)


def build_d_split(E, P, scale, hi, lo, n=None):
    """(hi, lo) = split of (E + E^T + E E^T) * scale from the lower triangles of E and P = E E^T."""
    call("dsvgp_build_d_split_f32", E, _ld(E), P, _ld(P), E.shape[0] if n is None else n, scale, hi, lo, _ld(hi))


def build_d_absmax(E, P, out_bits, n=None):
    """out_bits = max(out_bits, bits of max|E + E^T + E E^T|) from the lower triangles of E and P = E E^T."""
    call("dsvgp_build_d_absmax_f32", E, _ld(E), P, _ld(P), E.shape[0] if n is None else n, out_bits)


def kdir_fwd_half(x1, u1, p1, x2, w2, p2, hyp, K, Kh, Kl, hscale, canon=None, use_os=True):
    """K_zx assembly that writes only the two-half split of K * hscale; returns True if it did (else K was written)."""
    n1, d = x1.shape
    n2 = x2.shape[0]
    cidx, flag = canon if (canon is not None and p2) else (None, None)
    rc = call("dsvgp_kdir_fwd_half_f32", x1, u1 if p1 else None, n1, p1, x2, w2 if p2 else None, cidx, flag, n2, p2, d, hyp,
              int(use_os), 0.0, K, _ld(K), Kh, Kl, _ld(Kh), hscale)
    return rc == 2


def dA_apply_half(A, C, rows, nq, m, gmu, gvar, tp, t, dAh, dAl, Agh, Agl, s_dA, s_Ag, A_half=None, a_scale=None):
    """dA and A_g as two-half splits; A as the fp32 matrix, or (A_half = (Ah, Al), a_scale) as the split of A * a_scale."""
    if A_half is not None:
        call("dsvgp_dA_half_h_f32", A_half[0], A_half[1], a_scale, C, _ld(C), rows, nq, m, gmu, gvar, tp, tp.shape[0], t, dAh, dAl,
             Agh, Agl, _ld(dAh), s_dA, s_Ag)
        return
    call("dsvgp_dA_half_f32", A, C, _ld(A), rows, nq, m, gmu, gvar, tp, tp.shape[0], t, dAh, dAl, Agh, Agl, _ld(dAh), s_dA, s_Ag)


def set_kdir_fwd_knobs(tib=-1, stream_stores=-1):
    """benchmarking knobs of the fp32 assembly kernel (row points per CTA, evict-first stores)."""
    return call_raw("dsvgp_set_kdir_fwd_knobs", int(tib), int(stream_stores))


def gemm_tc_supported(A, B, b_kmajor, N):
    return bool(call_raw("dsvgp_gemm_tc_supported_f32", A, _ld(A), B, _ld(B), int(b_kmajor), int(N)))


def gemm_tc(A, A_lo, B, B_lo, C, M, N, K, b_kmajor=False, alpha=1.0, beta=0.0, D=None, C2=None, D2=None, a_tri=TRI_NONE,
            c_lower=False, chunk=2, C_lo=None, C2_lo=None, nsplit=1, split_ws=None):
    """tcgen05 3xTF32 product C[:M,:N] = alpha * A[:M,:K] @ (B[:K,:N] or B[:N,:K]^T) + beta*D (+ C2 = C + D2)."""
    call("dsvgp_gemm_tc_f32", A, A_lo, _ld(A), B, B_lo, _ld(B), int(b_kmajor), M, N, K, float(alpha), float(beta), C, _ld(C),
         D, _ld(D) if D is not None else 0, C2, _ld(C2) if C2 is not None else 0, D2, _ld(D2) if D2 is not None else 0,
         a_tri, int(c_lower), chunk, C_lo, C2_lo, int(nsplit), split_ws)
    return C


def chol_plan(Mq):
    return _lib.chol_plan(Mq)


def pad_identity(A, Mq):
    call("dsvgp_pad_identity_f64", A, _ld(A), Mq, A.shape[0])


def cholesky_inverse(Awork, L, W, nb0, nlev, info):
    """Awork (Mp x Mp fp64, destroyed) -> L, W = L^-1; info: device int32[1]."""
    call("dsvgp_chol_f64", Awork, _ld(Awork), L, _ld(L), W, _ld(W), Awork.shape[0], nb0, nlev, info)


def chol_backward(L, W, Lbar, out, n=None):
    """out[:n,:n] = sym(W^T Phi(L^T Lbar) W): the gradient w.r.t. A = L L^T given Lbar = dloss/dL (fp64; the lower
    triangles of L, W = L^-1 and Lbar are read)."""
    n = L.shape[0] if n is None else n
    ws = _workspace(call_raw("dsvgp_chol_bwd_workspace_f64", int(n)), L.device, "chol_bwd")
    call("dsvgp_chol_bwd_f64", L, _ld(L), W, _ld(W), Lbar, _ld(Lbar), out, _ld(out), int(n), ws, ws.numel())
    return out


def cast2d(src, dst, rows=None, cols=None, tril=False):
    rows = src.shape[0] if rows is None else rows
    cols = src.shape[1] if cols is None else cols
    call(f"dsvgp_cast_{suffix(src.dtype)}_{suffix(dst.dtype)}", src, _ld(src), dst, _ld(dst), rows, cols, int(tril))
    return dst


def mirror_lower(A, n=None):
    call("dsvgp_mirror_lower_" + suffix(A.dtype), A, _ld(A), A.shape[0] if n is None else n)
    return A


def add_outer(A, u, v, alpha=1.0, n=None):
    call("dsvgp_add_outer_" + suffix(A.dtype), A, _ld(A), A.shape[0] if n is None else n, u, v, float(alpha))
    return A


def tril_minus_eye(Ls_raw, E):
    """E = tril(Ls_raw) - I."""
    call("dsvgp_tril_minus_eye_" + suffix(E.dtype), Ls_raw, _ld(Ls_raw), E, _ld(E), E.shape[0])
    return E


def sym_phi(Y, P, n):
    call("dsvgp_sym_phi_f64", Y, _ld(Y), P, _ld(P), n)
    return P


def phi_outer(X, u, v, P, n):
    """lower triangle of P (fp64) = Phi(X + u v^T); the upper triangle of P is left as it is"""
    call("dsvgp_phi_outer_" + suffix(X.dtype), X, _ld(X), u, v, P, _ld(P), n)


def phi_lower(Y, P, n):
    call("dsvgp_phi_lower_f64", Y, _ld(Y), P, _ld(P), n)
    return P


def symmetrize(A, n):
    call("dsvgp_symmetrize_f64", A, _ld(A), n)
    return A


def reduce_slabs(rows, cols):
    return call_raw("dsvgp_reduce_slabs", rows, cols)


def col_dots(A, m, pm, pv, rows, nq, C=None, Bp=None, cmax=None):
    """pm = A^T m partials; pv = sum A*C (C given) or sum Bp*(2A + Bp) (Bp = B - A given).
    cmax (1-element int32 device tensor, zeroed by the caller): receives the bits of max|C|."""
    B = Bp
    nslab = pm.shape[0]
    call("dsvgp_col_dots_" + suffix(A.dtype), A, C, B, _ld(A), rows, nq, m, pm, pv, nslab, cmax if C is not None else None)


def col_dots_half(A_half, a_scale, m, pm, pv, rows, nq, C, cmax=None):
    """col_dots with A given only as the two-half split (Ah, Al) of A * a_scale (1-element device tensor)."""
    call("dsvgp_col_dots_h_f32", A_half[0], A_half[1], _ld(A_half[0]), a_scale, C, _ld(C), rows, nq, m, pm, pv, pm.shape[0], cmax)


def collect_grads(small, nZ, nV, hyp, noise_mode, out):
    """out = [dZ | dV_z | d c | d raw_os | d raw_ell | d raw_noise] (model dtype) from the engine's fp64 buffer, one launch."""
    call("dsvgp_collect_grads_" + suffix(out.dtype), small, int(nZ), int(nV), hyp, int(noise_mode), out)
    return out


def predict_finish(pm, pv, nq, p2, hyp, mu, var, add_noise, pred_jitter=1e-4):
    min_var = 1e-10 if mu.dtype == F64 else 1e-6      # gpytorch settings.min_variance
    call("dsvgp_predict_finish_" + suffix(mu.dtype), pm, pv, pm.shape[0], nq, p2, hyp, float(pred_jitter),
         int(add_noise), min_var, mu, var)


def elbo_terms(mu, var, y, hyp, w, gmu, gvar, sc, ws):
    min_var = 1e-10 if mu.dtype == F64 else 1e-6
    call("dsvgp_elbo_terms_" + suffix(mu.dtype), mu, var, y, mu.numel(), hyp, float(w), min_var, gmu, gvar, sc, ws)


def pll_terms(mu, var, y, w, gmu, gvar, sc, ws):
    min_var = 1e-10 if mu.dtype == F64 else 1e-6
    call("dsvgp_pll_terms_" + suffix(mu.dtype), mu, var, y, mu.numel(), float(w), min_var, gmu, gvar, sc, ws)


def pred_bwd_scalars(gmu, gvar, p2, hyp, add_noise, gsc, ws):
    call("dsvgp_pred_bwd_scalars_" + suffix(gmu.dtype), gmu, gvar, gmu.numel(), p2, hyp, int(add_noise), gsc, ws)


def dA_apply(A, C, Ag, rows, nq, m, gmu, gvar, tp, t, C_lo=None, Ag_lo=None):
    call("dsvgp_dA_" + suffix(A.dtype), A, C, Ag, _ld(A), rows, nq, m, gmu, gvar, tp, tp.shape[0], t, C_lo, Ag_lo)


def kl_divergence(m, Ls_raw, out, ws):
    call("dsvgp_kl_" + suffix(m.dtype), m, Ls_raw, _ld(Ls_raw), m.numel(), out, ws)


def var_grads(H, Ls_raw, t, m, inv_num_data, gm, gLs):
    call("dsvgp_var_grads_" + suffix(m.dtype), H, _ld(H), Ls_raw, _ld(Ls_raw), t, m, m.numel(), float(inv_num_data),
         gm, gLs, _ld(gLs))
