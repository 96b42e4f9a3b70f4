// extern "C" surface of libdsvgp_b200.so -- see include/dsvgp_b200.h for the contract of every entry point.
#include "../../include/dsvgp_b200.h"
#include "chol.cuh"
#include "common.cuh"
#include "data.cuh"
#include "gemm.cuh"
#include "kdir.cuh"
#include "misc.cuh"
#include "optim.cuh"
#include "tc_prep.cuh"
#include "trmm_tc.cuh"

using namespace dsvgp;
#define ST(s) reinterpret_cast<cudaStream_t>(s)

namespace dsvgp { unsigned long long g_launch_count = 0; }
namespace dsvgp { extern int g_fwd_tib, g_fwd_stream_stores, g_bwd_vpl; }

extern "C" {

int dsvgp_version(void) { return 100; }
int64_t dsvgp_launch_count(void) { return (int64_t)dsvgp::g_launch_count; }
int dsvgp_set_kdir_bwd_vpl(int vpl) {
  if (vpl == 2 || vpl == 4) dsvgp::g_bwd_vpl = vpl;
  return dsvgp::g_bwd_vpl;
}
int dsvgp_set_kdir_fwd_knobs(int tib, int stream_stores) {
  const int old = dsvgp::g_fwd_tib * 4 + dsvgp::g_fwd_stream_stores;
  if (tib == 0 || (tib >= 8 && tib <= 64 && tib % 8 == 0)) dsvgp::g_fwd_tib = tib;      /* 0 = adaptive (default) */
  if (stream_stores >= 0 && stream_stores <= 2) dsvgp::g_fwd_stream_stores = stream_stores;
  return old;
}
int dsvgp_built_for_sm(void) { return 100; }

int dsvgp_hyp_from_raw_f32(const float* a, const float* b, const float* c, const float* d, double* hyp, dsvgp_stream_t s) { return hyp_from_raw<float>(a, b, c, d, hyp, ST(s)); }
int dsvgp_hyp_from_raw_f64(const double* a, const double* b, const double* c, const double* d, double* hyp, dsvgp_stream_t s) { return hyp_from_raw<double>(a, b, c, d, hyp, ST(s)); }

int dsvgp_normalize_dirs_f32(const float* v, int rows, int d, float* vh, float* inv, dsvgp_stream_t s) { return normalize_dirs<float, float>(v, rows, d, vh, inv, ST(s)); }
int dsvgp_normalize_dirs_f64(const double* v, int rows, int d, double* vh, double* inv, dsvgp_stream_t s) { return normalize_dirs<double, double>(v, rows, d, vh, inv, ST(s)); }
int dsvgp_normalize_dirs_f32f64(const float* v, int rows, int d, double* vh, double* inv, dsvgp_stream_t s) { return normalize_dirs<float, double>(v, rows, d, vh, inv, ST(s)); }

int dsvgp_normalize_dirs_canon_f32(const float* v, int rows, int d, float* vh, float* inv, int* cidx, int* canon_flag, dsvgp_stream_t s) {
  if (!cidx || !canon_flag) return DSVGP_ERR_ARG;
  return normalize_dirs<float, float>(v, rows, d, vh, inv, ST(s), cidx, canon_flag);
}
int dsvgp_kdir_fwd_canon_f32(const float* x1, const float* u1, int n1, int p1, const float* x2, const float* w2, const int* cidx2, const int* canon_flag, int n2, int p2, int d, const double* hyp, int use_os, double diag_add, float* K, int64_t ldk, float* Klo, dsvgp_stream_t s) {
  if (!x1 || !x2 || !hyp || !K || (p1 > 0 && !u1) || (p2 > 0 && !w2)) return DSVGP_ERR_ARG;
  return kdir_fwd<float, float>(x1, u1, n1, p1, x2, w2, n2, p2, d, hyp, use_os, diag_add, K, ldk, ST(s), cidx2, canon_flag, Klo);
}

#define KFWD(NAME, T, TK)                                                                                          \
  int NAME(const T* x1, const TK* u1, int n1, int p1, const T* x2, const TK* w2, int n2, int p2, int d,            \
           const double* hyp, int use_os, double diag_add, TK* K, int64_t ldk, dsvgp_stream_t s) {                 \
    if (!x1 || !x2 || !hyp || !K || (p1 > 0 && !u1) || (p2 > 0 && !w2)) return DSVGP_ERR_ARG;                     \
    return kdir_fwd<T, TK>(x1, u1, n1, p1, x2, w2, n2, p2, d, hyp, use_os, diag_add, K, ldk, ST(s));               \
  }
KFWD(dsvgp_kdir_fwd_f32, float, float)
KFWD(dsvgp_kdir_fwd_f64, double, double)
KFWD(dsvgp_kdir_fwd_f32f64, float, double)

int dsvgp_kdir_diag_f32(int n, int p, const double* hyp, int use_os, float* out, dsvgp_stream_t s) { return kdir_diag<float>(n, p, hyp, use_os, out, ST(s)); }
int dsvgp_kdir_diag_f64(int n, int p, const double* hyp, int use_os, double* out, dsvgp_stream_t s) { return kdir_diag<double>(n, p, hyp, use_os, out, ST(s)); }

size_t dsvgp_kdir_bwd_workspace_f32(int n1, int p1, int n2, int p2, int d) { return kdir_bwd_workspace<float>(n1, p1, n2, p2, d); }
size_t dsvgp_kdir_bwd_workspace_f64(int n1, int p1, int n2, int p2, int d) { return kdir_bwd_workspace<double>(n1, p1, n2, p2, d); }

#define KBWD(NAME, T, TK)                                                                                          \
  int NAME(const T* x1, const TK* u1, const TK* inv1, int n1, int p1, const T* x2, const TK* w2, int n2, int p2,   \
           int d, const double* hyp, int use_os, const TK* dK, int64_t lddk, int dk_trans, double scale,           \
           double* gx, double* gv, double* gsc, void* ws, size_t ws_bytes, dsvgp_stream_t s) {                     \
    /* (inv1 = 1/|v1| is read only by the normalisation chain of gv) */                                            \
    if (!x1 || !x2 || !hyp || !dK || !ws || (p1 > 0 && (!u1 || (gv && !inv1))) || (p2 > 0 && !w2)) return DSVGP_ERR_ARG; \
    return kdir_bwd<T, TK>(x1, u1, inv1, n1, p1, x2, w2, n2, p2, d, hyp, use_os, dK, lddk, dk_trans, scale, gx,    \
                           gv, gsc, ws, ws_bytes, ST(s));                                                          \
  }
KBWD(dsvgp_kdir_bwd_f32, float, float)
KBWD(dsvgp_kdir_bwd_f64, double, double)
KBWD(dsvgp_kdir_bwd_f32f64, float, double)

size_t dsvgp_kdir_bwd_cols_workspace_f32(int n1, int p1, int n2, int p2, int d) { return kdir_bwd_cols_workspace<float>(n1, p1, n2, p2, d); }
size_t dsvgp_kdir_bwd_cols_workspace_f64(int n1, int p1, int n2, int p2, int d) { return kdir_bwd_cols_workspace<double>(n1, p1, n2, p2, d); }

#define KBWDC(NAME, T)                                                                                             \
  int NAME(const T* x1, const T* u1, int n1, int p1, const T* x2, const T* w2, const T* inv2, int n2, int p2, int d, \
           const double* hyp, int use_os, const T* dK, int64_t lddk, double scale, double* gx, double* gv, void* ws, \
           size_t ws_bytes, dsvgp_stream_t s) {                                                                    \
    if (!x1 || !x2 || !hyp || !dK || !ws || (p1 > 0 && !u1) || (p2 > 0 && (!w2 || (gv && !inv2)))) return DSVGP_ERR_ARG; \
    return kdir_bwd_cols<T, T>(x1, u1, n1, p1, x2, w2, inv2, n2, p2, d, hyp, use_os, dK, lddk, scale, gx, gv, ws,    \
                               ws_bytes, ST(s));                                                                   \
  }
KBWDC(dsvgp_kdir_bwd_cols_f32, float)
KBWDC(dsvgp_kdir_bwd_cols_f64, double)

void dsvgp_chol_plan(int Mq, int* Mp, int* nb0, int* nlev) { chol_plan(Mq, Mp, nb0, nlev); }
int dsvgp_pad_identity_f64(double* A, int64_t ld, int Mq, int Mp, dsvgp_stream_t s) { return pad_identity(A, ld, Mq, Mp, ST(s)); }
int dsvgp_chol_f64(double* Awork, int64_t lda, double* L, int64_t ldl, double* W, int64_t ldw, int Mp, int nb0, int nlev, int* info, dsvgp_stream_t s) {
  return chol_factor_inverse(Awork, lda, L, ldl, W, ldw, Mp, nb0, nlev, info, ST(s));
}
size_t dsvgp_chol_bwd_workspace_f64(int n) { return chol_bwd_workspace(n); }
int dsvgp_chol_bwd_f64(const double* L, int64_t ldl, const double* W, int64_t ldw, const double* Lbar, int64_t ldlb, double* Abar, int64_t lda, int n, void* ws, size_t ws_bytes, dsvgp_stream_t s) {
  return chol_backward(L, ldl, W, ldw, Lbar, ldlb, Abar, lda, n, ws, ws_bytes, ST(s));
}

int dsvgp_set_potrf_debug(void* p) { set_potrf_debug(static_cast<long long*>(p)); return 0; }
int dsvgp_collect_grads_f32(const double* small, int nZ, int nV, const double* hyp, int noise_mode, float* out, dsvgp_stream_t s) { return collect_grads<float>(small, nZ, nV, hyp, noise_mode, out, ST(s)); }
int dsvgp_collect_grads_f64(const double* small, int nZ, int nV, const double* hyp, int noise_mode, double* out, dsvgp_stream_t s) { return collect_grads<double>(small, nZ, nV, hyp, noise_mode, out, ST(s)); }
int dsvgp_set_gemm64_async(int on) { set_gemm64_async(on); return get_gemm64_async(); }
int dsvgp_set_rank_update(int on) { set_rank_update(on); return get_rank_update(); }
int dsvgp_set_chol_variant(int v) { set_chol_variant(v); return get_chol_variant(); }
int dsvgp_set_chol_lookahead(int on) { set_chol_lookahead(on); return get_chol_lookahead(); }
int dsvgp_set_chol_mid_link(int k) { set_chol_mid_link(k); return get_chol_mid_link(); }
int dsvgp_chol_wait_mid(dsvgp_stream_t s) { return chol_wait_mid(reinterpret_cast<cudaStream_t>(s)); }
int dsvgp_set_chol_inv_streams(int n) { set_chol_inv_streams(n); return get_chol_inv_streams(); }
int dsvgp_set_chol_graph(int on) { set_chol_graph(on); return get_chol_graph(); }
int dsvgp_set_chol_priority(int on) { set_chol_priority(on); return get_chol_priority(); }

int dsvgp_gemm_f32(int ta, int tb, int M, int N, int K, double alpha, const float* A, int64_t lda, const float* B, int64_t ldb, double beta, float* C, int64_t ldc, int a_tri, int b_tri, int c_tri, int batch, int64_t sA, int64_t sB, int64_t sC, const float* D, int64_t ldd, float* C2, int64_t ldc2, const float* D2, int64_t ldd2, dsvgp_stream_t s) {
  return gemm<float>(ta != 0, tb != 0, M, N, K, (float)alpha, A, lda, B, ldb, (float)beta, C, ldc, a_tri, b_tri, c_tri, batch, sA, sB, sC, ST(s), D, ldd, C2, ldc2, D2, ldd2);
}
int dsvgp_gemm_f64(int ta, int tb, int M, int N, int K, double alpha, const double* A, int64_t lda, const double* B, int64_t ldb, double beta, double* C, int64_t ldc, int a_tri, int b_tri, int c_tri, int batch, int64_t sA, int64_t sB, int64_t sC, const double* D, int64_t ldd, double* C2, int64_t ldc2, const double* D2, int64_t ldd2, dsvgp_stream_t s) {
  return gemm<double>(ta != 0, tb != 0, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, a_tri, b_tri, c_tri, batch, sA, sB, sC, ST(s), D, ldd, C2, ldc2, D2, ldd2);
}

int dsvgp_absmax_f32(const float* x, int64_t ld, int rows, int cols, int mode, unsigned int* out_bits, dsvgp_stream_t s) { return absmax<float>(x, ld, rows, cols, mode, out_bits, ST(s)); }
int dsvgp_absmax_f64(const double* x, int64_t ld, int rows, int cols, int mode, unsigned int* out_bits, dsvgp_stream_t s) { return absmax<double>(x, ld, rows, cols, mode, out_bits, ST(s)); }
int dsvgp_tc_scales_f32(const double* hyp, double jitter, const unsigned int* maxbits, int Mq, float* scales, int stage, dsvgp_stream_t s) { return tc_scales(hyp, jitter, maxbits, Mq, scales, stage, ST(s)); }
int dsvgp_split_half_f32(const float* src, int64_t lds, int rows, int cols, int mode, const float* scale, void* hi, void* lo, int64_t ldh, void* hiT, void* loT, int64_t ldhT, dsvgp_stream_t s) { return split_half<float>(src, lds, rows, cols, mode, scale, hi, lo, ldh, hiT, loT, ldhT, ST(s)); }
int dsvgp_split_half_f64(const double* src, int64_t lds, int rows, int cols, int mode, const float* scale, void* hi, void* lo, int64_t ldh, void* hiT, void* loT, int64_t ldhT, dsvgp_stream_t s) { return split_half<double>(src, lds, rows, cols, mode, scale, hi, lo, ldh, hiT, loT, ldhT, ST(s)); }
int dsvgp_build_d_split_f32(const float* E, int64_t lde, const float* P, int64_t ldp, int n, const float* scale, void* hi, void* lo, int64_t ldh, dsvgp_stream_t s) { return build_d_split(E, lde, P, ldp, n, scale, hi, lo, ldh, ST(s)); }
int dsvgp_build_d_absmax_f32(const float* E, int64_t lde, const float* P, int64_t ldp, int n, unsigned int* out_bits, dsvgp_stream_t s) { return build_d_absmax(E, lde, P, ldp, n, out_bits, ST(s)); }
int dsvgp_kdir_fwd_half_f32(const float* x1, const float* u1, int n1, int p1, const float* x2, const float* w2, const int* cidx2, const int* canon_flag, int n2, int p2, int d, const double* hyp, int use_os, double diag_add, float* K, int64_t ldk, void* Kh, void* Kl, int64_t ldkh, const float* hscale, dsvgp_stream_t s) {
  if (!x1 || !x2 || !hyp || !K || !Kh || !Kl || !hscale || (p1 > 0 && !u1) || (p2 > 0 && !w2)) return DSVGP_ERR_ARG;
  return kdir_fwd<float, float>(x1, u1, n1, p1, x2, w2, n2, p2, d, hyp, use_os, diag_add, K, ldk, ST(s), cidx2, canon_flag, nullptr, Kh, Kl, ldkh, hscale);
}
int dsvgp_dA_half_f32(const float* A, const float* C, int64_t ld, int rows, int nq, const float* m, const float* gmu, const float* gvar, float* tp, int nslab, float* t, void* dAh, void* dAl, void* Agh, void* Agl, int64_t ldh, const float* s_dA, const float* s_Ag, dsvgp_stream_t s) {
  if (!A || !C || !m || !gmu || !gvar || !tp || !t || !dAh || !dAl || !Agh || !Agl || !s_dA || !s_Ag) return DSVGP_ERR_ARG;
  return dA_apply_half(A, C, ld, rows, nq, m, gmu, gvar, tp, nslab, t, dAh, dAl, Agh, Agl, ldh, s_dA, s_Ag, nullptr, nullptr, nullptr, ST(s));
}
int dsvgp_dA_half_h_f32(const void* Ah, const void* Al, const float* a_scale, const float* C, int64_t ld, int rows, int nq, const float* m, const float* gmu, const float* gvar, float* tp, int nslab, float* t, void* dAh, void* dAl, void* Agh, void* Agl, int64_t ldh, const float* s_dA, const float* s_Ag, dsvgp_stream_t s) {
  if (!Ah || !Al || !a_scale || !C || !m || !gmu || !gvar || !tp || !t || !dAh || !dAl || !Agh || !Agl || !s_dA || !s_Ag) return DSVGP_ERR_ARG;
  return dA_apply_half(nullptr, C, ld, rows, nq, m, gmu, gvar, tp, nslab, t, dAh, dAl, Agh, Agl, ldh, s_dA, s_Ag, Ah, Al, a_scale, ST(s));
}
int dsvgp_col_dots_h_f32(const void* Ah, const void* Al, int64_t ldh, const float* a_scale, const float* C, int64_t ld, int rows, int nq, const float* m, float* pm, float* pv, int nslab, unsigned int* cmax_bits, dsvgp_stream_t s) {
  if (!m || !pm || !pv) return DSVGP_ERR_ARG;
  return col_dots_half(Ah, Al, ldh, a_scale, C, ld, rows, nq, m, pm, pv, nslab, cmax_bits, ST(s));
}
int dsvgp_gemm_tch_supported_f32(const void* A, int64_t lda, const void* B, int64_t ldb, int b_kmajor, int N) { return gemm_tch_supported(A, lda, B, ldb, b_kmajor, N); }
int dsvgp_gemm_tch_f32(const void* Ah, const void* Al, int64_t lda, const void* Bh, const void* Bl, int64_t ldb, int b_kmajor, int M, int N, int K, double alpha, double beta, const float* ab_inv, float* C, int64_t ldc, const float* D, int64_t ldd, float* C2, int64_t ldc2, const float* D2, int64_t ldd2, void* Ch, void* Cl, int64_t ldch, const float* c_scale, void* C2h, void* C2l, int64_t ldc2h, const float* c2_scale, int a_tri, int c_lower, int chunk, int nsplit, float* split_ws, dsvgp_stream_t s) {
  return gemm_tch(Ah, Al, lda, Bh, Bl, ldb, b_kmajor, M, N, K, (float)alpha, (float)beta, ab_inv, C, ldc, D, ldd, C2, ldc2, D2, ldd2, Ch, Cl, ldch, c_scale, C2h, C2l, ldc2h, c2_scale, a_tri, c_lower, chunk, nsplit, split_ws, ST(s));
}
int dsvgp_gemm_tc_supported_f32(const float* A, int64_t lda, const float* B, int64_t ldb, int b_kmajor, int N) { return gemm_tc_supported(A, lda, B, ldb, b_kmajor, N); }
int dsvgp_gemm_tc_f32(const float* Ah, const float* Al, int64_t lda, const float* Bh, const float* Bl, int64_t ldb, int b_kmajor, int M, int N, int K, double alpha, double beta, float* C, int64_t ldc, const float* D, int64_t ldd, float* C2, int64_t ldc2, const float* D2, int64_t ldd2, int a_tri, int c_lower, int chunk, float* Clo, float* C2lo, int nsplit, float* split_ws, dsvgp_stream_t s) {
  return gemm_tc(Ah, Al, lda, Bh, Bl, ldb, b_kmajor, M, N, K, (float)alpha, (float)beta, C, ldc, D, ldd, C2, ldc2, D2, ldd2, a_tri, c_lower, chunk, Clo, C2lo, nsplit, split_ws, ST(s));
}
int dsvgp_set_tc_tile_n(int n) { set_tc_tile_n(n); return get_tc_tile_n(); }
int dsvgp_set_tc_max_pairs(int n) { set_tc_max_pairs(n); return get_tc_max_pairs(); }
int dsvgp_set_tc_persistent(int on) { set_tc_persistent(on); return get_tc_persistent(); }
int dsvgp_set_tc_trace(void* buf, int cap_items) { set_tc_trace(static_cast<long long*>(buf), cap_items); return DSVGP_OK; }
int dsvgp_tc_work_list(int M, int N, int K, int a_tri, int c_lower, int nsplit, int pairs, int bke, int* out, int cap) {
  if (M <= 0 || N <= 0 || K <= 0 || nsplit < 1 || pairs < 1 || bke < 1 || cap < 0 || (cap > 0 && !out)) return DSVGP_ERR_ARG;
  const std::vector<int> t = tc::build_sched(M, N, K, a_tri, c_lower, nsplit, pairs, bke, nullptr);
  for (int i = 0; i < cap && i < (int)t.size(); ++i) out[i] = t[i];
  return (int)t.size();
}
int dsvgp_set_tc_cta_group(int cg) { set_tc_cta_group(cg); return get_tc_cta_group(); }
int dsvgp_split_lo_f32(const float* x, int64_t ldx, float* lo, int64_t ldl, int rows, int cols, dsvgp_stream_t s) { return split_lo(x, ldx, lo, ldl, rows, cols, ST(s)); }
int dsvgp_transpose_f32(const float* src, int64_t lds, float* dst, int64_t ldd, int rows, int cols, dsvgp_stream_t s) { return transpose_f32(src, lds, dst, ldd, rows, cols, ST(s)); }

int dsvgp_cast_f64_f32(const double* a, int64_t lda, float* b, int64_t ldb, int r, int c, int tril, dsvgp_stream_t s) { return cast2d<double, float>(a, lda, b, ldb, r, c, tril, ST(s)); }
int dsvgp_cast_f32_f64(const float* a, int64_t lda, double* b, int64_t ldb, int r, int c, int tril, dsvgp_stream_t s) { return cast2d<float, double>(a, lda, b, ldb, r, c, tril, ST(s)); }
int dsvgp_cast_f64_f64(const double* a, int64_t lda, double* b, int64_t ldb, int r, int c, int tril, dsvgp_stream_t s) { return cast2d<double, double>(a, lda, b, ldb, r, c, tril, ST(s)); }
int dsvgp_cast_f32_f32(const float* a, int64_t lda, float* b, int64_t ldb, int r, int c, int tril, dsvgp_stream_t s) { return cast2d<float, float>(a, lda, b, ldb, r, c, tril, ST(s)); }
int dsvgp_mirror_lower_f32(float* A, int64_t ld, int n, dsvgp_stream_t s) { return mirror_lower<float>(A, ld, n, ST(s)); }
int dsvgp_mirror_lower_f64(double* A, int64_t ld, int n, dsvgp_stream_t s) { return mirror_lower<double>(A, ld, n, ST(s)); }
int dsvgp_add_outer_f32(float* A, int64_t ld, int n, const float* u, const float* v, double alpha, dsvgp_stream_t s) { return add_outer<float>(A, ld, n, u, v, alpha, ST(s)); }
int dsvgp_add_outer_f64(double* A, int64_t ld, int n, const double* u, const double* v, double alpha, dsvgp_stream_t s) { return add_outer<double>(A, ld, n, u, v, alpha, ST(s)); }
int dsvgp_tril_minus_eye_f32(const float* Ls, int64_t ldl, float* E, int64_t lde, int n, dsvgp_stream_t s) { return tril_minus_eye<float>(Ls, ldl, E, lde, n, ST(s)); }
int dsvgp_tril_minus_eye_f64(const double* Ls, int64_t ldl, double* E, int64_t lde, int n, dsvgp_stream_t s) { return tril_minus_eye<double>(Ls, ldl, E, lde, n, ST(s)); }
int dsvgp_sym_phi_f64(const double* Y, int64_t ldy, double* P, int64_t ldp, int n, dsvgp_stream_t s) { return sym_phi(Y, ldy, P, ldp, n, ST(s)); }

int dsvgp_phi_outer_f32(const float* X, int64_t ldx, const float* u, const float* v, double* P, int64_t ldp, int n, dsvgp_stream_t s) { return phi_outer<float>(X, ldx, u, v, P, ldp, n, ST(s)); }
int dsvgp_phi_outer_f64(const double* X, int64_t ldx, const double* u, const double* v, double* P, int64_t ldp, int n, dsvgp_stream_t s) { return phi_outer<double>(X, ldx, u, v, P, ldp, n, ST(s)); }
int dsvgp_phi_lower_f64(const double* Y, int64_t ldy, double* P, int64_t ldp, int n, dsvgp_stream_t s) { return phi_lower(Y, ldy, P, ldp, n, ST(s)); }
int dsvgp_symmetrize_f64(double* A, int64_t ld, int n, dsvgp_stream_t s) { return symmetrize(A, ld, n, ST(s)); }

int dsvgp_reduce_slabs(int rows, int cols) { return reduce_slabs(rows, cols); }

#define PER_T(SUF, T)                                                                                              \
  int dsvgp_col_dots_##SUF(const T* A, const T* C, const T* B, int64_t ld, int rows, int nq, const T* m, T* pm,    \
                           T* pv, int nslab, unsigned int* cmax_bits, dsvgp_stream_t s) {                          \
    if (!A || !m || !pm || !pv) return DSVGP_ERR_ARG;                                                              \
    return col_dots<T>(A, C, B, ld, rows, nq, m, pm, pv, nslab, cmax_bits, ST(s));                                 \
  }                                                                                                                \
  int dsvgp_predict_finish_##SUF(const T* pm, const T* pv, int nslab, int nq, int p2, const double* hyp,           \
                                 double pred_jitter, int add_noise, double min_var, T* mu, T* var,                 \
                                 dsvgp_stream_t s) {                                                               \
    if (!pm || !pv || !hyp || !mu || !var) return DSVGP_ERR_ARG;                                                   \
    return predict_finish<T>(pm, pv, nslab, nq, p2, hyp, pred_jitter, add_noise, min_var, mu, var, ST(s));         \
  }                                                                                                                \
  int dsvgp_elbo_terms_##SUF(const T* mu, const T* var, const T* y, int nq, const double* hyp, double w,           \
                             double min_var, T* gmu, T* gvar, double* sc, double* ws, dsvgp_stream_t s) {          \
    if (!mu || !var || !y || !hyp || !gmu || !gvar || !sc || !ws) return DSVGP_ERR_ARG;                            \
    return elbo_terms<T>(mu, var, y, nq, hyp, w, min_var, gmu, gvar, sc, ws, ST(s));                               \
  }                                                                                                                \
  int dsvgp_pll_terms_##SUF(const T* mu, const T* var, const T* y, int nq, double w, double min_var, T* gmu,       \
                            T* gvar, double* sc, double* ws, dsvgp_stream_t s) {                                   \
    if (!mu || !var || !y || !gmu || !gvar || !sc || !ws) return DSVGP_ERR_ARG;                                    \
    return pll_terms<T>(mu, var, y, nq, w, min_var, gmu, gvar, sc, ws, ST(s));                                     \
  }                                                                                                                \
  int dsvgp_pred_bwd_scalars_##SUF(const T* gmu, const T* gvar, int nq, int p2, const double* hyp, int add_noise,  \
                                   double* gsc, double* ws, dsvgp_stream_t s) {                                    \
    if (!gmu || !gvar || !hyp || !gsc || !ws) return DSVGP_ERR_ARG;                                                \
    return pred_bwd_scalars<T>(gmu, gvar, nq, p2, hyp, add_noise, gsc, ws, ST(s));                                 \
  }                                                                                                                \
  int dsvgp_dA_##SUF(const T* A, T* C, T* Ag, int64_t ld, int rows, int nq, const T* m, const T* gmu,              \
                     const T* gvar, T* tp, int nslab, T* t, T* Clo, T* Aglo, dsvgp_stream_t s) {                   \
    if (!A || !C || !m || !gmu || !gvar || !tp || !t || nslab < 1) return DSVGP_ERR_ARG;                           \
    return dA_apply<T>(A, C, Ag, ld, rows, nq, m, gmu, gvar, tp, nslab, t, Clo, Aglo, ST(s));                      \
  }                                                                                                                \
  int dsvgp_kl_##SUF(const T* m, const T* Ls, int64_t ld, int Mq, double* out, double* ws, dsvgp_stream_t s) {     \
    if (!m || !Ls || !out || !ws) return DSVGP_ERR_ARG;                                                            \
    return kl_divergence<T>(m, Ls, ld, Mq, out, ws, ST(s));                                                        \
  }                                                                                                                \
  int dsvgp_var_grads_##SUF(const T* H, int64_t ldh, const T* Ls, int64_t ldl, const T* t, const T* m, int Mq,     \
                            double inv_nd, T* gm, T* gLs, int64_t ldg, dsvgp_stream_t s) {                         \
    if (!H || !Ls || !t || !m || !gm || !gLs) return DSVGP_ERR_ARG;                                                \
    return var_grads<T>(H, ldh, Ls, ldl, t, m, Mq, inv_nd, gm, gLs, ldg, ST(s));                                   \
  }
PER_T(f32, float)
PER_T(f64, double)

int dsvgp_dmma_peak_f64(int iters, int ctas, double* out, double* flops_host, dsvgp_stream_t s) { return dmma_peak(iters, ctas, out, flops_host, ST(s)); }

int dsvgp_adam_step_f32(int ntensors, const int64_t* desc_host, int ngroups, const double* group_host, dsvgp_stream_t s) { return adam_step<float>(ntensors, desc_host, ngroups, group_host, ST(s)); }
int dsvgp_adam_step_f64(int ntensors, const int64_t* desc_host, int ngroups, const double* group_host, dsvgp_stream_t s) { return adam_step<double>(ntensors, desc_host, ngroups, group_host, ST(s)); }

int dsvgp_gather_batch_f32(const float* X, const float* Y, int64_t N, int d, int ycols, const int64_t* idx, int n, int p, const int* cols_host, float* xb, float* yb, float* V, dsvgp_stream_t s) { return gather_batch<float>(X, Y, N, d, ycols, idx, n, p, cols_host, xb, yb, V, ST(s)); }
int dsvgp_gather_batch_f64(const double* X, const double* Y, int64_t N, int d, int ycols, const int64_t* idx, int n, int p, const int* cols_host, double* xb, double* yb, double* V, dsvgp_stream_t s) { return gather_batch<double>(X, Y, N, d, ycols, idx, n, p, cols_host, xb, yb, V, ST(s)); }

}  // extern "C"
