// Host-callable launchers of the kernel-assembly kernels (definitions in kdir.cu).
#pragma once
#include "common.cuh"

namespace dsvgp {

int bwd_num_chunks(int n1, int n2);
bool bwd_v4_ok(int n1, int p1, int n2, int p2, int d);

template <typename T, typename TK>
int normalize_dirs(const T* v, int rows, int d, TK* vhat, TK* inv_norm, cudaStream_t st, int* cidx = nullptr,
                   int* canon_flag = nullptr);   // cidx/canon_flag: one-hot (canonical) row detection, see kdir.cu

// hyp: device double[8] = {ell, outputscale, noise, constant, sigmoid(raw_ell), sigmoid(raw_os), sigmoid(raw_noise), -}
template <typename T, typename TK>
int kdir_fwd(const T* x1, const TK* u1, int n1, int p1, const T* x2, const TK* w2, int n2, int p2, int d,
             const double* hyp, int use_os, double diag_add, TK* K, int64_t ldk, cudaStream_t st,
             const int* cidx2 = nullptr, const int* canon_flag = nullptr,   // canonical column-side fast path (fp32)
             TK* Klo = nullptr,    // fp32 only: also write the TF32 'lo' companion of K; returns 1 if it was written
             void* Kh = nullptr, void* Kl = nullptr, int64_t ldkh = 0, const float* hscale = nullptr);
// Kh/Kl (fp32 only): write ONLY the two-half split of K * *hscale (operands of the 3xFP16 product); returns 2 if the
// vectorised kernel took the shape and wrote them (K untouched), otherwise K is written as usual and 0/1 is returned.

template <typename TK>
int kdir_diag(int n, int p, const double* hyp, int use_os, TK* out, cudaStream_t st);

template <typename TK>
size_t kdir_bwd_workspace(int n1, int p1, int n2, int p2, int d);

template <typename T, typename TK>
int kdir_bwd(const T* x1, const TK* u1, const TK* inv1, int n1, int p1, const T* x2, const TK* w2, int n2, int p2,
             int d, const double* hyp, int use_os, const TK* dK, int64_t lddk, int dk_trans, double scale,
             double* gx, double* gv, double* gsc, void* ws, size_t ws_bytes, cudaStream_t st);

// data-side gradient (d/dx2, d/dv2) of the same product; returns 1 if the vectorised fp32 kernel ran, 0 for the blocked one
template <typename TK>
size_t kdir_bwd_cols_workspace(int n1, int p1, int n2, int p2, int d);

template <typename T, typename TK>
int kdir_bwd_cols(const T* x1, const TK* u1, int n1, int p1, const T* x2, const TK* w2, const TK* inv2, int n2, int p2, int d,
                  const double* hyp, int use_os, const TK* dK, int64_t lddk, double scale, double* gx, double* gv, void* ws,
                  size_t ws_bytes, cudaStream_t st);

}  // namespace dsvgp
