// Blocked fp64 Cholesky + explicit triangular inverse (definitions in chol.cu).
#pragma once
#include "common.cuh"

namespace dsvgp {

// Padded size Mp = nb0 << nlev >= Mq with nb0 <= 112, nb0 % 4 == 0.
void chol_plan(int Mq, int* Mp, int* nb0, int* nlev);

// Awork (Mp x Mp, lower part holds the SPD matrix, identity on the padding) is destroyed.
// L (lower, diagonal blocks have their upper part zeroed) and W = L^-1 (lower) are written.
// *info (device): 0 on success, else 1 + index of the first non-positive pivot.
int chol_factor_inverse(double* Awork, int64_t lda, double* L, int64_t ldl, double* W, int64_t ldw, int Mp, int nb0,
                        int nlev, int* info, cudaStream_t st);

// dA = sym(W^T Phi(L^T dL) W) from the lower triangles of L, W = L^-1 and dL (contract: include/dsvgp_b200.h)
size_t chol_bwd_workspace(int n);
int chol_backward(const double* L, int64_t ldl, const double* W, int64_t ldw, const double* Lbar, int64_t ldlb, double* dA,
                  int64_t lda, int n, void* ws, size_t ws_bytes, cudaStream_t st);

// 1: round-1 diagonal-block kernel (in-kernel DMMA prologue, scalar updates); 2 (default): diag_prepare + all-DMMA block kernel
void set_chol_variant(int v);
int get_chol_variant();
// 1: diagonal-block chain, panel / trailing-update chain and eager-inverse chain all on high-priority streams of the
// library (forked from and joined to the caller's stream); 0: the diagonal chain stays on the caller's stream
// 1: trailing update of a step split into the thin part the next two links need and the bulk on a stream of its own
void set_chol_lookahead(int on);
int get_chol_lookahead();
void set_chol_mid_link(int k);
int get_chol_mid_link();
int chol_wait_mid(cudaStream_t s);
void set_chol_inv_streams(int n);
int get_chol_inv_streams();
void set_chol_graph(int on);
int get_chol_graph();
void set_chol_priority(int on);
int get_chol_priority();
void set_potrf_debug(long long* p);   // profiling aid: device buffer of 64 clock64() stamps (nullptr = off)

}  // namespace dsvgp
