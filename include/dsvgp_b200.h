/* dsvgp_b200 -- C ABI of the B200-native DSVGP hot path (libdsvgp_b200.so, sm_100a only).
 *
 * The reference (mishapadidar/GP-Derivatives-Variational-Inference) has no FFI: its boundary is the Python
 * class API.  These entry points are what a Python binding of that API calls underneath; each one says which
 * reference code it replaces (paths are under directionalvi/ of the reference).  The ctypes stubs a maintainer
 * would add are in INTEGRATION.md and, in full, in gp-derivatives-variational-inference_b200/dsvgp_b200/_lib.py.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host; matrices are row-major with an explicit
 *     leading dimension (in elements); the caller owns every buffer (the library never allocates user-visible
 *     memory); scratch comes in through a workspace pointer whose size a *_workspace() function reports;
 *   - all work is enqueued on the cudaStream_t given (pass torch.cuda.current_stream().cuda_stream); there is
 *     no hidden synchronisation, so every call is CUDA-graph capturable;
 *   - return value: 0 = ok, <0 = DSVGP_ERR_* ; nothing throws;
 *   - suffixes: _f32 / _f64 = dtype of the model tensors; _f32f64 = fp32 inputs, fp64 matrix (K_zz of an fp32
 *     model is assembled and factorised in fp64, DirectionalGradVariationalStrategy.py:74);
 *   - `hyp` is a device double[8]: {lengthscale, outputscale, noise, mean constant,
 *     sigmoid(raw_lengthscale), sigmoid(raw_outputscale), sigmoid(raw_noise), 0}  (dsvgp_hyp_from_raw_*).
 *   - directions are passed ALREADY NORMALISED (dsvgp_normalize_dirs_*), point-major: p consecutive rows per
 *     point (RBFKernelDirectionalGrad.py:10-13).
 */
#ifndef DSVGP_B200_H
#define DSVGP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* dsvgp_stream_t; /* cudaStream_t */

#define DSVGP_OK 0
#define DSVGP_ERR_ARG -1
#define DSVGP_ERR_LAUNCH -2
#define DSVGP_ERR_WORKSPACE -3

#define DSVGP_TRI_NONE 0
#define DSVGP_TRI_LOWER 1
#define DSVGP_TRI_UPPER 2

/* library version (major*10000 + minor*100 + patch) and the compute capability it was built for (100) */
int dsvgp_version(void);
int dsvgp_built_for_sm(void);
/* number of CUDA kernels this library has launched in this process (host-side counter) */
int64_t dsvgp_launch_count(void);
/* benchmarking knobs of the fp32 assembly kernel: row points per CTA (0 = adaptive, the default: 64, or 32 when that leaves
 * fewer than 1024 CTAs -- small minibatches; or a fixed 8..64, multiple of 8) and
 * evict-first (st.global.cs) stores of the covariance rows (0 off, 1 on, 2 = when the output exceeds 64 MB, the
 * default).  Negative = leave unchanged.  Returns tib*4 + stream_stores as set before the call. */
int dsvgp_set_kdir_fwd_knobs(int tib, int stream_stores);
/* column points per lane of the vectorised fp32 assembly backward: 4 (default; 128-point column tiles, one CTA per SM) or 2
 * (64-point tiles, two CTAs per SM).  Returns the value in force. */
int dsvgp_set_kdir_bwd_vpl(int vpl);

/* Positive()/GreaterThan(1e-4) transforms of gpytorch that the reference reaches through
 * self.lengthscale (RBFKernelDirectionalGrad.py:67), ScaleKernel.outputscale (directional_vi.py:56) and
 * GaussianLikelihood.noise (directional_vi.py:172).  raw_os / raw_noise / c may be NULL. */
int dsvgp_hyp_from_raw_f32(const float* raw_ell, const float* raw_os, const float* raw_noise, const float* c, double* hyp, dsvgp_stream_t s);
int dsvgp_hyp_from_raw_f64(const double* raw_ell, const double* raw_os, const double* raw_noise, const double* c, double* hyp, dsvgp_stream_t s);

/* v / |v| row-wise and 1/|v|  -- RBFKernelDirectionalGrad.py:57-58 */
int dsvgp_normalize_dirs_f32(const float* v, int rows, int d, float* vhat, float* inv_norm, dsvgp_stream_t s);
int dsvgp_normalize_dirs_f64(const double* v, int rows, int d, double* vhat, double* inv_norm, dsvgp_stream_t s);
int dsvgp_normalize_dirs_f32f64(const float* v, int rows, int d, double* vhat, double* inv_norm, dsvgp_stream_t s);

/* K (n1(p1+1) x n2(p2+1), interleaved) = [outputscale *] RBFKernelDirectionalGrad.forward(x1, x2, v1=.., v2=..)
 * -- RBFKernelDirectionalGrad.py:41-108 (+ ScaleKernel).  p2 = 0 gives the value-only columns the DFree strategy
 * keeps (DFreeDirectionalGradVariationalStrategy.py:118).  diag_add is added to the diagonal (add_jitter,
 * DirectionalGradVariationalStrategy.py:144) and is only meaningful for x1 == x2. */
int dsvgp_kdir_fwd_f32(const float* x1, const float* u1, int n1, int p1, const float* x2, const float* w2, int n2, int p2, int d, const double* hyp, int use_os, double diag_add, float* K, int64_t ldk, dsvgp_stream_t s);
int dsvgp_kdir_fwd_f64(const double* x1, const double* u1, int n1, int p1, const double* x2, const double* w2, int n2, int p2, int d, const double* hyp, int use_os, double diag_add, double* K, int64_t ldk, dsvgp_stream_t s);
int dsvgp_kdir_fwd_f32f64(const float* x1, const double* u1, int n1, int p1, const float* x2, const double* w2, int n2, int p2, int d, const double* hyp, int use_os, double diag_add, double* K, int64_t ldk, dsvgp_stream_t s);

/* Canonical-direction fast path of the fp32 assembly.  dsvgp_normalize_dirs_canon_f32 additionally writes, per
 * direction row, the coordinate of its single non-zero entry (sign in bit 31) and clears *canon_flag (device int, set
 * to 1 by the caller) if any row is not one-hot.  dsvgp_kdir_fwd_canon_f32 takes those for the SECOND argument's
 * directions: when the flag is still set -- eye(d) rows, which is what train_gp / eval_gp pass (directional_vi.py:87-88,
 * :292-293) -- D.w and u.w become lookups.  Decided on the device, no host synchronisation; results are identical.
 * Klo (optional, same leading dimension as K): TF32 'lo' companion of K for dsvgp_gemm_tc_f32; the call returns 1
 * instead of 0 when it was written (the vectorised kernel took the shape), otherwise use dsvgp_split_lo_f32. */
int dsvgp_normalize_dirs_canon_f32(const float* v, int rows, int d, float* vhat, float* inv_norm, int* cidx, int* canon_flag, dsvgp_stream_t s);
int dsvgp_kdir_fwd_canon_f32(const float* x1, const float* u1, int n1, int p1, const float* x2, const float* w2, const int* cidx2, const int* canon_flag, int n2, int p2, int d, const double* hyp, int use_os, double diag_add, float* K, int64_t ldk, float* Klo, dsvgp_stream_t s);

/* diag=True branch -- RBFKernelDirectionalGrad.py:110-119 */
int dsvgp_kdir_diag_f32(int n, int p, const double* hyp, int use_os, float* out, dsvgp_stream_t s);
int dsvgp_kdir_diag_f64(int n, int p, const double* hyp, int use_os, double* out, dsvgp_stream_t s);

/* Backward of dsvgp_kdir_fwd_* (autograd of RBFKernelDirectionalGrad.py:57-107): given dK, ACCUMULATES
 *   gx   (n1,d)      += scale * dL/dx1         (NULL to skip)
 *   gv   (n1*p1,d)   += scale * dL/dv1 (chain rule through the normalisation included; NULL to skip)
 *   gsc[0] += dL/dlengthscale, gsc[1] += dL/doutputscale   (NULL to skip)
 * all double.  dk_trans != 0 reads dK transposed (gradients for the second argument: swap the roles).
 * K is recomputed, never re-read. */
size_t dsvgp_kdir_bwd_workspace_f32(int n1, int p1, int n2, int p2, int d);
size_t dsvgp_kdir_bwd_workspace_f64(int n1, int p1, int n2, int p2, int d);
int dsvgp_kdir_bwd_f32(const float* x1, const float* u1, const float* inv1, int n1, int p1, const float* x2, const float* w2, int n2, int p2, int d, const double* hyp, int use_os, const float* dK, int64_t lddk, int dk_trans, double scale, double* gx, double* gv, double* gsc, void* ws, size_t ws_bytes, dsvgp_stream_t s);
int dsvgp_kdir_bwd_f64(const double* x1, const double* u1, const double* inv1, int n1, int p1, const double* x2, const double* w2, int n2, int p2, int d, const double* hyp, int use_os, const double* dK, int64_t lddk, int dk_trans, double scale, double* gx, double* gv, double* gsc, void* ws, size_t ws_bytes, dsvgp_stream_t s);
int dsvgp_kdir_bwd_f32f64(const float* x1, const double* u1, const double* inv1, int n1, int p1, const float* x2, const double* w2, int n2, int p2, int d, const double* hyp, int use_os, const double* dK, int64_t lddk, int dk_trans, double scale, double* gx, double* gv, double* gsc, void* ws, size_t ws_bytes, dsvgp_stream_t s);

/* Data-side ("column") gradient of dsvgp_kdir_fwd_*: the gradient w.r.t. the SECOND argument (the data points x2 and their
 * directions v2 of K_zx), given dK laid out as the forward writes K (n1(p1+1) x n2(p2+1), row-major).  ACCUMULATES
 *   gx (n2,d)      += scale * dL/dx2         (NULL to skip)
 *   gv (n2*p2,d)   += scale * dL/dv2 (chain rule through the normalisation included, inv2 = 1/|v2|; NULL to skip)
 * in double.  fp32 with d <= 20, n2 >= 512 and (p1, p2) in {(0,0), (1,1), (2,2), (1,0), (2,0)} runs a dedicated kernel that
 * reads dK once, row by row and coalesced, recomputes K and sums fp64 partials in a fixed order (no atomics), and returns 1;
 * every other shape and fp64 run dsvgp_kdir_bwd_* with dk_trans = 1 on the swapped problem (dK read strided) and return 0.
 * Results agree to rounding.  No length- or outputscale gradient (dsvgp_kdir_bwd_* gives those). */
size_t dsvgp_kdir_bwd_cols_workspace_f32(int n1, int p1, int n2, int p2, int d);
size_t dsvgp_kdir_bwd_cols_workspace_f64(int n1, int p1, int n2, int p2, int d);
int dsvgp_kdir_bwd_cols_f32(const float* x1, const float* u1, int n1, int p1, const float* x2, const float* w2, const float* inv2, int n2, int p2, int d, const double* hyp, int use_os, const float* dK, int64_t lddk, double scale, double* gx, double* gv, void* ws, size_t ws_bytes, dsvgp_stream_t s);
int dsvgp_kdir_bwd_cols_f64(const double* x1, const double* u1, int n1, int p1, const double* x2, const double* w2, const double* inv2, int n2, int p2, int d, const double* hyp, int use_os, const double* dK, int64_t lddk, double scale, double* gx, double* gv, void* ws, size_t ws_bytes, dsvgp_stream_t s);

/* Cholesky of the jittered K_zz and the inverse factor -- _cholesky_factor / psd_safe_cholesky
 * (DirectionalGradVariationalStrategy.py:72-75) and TriangularLazyTensor.inv_matmul (:181,:183).
 * dsvgp_chol_plan: padded size Mp = nb0 << nlev for an Mq x Mq matrix.  dsvgp_pad_identity_f64 writes the identity
 * padding.  dsvgp_chol_f64: Awork (destroyed) -> L (lower), W = L^-1 (lower); *info (device int) = 0 or
 * 1 + index of the first pivot that is not a positive finite number (<= 0, NaN or +inf; a pivot pair whose determinant
 * a11 a22 - a21^2 overflows reports its second pivot).  Only the lower triangle of Awork is read.  The factorisation loads
 * Awork two doubles at a time from the start of every block column, so Awork must be 16-byte aligned, lda even and, when
 * nlev > 0, nb0 even; otherwise DSVGP_ERR_ARG and nothing is enqueued.  The nb0 of dsvgp_chol_plan is a multiple of 4 and
 * every Mp x Mp tensor the library allocates qualifies.  The panel / trailing-update GEMMs of the factorisation run on a
 * library-owned side stream (one per device) that is forked from and joined back into `s` with events: from the
 * caller's point of view everything is ordered on `s`, there is still no host synchronisation, and the call stays
 * CUDA-graph capturable.  Not re-entrant from two host threads on the same device at the same time. */
void dsvgp_chol_plan(int Mq, int* Mp_host, int* nb0_host, int* nlev_host);
int dsvgp_pad_identity_f64(double* A, int64_t ld, int Mq, int Mp, dsvgp_stream_t s);
/* A/B knob of the diagonal-block chain: 1 = the round-1 kernel (DMMA prologue inside the single-CTA block kernel, scalar
 * rank-8 updates and inverse) and the batched recursive inverse after the factorisation instead of the eager one;
 * 2 = a small multi-CTA kernel forms the update of the next diagonal block and the block kernel does every bulk operation
 * as 8x8 DMMA tiles; 3 (default) = that update and the block kernel as one launch of a 4-CTA thread-block cluster that sums
 * its partial updates through distributed shared memory.  A single block always takes kernel 1, and so does variant 2
 * below four blocks.  Out-of-range values select 3.  Returns the value in force.  Results agree to rounding. */
int dsvgp_set_chol_variant(int v);
/* 1: the factorisation's three chains (diagonal blocks; panels + trailing updates; eager inverse) run on high-priority
 * streams owned by the library, forked from / joined to the caller's stream, so that work the caller overlaps with the
 * latency-bound factorisation on other streams cannot delay it; 0 (default; measured equal): the diagonal chain stays on the
 * caller's stream.
 * Returns the value in force. */
int dsvgp_set_chol_priority(int on);
/* Deferring a caller's overlapped work to the latency-bound part of the factorisation: the first links of the chain are bound by
 * their trailing updates (which fill the GPU), the later ones leave most SMs idle.  dsvgp_chol_wait_mid makes stream s wait for
 * diagonal block min(k, last) (dsvgp_set_chol_mid_link, default k = 20, negative: never) of the factorisation enqueued
 * last on the current device; a no-op when that factorisation had fewer than 8 blocks.  (Measured at 32 blocks: release points 14 .. 31 equal within noise, 6 .. 10 worse.)  Capturable (an event edge inside the graph). */
int dsvgp_set_chol_mid_link(int k);
int dsvgp_chol_wait_mid(dsvgp_stream_t s);
/* 1: dsvgp_chol_f64 captures its ~230 launches / ~400 event calls ONCE per (buffers, sizes, scheduling knobs) into a CUDA graph of
 * its own and replays it with one cudaGraphLaunch (a cache of 8 per device); the mid-chain event of dsvgp_chol_wait_mid becomes an
 * external event node.  Ignored while the caller's stream is being captured.  0 (default: measured equal on this host -- the GPU
 * sets the factorisation's pace) = plain launches.  Results are bit-identical.  Returns the value in force. */
int dsvgp_set_chol_graph(int on);
/* Streams of the eager inverse W = L^-1 (for every pair of every level of the recursive doubling, T = L21 W11 is issued when the
 * pair's top half is complete and W21 = -W22 T when its bottom half is): 3 (default) = one stream per level, ordered across levels
 * by events -- on fewer streams the 72 / 177 us products of the upper levels sit in front of the short ones of the following blocks
 * and the inverse finishes ~0.3 ms after the factor instead of one five-product dependency chain after it (factorisation alone
 * 2.23 -> 1.93 ms at M' = 3072); 2 = T products on one extra stream; 1 = one stream.  Results bit-identical.  Returns the value in force. */
int dsvgp_set_chol_inv_streams(int n);
/* 1: while the trailing matrix is large, the update of step k is split into the first two block columns of the
 * trapezoid (all that the diagonal block k+2 and the panel k+1 read; side stream) and the rest (a low-priority stream of its
 * own, two links' time to finish);
 * 0 (default; the split measured no gain): one product per step, which the diagonal block k+2 waits for.  Returns the value
 * in force. */
int dsvgp_set_chol_lookahead(int on);
/* profiling aid: a device buffer of 64 int64 that one diagonal-block kernel fills with clock64() stamps at its phase
 * boundaries (NULL switches it off); see scratch/potrf_phases.py */
int dsvgp_set_potrf_debug(void* buf);
int dsvgp_chol_f64(double* Awork, int64_t lda, double* L, int64_t ldl, double* W, int64_t ldw, int Mp, int nb0, int nlev, int* info, dsvgp_stream_t s);

/* C = alpha*op(A)*op(B) + beta*C, triangle-aware, batched -- every dense product of the strategy
 * (DirectionalGradVariationalStrategy.py:181-205) and of its backward.  fp32 uses 3xTF32 (fp32-accurate).
 * D != NULL: C = alpha*op(A)*op(B) + beta*D (D not batched); D == NULL: the addend is C itself.
 * C2 != NULL: a second output C2 = C + D2 is written by the same epilogue (used for B' = E^T A, B = A + B'). */
int dsvgp_gemm_f32(int ta, int tb, int M, int N, int K, double alpha, const float* A, int64_t lda, const float* B, int64_t ldb, double beta, float* C, int64_t ldc, int a_tri, int b_tri, int c_tri, int batch, int64_t sA, int64_t sB, int64_t sC, const float* D, int64_t ldd, float* C2, int64_t ldc2, const float* D2, int64_t ldd2, dsvgp_stream_t s);
int dsvgp_gemm_f64(int ta, int tb, int M, int N, int K, double alpha, const double* A, int64_t lda, const double* B, int64_t ldb, double beta, double* C, int64_t ldc, int a_tri, int b_tri, int c_tri, int batch, int64_t sA, int64_t sB, int64_t sC, const double* D, int64_t ldd, double* C2, int64_t ldc2, const double* D2, int64_t ldd2, dsvgp_stream_t s);

/* A/B knob of dsvgp_gemm_f64: 1 (default) = cp.async-pipelined kernel (3 stages, k-major shared layouts for operands that are
 * contiguous along their non-contracted index: no staging stores, conflict-free DMMA fragments, one barrier per k-tile),
 * 0 = the register-staged kernel of round 1.  Returns the value in force. */
int dsvgp_set_gemm64_async(int on);
/* fp64 products op(A) = A, op(B) = B^T with a short contraction (8 <= K <= 128, even; no triangle flags on the operands, no
 * batch): 1 = rank-update kernel (whole K extent of both operand tiles in shared memory in one cp.async burst, one barrier) --
 * the trailing updates of the blocked Cholesky; 2 = that kernel only for launches of at most 640 tiles (the latency-bound late
 * links; the panel products then go through it as dense products, W11 carrying explicit zeros above its diagonal); 0 (default:
 * 1 measured slower, 2 equal within 0.02 ms) = the general kernel.  Returns the value in force. */
int dsvgp_set_rank_update(int on);

/* The same product on the 5th-generation tensor cores (tcgen05.mma kind::tf32, TMA-fed, accumulators in tensor memory)
 * for the fp32 model's big whitening products -- TriangularLazyTensor.inv_matmul and the L_s products of
 * DirectionalGradVariationalStrategy.py:181-205 and their backward.  A: M x K row-major with explicit zeros outside
 * its triangle; B: K x N row-major (b_kmajor = 0) or N x K row-major (b_kmajor = 1, Gram matrices).  Every operand is
 * given as the raw fp32 array plus lo = x - trunc_tf32(x) (dsvgp_split_lo_f32); 3 MMAs per k-step give fp32-grade
 * products, `chunk` (k-blocks of 32) bounds the length of the tensor-core accumulation chain.  a_tri trims the k-range
 * (1 lower, 2 upper), c_lower skips tiles above the diagonal.  Clo / C2lo (optional) receive the lo parts of C / C2 from
 * the same epilogue.  nsplit > 1: split-K over gridDim.z with an fp64 reduction of the partial sums held in split_ws
 * (nsplit * M * round_up(N,4) floats; requires C2 == Clo == NULL).  dsvgp_gemm_tc_supported_f32 tells whether the operands
 * meet the TMA constraints (otherwise use dsvgp_gemm_f32). */
int dsvgp_gemm_tc_supported_f32(const float* A, int64_t lda, const float* B, int64_t ldb, int b_kmajor, int N);
int dsvgp_gemm_tc_f32(const float* Ah, const float* Al, int64_t lda, const float* Bh, const float* Bl, int64_t ldb, int b_kmajor, int M, int N, int K, double alpha, double beta, float* C, int64_t ldc, const float* D, int64_t ldd, float* C2, int64_t ldc2, const float* D2, int64_t ldd2, int a_tri, int c_lower, int chunk, float* Clo, float* C2lo, int nsplit, float* split_ws, dsvgp_stream_t s);
/* 3xFP16 variant of dsvgp_gemm_tc_f32 (tcgen05 kind::f16, twice the tensor throughput of kind::tf32): every operand is
 * the two-half split (hi, lo: fp16 arrays, passed as void*) of x * s with a power-of-two scale s per matrix chosen from an
 * a-priori bound (dsvgp_tc_scales_f32) so that fp16's 5-bit exponent never overflows; hi + lo carry the same 22
 * significand bits as the tf32 split.  ab_inv (device float) = 1/(sA*sB).  Outputs, each optional: C (fp32),
 * C2 = C + D2 (fp32), Ch/Cl = split of C * *c_scale, C2h/C2l = split of C2 * *c2_scale.  Half leading dimensions % 8 == 0;
 * a K x N row-major B needs ldb >= round_up(N, 64). */
int dsvgp_gemm_tch_supported_f32(const void* A, int64_t lda, const void* B, int64_t ldb, int b_kmajor, int N);
int dsvgp_gemm_tch_f32(const void* Ah, const void* Al, int64_t lda, const void* Bh, const void* Bl, int64_t ldb, int b_kmajor, int M, int N, int K, double alpha, double beta, const float* ab_inv, float* C, int64_t ldc, const float* D, int64_t ldd, float* C2, int64_t ldc2, const float* D2, int64_t ldd2, void* Ch, void* Cl, int64_t ldch, const float* c_scale, void* C2h, void* C2l, int64_t ldc2h, const float* c2_scale, int a_tri, int c_lower, int chunk, int nsplit, float* split_ws, dsvgp_stream_t s);
/* Operand preparation for dsvgp_gemm_tch_f32.
 * dsvgp_absmax_*: *out_bits = max(*out_bits, max|x_ij|) as the bit pattern of a non-negative float (zero it first; NaN
 *   gives +inf); mode 0: all entries, 2: the entries of tril(x) - I.
 * dsvgp_tc_scales_f32: power-of-two scales (device float[16]) of every operand of a step from rigorous a-priori bounds
 *   (list in csrc/tc_prep.cu): [0] W [1] K_zx [2] E [3] A [4] B [5] dA [6] A_g [7] D = S - I, [8..13] the reciprocal products
 *   1/(sW sK), 1/(sE sA), 1/(sE sB), 1/(sW sdA), 1/(sAg sA), 1/(sD sA).  maxbits (device uint[8]) = absmax bits of E, m, g_mu,
 *   g_var, and the MEASURED maxima of D = S - I ([4]) and C = (S - I) A ([5]; 0 = fall back to the a-priori bound).
 *   stage 0 fills what the forward pass needs (hyp, jitter, maxbits[0]), stage 2 re-makes the scale of D from maxbits[4],
 *   stage 1 the backward scales (dA from max|m| max|g_mu| + 2 max|g_var| max|C|).
 * dsvgp_split_half_*: (hi, lo) = two-half split of op(src) * *scale, optionally also of its transpose (hiT, loT);
 *   mode 0: src, 1: tril(src), 2: tril(src) - I.
 * dsvgp_kdir_fwd_half_f32: dsvgp_kdir_fwd_canon_f32 that writes ONLY the split (Kh, Kl) of K * *hscale; returns 2 when
 *   it did, otherwise K (fp32) was written instead (shape not taken by the vectorised kernel) and 0 is returned.
 * dsvgp_dA_half_f32: dsvgp_dA_f32 whose outputs are only the splits of dA * *s_dA and A_g * *s_Ag (C is not modified).
 * dsvgp_dA_half_h_f32 / dsvgp_col_dots_h_f32: the same pass / dsvgp_col_dots_f32 with A given ONLY as the split (Ah, Al) of
 *   A * *a_scale (leading dimension ldh, the one of the outputs for dA_half_h): the training step's whitening product then
 *   writes no fp32 A at all -- half of its store phase, which is bound by the 32 B/clk write port of an SM. */
int dsvgp_absmax_f32(const float* x, int64_t ld, int rows, int cols, int mode, unsigned int* out_bits, dsvgp_stream_t s);
int dsvgp_absmax_f64(const double* x, int64_t ld, int rows, int cols, int mode, unsigned int* out_bits, dsvgp_stream_t s);
int dsvgp_tc_scales_f32(const double* hyp, double jitter, const unsigned int* maxbits, int Mq, float* scales, int stage, dsvgp_stream_t s);
int dsvgp_split_half_f32(const float* src, int64_t lds, int rows, int cols, int mode, const float* scale, void* hi, void* lo, int64_t ldh, void* hiT, void* loT, int64_t ldhT, dsvgp_stream_t s);
int dsvgp_split_half_f64(const double* src, int64_t lds, int rows, int cols, int mode, const float* scale, void* hi, void* lo, int64_t ldh, void* hiT, void* loT, int64_t ldhT, dsvgp_stream_t s);
/* (hi, lo) = two-half split of D * *scale with D = S - I = E + E^T + E E^T (symmetric), from the lower triangles of
 * E = tril(L_s) - I and P = E E^T: the operand of the single dense product C = (S - I) A of the training step. */
int dsvgp_build_d_split_f32(const float* E, int64_t lde, const float* P, int64_t ldp, int n, const float* scale, void* hi, void* lo, int64_t ldh, dsvgp_stream_t s);
/* *out_bits = max(*out_bits, max|D_ij|) for the same D (measured, so that the scale of D stays tight when q(u) is far from
 * N(0, I)); feed it to dsvgp_tc_scales_f32 as maxbits[4] with stage 2 before dsvgp_build_d_split_f32. */
int dsvgp_build_d_absmax_f32(const float* E, int64_t lde, const float* P, int64_t ldp, int n, unsigned int* out_bits, dsvgp_stream_t s);
int dsvgp_kdir_fwd_half_f32(const float* x1, const float* u1, int n1, int p1, const float* x2, const float* w2, const int* cidx2, const int* canon_flag, int n2, int p2, int d, const double* hyp, int use_os, double diag_add, float* K, int64_t ldk, void* Kh, void* Kl, int64_t ldkh, const float* hscale, dsvgp_stream_t s);
int dsvgp_dA_half_f32(const float* A, const float* C, int64_t ld, int rows, int nq, const float* m, const float* gmu, const float* gvar, float* tp, int nslab, float* t, void* dAh, void* dAl, void* Agh, void* Agl, int64_t ldh, const float* s_dA, const float* s_Ag, dsvgp_stream_t s);
int dsvgp_dA_half_h_f32(const void* Ah, const void* Al, const float* a_scale, const float* C, int64_t ld, int rows, int nq, const float* m, const float* gmu, const float* gvar, float* tp, int nslab, float* t, void* dAh, void* dAl, void* Agh, void* Agl, int64_t ldh, const float* s_dA, const float* s_Ag, dsvgp_stream_t s);
int dsvgp_col_dots_h_f32(const void* Ah, const void* Al, int64_t ldh, const float* a_scale, const float* C, int64_t ld, int rows, int nq, const float* m, float* pm, float* pv, int nslab, unsigned int* cmax_bits, dsvgp_stream_t s);
/* tile scheme of dsvgp_gemm_tc_f32: 1 = one CTA per 128x256 tile (cta_group::1), 2 = CTA pairs on 256x256 tiles
 * (cta_group::2: each CTA stages half of the operands, 2-SM TMA loads, multicast commits).  Returns the value in force. */
int dsvgp_set_tc_cta_group(int cg);
/* N extent of a CTA-pair tile of dsvgp_gemm_tch_f32: 256 = one pair per SM pair (3 stages of 64 KB, 512 columns of tensor
 * memory), 128 = TWO pairs resident per SM pair (2 stages of 48 KB, 256 columns each, 4 epilogue warps): one pair's fixed
 * phases (set-up, pipeline fill, store of its tile) run under the other pair's main loop.  Returns the value in force. */
int dsvgp_set_tc_tile_n(int n);
/* CTA-pair tensor-core products: 1 (default) = persistent CTA pairs (one per SM pair) walking a host-balanced list of
 * (256 x 256 tile, split-K slice) work items; 0 = one CTA pair per tile.  Returns the value in force.
 * The FIRST product of a given shape / triangle mode / split on a device builds its work list: one cudaMalloc and one
 * synchronous copy of a few KB (the only host synchronisation of these entry points; never during stream capture -- a
 * capturing call whose list does not exist yet takes the per-tile kernel). */
int dsvgp_set_tc_persistent(int on);
/* Persistent products: use at most n CTA pairs (0 = every pair the device can hold, the default), leaving the other SMs to
 * whatever runs beside the product.  Returns the value in force. */
int dsvgp_set_tc_max_pairs(int n);
/* Profiling aid of the persistent products: with buf != NULL (device memory, 8 * cap_items int64) the MMA warp and the first
 * epilogue warp of every pair leader stamp the SM clock for each work item with list index < cap_items: buf[8 i + 0..6] = MMA warp
 * reaches item i, its first k-block issued, its last k-block issued, epilogue reaches the item, first chunk complete, last
 * chunk added (store phase starts), tile stored.  buf = NULL switches it off. */
int dsvgp_set_tc_trace(void* buf, int cap_items);
/* The work list the persistent kernels would use for a product on `pairs` CTA pairs (host only, no GPU needed): writes
 * at most `cap` ints [offsets (pairs + 1, padded to a multiple of 4) | items {pair-tile row, tile column, slice, kb0 | kb1 << 16}]
 * to `out` and returns the number of ints of the full table (call with cap = 0 to size the buffer).  bke = elements per
 * k-block (64 for the 3xFP16 product, 32 for 3xTF32). */
int dsvgp_tc_work_list(int M, int N, int K, int a_tri, int c_lower, int nsplit, int pairs, int bke, int* out, int cap);
int dsvgp_split_lo_f32(const float* x, int64_t ldx, float* lo, int64_t ldl, int rows, int cols, dsvgp_stream_t s);
int dsvgp_transpose_f32(const float* src, int64_t lds, float* dst, int64_t ldd, int rows, int cols, dsvgp_stream_t s);

/* helpers on M' x M' matrices of the replicated tail */
int dsvgp_cast_f64_f32(const double* src, int64_t lds, float* dst, int64_t ldd, int rows, int cols, int tril, dsvgp_stream_t s);
int dsvgp_cast_f32_f64(const float* src, int64_t lds, double* dst, int64_t ldd, int rows, int cols, int tril, dsvgp_stream_t s);
int dsvgp_cast_f64_f64(const double* src, int64_t lds, double* dst, int64_t ldd, int rows, int cols, int tril, dsvgp_stream_t s);
int dsvgp_cast_f32_f32(const float* src, int64_t lds, float* dst, int64_t ldd, int rows, int cols, int tril, dsvgp_stream_t s);
int dsvgp_mirror_lower_f32(float* A, int64_t ld, int n, dsvgp_stream_t s);
int dsvgp_mirror_lower_f64(double* A, int64_t ld, int n, dsvgp_stream_t s);
int dsvgp_add_outer_f32(float* A, int64_t ld, int n, const float* u, const float* v, double alpha, dsvgp_stream_t s);
int dsvgp_add_outer_f64(double* A, int64_t ld, int n, const double* u, const double* v, double alpha, dsvgp_stream_t s);
/* E = tril(Ls_raw) - I: the variational factor enters every product as I + E so that (S - I) A = E B + E^T A is
 * formed without the cancellation of Ls (Ls^T A) - A  (S = Ls Ls^T, B = A + E^T A). */
int dsvgp_tril_minus_eye_f32(const float* Ls, int64_t ldl, float* E, int64_t lde, int n, dsvgp_stream_t s);
int dsvgp_tril_minus_eye_f64(const double* Ls, int64_t ldl, double* E, int64_t lde, int n, dsvgp_stream_t s);
int dsvgp_sym_phi_f64(const double* Y, int64_t ldy, double* P, int64_t ldp, int n, dsvgp_stream_t s);
/* Cholesky backward dK = sym(L^-T Phi(L^T dL) L^-1): Phi = tril with halved diagonal; A <- (A + A^T)/2 in place */
int dsvgp_phi_lower_f64(const double* Y, int64_t ldy, double* P, int64_t ldp, int n, dsvgp_stream_t s);
int dsvgp_symmetrize_f64(double* A, int64_t ld, int n, dsvgp_stream_t s);
/* LOWER TRIANGLE of P = Phi(X + u v^T) in fp64 from X in the model dtype (the upper triangle of P is not written: its consumers
 * take P with a lower-triangle flag): dsvgp_add_outer + dsvgp_cast2d + dsvgp_phi_lower of the Cholesky-backward tail in one pass. */
int dsvgp_phi_outer_f32(const float* X, int64_t ldx, const float* u, const float* v, double* P, int64_t ldp, int n, dsvgp_stream_t s);
int dsvgp_phi_outer_f64(const double* X, int64_t ldx, const double* u, const double* v, double* P, int64_t ldp, int n, dsvgp_stream_t s);

/* predictive mean / diagonal variance (DirectionalGradVariationalStrategy.py:188,:192-205):
 *   pm[s][j] = sum_{i in slab s} A_ij m_i ;  pv[s][j] = sum A_ij C_ij  (C given)  or, with B' = B - A given in
 *   the `B` slot, sum B'_ij (2 A_ij + B'_ij) = sum (B_ij^2 - A_ij^2)
 *   mu_j = sum_s pm + c ; var_j = kdiag_j + pred_jitter + sum_s pv [+ noise], clamped at min_var.
 *   cmax_bits (optional, C given): *cmax_bits = max(*cmax_bits, max|C_ij|) as float bits -- the measured bound the
 *   3xFP16 scale of dA is made from (dsvgp_tc_scales_f32 maxbits[5]). */
int dsvgp_reduce_slabs(int rows, int cols);
int dsvgp_col_dots_f32(const float* A, const float* C, const float* B, int64_t ld, int rows, int nq, const float* m, float* pm, float* pv, int nslab, unsigned int* cmax_bits, dsvgp_stream_t s);
int dsvgp_col_dots_f64(const double* A, const double* C, const double* B, int64_t ld, int rows, int nq, const double* m, double* pm, double* pv, int nslab, unsigned int* cmax_bits, dsvgp_stream_t s);
int dsvgp_predict_finish_f32(const float* pm, const float* pv, int nslab, int nq, int p2, const double* hyp, double pred_jitter, int add_noise, double min_var, float* mu, float* var, dsvgp_stream_t s);
int dsvgp_predict_finish_f64(const double* pm, const double* pv, int nslab, int nq, int p2, const double* hyp, double pred_jitter, int add_noise, double min_var, double* mu, double* var, dsvgp_stream_t s);

/* Gaussian expected log-likelihood summed with weight w (= 1/n') and its gradient w.r.t. mu, var
 * (gpytorch GaussianLikelihood.expected_log_prob / VariationalELBO, directional_vi.py:217,246).
 * sc[0] += sum_j term_j*w ; sc[1] += explicit d/dnoise.  ws: 2*ceil(nq/256) doubles. */
int dsvgp_elbo_terms_f32(const float* mu, const float* var, const float* y, int nq, const double* hyp, double w, double min_var, float* gmu, float* gvar, double* sc, double* ws, dsvgp_stream_t s);
int dsvgp_elbo_terms_f64(const double* mu, const double* var, const double* y, int nq, const double* hyp, double w, double min_var, double* gmu, double* gvar, double* sc, double* ws, dsvgp_stream_t s);

/* PredictiveLogLikelihood data term (mll_type="PLL", directional_vi.py:218-219; SURVEY.md section 8f rank 1):
 * sc[0] += w * sum_j log N(y_j; mu_j, var_j) and its gradient w.r.t. mu, var; `var` already holds the marginal
 * variance (noise added once per likelihood() application, i.e. twice in the reference loop -- quirk Q3).
 * sc[1] += 0 (the noise gradient flows through var).  ws: 2*ceil(nq/256) doubles. */
int dsvgp_pll_terms_f32(const float* mu, const float* var, const float* y, int nq, double w, double min_var, float* gmu, float* gvar, double* sc, double* ws, dsvgp_stream_t s);
int dsvgp_pll_terms_f64(const double* mu, const double* var, const double* y, int nq, double w, double min_var, double* gmu, double* gvar, double* sc, double* ws, dsvgp_stream_t s);

/* gsc[0..3] += {d lengthscale, d outputscale, d noise, d constant} flowing through +c and the K_xx diagonal.
 * ws: 4*296 doubles. */
int dsvgp_pred_bwd_scalars_f32(const float* gmu, const float* gvar, int nq, int p2, const double* hyp, int add_noise, double* gsc, double* ws, dsvgp_stream_t s);
int dsvgp_pred_bwd_scalars_f64(const double* gmu, const double* gvar, int nq, int p2, const double* hyp, int add_noise, double* gsc, double* ws, dsvgp_stream_t s);

/* In place C <- m gmu^T + 2 C diag(gvar) (= dL/dA); Ag <- A diag(gvar) (NULL to skip); t = A gmu.
 * tp: nslab*rows scratch.  Clo / Aglo (optional, fp32 only): TF32 'lo' companions of the new C and of Ag. */
int dsvgp_dA_f32(const float* A, float* C, float* Ag, int64_t ld, int rows, int nq, const float* m, const float* gmu, const float* gvar, float* tp, int nslab, float* t, float* Clo, float* Aglo, dsvgp_stream_t s);
int dsvgp_dA_f64(const double* A, double* C, double* Ag, int64_t ld, int rows, int nq, const double* m, const double* gmu, const double* gvar, double* tp, int nslab, double* t, double* Clo, double* Aglo, dsvgp_stream_t s);

/* KL(N(m, Ls Ls^T) || N(0, I)) with Ls = tril(raw) (_VariationalStrategy.kl_divergence, gpytorch);
 * out[0] += KL.  ws: 296 doubles. */
int dsvgp_kl_f32(const float* m, const float* Ls_raw, int64_t ld, int Mq, double* out, double* ws, dsvgp_stream_t s);
int dsvgp_kl_f64(const double* m, const double* Ls_raw, int64_t ld, int Mq, double* out, double* ws, dsvgp_stream_t s);

/* gm = t - m/num_data ; gLs = tril(2 H^T) - (tril(Ls) - diag(1/Ls_ii))/num_data  (H = Ls^T G) */
/* Every small gradient of a step in one launch: out (model dtype, nZ + nV + 4 elements) = [dZ | dV_z | d c | d raw_outputscale |
 * d raw_lengthscale | d raw_noise] from the engine's fp64 buffer small = [scalars(8) | dZ (nZ) | dV_z (nV)] and the softplus
 * derivatives hyp[4..6]; noise_mode 1: d noise = scalars[1] + scalars[6] (ELBO / PLL step), 0: scalars[6]. */
int dsvgp_collect_grads_f32(const double* small, int nZ, int nV, const double* hyp, int noise_mode, float* out, dsvgp_stream_t s);
int dsvgp_collect_grads_f64(const double* small, int nZ, int nV, const double* hyp, int noise_mode, double* out, dsvgp_stream_t s);
int dsvgp_var_grads_f32(const float* H, int64_t ldh, const float* Ls_raw, int64_t ldl, const float* t, const float* m, int Mq, double inv_num_data, float* gm, float* gLs, int64_t ldg, dsvgp_stream_t s);
int dsvgp_var_grads_f64(const double* H, int64_t ldh, const double* Ls_raw, int64_t ldl, const double* t, const double* m, int Mq, double inv_num_data, double* gm, double* gLs, int64_t ldg, dsvgp_stream_t s);

/* Measurement aid (bench.py): `ctas` CTAs of 8 warps each run `iters` rounds of 8 independent register-resident DMMA
 * m8n8k4 chains -- no memory traffic -- so that flops / elapsed time is the fp64 tensor-pipe peak of THIS device, the
 * roofline denominator of the fp64 products (Cholesky updates, Cholesky backward, every product of an fp64 model).
 * *flops_host (HOST double, optional) receives the flop count of the launch; out: device double[1] (never written). */
int dsvgp_dmma_peak_f64(int iters, int ctas, double* out, double* flops_host, dsvgp_stream_t s);

/* ---- optimiser step (SURVEY.md section 8f rank 2) ------------------------------------------------------------
 * One launch of a fused multi-tensor Adam over every tensor of an optimiser: replaces torch.optim.Adam.step() of the
 * reference's two optimisers (directional_vi.py:192-199, stepped at :251-254); arithmetic follows torch.optim.Adam
 * (amsgrad=False, maximize=False) operation by operation in the parameter dtype.
 *   desc_host  : HOST array, ntensors x 8 int64 = {param, grad, exp_avg, exp_avg_sq (device addresses), numel,
 *                group index, tri_n, 0}; tri_n > 0 marks an n x n matrix whose strictly-upper gradient is
 *                structurally zero (chol_variational_covar): only the lower triangle is visited.
 *   group_host : HOST array, ngroups (<= 4) x 8 double = {lr, beta1, beta2, eps, weight_decay, step, 0, 0}; `step` is
 *                the 1-based step count used for the bias corrections.
 * Both host arrays are consumed before the call returns. */
int dsvgp_adam_step_f32(int ntensors, const int64_t* desc_host, int ngroups, const double* group_host, dsvgp_stream_t s);
int dsvgp_adam_step_f64(int ntensors, const int64_t* desc_host, int ngroups, const double* group_host, dsvgp_stream_t s);

/* ---- input side (SURVEY.md section 8f rank 3) ------------------------------------------------------------------
 * Minibatch gather fused with select_cols_of_y (directional_vi.py:68-90, :229-241): for minibatch row i,
 * xb[i,:] = X[idx[i],:], yb[i*(p+1)+a] = Y[idx[i], cols[a]] (interleaved), V[i*p+b,:] = e_{cols[1+b]-1}.
 * X (N x d) and Y (N x ycols) are contiguous and resident on the device; idx = n int64 row indices on the device
 * (NULL = rows 0..n-1); cols_host = p+1 column indices of Y on the HOST (cols[0] is the function-value column),
 * consumed before the call returns; V may be NULL (no direction rows wanted, e.g. the derivative-free strategy). */
int dsvgp_gather_batch_f32(const float* X, const float* Y, int64_t N, int d, int ycols, const int64_t* idx, int n, int p, const int* cols_host, float* xb, float* yb, float* V, dsvgp_stream_t s);
int dsvgp_gather_batch_f64(const double* X, const double* Y, int64_t N, int d, int ycols, const int64_t* idx, int n, int p, const int* cols_host, double* xb, double* yb, double* V, dsvgp_stream_t s);

#ifdef __cplusplus
}
#endif
#endif /* DSVGP_B200_H */
