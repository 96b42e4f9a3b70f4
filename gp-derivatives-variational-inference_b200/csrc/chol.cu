// Blocked right-looking Cholesky of the jittered K_zz in fp64 plus the explicit inverse of the factor.
//
// Replaces psd_safe_cholesky(K_zz.double()) (DirectionalGradVariationalStrategy.py:72-75, cuSOLVER potrf in the
// reference) and turns both triangular solves (:181,:183) into one triangular matrix product W * K_zx with
// W = L^-1, which is what lets the whitening run as a plain tiled tensor-core GEMM.
//
// The matrix is padded with an identity block to Mp = nb0 * 2^nlev so that every level of the recursive
// inverse has uniform blocks:  for a 2x2 block-lower L = [[L11,0],[L21,L22]],
//     W = [[W11, 0], [-W22 * (L21 * W11), W22]],
// applied bottom-up; each level is two batched GEMMs.  Diagonal nb0 x nb0 blocks are factorised AND inverted
// inside one CTA in shared memory.  Status goes to a device int (0 ok, i+1 = first pivot that is not positive and finite), never to
// the host: the caller decides when to look (no hidden synchronisation).
//
// Known limitation (open): the panels are solved by multiplying with explicit inverses -- L21 = A21 W11^T across blocks
// (chol_enqueue) and A_panel D^T with D = inv(L11) on the 8x8 tiles inside a block (factor_invert_smem).  That is not
// backward stable when the diagonal block is ill-conditioned: a tiny pivot with more rows of its block after it makes
// the factor residual max|L L^T - A| / max|A| grow with cond(L11).  Measured on a B200, two adjacent rows at
// cos = 1 - 1e-10 (cond 7e10) give 2e-13 .. 5e-13 against LAPACK's 6e-16, unless the pair ends its block
// (tests/test_cholesky_gpu.py::test_adjacent_near_collinear_rows, strict xfail).  K_zz at the conditioning of trained
// states (cond <= 1e6) stays within 1.3x of LAPACK's residual.  A stable fix solves the panels by substitution (TRSM).
#include <algorithm>
#include <vector>

#include "chol.cuh"
#include "common.cuh"
#include "gemm.cuh"

namespace dsvgp {

constexpr int POTRF_THREADS = 512;
static_assert(POTRF_THREADS == 512, "potrf_inv_block: warp 0 + a named barrier of 480 threads (warps 1-15), 16 x 32 mappings");

void chol_plan(int Mq, int* Mp, int* nb0, int* nlev) {
  int k = 0;
  while (ceil_div(Mq, 1 << k) > 112) ++k;
  int b = ceil_div(Mq, 1 << k);
  b = ceil_div(b, 4) * 4;
  *Mp = b << k;
  *nb0 = b;
  *nlev = k;
}

// 1/sqrt(d) and sqrt(d) without the library sqrt + division (two long dependent sequences per pivot, 96 pivots on
// the critical path of every diagonal block): fp32 rsqrt seed (relative error e ~ 2^-21), one third-order step
// y <- y (1 + e/2 + 3e^2/8), e = 1 - d y^2 (error ~ e^3 = 2^-63), then l = d*y with one Newton correction.  Both
// results are within 1 ulp.  Only used for d inside the fp32 normal range; the caller keeps sqrt()/division outside it.
__device__ __forceinline__ void rsqrt_sqrt_f64(double d, double& rinv, double& root) {
  double y = (double)rsqrtf((float)d);
  const double e = fma(-d * y, y, 1.0);
  y = fma(y * e, fma(0.375, e, 0.5), y);
  double l = d * y;
  l = fma(fma(-l, l, d), 0.5 * y, l);
  rinv = y;
  root = l;
}

__device__ __forceinline__ void dmma884(double (&c)[2], double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c[0]), "+d"(c[1]) : "d"(a), "d"(b));
}

// 8-byte asynchronous global -> shared copy; bytes = 0 writes a zero instead (the source is not read).  The loads of a
// whole operand block are in flight together instead of one L2 round trip per loop iteration.
__device__ __forceinline__ void cp_async8(double* smem_dst, const double* gsrc, bool pred) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  const int bytes = pred ? 8 : 0;
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;\n" ::"r"(d), "l"(gsrc), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }

// Factorise the nb x nb diagonal block k and invert the factor, both inside one CTA in shared memory.
//
// Prologue (Aleft != null, i.e. k >= 1): the step-(k-1) update of THIS block is applied here instead of by separate
// panel / column-update launches, so that the chain  potrf(k-1) -> potrf(k)  is the whole critical path and the panel
// solve + trailing update of step k-1 run beside it on another stream (chol_factor_inverse):
//     Z = A[k,k-1] * W11(k-1)^T          (= L[k,k-1]; DMMA from shared memory, k-range cut by the triangle of W11)
//     A[k,k] <- A[k,k] - Z Z^T           (lower 8x8 tiles only)
// Operands are staged with a row stride of nbp+4 doubles (bank pair (4g + t) mod 16: conflict-free DMMA fragments).
//
// Factor / inverse, blocked by 8 columns so that almost all work is rank-8 updates and only 2 block barriers per 8
// columns are on the critical path:
//   factor : (A) one warp factors the 8x8 diagonal block in registers (pivots and multipliers move by shuffles),
//            (B) one thread per row solves the 8-column panel, (C) all threads apply the rank-8 trailing update.
//   inverse: block row I:  T = L[I,0:I] * W[0:I,0:I],  D = inv(L[I,I]) (one warp),  W[I,0:I] = -D * T,  W[I,I] = D.
// The block is padded to a multiple of 8 with the identity.  Writes L (upper part zeroed) and W = L^-1.
constexpr int POTRF_MAXBLK = 5;      // (nbp/8) * ceil(nbp/24) 8x24 output blocks over 16 warps, nbp <= 112

__global__ void __launch_bounds__(POTRF_THREADS)
potrf_inv_block(const double* __restrict__ A, int64_t lda, double* __restrict__ L, int64_t ldl,
                double* __restrict__ W, int64_t ldw, int nb, int* __restrict__ info, int row_offset,
                const double* __restrict__ Aleft, const double* __restrict__ Wprev) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int nbp = (nb + 7) & ~7, ld = nbp + 1, ldp = nbp + 4;
  double* R1 = reinterpret_cast<double*>(smem_raw);   // [nbp][ldp]  prologue: A[k,k-1] then Z ; afterwards Ws
  double* R2 = R1 + nbp * ldp;                        // [nbp][ldp]  prologue: W11(k-1)       ; afterwards Ls
  double* rdg = R2 + nbp * ldp;                       // [nbp] reciprocals of the diagonal of L
  double* Ls = R2;                                    // [nbp][ld]
  double* Ws = R1;                                    // [nbp][ld]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int tx = tid & 31, ty = tid >> 5;             // 32 x 16 mapping of the trailing update
  if (Aleft != nullptr) {
    for (int i = ty; i < nbp; i += 16)
      for (int c = tx; c < nbp; c += 32) {
        const bool in = i < nb && c < nb;
        cp_async8(R1 + i * ldp + c, in ? Aleft + (int64_t)i * lda + c : Aleft, in);
        cp_async8(R2 + i * ldp + c, (in && c <= i) ? Wprev + (int64_t)i * ldw + c : Wprev, in && c <= i);
      }
    cp_async_wait_all();
    __syncthreads();
    const int T = nbp >> 3, groups = (T + 2) / 3, nblocks = T * groups;
    const int g = lane >> 2, t = lane & 3;
    double acc[POTRF_MAXBLK][3][2];
#pragma unroll
    for (int b = 0; b < POTRF_MAXBLK; ++b) {            // Z = X Y^T, 8 x 24 blocks round-robin over the warps
#pragma unroll
      for (int q = 0; q < 3; ++q) acc[b][q][0] = acc[b][q][1] = 0.0;
      const int blk = warp + 16 * b;
      if (blk < nblocks) {
        const int ri = blk / groups, cg = blk % groups;
        const int kmax = 8 * min(3 * cg + 3, T);       // W11 is lower triangular: Y[j][k] = 0 for k > j
        const double* xa = R1 + (8 * ri + g) * ldp + t;
        for (int k0 = 0; k0 < kmax; k0 += 4) {
          const double a = xa[k0];
#pragma unroll
          for (int q = 0; q < 3; ++q)
            if (3 * cg + q < T) dmma884(acc[b][q], a, R2[(8 * (3 * cg + q) + g) * ldp + k0 + t]);
        }
      }
    }
    __syncthreads();                                   // X and Y are dead
    for (int i = ty; i < nbp; i += 16)                 // A[k,k] (lower) streams into the Ls region underneath the SYRK
      for (int c = tx; c < nbp; c += 32) {
        const bool in = i < nb && c <= i;
        cp_async8(Ls + i * ld + c, in ? A + (int64_t)i * lda + c : A, in);
      }
#pragma unroll
    for (int b = 0; b < POTRF_MAXBLK; ++b) {
      const int blk = warp + 16 * b;
      if (blk < nblocks) {
        const int ri = blk / groups, cg = blk % groups;
#pragma unroll
        for (int q = 0; q < 3; ++q)
          if (3 * cg + q < T) {
            double* z = R1 + (8 * ri + g) * ldp + 8 * (3 * cg + q) + 2 * t;
            z[0] = acc[b][q][0];
            z[1] = acc[b][q][1];
          }
      }
    }
    __syncthreads();
#pragma unroll
    for (int b = 0; b < POTRF_MAXBLK; ++b) {            // D = Z Z^T on the lower tiles (reuses acc)
#pragma unroll
      for (int q = 0; q < 3; ++q) acc[b][q][0] = acc[b][q][1] = 0.0;
      const int blk = warp + 16 * b;
      if (blk < nblocks) {
        const int ri = blk / groups, cg = blk % groups;
        if (3 * cg <= ri) {
          const double* za = R1 + (8 * ri + g) * ldp + t;
          for (int k0 = 0; k0 < nbp; k0 += 4) {
            const double a = za[k0];
#pragma unroll
            for (int q = 0; q < 3; ++q)
              if (3 * cg + q <= ri) dmma884(acc[b][q], a, R1[(8 * (3 * cg + q) + g) * ldp + k0 + t]);
          }
        }
      }
    }
    cp_async_wait_all();
    __syncthreads();                                   // A[k,k] has landed in Ls; Z is dead: its region becomes Ws
#pragma unroll
    for (int b = 0; b < POTRF_MAXBLK; ++b) {            // Ls = A[k,k] - D below / on the diagonal, identity on the padding
      const int blk = warp + 16 * b;
      if (blk < nblocks) {
        const int ri = blk / groups, cg = blk % groups;
#pragma unroll
        for (int q = 0; q < 3; ++q)
          if (3 * cg + q <= ri) {
            const int r = 8 * ri + g;
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              const int c = 8 * (3 * cg + q) + 2 * t + e;
              if (c <= r) Ls[r * ld + c] = (r < nb) ? Ls[r * ld + c] - acc[b][q][e] : (r == c ? 1.0 : 0.0);
            }
          }
      }
    }
    for (int i = ty; i < nbp; i += 16)
      for (int c = tx; c < nbp; c += 32) Ws[i * ld + c] = 0.0;
  } else {
    for (int i = ty; i < nbp; i += 16)
      for (int c = tx; c < nbp; c += 32) {
        const bool in = i < nb && c <= i;
        cp_async8(Ls + i * ld + c, in ? A + (int64_t)i * lda + c : A, in);
        Ws[i * ld + c] = 0.0;
      }
    cp_async_wait_all();
    __syncthreads();
    for (int i = nb + tid; i < nbp; i += POTRF_THREADS) Ls[i * ld + i] = 1.0;      // identity on the padding
  }
  // ------------------------------------------------------------------------------- factor + inverse, pipelined
  // The sequential pivot chain (A) runs on warp 0 only; instead of leaving the other 15 warps idle, block k+1's chain is
  // started as soon as its 8 columns are up to date ("thin" update), and the rest of step k's rank-8 update (C) plus the
  // inversion of block row k run beside it on warps 1-15 (their own named barrier).  Per 8 columns: thin | (A)(k+1) ||
  // (C)(k) + inverse row k | (B)(k+1), three block barriers as before, and no separate inverse phase afterwards.
  auto factor_diag = [&](int k0) {                     // (A) lanes r = lane & 7 hold row r of the diagonal block
      const int r = lane & 7;
      double a[8];
#pragma unroll
      for (int c = 0; c < 8; ++c) a[c] = Ls[(k0 + r) * ld + k0 + c];
      // Two pivots per step: with det = a11 a22 - a21^2 the second pivot is d2 = det / a11, so rsqrt(a11) and rsqrt(det)
      // are two INDEPENDENT chains (they overlap in the fp64 pipe) and 1/l22 = rsqrt(det) * l11 -- the sequential
      // pivot chain, a third of this kernel's time, has 4 links per 8x8 block instead of 8.  det has the same
      // cancellation as d2 = a22 - l21^2 (both lose log2(cond of the 2x2 block) bits).
#pragma unroll
      for (int k = 0; k < 8; k += 2) {
        const double a11 = __shfl_sync(0xffffffffu, a[k], k);
        const double a21 = __shfl_sync(0xffffffffu, a[k], k + 1);
        const double a22 = __shfl_sync(0xffffffffu, a[k + 1], k + 1);
        const double det = fma(a11, a22, -(a21 * a21));
        const bool ok1 = a11 > 0.0, ok2 = ok1 && det > 0.0;          // also false for NaN
        double l11, r1, sdet, rdet;
        if (ok2 && a11 > 1e-30 && a11 < 1e30 && det > 1e-30 && det < 1e30) {
          rsqrt_sqrt_f64(a11, r1, l11);
          rsqrt_sqrt_f64(det, rdet, sdet);
        } else if (ok2 && a11 < INFINITY && det < INFINITY) {
          l11 = sqrt(a11);
          r1 = 1.0 / l11;
          sdet = sqrt(det);
          rdet = 1.0 / sdet;
        } else {                                       // (+inf: l22 = inf, 1/l22 = 0 would pass as a factor with info 0)
          if (lane == 0) atomicCAS(info, 0, row_offset + k0 + k + ((ok1 && a11 < INFINITY) ? 2 : 1));
          l11 = r1 = sdet = rdet = nan("");
        }
        const double l21 = a21 * r1;
        const double r2 = rdet * l11;                                // 1 / l22
        const double l22 = sdet * r1;                                // sqrt(det / a11)
        if (r == k) {
          a[k] = l11;
        } else if (r == k + 1) {
          a[k] = l21;
          a[k + 1] = l22;
        } else if (r > k + 1) {
          a[k] = a[k] * r1;
          a[k + 1] = (a[k + 1] - a[k] * l21) * r2;
        }
        if (lane == k) rdg[k0 + k] = r1;
        if (lane == k + 1) rdg[k0 + k + 1] = r2;
#pragma unroll
        for (int c = k + 2; c < 8; ++c) {
          const double lck = __shfl_sync(0xffffffffu, a[k], c);
          const double lck1 = __shfl_sync(0xffffffffu, a[k + 1], c);
          if (r >= c) a[c] = fma(-a[k + 1], lck1, fma(-a[k], lck, a[c]));
        }
      }
      if (lane < 8) {
#pragma unroll
        for (int c = 0; c < 8; ++c)
          if (c <= r) Ls[(k0 + r) * ld + k0 + c] = a[c];
      }
  };
  auto panel_solve = [&](int k0) {                     // (B) rows below the diagonal block: x L11^T = a
    for (int i = k0 + 8 + tid; i < nbp; i += POTRF_THREADS) {
      double x[8];
#pragma unroll
      for (int c = 0; c < 8; ++c) x[c] = Ls[i * ld + k0 + c];
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        double sacc = x[c];
#pragma unroll
        for (int q = 0; q < c; ++q) sacc -= x[q] * Ls[(k0 + c) * ld + k0 + q];
        x[c] = sacc * rdg[k0 + c];
      }
#pragma unroll
      for (int c = 0; c < 8; ++c) Ls[i * ld + k0 + c] = x[c];
    }
  };
  __syncthreads();
  if (warp == 0) factor_diag(0);
  __syncthreads();
  panel_solve(0);
  __syncthreads();
  for (int k0 = 0; k0 < nbp; k0 += 8) {
    const int t0 = k0 + 8;
    // thin: rank-8 update of block column [t0, t0+8) only (all that (A) and (B) of the next step read)
    for (int e = tid; e < (nbp - t0) * 8; e += POTRF_THREADS) {
      const int i = t0 + (e >> 3), c = t0 + (e & 7);
      if (c <= i) {
        double sacc = Ls[i * ld + c];
#pragma unroll
        for (int q = 0; q < 8; ++q) sacc -= Ls[i * ld + k0 + q] * Ls[c * ld + k0 + q];
        Ls[i * ld + c] = sacc;
      }
    }
    __syncthreads();
    if (warp == 0) {
      if (t0 < nbp) factor_diag(t0);
    } else {
      // (C) rest of the rank-8 update of step k0: rows >= t0 + 8, columns [t0 + 8, i]
      for (int i = t0 + 8 + (warp - 1); i < nbp; i += 15) {
        double li[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) li[q] = Ls[i * ld + k0 + q];
        for (int c = t0 + 8 + lane; c <= i; c += 32) {
          double sacc = Ls[i * ld + c];
#pragma unroll
          for (int q = 0; q < 8; ++q) sacc -= li[q] * Ls[c * ld + k0 + q];
          Ls[i * ld + c] = sacc;
        }
      }
      // inverse, block row I0 = k0:  D = inv(L[I,I]),  T = L[I,0:I] * W[0:I,0:I],  W[I,0:I] = -D * T,  W[I,I] = D
      const int I0 = k0, u = tid - 32, r = u & 7;      // u: 0..479
      if (u < 8) {                                     // D: thread = column j of the 8x8 inverse
        const int j = u;
        double x[8], acc[8];                           // right-looking substitution: 8 x (mul + fma) on the critical path
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[i] = (i == j) ? 1.0 : 0.0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          x[k] = (k >= j) ? acc[k] * rdg[I0 + k] : 0.0;
#pragma unroll
          for (int i = k + 1; i < 8; ++i) acc[i] = fma(-Ls[(I0 + i) * ld + I0 + k], x[k], acc[i]);
        }
#pragma unroll
        for (int i = 0; i < 8; ++i)
          if (i >= j) Ws[(I0 + i) * ld + I0 + j] = x[i];
      }
      for (int c = u >> 3; c < I0; c += 60) {          // T[r][c] -> Ws[I0+r][c], c < I0
        double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;      // 4 independent chains (the range is a multiple of 8)
        const double* lrow = Ls + (I0 + r) * ld;
        for (int k = c & ~7; k < I0; k += 4) {
          s0 = fma(lrow[k], Ws[k * ld + c], s0);
          s1 = fma(lrow[k + 1], Ws[(k + 1) * ld + c], s1);
          s2 = fma(lrow[k + 2], Ws[(k + 2) * ld + c], s2);
          s3 = fma(lrow[k + 3], Ws[(k + 3) * ld + c], s3);
        }
        Ws[(I0 + r) * ld + c] = (s0 + s1) + (s2 + s3);
      }
      asm volatile("bar.sync 1, 480;" ::: "memory");  // warps 1-15 only: D and T complete
      for (int c0 = 0; c0 < I0; c0 += 60) {            // W[I0+r][c] = -sum_{q<=r} D[r][q] T[q][c]  (in place, per 8-lane group)
        const int c = c0 + (u >> 3);
        double t[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) t[q] = (c < I0) ? Ws[(I0 + q) * ld + c] : 0.0;
        __syncwarp();
        if (c < I0) {
          double sacc = 0.0;
#pragma unroll
          for (int q = 0; q < 8; ++q)
            if (q <= r) sacc -= Ws[(I0 + r) * ld + I0 + q] * t[q];
          Ws[(I0 + r) * ld + c] = sacc;
        }
        __syncwarp();
      }
    }
    __syncthreads();
    if (t0 < nbp) panel_solve(t0);
    __syncthreads();
  }
  __syncthreads();
  for (int i = ty; i < nb; i += 16)
    for (int c = tx; c < nb; c += 32) {
      L[(int64_t)i * ldl + c] = Ls[i * ld + c];
      W[(int64_t)i * ldw + c] = Ws[i * ld + c];
    }
}


// =====================================================================================================================
// Variant 2 of the diagonal-block chain (round 2).  ncu of variant 1 (profiles/r01_ncu_prof_potrf.txt): 142k cycles per
// block, issue slots 32 % busy, top stall = barrier -- ~39k cycles of DMMA prologue on ONE SM (two 96^3 products at that
// SM's own DMMA rate) and ~8.6k cycles per 8-column step whose long pole is scalar fp64 code fed from shared memory two
// loads per FMA (the inverse's T = L[I,0:I] W[0:I,0:I] and the rank-8 trailing update).  Here:
//   * diag_prepare (ncta CTAs, main stream, before the block kernel): CTA r forms the COLUMN slice Z[:, cols_r] of
//     Z = A[k,k-1] W11(k-1)^T and from it its share D_r = Z[:, cols_r] Z[:, cols_r]^T of the update of the diagonal block
//     (splitting the SYRK along its contraction index needs no exchange between CTAs); partials go to dead upper blocks of
//     the work matrix and the block kernel starts from A[k,k] - sum_r D_r;
//   * potrf_inv_block2: every bulk operation of the factorisation and of the inversion is an 8x8 DMMA tile product on
//     fragments with a row stride of nbp + 4 doubles (conflict-free): panel = A_panel D^T with D = inv(L11) (8x8, from
//     warp 0 right after the pivot chain) instead of a per-row substitution, thin and trailing rank-8 updates, the
//     inverse's block row T and -D T.  Warp 0 runs the sequential 8x8 pivot chain of block column j+1 while warps 1-15 do
//     the trailing update of step j and the inverse block row j.
constexpr int PREP_MAXC = 4;        // CTAs of diag_prepare = partial sums the block kernel adds up

struct PrepParts { double* p[PREP_MAXC]; };

__global__ void __launch_bounds__(POTRF_THREADS)
diag_prepare(const double* __restrict__ Aleft, int64_t lda, const double* __restrict__ Wprev, int64_t ldw, int nb,
             PrepParts parts, int64_t ldd, int ncta) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int nbp = (nb + 7) & ~7, ldp = nbp + 4, T = nbp >> 3;
  const int tcs = (T + ncta - 1) / ncta;                       // tile columns per CTA
  const int c0 = blockIdx.x * tcs, c1 = min(T, c0 + tcs), nc = max(c1 - c0, 0);
  const int ldz = 8 * tcs + 4;
  double* X = reinterpret_cast<double*>(smem_raw);             // [nbp][ldp]   A[k,k-1]
  double* Y = X + nbp * ldp;                                   // [8 tcs][ldp] rows 8 c0 .. 8 c1 of W11(k-1)
  double* Zs = Y + 8 * tcs * ldp;                              // [nbp][ldz]   Z[:, 8 c0 .. 8 c1)
  double* Dp = parts.p[blockIdx.x];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
  const int kmax_all = 8 * c1;                                 // W11 lower: column j of Z needs k <= j only
  for (int e = tid; e < nbp * (kmax_all >> 1); e += POTRF_THREADS) {        // 16-byte chunks
    const int i = e / (kmax_all >> 1), c = 2 * (e - i * (kmax_all >> 1));
    const bool in = i < nb && c + 1 < nb;
    if (in) {
      const uint32_t d = (uint32_t)__cvta_generic_to_shared(X + i * ldp + c);
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(Aleft + (int64_t)i * lda + c) : "memory");
    } else {
      X[i * ldp + c] = (i < nb && c < nb) ? Aleft[(int64_t)i * lda + c] : 0.0;
      X[i * ldp + c + 1] = 0.0;
    }
  }
  for (int e = tid; e < 8 * nc * kmax_all; e += POTRF_THREADS) {
    const int r = e / kmax_all, c = e - r * kmax_all, j = 8 * c0 + r;
    const bool in = j < nb && c <= j;
    cp_async8(Y + r * ldp + c, in ? Wprev + (int64_t)j * ldw + c : Wprev, in);
  }
  cp_async_wait_all();
  __syncthreads();
  // Z slice: 8 x (8 nc) output strips, one per (tile row, warp), up to PREP tile columns wide (nc <= 4 accumulators)
  for (int ti = warp; ti < T; ti += POTRF_THREADS / 32) {
    double acc[4][2];
#pragma unroll
    for (int q = 0; q < 4; ++q) acc[q][0] = acc[q][1] = 0.0;
    const double* xa = X + (8 * ti + g) * ldp + t;
    for (int k0 = 0; k0 < kmax_all; k0 += 4) {
      const double a = xa[k0];
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (q < nc && k0 < 8 * (c0 + q + 1)) dmma884(acc[q], a, Y[(8 * q + g) * ldp + k0 + t]);
    }
#pragma unroll
    for (int q = 0; q < 4; ++q)
      if (q < nc) {
        double* z = Zs + (8 * ti + g) * ldz + 8 * q + 2 * t;
        z[0] = acc[q][0];
        z[1] = acc[q][1];
      }
  }
  __syncthreads();
  // D_r = Zs Zs^T on the lower tiles (contraction over this CTA's 8 nc columns only)
  const int groups = (T + 2) / 3, nblocks = T * groups;
  for (int blk = warp; blk < nblocks; blk += POTRF_THREADS / 32) {
    const int ri = blk / groups, cg = blk % groups;
    if (3 * cg > ri) continue;
    double acc[3][2];
#pragma unroll
    for (int q = 0; q < 3; ++q) acc[q][0] = acc[q][1] = 0.0;
    const double* za = Zs + (8 * ri + g) * ldz + t;
    for (int k0 = 0; k0 < 8 * nc; k0 += 4) {
      const double a = za[k0];
#pragma unroll
      for (int q = 0; q < 3; ++q)
        if (3 * cg + q <= ri) dmma884(acc[q], a, Zs[(8 * (3 * cg + q) + g) * ldz + k0 + t]);
    }
#pragma unroll
    for (int q = 0; q < 3; ++q)
      if (3 * cg + q <= ri) {
        const int r = 8 * ri + g, c = 8 * (3 * cg + q) + 2 * t;
        if (r < nb) {
          if (c < nb) Dp[(int64_t)r * ldd + c] = acc[q][0];
          if (c + 1 < nb) Dp[(int64_t)r * ldd + c + 1] = acc[q][1];
        }
      }
  }
}

#ifndef POTRF_S0_IDLE
#define POTRF_S0_IDLE 1     // 1: warps 4, 8, 12 (warp 0's scheduler) take no leftover work during the pivot phase
#endif
template <int V> struct IntTag { static constexpr int value = V; };
__device__ long long* g_potrf_dbg = nullptr;     // profiling aid: clock64() at the phase boundaries of one block kernel
#define DBG_T(slot) do { if (dbg != nullptr && tid == 0) dbg[slot] = clock64(); } while (0)

// Factorise the nbp x nbp block held in shared memory (Ls, row stride ld) and invert the factor (Ws): the body shared by
// the single-CTA block kernel (variant 2) and the cluster kernel (variant 3).  Ends with L and W written to global memory.
__device__ __forceinline__ void factor_invert_smem(double* __restrict__ Ls, double* __restrict__ Ws, const int ld, const int nbp,
                                                   const int nb, int* __restrict__ info, const int row_offset,
                                                   double* __restrict__ L, const int64_t ldl, double* __restrict__ W,
                                                   const int64_t ldw, long long* dbg) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3, T = nbp >> 3;
  // The 8x8 diagonal block, entirely in registers and redundantly in every lane of warp 0: no shuffles, no shared-memory
  // round trips inside the sequential pivot chain (measured: the shuffle-based version + the 8x8 inverse through shared memory
  // took 4.0k cycles per 8 columns = 49k of the 65k cycles between the first and the last barrier of this kernel).
  // Two pivots per link (det = a11 a22 - a21^2: rsqrt(a11) and rsqrt(det) are independent chains), then D = inv(L11) by a
  // right-looking substitution on the registers, lane j < 8 doing column j.  L11 -> Ls, D -> diagonal block of Ws.
  auto factor_diag = [&](int k0) {
    double a[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int c = 0; c <= i; ++c) a[i][c] = Ls[(k0 + i) * ld + k0 + c];
    double rd[8];
#pragma unroll
    for (int k = 0; k < 8; k += 2) {
      const double a11 = a[k][k], a21 = a[k + 1][k], a22 = a[k + 1][k + 1];
      const double det = fma(a11, a22, -(a21 * a21));
      const bool ok1 = a11 > 0.0, ok2 = ok1 && det > 0.0;          // also false for NaN
      double l11, r1, sdet, rdet;
      if (ok2 && a11 > 1e-30 && a11 < 1e30 && det > 1e-30 && det < 1e30) {
        rsqrt_sqrt_f64(a11, r1, l11);
        rsqrt_sqrt_f64(det, rdet, sdet);
      } else if (ok2 && a11 < INFINITY && det < INFINITY) {
        l11 = sqrt(a11);
        r1 = 1.0 / l11;
        sdet = sqrt(det);
        rdet = 1.0 / sdet;
      } else {                                           // (+inf: l22 = inf, 1/l22 = 0 would pass as a factor with info 0)
        if (lane == 0) atomicCAS(info, 0, row_offset + k0 + k + ((ok1 && a11 < INFINITY) ? 2 : 1));
        l11 = r1 = sdet = rdet = nan("");
      }
      const double l21 = a21 * r1;
      const double r2 = rdet * l11;                                // 1 / l22
      a[k][k] = l11;
      a[k + 1][k] = l21;
      a[k + 1][k + 1] = sdet * r1;                                 // sqrt(det / a11)
      rd[k] = r1;
      rd[k + 1] = r2;
#pragma unroll
      for (int i = k + 2; i < 8; ++i) {
        a[i][k] *= r1;
        a[i][k + 1] = (a[i][k + 1] - a[i][k] * l21) * r2;
      }
#pragma unroll
      for (int i = k + 2; i < 8; ++i)
#pragma unroll
        for (int c = k + 2; c <= i; ++c) a[i][c] = fma(-a[i][k + 1], a[c][k + 1], fma(-a[i][k], a[c][k], a[i][c]));
    }
    // D = inv(L11), column j on lane j (lanes >= 8 compute a copy of column lane & 7 and do not store)
    const int j = lane & 7;
    double x[8], acc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = (i == j) ? 1.0 : 0.0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      x[k] = (k >= j) ? acc[k] * rd[k] : 0.0;
#pragma unroll
      for (int i = k + 1; i < 8; ++i) acc[i] = fma(-a[i][k], x[k], acc[i]);
    }
    __syncwarp();                                         // all 32 lanes have read the block before 8 of them overwrite it
    if (lane < 8) {
#pragma unroll
      for (int i = 0; i < 8; ++i) Ws[(k0 + i) * ld + k0 + j] = x[i];       // (x[i] = 0 above the diagonal)
    }
    // L11: every lane holds the whole block, so ONE lane writes it, two entries per 16-byte store (rows are 16-byte aligned:
    // ld and k0 are even).  "lane c writes column c" compiled to 64 compare-and-branch sequences, whose branch-resolution stalls
    // were 60 % of this warp's samples in the pivot chain (ncu source page, --warp-sampling-interval 0).
    if (lane == 8) {
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int c = 0; c < 8; c += 2)
          *reinterpret_cast<double2*>(Ls + (k0 + i) * ld + k0 + c) =
              make_double2((c <= i) ? a[i][c] : 0.0, (c + 1 <= i) ? a[i][c + 1] : 0.0);
    }
  };
  // one tile of the inverse's block row jp: Tt = L[jp, tc..jp) W[tc..jp, tc] on two independent accumulators (half the
  // dependent-DMMA chain), then W[jp, tc] = -D_jp Tt through the warp's own 8x8 patch of Ws
  auto inverse_tile = [&](int jp, int tc) {
    const int kp = 8 * jp;
    double acc0[2] = {0.0, 0.0}, acc1[2] = {0.0, 0.0};
    const double* la = Ls + (kp + g) * ld + t;
    int kk = 8 * tc;
    for (; kk + 4 < kp; kk += 8) {
      dmma884(acc0, la[kk], Ws[(kk + t) * ld + 8 * tc + g]);
      dmma884(acc1, la[kk + 4], Ws[(kk + 4 + t) * ld + 8 * tc + g]);
    }
    if (kk < kp) dmma884(acc0, la[kk], Ws[(kk + t) * ld + 8 * tc + g]);
    double* wt = Ws + (kp + g) * ld + 8 * tc + 2 * t;
    wt[0] = acc0[0] + acc1[0];
    wt[1] = acc0[1] + acc1[1];
    __syncwarp();
    double out[2] = {0.0, 0.0};
#pragma unroll
    for (int s = 0; s < 2; ++s)
      dmma884(out, -Ws[(kp + g) * ld + kp + 4 * s + t], Ws[(kp + 4 * s + t) * ld + 8 * tc + g]);
    __syncwarp();
    wt[0] = out[0];
    wt[1] = out[1];
  };
  DBG_T(0);
  __syncthreads();
  DBG_T(1);
  for (int j = 0; j < T; ++j) {
    const int k0 = 8 * j;
    // ---- S1: pivot chain + 8x8 inverse of block column j (warp 0)  ||  leftovers of step j-1 (warps 1-15)
    if (warp == 0) {
      factor_diag(k0);
      DBG_T(2 + 4 * j);
    } else if ((POTRF_S0_IDLE ? (warp & 3) != 0 : true) && j > 0) {
      // (warps 4, 8, 12 share warp 0's scheduler and with it the fp64 pipe: their DMMAs, 16 pipe cycles each, were what the pivot
      //  chain's dependent DFMAs waited for -- the chain took 4.3k cycles per 8 columns against ~2k alone.  They sit this phase out.)
      const int jp = j - 1, kp = 8 * jp;               // previous step: panel jp is final, D_jp sits in Ws[jp,jp]
      // items: [0, jp)  inverse block row jp, tile column tc (longest chains first);
      //        [jp, jp + ntr)  trailing tiles (ti >= tj >= j + 1)
      const int nt = T - (j + 1), ntr = nt * (nt + 1) / 2, nitems = jp + ntr;
      constexpr int NWORK = POTRF_S0_IDLE ? (POTRF_THREADS / 32 / 4) * 3 : POTRF_THREADS / 32 - 1;
      for (int it = POTRF_S0_IDLE ? (warp >> 2) * 3 + (warp & 3) - 1 : warp - 1; it < nitems; it += NWORK) {
        if (it < jp) {
          inverse_tile(jp, it);
        } else {
          int q = it - jp, ti = 0;                       // q-th lower tile of the trailing nt x nt tile triangle
          while (q > ti) { q -= ti + 1; ++ti; }
          const int tj = q;
          const int ri = 8 * (j + 1 + ti), rj = 8 * (j + 1 + tj);
          double acc[2] = {0.0, 0.0};
#pragma unroll
          for (int s = 0; s < 2; ++s) dmma884(acc, Ls[(ri + g) * ld + kp + 4 * s + t], Ls[(rj + g) * ld + kp + 4 * s + t]);
          double* c = Ls + (ri + g) * ld + rj + 2 * t;
          c[0] -= acc[0];
          c[1] -= acc[1];
        }
      }
    }
    __syncthreads();
    DBG_T(3 + 4 * j);
    if (j + 1 < T) {
      // ---- S2: panel j = (rows below the diagonal block, columns of block j) * D_j^T, one 8x8 tile per warp
      for (int ti = j + 1 + warp; ti < T; ti += POTRF_THREADS / 32) {
        double* pa = Ls + (8 * ti + g) * ld + k0;
        const double a0 = pa[t], a1 = pa[4 + t];
        double acc[2] = {0.0, 0.0};
        dmma884(acc, a0, Ws[(k0 + g) * ld + k0 + t]);
        dmma884(acc, a1, Ws[(k0 + g) * ld + k0 + 4 + t]);
        __syncwarp();                                     // every lane's fragment loads of this tile precede the in-place stores
        pa[2 * t] = acc[0];
        pa[2 * t + 1] = acc[1];
      }
      __syncthreads();
      DBG_T(4 + 4 * j);
      // ---- S3: thin update of block column j+1 (all that the next pivot chain and the next panel read)
      const int t0 = k0 + 8;
      for (int ti = j + 1 + warp; ti < T; ti += POTRF_THREADS / 32) {
        double acc[2] = {0.0, 0.0};
#pragma unroll
        for (int s = 0; s < 2; ++s) dmma884(acc, Ls[(8 * ti + g) * ld + k0 + 4 * s + t], Ls[(t0 + g) * ld + k0 + 4 * s + t]);
        double* c = Ls + (8 * ti + g) * ld + t0 + 2 * t;
        c[0] -= acc[0];
        c[1] -= acc[1];
      }
      __syncthreads();
      DBG_T(5 + 4 * j);
    }
  }
  // inverse block row T-1 (all warps; the trailing triangle of the last step is empty)
  for (int tc = warp; tc < T - 1; tc += POTRF_THREADS / 32) inverse_tile(T - 1, tc);
  __syncthreads();
  DBG_T(62);
  for (int i = warp; i < nb; i += POTRF_THREADS / 32)
    for (int c = lane; c < nb; c += 32) {
      const bool low = c <= i;
      L[(int64_t)i * ldl + c] = low ? Ls[i * ld + c] : 0.0;
      W[(int64_t)i * ldw + c] = low ? Ws[i * ld + c] : 0.0;
    }
  DBG_T(63);
}

__global__ void __launch_bounds__(POTRF_THREADS)
potrf_inv_block2(const double* __restrict__ A, int64_t lda, double* __restrict__ L, int64_t ldl,
                 double* __restrict__ W, int64_t ldw, int nb, int* __restrict__ info, int row_offset,
                 PrepParts parts, int64_t ldd, int nparts) {
  long long* dbg = (row_offset == 0) ? nullptr : g_potrf_dbg;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int nbp = (nb + 7) & ~7, ld = nbp + 4, T = nbp >> 3;
  double* Ls = reinterpret_cast<double*>(smem_raw);   // [nbp][ld]
  double* Ws = Ls + nbp * ld;                         // [nbp][ld]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
  DBG_T(61);
  // ---- start: Ls = A[k,k] - sum_r D_r (lower), identity on the padding; Ws = 0.
  // (measured, round 2: one element at a time with its five dependent-latency loads cost 27k of this kernel's 93k cycles.
  // A warp owns rows warp, warp+16, ..; lanes own columns lane, lane+32, lane+64, lane+96; all loads of two rows -- up to
  // 2 x 4 x 5 -- are in flight together.)
  for (int e = tid; e < nbp * ld; e += POTRF_THREADS) Ws[e] = 0.0;
  for (int i0 = warp; i0 < nbp; i0 += 2 * (POTRF_THREADS / 32)) {
    double v[2][4];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int i = i0 + u * (POTRF_THREADS / 32);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int c = lane + 32 * q;
        v[u][q] = (i < nb && c <= i) ? A[(int64_t)i * lda + c] : ((i < nbp && i == c) ? 1.0 : 0.0);
      }
    }
    for (int r = 0; r < nparts; r += 2) {             // two partial sums per round: 16 more loads in flight
      const double* pr0 = parts.p[r];
      const double* pr1 = parts.p[r + 1 < nparts ? r + 1 : r];
      const bool two = r + 1 < nparts;
      double w0[2][4], w1[2][4];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int i = i0 + u * (POTRF_THREADS / 32);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int c = lane + 32 * q;
          const bool in = i < nb && c <= i;
          w0[u][q] = in ? pr0[(int64_t)i * ldd + c] : 0.0;
          w1[u][q] = (in && two) ? pr1[(int64_t)i * ldd + c] : 0.0;
        }
      }
#pragma unroll
      for (int u = 0; u < 2; ++u)
#pragma unroll
        for (int q = 0; q < 4; ++q) v[u][q] = (v[u][q] - w0[u][q]) - w1[u][q];
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int i = i0 + u * (POTRF_THREADS / 32);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int c = lane + 32 * q;
        if (i < nbp && c < nbp) Ls[i * ld + c] = v[u][q];
      }
    }
  }
  factor_invert_smem(Ls, Ws, ld, nbp, nb, info, row_offset, L, ldl, W, ldw, dbg);
}

// ---------------------------------------------------------------------------------------------------------------------
// Variant 3: diag_prepare and the block kernel as ONE launch of a 4-CTA thread-block cluster.  CTA r forms its column slice
// of Z = A[k,k-1] W11(k-1)^T and its partial update D_r = Z_r Z_r^T in its OWN shared memory; after a cluster barrier CTA 0
// gathers  A[k,k] - D_0 - D_1 - D_2 - D_3  straight from the four shared memories (distributed shared memory,
// ld.shared::cluster) and factorises; CTAs 1-3 leave after a second barrier.  Against variant 2 this drops a launch gap
// and the round trip of the partial sums through global memory (9 dependent L2 round trips, ~10k cycles per block).
__device__ __forceinline__ uint32_t cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_barrier() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ double ld_dsmem_f64(const double* local_ptr, uint32_t rank) {
  const uint32_t a = (uint32_t)__cvta_generic_to_shared(local_ptr);
  uint32_t ra;
  double v;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(a), "r"(rank));
  asm volatile("ld.shared::cluster.f64 %0, [%1];" : "=d"(v) : "r"(ra) : "memory");
  return v;
}

constexpr int CL = 4;               // cluster size = column slices of Z

__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(POTRF_THREADS)
potrf_cluster(const double* __restrict__ A, int64_t lda, double* __restrict__ L, int64_t ldl, double* __restrict__ W,
              int64_t ldw, int nb, int* __restrict__ info, int row_offset, const double* __restrict__ Aleft,
              const double* __restrict__ Wprev) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int nbp = (nb + 7) & ~7, ld = nbp + 4, T = nbp >> 3;
  const int tcs = (T + CL - 1) / CL, ldz = 8 * tcs + 4;
  // two regions of nbp x ld doubles:  R0 = X = A[k,k-1]  ->  D_r (lower tiles; X is dead once Z is formed)  ->  Ls (in place)
  //                                    R1 = Y (rows of W11(k-1)) + Zs (column slice of Z)  ->  Ws
  double* R0 = reinterpret_cast<double*>(smem_raw);
  double* R1 = R0 + nbp * ld;
  double* R2 = R0;                                     // D_r
  double* Y = R1;                                      // [8 tcs][ld]
  double* Zs = Y + 8 * tcs * ld;                       // [nbp][ldz]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
  const uint32_t rank = cluster_rank();
  long long* dbg = (row_offset == 0 || rank != 0) ? nullptr : g_potrf_dbg;
  DBG_T(61);
  const bool upd = Aleft != nullptr;
  if (upd) {
    // tile columns of this CTA, dealt out boustrophedon (0 1 2 3 3 2 1 0 0 1 ..): column j of Z needs k <= j only (W11 is
    // lower triangular), so contiguous slices would give the last CTA 5x the work of the first (measured: 6.3k cycles of
    // the leader waiting at the cluster barrier)
    int tcol[4] = {0, 0, 0, 0}, nc = 0;
    for (int c = 0; c < T; ++c) {
      const int rnd = c / CL, pos = c % CL;
      if ((uint32_t)((rnd & 1) ? CL - 1 - pos : pos) == rank && nc < 4) tcol[nc++] = c;
    }
    const int kmax_all = nc > 0 ? 8 * (tcol[nc - 1] + 1) : 0;
    if (nc > 0) {
      // (a warp per row, lanes along the row: no per-element division -- the index arithmetic of the flat loops was most of
      //  this phase's 5k cycles)
      for (int i = warp; i < nbp; i += POTRF_THREADS / 32)                       // X = A[k,k-1], 16-byte chunks
        for (int c = 2 * lane; c < kmax_all; c += 64) {
          if (i < nb && c + 1 < nb) {
            const uint32_t d = (uint32_t)__cvta_generic_to_shared(R0 + i * ld + c);
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(Aleft + (int64_t)i * lda + c) : "memory");
          } else {
            R0[i * ld + c] = (i < nb && c < nb) ? Aleft[(int64_t)i * lda + c] : 0.0;
            R0[i * ld + c + 1] = 0.0;
          }
        }
      for (int r = warp; r < 8 * nc; r += POTRF_THREADS / 32) {                  // Y = this CTA's rows of W11(k-1)
        const int j = 8 * tcol[r >> 3] + (r & 7);
        for (int c = lane; c < kmax_all; c += 32) {
          const bool in = j < nb && c <= j;
          cp_async8(Y + r * ld + c, in ? Wprev + (int64_t)j * ldw + c : Wprev, in);
        }
      }
    }
    cp_async_wait_all();
    __syncthreads();
    DBG_T(52);
    // Z slice: 8 x (8 nc) strips.  No conditions inside the k loops of this prologue: with `if (k0 < 8 (tcol[q] + 1)) dmma` /
    // `if (3 cg + q <= ri) dmma` each DMMA sat behind its own branch and its operand load behind that -- load latency + DMMA
    // latency serialised per accumulator (4.3k + 5.6k cycles for the two phases).  Y is zero beyond the triangle (zero-filled
    // above); the accumulator count is a compile-time constant per call and the k range is cut per SEGMENT, outside the loops.
    auto z_strips = [&](auto nc_tag) {
      constexpr int NC = decltype(nc_tag)::value;
      for (int ti = warp; ti < T; ti += POTRF_THREADS / 32) {
        double acc[NC][2];
#pragma unroll
        for (int q = 0; q < NC; ++q) acc[q][0] = acc[q][1] = 0.0;
        const double* xa = R0 + (8 * ti + g) * ld + t;
        const double* yb = Y + g * ld + t;
        // column q of this CTA needs k < 8 (tcol[q] + 1) only (W11 is lower triangular; tcol ascending): segment s of the k range
        // feeds accumulators s .. NC-1 -- half the DMMAs of the full range, and this phase is bound by the SM's DMMA pipe
        int k0 = 0;
#pragma unroll
        for (int sgm = 0; sgm < NC; ++sgm) {
          const int kend = 8 * (tcol[sgm] + 1);
#pragma unroll 2
          for (; k0 < kend; k0 += 4) {
            const double a = xa[k0];
#pragma unroll
            for (int q = sgm; q < NC; ++q) dmma884(acc[q], a, yb[8 * q * ld + k0]);
          }
        }
#pragma unroll
        for (int q = 0; q < NC; ++q) {
          double* z = Zs + (8 * ti + g) * ldz + 8 * q + 2 * t;
          z[0] = acc[q][0];
          z[1] = acc[q][1];
        }
      }
    };
    if (nc == 3) z_strips(IntTag<3>{});
    else if (nc == 4) z_strips(IntTag<4>{});
    else if (nc == 2) z_strips(IntTag<2>{});
    else if (nc == 1) z_strips(IntTag<1>{});
    __syncthreads();
    DBG_T(53);
    // D_r = Zs Zs^T on the lower tiles (contraction over this CTA's 8 nc columns), into R2 = R0 (X is dead).  Only the
    // blocks (tile row ri, group of 3 tile columns cg <= ri / 3) that touch the lower triangle are dealt out.
    auto syrk_block = [&](auto nq_tag, int ri, int cg) {
      constexpr int NQ = decltype(nq_tag)::value;
      double acc[NQ][2];
#pragma unroll
      for (int q = 0; q < NQ; ++q) acc[q][0] = acc[q][1] = 0.0;
      const double* za = Zs + (8 * ri + g) * ldz + t;
      const double* zb = Zs + (8 * 3 * cg + g) * ldz + t;
#pragma unroll 2
      for (int k0 = 0; k0 < 8 * nc; k0 += 4) {
        const double a = za[k0];
#pragma unroll
        for (int q = 0; q < NQ; ++q) dmma884(acc[q], a, zb[8 * q * ldz + k0]);
      }
#pragma unroll
      for (int q = 0; q < NQ; ++q) {
        double* dd = R2 + (8 * ri + g) * ld + 8 * (3 * cg + q) + 2 * t;
        dd[0] = acc[q][0];
        dd[1] = acc[q][1];
      }
    };
    int idx = 0;
    for (int ri = 0; ri < T; ++ri)
      for (int cg = 0; 3 * cg <= ri; ++cg, ++idx) {
        if ((idx & 15) != warp) continue;
        const int nq = min(3, ri - 3 * cg + 1);
        if (nq == 3) syrk_block(IntTag<3>{}, ri, cg);
        else if (nq == 2) syrk_block(IntTag<2>{}, ri, cg);
        else syrk_block(IntTag<1>{}, ri, cg);
      }
  }
  DBG_T(54);
  cluster_barrier();                                   // every partial is in place (release / acquire at cluster scope)
  DBG_T(55);
  // A[k,k] - D_0 - D_1 - D_2 - D_3 on the lower triangle (identity on the padding), rows dealt out round-robin over the
  // four CTAs (each reads one local and three remote partials -- the leader alone took 9.8k cycles for it), written into
  // the LEADER's second region (Y / Zs are dead everywhere), which becomes Ls.
  {
    const uint32_t r1a = (uint32_t)__cvta_generic_to_shared(R1);
    uint32_t r1lead;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r1lead) : "r"(r1a), "r"(0u));
    const int rows_cta = (nbp - (int)rank + CL - 1) / CL;                      // rows rank, rank + 4, ..
    for (int m0 = warp; m0 < rows_cta; m0 += 2 * (POTRF_THREADS / 32)) {
      double v[2][4];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int m = m0 + u * (POTRF_THREADS / 32), i = (int)rank + CL * m;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int c = lane + 32 * q;
          const bool in = m < rows_cta && i < nb && c <= i;
          double a = in ? A[(int64_t)i * lda + c] : ((m < rows_cta && i == c) ? 1.0 : 0.0);
          if (in && upd) {
            const double* dp = R2 + i * ld + c;
            const double d0 = ld_dsmem_f64(dp, 0), d1 = ld_dsmem_f64(dp, 1), d2 = ld_dsmem_f64(dp, 2), d3 = ld_dsmem_f64(dp, 3);
            a = (((a - d0) - d1) - d2) - d3;
          }
          v[u][q] = a;
        }
      }
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int m = m0 + u * (POTRF_THREADS / 32), i = (int)rank + CL * m;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int c = lane + 32 * q;
          if (m < rows_cta && i < nbp && c <= i) {
            const uint32_t dst = r1lead + (uint32_t)((i * ld + c) * sizeof(double));
            asm volatile("st.shared::cluster.f64 [%0], %1;" ::"r"(dst), "d"(v[u][q]) : "memory");
          }
        }
      }
    }
  }
  DBG_T(56);
  cluster_barrier();                                   // the leader's Ls is complete; nobody reads a partial any more
  DBG_T(57);
  if (rank != 0) return;
  for (int e = tid; e < nbp * ld; e += POTRF_THREADS) R0[e] = 0.0;              // D_0 is dead: its region becomes Ws
  factor_invert_smem(R1, R0, ld, nbp, nb, info, row_offset, L, ldl, W, ldw, dbg);
}

void set_potrf_debug(long long* p) { cudaMemcpyToSymbol(g_potrf_dbg, &p, sizeof(p)); }

static int g_chol_variant = 3;
void set_chol_variant(int v) { g_chol_variant = (v >= 1 && v <= 3) ? v : 3; }
int get_chol_variant() { return g_chol_variant; }
static int g_chol_lookahead = 0;  // 1: trailing update split into the part the next two links need (side stream) and the bulk (own stream);
                                  // measured: no gain (C3 step 11.43 -> 11.46 ms, A/B in one process) -- off
void set_chol_lookahead(int on) { g_chol_lookahead = on ? 1 : 0; }
int get_chol_lookahead() { return g_chol_lookahead; }
static int g_chol_mid_link = 20;  // chol_wait_mid(): the diagonal block whose completion releases work the caller deferred (see there); < 0: none
void set_chol_mid_link(int k) { g_chol_mid_link = k; }
int get_chol_mid_link() { return g_chol_mid_link; }
static int g_chol_inv_streams = 3; // eager inverse: 3 = one stream per level of the recursive doubling (default), 2 = T products on a second stream, 1 = one stream
void set_chol_inv_streams(int n) { g_chol_inv_streams = n >= 3 ? 3 : (n == 2 ? 2 : 1); }
int get_chol_inv_streams() { return g_chol_inv_streams; }
static int g_chol_priority = 0;   // 1: the three chains of the factorisation on the library's high-priority streams; 0: diagonal chain on the caller's
                                  // stream (measured: no difference on any workload -- off)
void set_chol_priority(int on) { g_chol_priority = on ? 1 : 0; }
int get_chol_priority() { return g_chol_priority; }

struct SideCtx { cudaStream_t diag = nullptr, side = nullptr, inv = nullptr, inv2 = nullptr, bulk = nullptr, lvl[8] = {}; cudaEvent_t ev_lvl[8], ev_main[64], ev_side[64], ev_panel[64], ev_bulk[64], ev_T[8], ev_inv, ev_inv2, ev_pre, ev_entry, ev_done, ev_mid; bool ready = false, mid_valid = false; };
static SideCtx g_side_ctxs[16];                         // one set of side streams + event pool per device

// The first links of the chain are throughput-bound (their rank-nb0 trailing updates fill the GPU: potrf(k+2) waits for update(k)),
// the later ones latency-bound (most SMs idle).  Work a caller overlaps with the factorisation on another stream therefore only
// costs nothing when it runs beside the LATER links: chol_wait_mid makes stream s wait for diagonal block g_chol_mid_link of the
// factorisation enqueued last on this device (no-op when that call had fewer blocks, or the knob is negative).
int chol_wait_mid(cudaStream_t s) {
  int dev = 0;
  cudaGetDevice(&dev);
  SideCtx& sc = g_side_ctxs[dev & 15];
  if (sc.ready && sc.mid_valid) cudaStreamWaitEvent(s, sc.ev_mid, 0);
  return DSVGP_OK;
}

static thread_local bool tl_own_capture = false;       // chol_enqueue runs inside the capture of the factorisation's own graph

static int chol_enqueue(double* Awork, int64_t lda, double* L, int64_t ldl, double* W, int64_t ldw, int Mp, int nb0,
                        int nlev, int* info, cudaStream_t st) {
  if (Mp <= 0) return DSVGP_OK;
  if (!Awork || !L || !W || !info || nb0 <= 0 || nb0 > 112 || (nb0 << nlev) != Mp) return DSVGP_ERR_ARG;
  // diag_prepare and potrf_cluster read A[k,k-1] two doubles at a time: 16-byte cp.async at Aleft + i lda + c with c even and
  // Aleft = Awork + k nb0 lda + (k-1) nb0.  That address is 16-byte aligned for every block k and row i exactly when Awork is
  // 16-byte aligned, lda is even and, once there is more than one block, nb0 is even (chol_plan's nb0 is a multiple of 4).
  // Every other global access of the factorisation, the inverse and their GEMMs is 8 bytes wide or checks its own alignment.
  if ((lda & 1) != 0 || ((uintptr_t)Awork & 15) != 0 || (nlev > 0 && (nb0 & 1) != 0)) return DSVGP_ERR_ARG;
  const int nblk = 1 << nlev;
  const int nbp = (nb0 + 7) & ~7;
  if ((nbp >> 3) * (((nbp >> 3) + 2) / 3) > 16 * POTRF_MAXBLK) return DSVGP_ERR_ARG;
  const size_t smem = sizeof(double) * (size_t)(2 * nbp * (nbp + 4) + nbp);
  const bool v3 = g_chol_variant == 3 && nblk >= 2;     // cluster kernel: no scratch in global memory at all
  const bool v2 = g_chol_variant == 2 && nblk >= 4;    // (one or two blocks: nothing to gain, and only one dead block to hold partials)
  // variant 2: partial sums of the diagonal-block update live in dead blocks of the work matrix above its diagonal
  // (the factorisation only touches the lower triangle; the inverse's scratch is below it too)
  PrepParts parts{};
  int nparts = 0;
  if (v2) {
    if (nblk >= 5) {
      for (int r = 0; r < 4; ++r) parts.p[nparts++] = Awork + (int64_t)(r + 1) * nb0;             // blocks (0,1) .. (0,4)
    } else {
      for (int r = 0; r < 3; ++r) parts.p[nparts++] = Awork + (int64_t)(r + 1) * nb0;             // (0,1) (0,2) (0,3)
      parts.p[nparts++] = Awork + (int64_t)nb0 * lda + 2 * nb0;                                    // (1,2)
    }
    const int T = nbp >> 3;
    if (nparts > T) nparts = T;
  }
  const int tcs = nparts ? ((nbp >> 3) + nparts - 1) / nparts : 0;
  const size_t smem_prep = sizeof(double) * (size_t)(nbp * (nbp + 4) + 8 * tcs * (nbp + 4) + nbp * (8 * tcs + 4));
  if (smem > 48 * 1024) {
    cudaFuncSetAttribute(potrf_inv_block, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    cudaFuncSetAttribute(potrf_inv_block2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  }
  if (smem_prep > 48 * 1024) cudaFuncSetAttribute(diag_prepare, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_prep);
  const int tcs_cl = ((nbp >> 3) + CL - 1) / CL;
  const size_t smem_cl = sizeof(double) * (size_t)(nbp * (nbp + 4)) +
                         sizeof(double) * (size_t)std::max(nbp * (nbp + 4), 8 * tcs_cl * (nbp + 4) + nbp * (8 * tcs_cl + 4));
  if (v3 && smem_cl > 48 * 1024) cudaFuncSetAttribute(potrf_cluster, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_cl);
  cudaMemsetAsync(info, 0, sizeof(int), st);
  // Two chains.  Main stream: the diagonal blocks only -- potrf(k) applies the step-(k-1) update to its own block in
  // its prologue, so it needs W11(k-1) (stream order) and block row k updated through step k-2 (event from the side
  // stream).  Side stream, per step k: panel  L[k+1:, k] = A[k+1:, k] W11(k)^T  (after potrf(k)), then the trailing
  // update of everything below block row k+1 (a lower trapezoid: block column k+1 included, the diagonal block (k+1,k+1)
  // excluded -- potrf(k+1) owns it).  The 32 latency-bound single-CTA kernels overlap the throughput-bound GEMMs.
  // Fork/join with events keeps the whole factorisation capturable in a CUDA graph.
  // All three chains run on the library's own HIGH-PRIORITY streams (the diagonal chain forks from the caller's stream and joins
  // it at the end): the engine fills the SMs this latency-bound phase leaves idle with the K_zx assembly and the L_s operand
  // products on another stream, and at equal priority those filler CTAs delayed the first links of the chain by 0.1 - 0.2 ms
  // each (torch.profiler trace of the C3 step: 0.49 ms of gaps between the first six diagonal blocks).
  int dev = 0;
  cudaGetDevice(&dev);
  SideCtx& sc = g_side_ctxs[dev & 15];
  sc.mid_valid = false;
  if (!sc.ready) {
    int prio_least = 0, prio_greatest = 0;
    cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest);
    if (cudaStreamCreateWithPriority(&sc.diag, cudaStreamNonBlocking, prio_greatest) != cudaSuccess) return DSVGP_ERR_LAUNCH;
    if (cudaStreamCreateWithPriority(&sc.side, cudaStreamNonBlocking, prio_greatest) != cudaSuccess) return DSVGP_ERR_LAUNCH;
    if (cudaStreamCreateWithPriority(&sc.inv, cudaStreamNonBlocking, prio_greatest) != cudaSuccess) return DSVGP_ERR_LAUNCH;
    if (cudaStreamCreateWithPriority(&sc.inv2, cudaStreamNonBlocking, prio_greatest) != cudaSuccess) return DSVGP_ERR_LAUNCH;
    if (cudaStreamCreateWithPriority(&sc.bulk, cudaStreamNonBlocking, prio_least) != cudaSuccess) return DSVGP_ERR_LAUNCH;
    for (int i = 0; i < 64; ++i) {
      cudaEventCreateWithFlags(&sc.ev_main[i], cudaEventDisableTiming);
      cudaEventCreateWithFlags(&sc.ev_side[i], cudaEventDisableTiming);
      cudaEventCreateWithFlags(&sc.ev_panel[i], cudaEventDisableTiming);
      cudaEventCreateWithFlags(&sc.ev_bulk[i], cudaEventDisableTiming);
    }
    cudaEventCreateWithFlags(&sc.ev_inv, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&sc.ev_entry, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&sc.ev_done, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&sc.ev_mid, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&sc.ev_inv2, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&sc.ev_pre, cudaEventDisableTiming);
    for (int i = 0; i < 8; ++i) cudaEventCreateWithFlags(&sc.ev_T[i], cudaEventDisableTiming);
    for (int i = 0; i < 8; ++i) {
      if (cudaStreamCreateWithPriority(&sc.lvl[i], cudaStreamNonBlocking, prio_greatest) != cudaSuccess) return DSVGP_ERR_LAUNCH;
      cudaEventCreateWithFlags(&sc.ev_lvl[i], cudaEventDisableTiming);
    }
    sc.ready = true;
  }
  cudaStream_t side = sc.side, inv = sc.inv;
  const bool two_chains = nblk <= 64;
  cudaStream_t caller = st;
  if (two_chains && g_chol_priority) {                  // the diagonal chain moves to the high-priority stream
    cudaEventRecord(sc.ev_entry, caller);
    cudaStreamWaitEvent(sc.diag, sc.ev_entry, 0);
    st = sc.diag;
  }
  // Eager inverse (round 2): the recursive-doubling inverse W = [[W11, 0], [-W22 (L21 W11), W22]] does not wait for the end
  // of the factorisation.  For every pair of every level, T = L21 W11 is issued (third stream) as soon as the pair's top half
  // is factorised and inverted, and W21 = -W22 T as soon as its bottom half is: after the last diagonal block only ONE product
  // per level is left (96, 192, .. 1536 wide) instead of the ten batched level products of round 1 (0.72 ms at M' = 3072).
  // T lives in the dead upper-right quadrant of the pair inside W (the work matrix' lower-left quadrant is still read by the
  // next diag_prepare).
  const bool eager_inv = two_chains && nlev >= 1 && g_chol_variant >= 2;
  int last_side = -1, last_bulk = -1;
  unsigned t_pending = 0;                               // levels whose T product (second inverse stream) no W21 has waited for yet
  const bool per_level = g_chol_inv_streams >= 3 && nlev <= 8;
  unsigned lvl_used = 0;                                // level streams that carry work of this factorisation (joined at the end)
  for (int k = 0; k < nblk; ++k) {
    const int64_t o = (int64_t)k * nb0;
    // (more than 64 blocks: more steps than pooled events -- everything goes on the caller's stream, in order)
    if (two_chains && k >= 2 && last_side >= k - 2) cudaStreamWaitEvent(st, sc.ev_side[k - 2], 0);
    const double* Aleft = k > 0 ? Awork + o * lda + (o - nb0) : nullptr;
    const double* Wprev = k > 0 ? W + (o - nb0) * ldw + (o - nb0) : nullptr;
    if (v3) {
      potrf_cluster<<<CL, POTRF_THREADS, smem_cl, st>>>(Awork + o * lda + o, lda, L + o * ldl + o, ldl, W + o * ldw + o, ldw, nb0,
                                                        info, (int)o, Aleft, Wprev);
    } else if (v2) {
      if (k > 0) {
        diag_prepare<<<nparts, POTRF_THREADS, smem_prep, st>>>(Aleft, lda, Wprev, ldw, nb0, parts, lda, nparts);
        CHECK_LAUNCH();
      }
      potrf_inv_block2<<<1, POTRF_THREADS, smem, st>>>(Awork + o * lda + o, lda, L + o * ldl + o, ldl, W + o * ldw + o, ldw,
                                                       nb0, info, (int)o, parts, lda, k > 0 ? nparts : 0);
    } else {
      potrf_inv_block<<<1, POTRF_THREADS, smem, st>>>(Awork + o * lda + o, lda, L + o * ldl + o, ldl, W + o * ldw + o, ldw,
                                                      nb0, info, (int)o, Aleft, Wprev);
    }
    CHECK_LAUNCH();
    const int m = Mp - (int)o - nb0;
    if (two_chains) cudaEventRecord(sc.ev_main[k], st);
    if (two_chains && nblk >= 8 && k == std::min(g_chol_mid_link, nblk - 1)) {
      // (inside the factorisation's own graph the record is an EXTERNAL event node: streams outside the graph may wait for it)
      if (tl_own_capture) cudaEventRecordWithFlags(sc.ev_mid, st, cudaEventRecordExternal);
      else cudaEventRecord(sc.ev_mid, st);
      sc.mid_valid = true;
    }
    if (m > 0) {
      cudaStream_t gs = two_chains ? side : st;
      if (two_chains) cudaStreamWaitEvent(side, sc.ev_main[k], 0);
      double* L21 = L + (o + nb0) * ldl + o;
      // panel  L21 = A21 * W11^T   (op(B) = W11^T is upper triangular; explicit inverse: see the limitation at the top)
      // (W11 carries explicit zeros above its diagonal, so the triangle flag only saves flops: with the rank-K kernel on, which
      //  takes dense operands only, the panel goes through it as a dense product)
      int rc = gemm1<double>(false, true, m, nb0, nb0, 1.0, Awork + (o + nb0) * lda + o, lda, W + o * ldw + o, ldw, 0.0,
                             L21, ldl, TRI_NONE, get_rank_update() ? TRI_NONE : TRI_UPPER, 0, gs);
      if (rc) return rc;
      if (eager_inv) cudaEventRecord(sc.ev_panel[k], side);
      const int m2 = m - nb0;
      // (worth it only while the bulk is long: one product per step keeps up with the chain once panel + update fit into one link)
      const bool split = two_chains && g_chol_lookahead && m2 >= 16 * nb0;
      if (m2 > 0 && split) {
        // Trailing update with a lookahead of two.  Of the lower trapezoid below block row k+1, the next two links of the chain
        // need only its first two block COLUMNS (k+1: the input of panel(k+1); tiles (k+2, k+1) and (k+2, k+2): read by
        // potrf(k+2)).  That thin product (m2 x 192 x 96) stays on the side stream; the rest -- the lower triangle from block
        // (k+3, k+3) on, 0.8 GFLOP / 60 us at the first links of M' = 3072 -- goes to a low-priority stream of its own and has two
        // links' time to finish: the next thin product (which accumulates onto tiles it writes) waits for it, nobody else.  With
        // one product per step, potrf(k+2) waited for all of it and the first ten links ran at 75 - 100 us instead of 50.
        const double* L21b = L21 + (int64_t)nb0 * ldl;
        double* A22b = Awork + (o + 2 * nb0) * lda + (o + nb0);
        if (last_bulk >= 0) cudaStreamWaitEvent(side, sc.ev_bulk[last_bulk], 0);
        rc = gemm<double>(false, true, m2, 2 * nb0, nb0, -1.0, L21b, ldl, L21, ldl, 1.0, A22b, lda, TRI_NONE, TRI_NONE, 0, 1, 0, 0, 0,
                          side);
        if (rc) return rc;
        cudaEventRecord(sc.ev_side[k], side);             // what potrf(k+2) waits for
        last_side = k;
        cudaStreamWaitEvent(sc.bulk, sc.ev_side[k], 0);   // (after the thin product: they share the SMs)
        const double* L21c = L21b + (int64_t)nb0 * ldl;   // rows from block k+3
        rc = gemm<double>(false, true, m2 - nb0, m2 - nb0, nb0, -1.0, L21c, ldl, L21c, ldl, 1.0,
                          A22b + (int64_t)nb0 * lda + 2 * nb0, lda, TRI_NONE, TRI_NONE, 1, 1, 0, 0, 0, sc.bulk);
        if (rc) return rc;
        cudaEventRecord(sc.ev_bulk[k], sc.bulk);
        last_bulk = k;
      } else if (m2 > 0) {
        // trailing update below block row k+1:  A22[nb0:, :] -= L21[nb0:, :] * L21^T  on the tiles with col <= row + nb0
        const double* L21b = L21 + (int64_t)nb0 * ldl;
        double* A22b = Awork + (o + 2 * nb0) * lda + (o + nb0);
        if (last_bulk >= 0) {
          cudaStreamWaitEvent(gs, sc.ev_bulk[last_bulk], 0);
          last_bulk = -1;
        }
        rc = gemm<double>(false, true, m2, m, nb0, -1.0, L21b, ldl, L21, ldl, 1.0, A22b, lda, TRI_NONE, TRI_NONE, 1, 1, 0, 0, 0,
                          gs, nullptr, 0, nullptr, 0, nullptr, 0, nb0);
        if (rc) return rc;
      }
      if (two_chains && !(m2 > 0 && split)) {
        cudaEventRecord(sc.ev_side[k], side);
        last_side = k;
      }
    }
    if (eager_inv && per_level) {
      // One stream PER LEVEL of the recursive doubling.  On one stream (or two: T products / W21 products) the long products of
      // the upper levels (T and W21 of the 768- and 1536-wide pairs: 72 / 177 us) sit in front of the short ones of the blocks that
      // follow, every such delay is inherited by everything after it, and by the last diagonal block the inverse is ten blocks
      // behind: ~20 kernels (0.5 - 0.66 ms) ran after the factor was complete where the true dependency chain is five
      // (W21 of 96, 192, .., 1536: 0.32 ms).  Per level, T(lev) and W21(lev) of consecutive pairs alternate on lvl[lev]; across
      // levels the order is carried by events: the first product of block k waits for the diagonal block, every product of level
      // lev for the W21 of level lev - 1 issued just before it (which completes the group it reads).
      for (int lev = 0; lev < nlev && ((k + 1) & ((1 << lev) - 1)) == 0; ++lev) {
        const int idx = (k + 1) >> lev;
        const int b = nb0 << lev;
        cudaStream_t ls = sc.lvl[lev];
        if (lev == 0) cudaStreamWaitEvent(ls, sc.ev_main[k], 0);        // block k is factorised and inverted
        else cudaStreamWaitEvent(ls, sc.ev_lvl[lev - 1], 0);            // the group below is complete (it waited for block k in turn)
        lvl_used |= 1u << lev;
        if (idx & 1) {                                   // TOP half ended: T = L21 W11 (needs the panel of column k)
          const int64_t s0 = (int64_t)(idx - 1) * b;
          cudaStreamWaitEvent(ls, sc.ev_panel[k], 0);
          int rc = gemm<double>(false, false, b, b, b, 1.0, L + (s0 + b) * ldl + s0, ldl, W + s0 * ldw + s0, ldw, 0.0,
                                W + s0 * ldw + (s0 + b), ldw, TRI_NONE, TRI_LOWER, 0, 1, 0, 0, 0, ls);
          if (rc) return rc;
          break;
        }
        const int64_t s0 = (int64_t)(idx - 2) * b;       // BOTTOM half ended: W21 = -W22 T (T: earlier on this same stream)
        int rc = gemm<double>(false, false, b, b, b, -1.0, W + (s0 + b) * ldw + (s0 + b), ldw, W + s0 * ldw + (s0 + b), ldw, 0.0,
                              W + (s0 + b) * ldw + s0, ldw, TRI_LOWER, TRI_NONE, 0, 1, 0, 0, 0, ls);
        if (rc) return rc;
        cudaEventRecord(sc.ev_lvl[lev], ls);
      }
    } else if (eager_inv) {
      bool waited = false;
      for (int lev = 0; lev < nlev && ((k + 1) & ((1 << lev) - 1)) == 0; ++lev) {
        const int idx = (k + 1) >> lev;                  // groups of 2^lev blocks finished so far
        const int b = nb0 << lev;
        if (!waited) {
          cudaStreamWaitEvent(inv, sc.ev_main[k], 0);    // block k is factorised and inverted
          waited = true;
        }
        if (idx & 1) {                                   // a TOP half just ended: T = L21 W11 (needs the panel of column k)
          // (mode 2) T products on a stream of their own: measured equal to one stream -- the long T products still sit in front
          // of the short ones; the per-level layout above is what removes the backlog.
          const int64_t s0 = (int64_t)(idx - 1) * b;
          cudaStream_t ts = (g_chol_inv_streams >= 2 && lev < 8) ? sc.inv2 : inv;
          if (ts != inv) {
            cudaEventRecord(sc.ev_pre, inv);             // W11 of this group is complete (its lower-level W21 were just issued on inv)
            cudaStreamWaitEvent(ts, sc.ev_pre, 0);
          }
          cudaStreamWaitEvent(ts, sc.ev_panel[k], 0);
          int rc = gemm<double>(false, false, b, b, b, 1.0, L + (s0 + b) * ldl + s0, ldl, W + s0 * ldw + s0, ldw, 0.0,
                                W + s0 * ldw + (s0 + b), ldw, TRI_NONE, TRI_LOWER, 0, 1, 0, 0, 0, ts);
          if (rc) return rc;
          if (ts != inv) {
            cudaEventRecord(sc.ev_T[lev], ts);
            t_pending |= 1u << lev;
          }
          break;
        }
        const int64_t s0 = (int64_t)(idx - 2) * b;       // a BOTTOM half just ended: W21 = -W22 T, the pair is complete
        if (t_pending & (1u << lev)) {
          cudaStreamWaitEvent(inv, sc.ev_T[lev], 0);
          t_pending &= ~(1u << lev);
        }
        int rc = gemm<double>(false, false, b, b, b, -1.0, W + (s0 + b) * ldw + (s0 + b), ldw, W + s0 * ldw + (s0 + b), ldw, 0.0,
                              W + (s0 + b) * ldw + s0, ldw, TRI_LOWER, TRI_NONE, 0, 1, 0, 0, 0, inv);
        if (rc) return rc;
      }
    }
  }
  if (st != caller) {                                   // join: the caller's stream continues after all three chains
    cudaEventRecord(sc.ev_done, st);
    cudaStreamWaitEvent(caller, sc.ev_done, 0);
    st = caller;
  }
  if (two_chains && last_side >= 0) cudaStreamWaitEvent(st, sc.ev_side[last_side], 0);
  if (last_bulk >= 0) cudaStreamWaitEvent(st, sc.ev_bulk[last_bulk], 0);
  if (eager_inv && per_level) {
    for (int lev = 0; lev < nlev; ++lev)
      if (lvl_used & (1u << lev)) {
        cudaEventRecord(sc.ev_lvl[lev], sc.lvl[lev]);
        cudaStreamWaitEvent(st, sc.ev_lvl[lev], 0);
      }
    return DSVGP_OK;
  }
  if (eager_inv) {
    cudaEventRecord(sc.ev_inv, inv);
    cudaStreamWaitEvent(st, sc.ev_inv, 0);
    if (g_chol_inv_streams >= 2) {                      // (every T has been consumed by a W21 on inv; the join keeps the fork/join
      cudaEventRecord(sc.ev_inv2, sc.inv2);             //  structure explicit for graph capture)
      cudaStreamWaitEvent(st, sc.ev_inv2, 0);
    }
    return DSVGP_OK;
  }
  // recursive inverse; Awork (no longer needed) is the scratch for T = L21 * W11
  for (int lev = 0; lev < nlev; ++lev) {
    const int b = nb0 << lev, npairs = nblk >> (lev + 1);
    const int64_t sL = (int64_t)2 * b * ldl + 2 * b, sW = (int64_t)2 * b * ldw + 2 * b, sT = (int64_t)2 * b * lda + 2 * b;
    int rc = gemm<double>(false, false, b, b, b, 1.0, L + (int64_t)b * ldl, ldl, W, ldw, 0.0, Awork + (int64_t)b * lda,
                          lda, TRI_NONE, TRI_LOWER, 0, npairs, sL, sW, sT, st);
    if (rc) return rc;
    rc = gemm<double>(false, false, b, b, b, -1.0, W + (int64_t)b * ldw + b, ldw, Awork + (int64_t)b * lda, lda, 0.0,
                      W + (int64_t)b * ldw, ldw, TRI_LOWER, TRI_NONE, 0, npairs, sW, sT, sW, st);
    if (rc) return rc;
  }
  return DSVGP_OK;
}

// ---- the factorisation as a cached CUDA graph (knob, off by default) --------------------------------------------------------
// One factorisation is ~230 kernel launches and ~400 event calls.  The buffers of a model's factor are allocated once, so the whole
// fork/join structure can be captured ONCE per (buffers, sizes, scheduling knobs) and replayed with a single cudaGraphLaunch.
// Measured: the factorisation alone takes the same 1.93 ms replayed or launched (the GPU, not the host, sets its pace), so this stays
// a knob for hosts slower than this box's.  Not used while the caller's
// stream is itself being captured (graphs.GraphedStep): there the launches simply become part of the caller's graph.
static int g_chol_graph = 0;
void set_chol_graph(int on) { g_chol_graph = on ? 1 : 0; }
int get_chol_graph() { return g_chol_graph; }

struct CholGraphKey {
  double *Awork, *L, *W;
  int64_t lda, ldl, ldw;
  int Mp, nb0, nlev;
  int* info;
  int knobs[8];
  bool operator==(const CholGraphKey& o) const {
    if (Awork != o.Awork || L != o.L || W != o.W || lda != o.lda || ldl != o.ldl || ldw != o.ldw || Mp != o.Mp || nb0 != o.nb0 ||
        nlev != o.nlev || info != o.info)
      return false;
    for (int i = 0; i < 8; ++i)
      if (knobs[i] != o.knobs[i]) return false;
    return true;
  }
};
struct CholGraphEntry { CholGraphKey key; cudaGraphExec_t exec; bool mid_valid; unsigned long long used; };
static std::vector<CholGraphEntry> g_chol_graphs[16];
static unsigned long long g_chol_graph_clock = 0;

int chol_factor_inverse(double* Awork, int64_t lda, double* L, int64_t ldl, double* W, int64_t ldw, int Mp, int nb0,
                        int nlev, int* info, cudaStream_t st) {
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  if (!g_chol_graph || Mp <= 0 || cudaStreamIsCapturing(st, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone)
    return chol_enqueue(Awork, lda, L, ldl, W, ldw, Mp, nb0, nlev, info, st);
  int dev = 0;
  cudaGetDevice(&dev);
  std::vector<CholGraphEntry>& cache = g_chol_graphs[dev & 15];
  CholGraphKey key{Awork, L, W, lda, ldl, ldw, Mp, nb0, nlev, info,
                   {g_chol_variant, g_chol_lookahead, g_chol_priority, g_chol_inv_streams, g_chol_mid_link, get_rank_update(),
                    get_gemm64_async(), 0}};
  CholGraphEntry* hit = nullptr;
  for (auto& e : cache)
    if (e.key == key) hit = &e;
  if (!hit) {
    // make sure everything with per-process one-time setup (streams, events, function attributes) has run eagerly once
    static bool warmed[16] = {};
    if (!warmed[dev & 15]) {
      warmed[dev & 15] = true;
      return chol_enqueue(Awork, lda, L, ldl, W, ldw, Mp, nb0, nlev, info, st);
    }
    if (cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
      cudaGetLastError();
      return chol_enqueue(Awork, lda, L, ldl, W, ldw, Mp, nb0, nlev, info, st);
    }
    tl_own_capture = true;
    const int rc = chol_enqueue(Awork, lda, L, ldl, W, ldw, Mp, nb0, nlev, info, st);
    tl_own_capture = false;
    cudaGraph_t graph = nullptr;
    const cudaError_t ce = cudaStreamEndCapture(st, &graph);
    cudaGraphExec_t exec = nullptr;
    if (rc != DSVGP_OK || ce != cudaSuccess || graph == nullptr || cudaGraphInstantiate(&exec, graph, 0) != cudaSuccess) {
      if (graph) cudaGraphDestroy(graph);
      cudaGetLastError();
      if (rc != DSVGP_OK) return rc;
      return chol_enqueue(Awork, lda, L, ldl, W, ldw, Mp, nb0, nlev, info, st);     // (nothing was enqueued by the failed capture)
    }
    cudaGraphDestroy(graph);
    if (cache.size() >= 8) {                              // evict the least recently used graph
      size_t lru = 0;
      for (size_t i = 1; i < cache.size(); ++i)
        if (cache[i].used < cache[lru].used) lru = i;
      cudaGraphExecDestroy(cache[lru].exec);
      cache.erase(cache.begin() + lru);
    }
    cache.push_back(CholGraphEntry{key, exec, g_side_ctxs[dev & 15].mid_valid, 0});
    hit = &cache.back();
  }
  hit->used = ++g_chol_graph_clock;
  g_side_ctxs[dev & 15].mid_valid = hit->mid_valid;
  if (cudaGraphLaunch(hit->exec, st) != cudaSuccess) {
    cudaGetLastError();
    return DSVGP_ERR_LAUNCH;
  }
  return DSVGP_OK;
}

}  // namespace dsvgp
