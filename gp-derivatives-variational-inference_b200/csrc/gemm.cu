// Triangle-aware batched GEMM on the legacy warp-level tensor path (mma.sync), fp64 (DMMA m8n8k4) and
// fp32-accurate 3xTF32 (m16n8k8).  This is the general-shape workhorse for everything around the hot whitening
// GEMMs: Cholesky panel / trailing updates, the recursive triangular inverse, the replicated M'^3 backward
// tail, and -- until/unless the tcgen05 kernel in trmm_tc.cu takes a shape -- the whitening products themselves.
//
//   C = alpha * op(A) * op(B) + beta * C         op(A): M x K, op(B): K x N, all row-major with leading dims
//
// a_tri / b_tri say that op(A) / op(B) is lower (1) or upper (2) triangular *as an operand of the product*:
// whole k-ranges that multiply structural zeros are skipped and the elements on the wrong side of the diagonal
// are masked to zero at load time, so a buffer whose other triangle holds garbage (the raw chol_variational_covar
// parameter, a Cholesky factor written in place) can be passed as is.  c_tri = 1 computes only the tiles that
// touch the lower triangle of C (SYRK-like results).
#include "common.cuh"
#include "gemm.cuh"

namespace dsvgp {

constexpr int BM = 64, BN = 64, BK = 16, LDS_ = BK + 4, GEMM_THREADS = 128;

__device__ __forceinline__ void mma_f64(double (&c)[2], double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c[0]), "+d"(c[1]) : "d"(a), "d"(b));
}

__device__ __forceinline__ uint32_t to_tf32(float x) {
  uint32_t r;
  asm volatile("cvt.rna.tf32.f32 %0, %1;\n" : "=r"(r) : "f"(x));
  return r;
}

__device__ __forceinline__ void mma_tf32(float (&c)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

template <typename T>
struct GemmParams {
  const T* A; const T* B; T* C; const T* D;   // D: addend scaled by beta (== C unless given)
  T* C2; const T* D2;                          // optional second output C2 = C + D2 (not batched)
  int M, N, K;
  int64_t lda, ldb, ldc, ldd, ldc2, ldd2, sA, sB, sC;
  T alpha, beta;
  int a_tri, b_tri, c_tri;
  int c_off;   // c_tri == 1: tiles with n0 >= m0 + BM + c_off are skipped (c_off > 0: lower trapezoid)
};

// element (r, k) of op(A) (r in M, k in K) lives at A[r*lda + k] (TA=false) or A[k*lda + r] (TA=true)
template <typename T, bool TA, bool TB>
__global__ void __launch_bounds__(GEMM_THREADS)
gemm_kernel(GemmParams<T> p) {
  __shared__ __align__(16) T As[2][BM * LDS_];
  __shared__ __align__(16) T Bs[2][BN * LDS_];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // Heavy tiles first: with a triangular operand the k-range of a tile grows with its row (a lower: k <= r) or column
  // (b upper: k <= c); CUDA hands out blockIdx in increasing order, so the longest tiles would start last and run alone at
  // the end of the launch.  Reversing that index starts them first.
  const int by = (p.a_tri == 1) ? (int)(gridDim.y - 1 - blockIdx.y) : (int)blockIdx.y;
  const int bx = (p.b_tri == 2) ? (int)(gridDim.x - 1 - blockIdx.x) : (int)blockIdx.x;
  const int m0 = by * BM, n0 = bx * BN;
  if (p.c_tri == 1 && n0 >= m0 + BM + p.c_off) return;     // tile strictly above the (shifted) diagonal
  const T* A = p.A + (int64_t)blockIdx.z * p.sA;
  const T* B = p.B + (int64_t)blockIdx.z * p.sB;
  T* C = p.C + (int64_t)blockIdx.z * p.sC;
  const T* D = p.D ? p.D : C;   // an explicit addend is not batched
  const int64_t ldd = p.D ? p.ldd : p.ldc;

  // k-range that can be non-zero for this tile
  int kbeg = 0, kend = p.K;
  if (p.a_tri == 1) kend = min(kend, m0 + BM);          // lower: k <= r
  if (p.a_tri == 2) kbeg = max(kbeg, m0);               // upper: k >= r
  if (p.b_tri == 1) kbeg = max(kbeg, n0);               // lower: k >= c
  if (p.b_tri == 2) kend = min(kend, n0 + BN);          // upper: k <= c
  kbeg = (kbeg / BK) * BK;

  constexpr int PER = BM * BK / GEMM_THREADS;   // 8 elements of each operand per thread per stage
  T ra[PER], rb[PER];

  auto load_tiles = [&](int k0) {
#pragma unroll
    for (int q = 0; q < PER; ++q) {
      const int e = tid + q * GEMM_THREADS;
      int r, k;
      if (!TA) { r = e / BK; k = e % BK; } else { k = e / BM; r = e % BM; }
      const int gr = m0 + r, gk = k0 + k;
      bool ok = gr < p.M && gk < p.K;
      if (p.a_tri == 1) ok = ok && gk <= gr;
      if (p.a_tri == 2) ok = ok && gk >= gr;
      ra[q] = ok ? (TA ? A[(int64_t)gk * p.lda + gr] : A[(int64_t)gr * p.lda + gk]) : T(0);
    }
#pragma unroll
    for (int q = 0; q < PER; ++q) {
      const int e = tid + q * GEMM_THREADS;
      int c, k;
      if (TB) { c = e / BK; k = e % BK; } else { k = e / BN; c = e % BN; }
      const int gc = n0 + c, gk = k0 + k;
      bool ok = gc < p.N && gk < p.K;
      if (p.b_tri == 1) ok = ok && gk >= gc;
      if (p.b_tri == 2) ok = ok && gk <= gc;
      rb[q] = ok ? (TB ? B[(int64_t)gc * p.ldb + gk] : B[(int64_t)gk * p.ldb + gc]) : T(0);
    }
  };
  auto store_tiles = [&](int buf) {
#pragma unroll
    for (int q = 0; q < PER; ++q) {
      const int e = tid + q * GEMM_THREADS;
      int r, k;
      if (!TA) { r = e / BK; k = e % BK; } else { k = e / BM; r = e % BM; }
      As[buf][r * LDS_ + k] = ra[q];
    }
#pragma unroll
    for (int q = 0; q < PER; ++q) {
      const int e = tid + q * GEMM_THREADS;
      int c, k;
      if (TB) { c = e / BK; k = e % BK; } else { k = e / BN; c = e % BN; }
      Bs[buf][c * LDS_ + k] = rb[q];
    }
  };

  const int wm = (warp >> 1) * 32, wn = (warp & 1) * 32;   // warp tile origin inside the CTA tile
  const int g = lane >> 2, t = lane & 3;

  constexpr bool F64 = sizeof(T) == 8;
  // accumulators: fp64 4x4 m8n8 tiles x 2 ; fp32 2x4 m16n8 tiles x 4
  // fp32 path: the tensor-core accumulation chain is kept to ONE k-tile (2 mma steps); the running sum lives in
  // fp64 registers.  A long fp32 tensor-core chain loses ~1e-6 of |A||B| (measured, K = 3072), which the
  // ill-conditioned whitening product W*K_zx amplifies ~400x; with the fp64 master sum the error is set by the
  // 3xTF32 products alone.
  double acc64[F64 ? 4 : 2][4][F64 ? 2 : 4];
  float acc32[F64 ? 1 : 2][F64 ? 1 : 4][4];
  if constexpr (F64) {
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc64[i][j][0] = acc64[i][j][1] = 0.0;
  } else {
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int q = 0; q < 4; ++q) acc64[i][j][q] = 0.0;
  }

  if (kbeg < kend) {
    load_tiles(kbeg);
    store_tiles(0);
    __syncthreads();
    int buf = 0;
    for (int k0 = kbeg; k0 < kend; k0 += BK) {
      const bool more = k0 + BK < kend;
      if (more) load_tiles(k0 + BK);
      const T* as = As[buf];
      const T* bs = Bs[buf];
      if constexpr (F64) {
#pragma unroll
        for (int kk = 0; kk < BK; kk += 4) {
          double af[4], bf[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) af[i] = as[(wm + 8 * i + g) * LDS_ + kk + t];
#pragma unroll
          for (int j = 0; j < 4; ++j) bf[j] = bs[(wn + 8 * j + g) * LDS_ + kk + t];
#pragma unroll
          for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) mma_f64(acc64[i][j], af[i], bf[j]);
        }
      } else {
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int q = 0; q < 4; ++q) acc32[i][j][q] = 0.f;
#pragma unroll
        for (int kk = 0; kk < BK; kk += 8) {
          uint32_t ah[2][4], al[2][4], bh[4][2], bl[4][2];
#pragma unroll
          for (int i = 0; i < 2; ++i) {
            const int r = wm + 16 * i + g;
            const float v[4] = {(float)as[r * LDS_ + kk + t], (float)as[(r + 8) * LDS_ + kk + t],
                                (float)as[r * LDS_ + kk + t + 4], (float)as[(r + 8) * LDS_ + kk + t + 4]};
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              ah[i][q] = to_tf32(v[q]);
              al[i][q] = to_tf32(v[q] - __uint_as_float(ah[i][q]));
            }
          }
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int c = wn + 8 * j + g;
            const float v[2] = {(float)bs[c * LDS_ + kk + t], (float)bs[c * LDS_ + kk + t + 4]};
#pragma unroll
            for (int q = 0; q < 2; ++q) {
              bh[j][q] = to_tf32(v[q]);
              bl[j][q] = to_tf32(v[q] - __uint_as_float(bh[j][q]));
            }
          }
#pragma unroll
          for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              mma_tf32(acc32[i][j], al[i], bh[j]);   // small terms first
              mma_tf32(acc32[i][j], ah[i], bl[j]);
              mma_tf32(acc32[i][j], ah[i], bh[j]);
            }
        }
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int q = 0; q < 4; ++q) acc64[i][j][q] += (double)acc32[i][j][q];
      }
      if (more) {
        store_tiles(buf ^ 1);
        __syncthreads();
        buf ^= 1;
      }
    }
  }

  // epilogue
  auto put = [&](int r, int c, T v) {
    if (r < p.M && c < p.N) {
      T* dst = C + (int64_t)r * p.ldc + c;
      const T res = (p.beta == T(0)) ? p.alpha * v : p.alpha * v + p.beta * D[(int64_t)r * ldd + c];
      *dst = res;
      if (p.C2) p.C2[(int64_t)r * p.ldc2 + c] = res + p.D2[(int64_t)r * p.ldd2 + c];
    }
  };
  if constexpr (F64) {
    // a lane holds two adjacent columns of each 8x8 tile: 16-byte loads / stores when everything is 16-byte aligned
    const bool v2 = ((p.ldc | ldd | (p.C2 ? (p.ldc2 | p.ldd2) : 0)) & 1) == 0 && (((uintptr_t)C | (uintptr_t)D) & 15) == 0 &&
                    (!p.C2 || ((((uintptr_t)p.C2 | (uintptr_t)p.D2) & 15) == 0));
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int r = m0 + wm + 8 * i + g, c = n0 + wn + 8 * j + 2 * t;
        if (v2 && r < p.M && c + 1 < p.N) {
          double2 res = make_double2((double)p.alpha * acc64[i][j][0], (double)p.alpha * acc64[i][j][1]);
          if (p.beta != T(0)) {
            const double2 dd = *reinterpret_cast<const double2*>(D + (int64_t)r * ldd + c);
            res.x += (double)p.beta * dd.x;
            res.y += (double)p.beta * dd.y;
          }
          *reinterpret_cast<double2*>(C + (int64_t)r * p.ldc + c) = res;
          if (p.C2) {
            const double2 ee = *reinterpret_cast<const double2*>(p.D2 + (int64_t)r * p.ldd2 + c);
            *reinterpret_cast<double2*>(p.C2 + (int64_t)r * p.ldc2 + c) = make_double2(res.x + ee.x, res.y + ee.y);
          }
        } else {
          put(r, c, (T)acc64[i][j][0]);
          put(r, c + 1, (T)acc64[i][j][1]);
        }
      }
  } else {
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int r = m0 + wm + 16 * i + g, c = n0 + wn + 8 * j + 2 * t;
        put(r, c, (T)acc64[i][j][0]);
        put(r, c + 1, (T)acc64[i][j][1]);
        put(r + 8, c, (T)acc64[i][j][2]);
        put(r + 8, c + 1, (T)acc64[i][j][3]);
      }
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// fp64 variant with an asynchronous operand pipeline (round 2).  ncu of the kernel above on the Cholesky-backward products
// (profiles/r01_ncu_prof_tail.txt): DMMA pipe 73 % busy, 30 M shared-memory bank conflicts per launch -- all of them in the
// register -> shared staging stores of the TRANSPOSED operand layouts (stride 20 doubles: 4-way) -- and a barrier pair per
// 16-wide k-tile.  Here the operands go global -> shared with cp.async (no register staging, no staging stores), a k-major
// shared layout (row stride 68 doubles: conflict-free DMMA fragments) is used whenever the operand is contiguous along its
// non-contracted index, three stages are in flight and there is ONE barrier per k-tile.
constexpr int AS_STAGES = 3;
constexpr int AS_LDK = BK + 4;       // [row][k] layout (operand contiguous along k):   row stride 20 doubles
constexpr int AS_LDM = BM + 4;       // [k][row] layout (operand contiguous along rows): row stride 68 doubles
constexpr int AS_TILE = (BM * AS_LDK > BK * AS_LDM) ? BM * AS_LDK : BK * AS_LDM;    // doubles per operand per stage

__device__ __forceinline__ void cp_async8_zfill(double* smem_dst, const double* gsrc, bool pred) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  const int bytes = pred ? 8 : 0;
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;\n" ::"r"(d), "l"(gsrc), "r"(bytes) : "memory");
}

template <bool TA, bool TB>
__global__ void __launch_bounds__(GEMM_THREADS, 3)
gemm64_async_kernel(GemmParams<double> p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* As = reinterpret_cast<double*>(smem_raw);                  // [AS_STAGES][AS_TILE]
  double* Bs = As + AS_STAGES * AS_TILE;                             // [AS_STAGES][AS_TILE]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int by = (p.a_tri == 1) ? (int)(gridDim.y - 1 - blockIdx.y) : (int)blockIdx.y;      // heavy tiles first
  const int bx = (p.b_tri == 2) ? (int)(gridDim.x - 1 - blockIdx.x) : (int)blockIdx.x;
  const int m0 = by * BM, n0 = bx * BN;
  if (p.c_tri == 1 && n0 >= m0 + BM + p.c_off) return;
  const double* A = p.A + (int64_t)blockIdx.z * p.sA;
  const double* B = p.B + (int64_t)blockIdx.z * p.sB;
  double* C = p.C + (int64_t)blockIdx.z * p.sC;
  const double* D = p.D ? p.D : C;
  const int64_t ldd = p.D ? p.ldd : p.ldc;

  int kbeg = 0, kend = p.K;
  if (p.a_tri == 1) kend = min(kend, m0 + BM);
  if (p.a_tri == 2) kbeg = max(kbeg, m0);
  if (p.b_tri == 1) kbeg = max(kbeg, n0);
  if (p.b_tri == 2) kend = min(kend, n0 + BN);
  kbeg = (kbeg / BK) * BK;
  const int nkt = kbeg < kend ? (kend - kbeg + BK - 1) / BK : 0;

  // element (r, k) of op(A): TA ? A[k*lda + r] : A[r*lda + k].  Shared: TA ? [k][r] (stride AS_LDM) : [r][k] (stride AS_LDK).
  auto issue = [&](int kt, int stage) {
    const int k0 = kbeg + kt * BK;
    double* as = As + stage * AS_TILE;
    double* bs = Bs + stage * AS_TILE;
#pragma unroll
    for (int q = 0; q < BM * BK / GEMM_THREADS; ++q) {
      const int e = tid + q * GEMM_THREADS;
      int r, k;
      if (!TA) { r = e / BK; k = e % BK; } else { k = e / BM; r = e % BM; }
      const int gr = m0 + r, gk = k0 + k;
      bool ok = gr < p.M && gk < p.K;
      if (p.a_tri == 1) ok = ok && gk <= gr;
      if (p.a_tri == 2) ok = ok && gk >= gr;
      const double* src = ok ? (TA ? A + (int64_t)gk * p.lda + gr : A + (int64_t)gr * p.lda + gk) : A;
      cp_async8_zfill(TA ? as + k * AS_LDM + r : as + r * AS_LDK + k, src, ok);
    }
#pragma unroll
    for (int q = 0; q < BN * BK / GEMM_THREADS; ++q) {
      const int e = tid + q * GEMM_THREADS;
      int c, k;
      if (TB) { c = e / BK; k = e % BK; } else { k = e / BN; c = e % BN; }
      const int gc = n0 + c, gk = k0 + k;
      bool ok = gc < p.N && gk < p.K;
      if (p.b_tri == 1) ok = ok && gk >= gc;
      if (p.b_tri == 2) ok = ok && gk <= gc;
      const double* src = ok ? (TB ? B + (int64_t)gc * p.ldb + gk : B + (int64_t)gk * p.ldb + gc) : B;
      cp_async8_zfill(TB ? bs + c * AS_LDK + k : bs + k * AS_LDM + c, src, ok);
    }
  };

  const int wm = (warp >> 1) * 32, wn = (warp & 1) * 32;
  const int g = lane >> 2, t = lane & 3;
  double acc[4][4][2];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

#pragma unroll
  for (int s = 0; s < AS_STAGES - 1; ++s) {
    if (s < nkt) issue(s, s);
    asm volatile("cp.async.commit_group;\n" ::: "memory");
  }
  for (int kt = 0; kt < nkt; ++kt) {
    asm volatile("cp.async.wait_group %0;\n" ::"n"(AS_STAGES - 2) : "memory");      // tile kt has landed (this thread's part)
    __syncthreads();                                     // ... everybody's part; and everybody is done with tile kt-1's buffer
    if (kt + AS_STAGES - 1 < nkt) issue(kt + AS_STAGES - 1, (kt + AS_STAGES - 1) % AS_STAGES);
    asm volatile("cp.async.commit_group;\n" ::: "memory");
    const double* as = As + (kt % AS_STAGES) * AS_TILE;
    const double* bs = Bs + (kt % AS_STAGES) * AS_TILE;
#pragma unroll
    for (int kk = 0; kk < BK; kk += 4) {
      double af[4], bf[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) af[i] = TA ? as[(kk + t) * AS_LDM + wm + 8 * i + g] : as[(wm + 8 * i + g) * AS_LDK + kk + t];
#pragma unroll
      for (int j = 0; j < 4; ++j) bf[j] = TB ? bs[(wn + 8 * j + g) * AS_LDK + kk + t] : bs[(kk + t) * AS_LDM + wn + 8 * j + g];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) mma_f64(acc[i][j], af[i], bf[j]);
    }
  }
  asm volatile("cp.async.wait_all;\n" ::: "memory");

  auto put = [&](int r, int c, double v) {
    if (r < p.M && c < p.N) {
      const double res = (p.beta == 0.0) ? p.alpha * v : p.alpha * v + p.beta * D[(int64_t)r * ldd + c];
      C[(int64_t)r * p.ldc + c] = res;
      if (p.C2) p.C2[(int64_t)r * p.ldc2 + c] = res + p.D2[(int64_t)r * p.ldd2 + c];
    }
  };
  const bool v2 = ((p.ldc | ldd | (p.C2 ? (p.ldc2 | p.ldd2) : 0)) & 1) == 0 && (((uintptr_t)C | (uintptr_t)D) & 15) == 0 &&
                  (!p.C2 || ((((uintptr_t)p.C2 | (uintptr_t)p.D2) & 15) == 0));
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int r = m0 + wm + 8 * i + g, c = n0 + wn + 8 * j + 2 * t;
      if (v2 && r < p.M && c + 1 < p.N) {
        double2 res = make_double2(p.alpha * acc[i][j][0], p.alpha * acc[i][j][1]);
        if (p.beta != 0.0) {
          const double2 dd = *reinterpret_cast<const double2*>(D + (int64_t)r * ldd + c);
          res.x += p.beta * dd.x;
          res.y += p.beta * dd.y;
        }
        *reinterpret_cast<double2*>(C + (int64_t)r * p.ldc + c) = res;
        if (p.C2) {
          const double2 ee = *reinterpret_cast<const double2*>(p.D2 + (int64_t)r * p.ldd2 + c);
          *reinterpret_cast<double2*>(p.C2 + (int64_t)r * p.ldc2 + c) = make_double2(res.x + ee.x, res.y + ee.y);
        }
      } else {
        put(r, c, acc[i][j][0]);
        put(r, c + 1, acc[i][j][1]);
      }
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// fp64 rank-K update  C = alpha * A * B^T + beta * C  with a SHORT contraction (K <= 128: the rank-96 trailing updates of the
// blocked Cholesky).  An EXPERIMENT, off by default (see g_rank_update below).  The general kernel spends a barrier pair and a register-staged, bank-conflicted store per 16-wide k-tile and
// ran these updates at 10-12 TFLOP/s (66-78 us for the 0.8 GFLOP update of the first links at M' = 3072 -- longer than the diagonal
// block beside it, so the panel/update chain, not the diagonal chain, set the pace of the first ten links).  Here the whole
// K extent of both operand tiles goes global -> shared in ONE cp.async burst ([row][k] layout, row stride = K rounded up to 16
// plus 4 doubles: conflict-free DMMA fragments), one barrier, then every warp runs its K/4 DMMA steps back to back.
constexpr int RK_MAXK = 128;
constexpr int RK_SMALL_GRID = 640;
__host__ __device__ constexpr int rk_ld(int K) { return ((K + 15) & ~15) + 4; }

__device__ __forceinline__ void cp_async16_zfill(double* smem_dst, const double* gsrc, bool pred) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  const int bytes = pred ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(d), "l"(gsrc), "r"(bytes) : "memory");
}

__global__ void __launch_bounds__(GEMM_THREADS, 2)
rank_update64_kernel(GemmParams<double> p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int LD = rk_ld(p.K), K4 = (p.K + 3) & ~3;
  double* As = reinterpret_cast<double*>(smem_raw);                  // [BM][LD]
  double* Bs = As + BM * LD;                                         // [BN][LD]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  if (p.c_tri == 1 && n0 >= m0 + BM + p.c_off) return;
  double* C = p.C;
  const double* D = p.D ? p.D : C;
  const int64_t ldd = p.D ? p.ldd : p.ldc;
  // operands: K contiguous; two doubles per cp.async (K, leading dimensions even and bases 16-byte aligned: checked by the host)
  const int kp = K4 / 2;                                             // 16-byte pieces per row (zero-filled beyond K)
  for (int e = tid; e < BM * kp; e += GEMM_THREADS) {
    const int r = e / kp, k = (e % kp) * 2;
    const bool ok = (m0 + r < p.M) && (k < p.K);
    cp_async16_zfill(As + r * LD + k, ok ? p.A + (int64_t)(m0 + r) * p.lda + k : p.A, ok);
  }
  for (int e = tid; e < BN * kp; e += GEMM_THREADS) {
    const int c = e / kp, k = (e % kp) * 2;
    const bool ok = (n0 + c < p.N) && (k < p.K);
    cp_async16_zfill(Bs + c * LD + k, ok ? p.B + (int64_t)(n0 + c) * p.ldb + k : p.B, ok);
  }
  asm volatile("cp.async.commit_group;\n" ::: "memory");
  const int wm = (warp >> 1) * 32, wn = (warp & 1) * 32;
  const int g = lane >> 2, t = lane & 3;
  double acc[4][4][2];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
  asm volatile("cp.async.wait_all;\n" ::: "memory");
  __syncthreads();
#pragma unroll 2
  for (int kk = 0; kk < K4; kk += 4) {
    double af[4], bf[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) af[i] = As[(wm + 8 * i + g) * LD + kk + t];
#pragma unroll
    for (int j = 0; j < 4; ++j) bf[j] = Bs[(wn + 8 * j + g) * LD + kk + t];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) mma_f64(acc[i][j], af[i], bf[j]);
  }
  const bool v2 = ((p.ldc | ldd) & 1) == 0 && (((uintptr_t)C | (uintptr_t)D) & 15) == 0;
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int r = m0 + wm + 8 * i + g, c = n0 + wn + 8 * j + 2 * t;
      if (r >= p.M) continue;
      if (v2 && c + 1 < p.N) {
        double2 res = make_double2(p.alpha * acc[i][j][0], p.alpha * acc[i][j][1]);
        if (p.beta != 0.0) {
          const double2 dd = *reinterpret_cast<const double2*>(D + (int64_t)r * ldd + c);
          res.x += p.beta * dd.x;
          res.y += p.beta * dd.y;
        }
        *reinterpret_cast<double2*>(C + (int64_t)r * p.ldc + c) = res;
      } else {
#pragma unroll
        for (int z = 0; z < 2; ++z)
          if (c + z < p.N) {
            const double v = p.alpha * acc[i][j][z];
            C[(int64_t)r * p.ldc + c + z] = (p.beta == 0.0) ? v : v + p.beta * D[(int64_t)r * ldd + c + z];
          }
      }
    }
}

static int g_rank_update = 0;   // measured (scratch/rank_update_ab.py, scratch/prio_ab.py): 65 vs 58 us on the first link's update, equal
                                // later -- both kernels are ramp-bound at K = 96 (13 TFLOP/s) -- and its 100 KB of shared memory per
                                // CTA crowds the diagonal-block cluster running beside it: the step is 0.1 ms SLOWER.  Off.
void set_rank_update(int on) { g_rank_update = (on >= 0 && on <= 2) ? on : 0; }   // 2: only launches of at most RK_SMALL_GRID tiles (the latency-bound late links)
int get_rank_update() { return g_rank_update; }

static int g_gemm64_async = 1;
void set_gemm64_async(int on) { g_gemm64_async = on ? 1 : 0; }
int get_gemm64_async() { return g_gemm64_async; }

template <bool TA, bool TB>
static int launch_gemm64_async(const GemmParams<double>& p, dim3 grid, cudaStream_t st) {
  constexpr int smem = 2 * AS_STAGES * AS_TILE * (int)sizeof(double);
  static bool attr[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (!attr[dev & 63]) {
    if (cudaFuncSetAttribute(gemm64_async_kernel<TA, TB>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess)
      return DSVGP_ERR_LAUNCH;
    attr[dev & 63] = true;
  }
  gemm64_async_kernel<TA, TB><<<grid, GEMM_THREADS, smem, st>>>(p);
  return DSVGP_OK;
}

template <typename T>
int gemm(bool ta, bool tb, int M, int N, int K, T alpha, const T* A, int64_t lda, const T* B, int64_t ldb, T beta,
         T* C, int64_t ldc, int a_tri, int b_tri, int c_tri, int batch, int64_t sA, int64_t sB, int64_t sC,
         cudaStream_t st, const T* D, int64_t ldd, T* C2, int64_t ldc2, const T* D2, int64_t ldd2, int c_off) {
  if (M <= 0 || N <= 0 || batch <= 0) return DSVGP_OK;
  // K = 0 reads neither operand (C = beta * D): an empty operand, whose pointer torch reports as NULL, is accepted there
  if (!C || K < 0 || (K > 0 && (!A || !B)) || (C2 && !D2)) return DSVGP_ERR_ARG;
  GemmParams<T> p{A, B, C, D, C2, D2, M, N, K, lda, ldb, ldc, ldd, ldc2, ldd2, sA, sB, sC, alpha, beta, a_tri, b_tri, c_tri, c_off};
  dim3 grid(ceil_div(N, BN), ceil_div(M, BM), batch);
  if constexpr (sizeof(T) == 8) {
    if ((g_rank_update == 1 || (g_rank_update == 2 && (int64_t)grid.x * grid.y <= RK_SMALL_GRID)) && !ta && tb && K >= 8 && K <= RK_MAXK && (K & 1) == 0 && batch == 1 && a_tri == 0 && b_tri == 0 && !C2 &&
        ((lda | ldb) & 1) == 0 && (((uintptr_t)A | (uintptr_t)B) & 15) == 0) {
      const int smem = (BM + BN) * rk_ld(K) * (int)sizeof(double);
      static bool attr[64] = {};
      int dev = 0;
      cudaGetDevice(&dev);
      if (!attr[dev & 63]) {
        if (cudaFuncSetAttribute(rank_update64_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (BM + BN) * rk_ld(RK_MAXK) * (int)sizeof(double)) != cudaSuccess)
          return DSVGP_ERR_LAUNCH;
        attr[dev & 63] = true;
      }
      rank_update64_kernel<<<grid, GEMM_THREADS, smem, st>>>(p);
      CHECK_LAUNCH();
      return DSVGP_OK;
    }
    if (g_gemm64_async && K > 128) {      // (short contractions -- the rank-96 Cholesky updates -- do not amortise the pipeline fill)
      int rc;
      if (!ta && !tb) rc = launch_gemm64_async<false, false>(p, grid, st);
      else if (!ta && tb) rc = launch_gemm64_async<false, true>(p, grid, st);
      else if (ta && !tb) rc = launch_gemm64_async<true, false>(p, grid, st);
      else rc = launch_gemm64_async<true, true>(p, grid, st);
      if (rc) return rc;
      CHECK_LAUNCH();
      return DSVGP_OK;
    }
  }
  if (!ta && !tb) gemm_kernel<T, false, false><<<grid, GEMM_THREADS, 0, st>>>(p);
  else if (!ta && tb) gemm_kernel<T, false, true><<<grid, GEMM_THREADS, 0, st>>>(p);
  else if (ta && !tb) gemm_kernel<T, true, false><<<grid, GEMM_THREADS, 0, st>>>(p);
  else gemm_kernel<T, true, true><<<grid, GEMM_THREADS, 0, st>>>(p);
  CHECK_LAUNCH();
  return DSVGP_OK;
}

template int gemm<float>(bool, bool, int, int, int, float, const float*, int64_t, const float*, int64_t, float, float*,
                         int64_t, int, int, int, int, int64_t, int64_t, int64_t, cudaStream_t, const float*, int64_t, float*, int64_t,
                         const float*, int64_t, int);
template int gemm<double>(bool, bool, int, int, int, double, const double*, int64_t, const double*, int64_t, double,
                          double*, int64_t, int, int, int, int, int64_t, int64_t, int64_t, cudaStream_t, const double*, int64_t,
                          double*, int64_t, const double*, int64_t, int);

}  // namespace dsvgp
