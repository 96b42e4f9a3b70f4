// Fused RBF directional-gradient kernel assembly (forward, backward, diag) for sm_100a.
//
// Replaces the ~45 eager ops of the reference's RBFKernelDirectionalGrad.forward
// (/root/reference/directionalvi/RBFKernelDirectionalGrad.py:41-108) and their autograd backward:
// with D = x1_i - x2_j, k = os*exp(-|D|^2 / 2l^2), u = v1[i,a-1]/|v1[i,a-1]|, w = v2[j,b-1]/|v2[j,b-1]|,
//   K[i(p1+1)+a, j(p2+1)+b] = k                                   a=b=0
//                             k (D.w)/l^2                          a=0,b>0
//                            -k (D.u)/l^2                          a>0,b=0
//                             k (u.w/l^2 - (D.u)(D.w)/l^4)         a,b>0
// written ONCE, directly in the interleaved layout the reference reaches through two full-matrix gathers
// (:105-107).  Inputs are staged through shared memory in d-chunks; the output tile is staged in shared
// memory so every global store is a full coalesced row segment.
//
// T  = dtype of x (model dtype); TK = dtype of K / dK and of all arithmetic (double for K_zz always, because
// the reference factorises K_zz in fp64, DirectionalGradVariationalStrategy.py:74).
#include <cuda_fp16.h>

#include "common.cuh"
#include "kdir.cuh"

namespace dsvgp {

// ------------------------------------------------------------------------------------------------ prep
// One warp per direction row: vhat = v / |v|, inv_norm = 1/|v|   (RBFKernelDirectionalGrad.py:57-58)
// cidx (optional): per row, the coordinate of its single non-zero entry with the sign in bit 31, and *canon_flag is
// cleared if any row is not one-hot (the flag must be set to 1 by the caller beforehand).
template <typename T, typename TK>
__global__ void normalize_dirs_kernel(const T* __restrict__ v, int rows, int d, TK* __restrict__ vhat,
                                      TK* __restrict__ inv_norm, int* __restrict__ cidx, int* __restrict__ canon_flag) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  TK s = 0;
  int nnz = 0, pos = 0, neg = 0;
  for (int c = lane; c < d; c += 32) {
    TK a = (TK)v[(int64_t)row * d + c];
    s += a * a;
    if (a != TK(0)) {
      ++nnz;
      pos = c;
      neg = a < TK(0);
    }
  }
  s = warp_sum(s);
  if (cidx) {
    const int tot = warp_sum(nnz);
    const int code = warp_sum(nnz ? (pos | (neg ? (int)0x80000000 : 0)) : 0);    // exact when tot == 1
    if (lane == 0) {
      cidx[row] = (tot == 1) ? code : 0;
      if (tot != 1 && canon_flag) *canon_flag = 0;
    }
  }
  const TK inv = TK(1) / dsqrt<TK>(s);
  for (int c = lane; c < d; c += 32) vhat[(int64_t)row * d + c] = (TK)v[(int64_t)row * d + c] * inv;
  if (lane == 0 && inv_norm) inv_norm[row] = inv;
}

// --------------------------------------------------------------------------------------- forward (blocked)
template <typename TK> struct FwdTile { static constexpr int TI = 32; };
template <> struct FwdTile<double> { static constexpr int TI = 16; };
constexpr int FWD_TJ = 32;
constexpr int FWD_DC = 16;
constexpr int FWD_LDX = FWD_TJ + 1;   // padded row of the transposed column-side staging

template <typename TK, int P1, int P2>
constexpr size_t fwd_smem_bytes() {
  constexpr int TI = FwdTile<TK>::TI;
  return sizeof(TK) * (size_t)(TI * FWD_DC + TI * P1 * FWD_DC + FWD_DC * FWD_LDX + P2 * FWD_DC * FWD_LDX +
                               TI * (P1 + 1) * (FWD_TJ * (P2 + 1) + 1));
}

template <typename T, typename TK, int P1, int P2>
__global__ void __launch_bounds__(256)
kdir_fwd_blocked(const T* __restrict__ x1, const TK* __restrict__ u1, int n1, const T* __restrict__ x2,
                 const TK* __restrict__ w2, int n2, int d, const double* __restrict__ hyp, int use_os,
                 TK diag_add, TK* __restrict__ K, int64_t ldk) {
  constexpr int TI = FwdTile<TK>::TI, TJ = FWD_TJ, DC = FWD_DC, RP = TI / 8;
  constexpr int Q1 = P1 + 1, Q2 = P2 + 1, LDS = TJ * Q2 + 1, LDX = FWD_LDX;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  TK* x1s = reinterpret_cast<TK*>(smem_raw);      // [TI][DC]
  TK* u1s = x1s + TI * DC;                        // [TI*P1][DC]
  TK* x2s = u1s + TI * P1 * DC;                   // [DC][LDX]
  TK* w2s = x2s + DC * LDX;                       // [P2][DC][LDX]
  TK* Ks = w2s + P2 * DC * LDX;                    // [TI*Q1][LDS]

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int i0 = blockIdx.y * TI, j0 = blockIdx.x * TJ;

  TK r2[RP], al[RP][P1 > 0 ? P1 : 1], be[RP][P2 > 0 ? P2 : 1], ga[RP][P1 > 0 ? P1 : 1][P2 > 0 ? P2 : 1];
#pragma unroll
  for (int r = 0; r < RP; ++r) {
    r2[r] = 0;
#pragma unroll
    for (int a = 0; a < P1; ++a) al[r][a] = 0;
#pragma unroll
    for (int b = 0; b < P2; ++b) be[r][b] = 0;
#pragma unroll
    for (int a = 0; a < P1; ++a)
#pragma unroll
      for (int b = 0; b < P2; ++b) ga[r][a][b] = 0;
  }

  for (int c0 = 0; c0 < d; c0 += DC) {
    __syncthreads();
    for (int e = tid; e < TI * DC; e += 256) {
      const int i = e / DC, cc = e % DC;
      const bool ok = (i0 + i < n1) && (c0 + cc < d);
      x1s[e] = ok ? (TK)x1[(int64_t)(i0 + i) * d + c0 + cc] : TK(0);
    }
    for (int e = tid; e < TI * P1 * DC; e += 256) {
      const int ia = e / DC, cc = e % DC;
      const bool ok = (i0 * P1 + ia < n1 * P1) && (c0 + cc < d);
      u1s[e] = ok ? u1[(int64_t)(i0 * P1 + ia) * d + c0 + cc] : TK(0);
    }
    for (int e = tid; e < TJ * DC; e += 256) {
      const int j = e / DC, cc = e % DC;
      const bool ok = (j0 + j < n2) && (c0 + cc < d);
      x2s[cc * LDX + j] = ok ? (TK)x2[(int64_t)(j0 + j) * d + c0 + cc] : TK(0);
    }
    for (int e = tid; e < TJ * P2 * DC; e += 256) {
      const int jb = e / DC, cc = e % DC, j = jb / (P2 > 0 ? P2 : 1), b = jb % (P2 > 0 ? P2 : 1);
      const bool ok = (j0 + j < n2) && (c0 + cc < d);
      w2s[(b * DC + cc) * LDX + j] = ok ? w2[(int64_t)((j0 + j) * P2 + b) * d + c0 + cc] : TK(0);
    }
    __syncthreads();
#pragma unroll
    for (int cc = 0; cc < DC; ++cc) {
      const TK xj = x2s[cc * LDX + lane];
      TK wj[P2 > 0 ? P2 : 1];
#pragma unroll
      for (int b = 0; b < P2; ++b) wj[b] = w2s[(b * DC + cc) * LDX + lane];
#pragma unroll
      for (int r = 0; r < RP; ++r) {
        const int i = warp + 8 * r;
        const TK dl = x1s[i * DC + cc] - xj;
        r2[r] += dl * dl;
#pragma unroll
        for (int b = 0; b < P2; ++b) be[r][b] += dl * wj[b];
#pragma unroll
        for (int a = 0; a < P1; ++a) {
          const TK ui = u1s[(i * P1 + a) * DC + cc];
          al[r][a] += dl * ui;
#pragma unroll
          for (int b = 0; b < P2; ++b) ga[r][a][b] += ui * wj[b];
        }
      }
    }
  }

  const TK ell = (TK)hyp[0], os = use_os ? (TK)hyp[1] : TK(1);
  const TK il2 = TK(1) / (ell * ell);
#pragma unroll
  for (int r = 0; r < RP; ++r) {
    const int i = warp + 8 * r;
    const TK k = os * dexp<TK>(TK(-0.5) * r2[r] * il2);
    const bool dg = (diag_add != TK(0)) && (i0 + i == j0 + lane);
    TK* row0 = Ks + (i * Q1) * LDS + lane * Q2;
    row0[0] = k + (dg ? diag_add : TK(0));
#pragma unroll
    for (int b = 0; b < P2; ++b) row0[1 + b] = k * be[r][b] * il2;
#pragma unroll
    for (int a = 0; a < P1; ++a) {
      TK* rowa = row0 + (1 + a) * LDS;
      const TK aa = al[r][a] * il2;
      rowa[0] = -k * aa;
#pragma unroll
      for (int b = 0; b < P2; ++b)
        rowa[1 + b] = k * (ga[r][a][b] * il2 - aa * be[r][b] * il2) + ((dg && a == b) ? diag_add : TK(0));
    }
  }
  __syncthreads();
  // coalesced write-out: each row of the tile is a contiguous TJ*Q2 segment of the output row
  const int rows = min(TI * Q1, n1 * Q1 - i0 * Q1);
  const int cols = min(TJ * Q2, n2 * Q2 - j0 * Q2);
  TK* Kt = K + (int64_t)(i0 * Q1) * ldk + (int64_t)j0 * Q2;
  for (int e = tid; e < rows * (TJ * Q2); e += 256) {
    const int rr = e / (TJ * Q2), cc = e % (TJ * Q2);
    if (cc < cols) Kt[(int64_t)rr * ldk + cc] = Ks[rr * LDS + cc];
  }
}

// lo = rn_tf32(x - trunc_tf32(x)): the part of x a TF32 tensor core does not see (see trmm_tc.cu)
// Packed fp32 pairs (Blackwell FFMA2 / FADD2 / FMUL2: one issue slot for two lanes of work, and an operand may be a plain
// fp32 register broadcast to both halves -- make_float2(x, x) costs nothing).  The vectorised assembly kernels are bound by
// instruction issue on their dot products (ncu: FMA pipe 36 % busy, issue-active 47-74 % with 2-3 warps per scheduler), and
// a lane's four column points are two such pairs.
__device__ __forceinline__ float2 f2fma(float2 a, float2 b, float2 c) {
  float2 r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;"
      : "=l"(reinterpret_cast<unsigned long long&>(r))
      : "l"(reinterpret_cast<const unsigned long long&>(a)), "l"(reinterpret_cast<const unsigned long long&>(b)),
        "l"(reinterpret_cast<const unsigned long long&>(c)));
  return r;
}
__device__ __forceinline__ float2 f2sub(float2 a, float2 b) {
  float2 r;
  asm("sub.rn.f32x2 %0, %1, %2;"
      : "=l"(reinterpret_cast<unsigned long long&>(r))
      : "l"(reinterpret_cast<const unsigned long long&>(a)), "l"(reinterpret_cast<const unsigned long long&>(b)));
  return r;
}
__device__ __forceinline__ float2 f2bc(float x) { return make_float2(x, x); }

__device__ __forceinline__ float tf32_lo_part(float x) {
  const float r = x - __uint_as_float(__float_as_uint(x) & 0xFFFFE000u);
  uint32_t t;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(t) : "f"(r));
  return __uint_as_float(t);
}

// ---------------------------------------------------------------------------------- forward (fp32, vectorised)
// The hot assembly (K_zx of an fp32 model).  A lane owns 4 CONSECUTIVE column points, a warp 128 of them, so
//   * column-side operands are read from shared memory as one LDS.128 per (c, plane) [layout (plane, c, j), j contiguous],
//     row-side operands as broadcast LDS.128 over 4 c's [layout (row, plane, c), c contiguous];
//   * each output row segment of a warp (128 points x (P2+1) floats, contiguous in memory) is transposed through a
//     per-warp shared-memory strip so that every global store instruction writes 512 contiguous bytes.
// One CTA keeps ONE 128-point column tile (all d coordinates) resident and sweeps V4_TIB = 64 row points over it, one
// row point per warp per pass, so the tile load is amortised over 8192 point pairs and the sweep has no block barriers.
// Canonical column-side directions (every row of v2 one-hot: what train_gp / eval_gp pass, directional_vi.py:87-88,
// :292-293) are detected on the device by normalize_dirs (no host sync): then D.w and u.w are lookups, not dot
// products, and the per-pair work drops from (1+p1)(1+p2) to (1+p1) FMAs per coordinate.
// p1 = p2 = 0 is the plain RBF kernel (K_zx of the SVGP baseline, K_xx of a predictive covariance without directions): one
// output row per row point, one FMA pair per coordinate and pair, the same tiles, strips and stores with Q1 = Q2 = 1.  (Its
// backward, kdir_bwd_v4<0, 0>, takes d <= 20 like the other cases: see bwd_v4_ok.)
constexpr int V4_TJ = 128, V4_TIB = 64;

int g_bwd_vpl = 4;             // column points per lane of kdir_bwd_v4: 4, or 2 = two CTAs per SM (benchmarking knob; measured equal:
                               // 0.50 / 0.54 ms at C3 -- the kernel is bound by shared-memory reads + FMA issue, not by latency)
int g_fwd_tib = 0;             // row points per CTA of kdir_fwd_v4: 0 (default) = 64, or 32 when that leaves fewer than 1024 CTAs (small
                               // minibatches: C4 n = 2048 130 -> 107 us, n = 512 69 -> 40 us; scratch/tib_sweep.py); else a fixed multiple of 8 <= 64
int g_fwd_stream_stores = 2;   // 1: st.global.cs (evict-first) for the K / K_lo rows; 2 (default): when the output is
                               // larger than half of the 126 MB L2 (measured on C3: K only 0.144 -> 0.136 ms, K + lo 0.209 -> 0.195 ms)

template <int P1, int P2>
size_t fwd_v4_smem_bytes(int dpad, int tib = V4_TIB) {
  return sizeof(float) * (size_t)(tib * (P1 + 1) * dpad + (P2 + 1) * dpad * V4_TJ + 8 * V4_TJ * (P2 + 1));
}

__device__ __forceinline__ void cp_async4_zfill(float* smem_dst, const float* gsrc, bool pred) {   // pred false: writes 0, reads nothing
  const uint32_t dst = (uint32_t)__cvta_generic_to_shared(smem_dst);
  const int bytes = pred ? 4 : 0;
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;\n" ::"r"(dst), "l"(gsrc), "r"(bytes) : "memory");
}

// MODE 0: general directions only (returns at once if the device flag says canonical); MODE 1: canonical only (returns
// at once otherwise).  Both are launched back to back when a flag is supplied: the choice is made on the device without
// a host synchronisation, and the canonical variant compiles to far fewer registers (3 CTAs per SM instead of 2).
// OUT 0: K (fp32).  OUT 1: K and its TF32 lo part (operands of the 3xTF32 product).  OUT 2: no fp32 matrix at all, only
// the two-half split (Kh, Kl) of K * *hscale -- the operands of the 3xFP16 product (trmm_tc.cu), same bytes as K alone.
template <int P1, int P2, int OUT, int MODE>
__global__ void __launch_bounds__(256, MODE == 1 ? 3 : 2)
kdir_fwd_v4(const float* __restrict__ x1, const float* __restrict__ u1, int n1, const float* __restrict__ x2,
            const float* __restrict__ w2, const int* __restrict__ cidx2, const int* __restrict__ canon_flag, int n2, int d,
            const double* __restrict__ hyp, int use_os, float diag_add, float* __restrict__ K, int64_t ldk,
            float* __restrict__ Klo, int TIB, int stream_stores, __half* __restrict__ Kh, __half* __restrict__ Kl,
            int64_t ldkh, const float* __restrict__ hscale) {
  constexpr bool WITH_LO = OUT == 1;
  constexpr int Q1 = P1 + 1, Q2 = P2 + 1, TJ = V4_TJ;
  const int dpad = (d + 3) & ~3;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* rs = reinterpret_cast<float*>(smem_raw);          // [TIB][Q1][dpad]   row point i: x1_i then u_i1..u_iP1
  float* cs = rs + TIB * Q1 * dpad;                        // [Q2][dpad][TJ]    plane 0: x2, plane 1+b: w_b
  float* strip = cs + Q2 * dpad * TJ;                      // [8 warps][TJ*Q2]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int i0 = blockIdx.y * TIB, j0 = blockIdx.x * TJ;
  const bool flag_set = (P2 > 0) && cidx2 != nullptr && canon_flag != nullptr && (*canon_flag != 0);
  if ((MODE == 1) != flag_set) return;                      // grid-uniform
  constexpr bool canon = MODE == 1;

  // (zero-filling 4-byte cp.async: every element of both tiles in flight at once instead of one global round trip per loop pass)
  for (int e = tid; e < TIB * Q1 * dpad; e += 256) {       // row side: consecutive threads -> consecutive c
    const int cc = e % dpad, ia = e / dpad, i = ia / Q1, a = ia % Q1;
    const bool ok = i0 + i < n1 && cc < d;
    const float* src = !ok ? x1 : (a == 0) ? x1 + (int64_t)(i0 + i) * d + cc : u1 + (int64_t)((i0 + i) * P1 + a - 1) * d + cc;
    cp_async4_zfill(rs + e, src, ok);
  }
  {                                                        // column side: consecutive threads -> consecutive j
    const int j = tid & 127, planes = canon ? 1 : Q2;
    for (int row = tid >> 7; row < planes * dpad; row += 2) {
      const int b = row / dpad, cc = row % dpad;
      const bool ok = j0 + j < n2 && cc < d;
      const float* src = !ok ? x2 : (b == 0) ? x2 + (int64_t)(j0 + j) * d + cc : w2 + (int64_t)((j0 + j) * P2 + b - 1) * d + cc;
      cp_async4_zfill(cs + row * TJ + j, src, ok);
    }
  }
  asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;\n" ::: "memory");
  __syncthreads();

  // canonical column directions: coordinate index / sign of this lane's 4 points, and x2 at that coordinate
  int cix[P2 > 0 ? P2 : 1][4];
  float csg[P2 > 0 ? P2 : 1][4], xjc[P2 > 0 ? P2 : 1][4];
  if constexpr (canon) {
#pragma unroll
    for (int b = 0; b < P2; ++b)
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int j = j0 + 4 * lane + q;
        const int code = (j < n2) ? cidx2[(int64_t)j * P2 + b] : 0;
        cix[b][q] = code & 0x7fffffff;
        csg[b][q] = (code < 0) ? -1.f : 1.f;
        xjc[b][q] = cs[cix[b][q] * TJ + 4 * lane + q];
      }
  }

  const float ell = (float)hyp[0], os = use_os ? (float)hyp[1] : 1.f;
  const float il2 = 1.f / (ell * ell);
  float* mystrip = strip + warp * (TJ * Q2);
  const bool vec_ok = OUT == 2 ? (((ldkh & 3) == 0) && (((reinterpret_cast<uintptr_t>(Kh) | reinterpret_cast<uintptr_t>(Kl)) & 7) == 0))
                               : (((ldk & 3) == 0) && ((reinterpret_cast<uintptr_t>(K) & 15) == 0));
  const float hs = OUT == 2 ? *hscale : 1.f;
  const int cols = min(TJ * Q2, (n2 - j0) * Q2);

  for (int it = 0; it < TIB / 8; ++it) {
    const int il = it * 8 + warp, gi = i0 + il;
    if (gi >= n1) break;                                   // warp-uniform
    const float* rbase = rs + (il * Q1) * dpad;
    float r2[4], al[P1 > 0 ? P1 : 1][4], be[P2 > 0 ? P2 : 1][4], ga[P1 > 0 ? P1 : 1][P2 > 0 ? P2 : 1][4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      r2[q] = 0.f;
#pragma unroll
      for (int a = 0; a < P1; ++a) al[a][q] = 0.f;
#pragma unroll
      for (int b = 0; b < P2; ++b) be[b][q] = 0.f;
#pragma unroll
      for (int a = 0; a < P1; ++a)
#pragma unroll
        for (int b = 0; b < P2; ++b) ga[a][b][q] = 0.f;
    }
    // (dot products on packed pairs: pair h holds this lane's column points 2h, 2h + 1)
    float2 r2p[2], alp[P1 > 0 ? P1 : 1][2], bep[P2 > 0 ? P2 : 1][2], gap[P1 > 0 ? P1 : 1][P2 > 0 ? P2 : 1][2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      r2p[h] = make_float2(0.f, 0.f);
#pragma unroll
      for (int a = 0; a < P1; ++a) alp[a][h] = make_float2(0.f, 0.f);
#pragma unroll
      for (int b = 0; b < P2; ++b) bep[b][h] = make_float2(0.f, 0.f);
#pragma unroll
      for (int a = 0; a < P1; ++a)
#pragma unroll
        for (int b = 0; b < P2; ++b) gap[a][b][h] = make_float2(0.f, 0.f);
    }
    if constexpr (!canon) {
      for (int c4 = 0; c4 < dpad; c4 += 4) {
        const float4 xr = *reinterpret_cast<const float4*>(rbase + c4);
        float4 ur[P1 > 0 ? P1 : 1];
#pragma unroll
        for (int a = 0; a < P1; ++a) ur[a] = *reinterpret_cast<const float4*>(rbase + (1 + a) * dpad + c4);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float4 xj4 = *reinterpret_cast<const float4*>(cs + (c4 + k) * TJ + 4 * lane);
          const float2 xj[2] = {make_float2(xj4.x, xj4.y), make_float2(xj4.z, xj4.w)};
          float2 wj[P2 > 0 ? P2 : 1][2];
#pragma unroll
          for (int b = 0; b < P2; ++b) {
            const float4 t = *reinterpret_cast<const float4*>(cs + ((1 + b) * dpad + c4 + k) * TJ + 4 * lane);
            wj[b][0] = make_float2(t.x, t.y);
            wj[b][1] = make_float2(t.z, t.w);
          }
          const float2 xi = f2bc(k == 0 ? xr.x : k == 1 ? xr.y : k == 2 ? xr.z : xr.w);
          float2 ui[P1 > 0 ? P1 : 1];
#pragma unroll
          for (int a = 0; a < P1; ++a) ui[a] = f2bc(k == 0 ? ur[a].x : k == 1 ? ur[a].y : k == 2 ? ur[a].z : ur[a].w);
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const float2 dl = f2sub(xi, xj[h]);
            r2p[h] = f2fma(dl, dl, r2p[h]);
#pragma unroll
            for (int b = 0; b < P2; ++b) bep[b][h] = f2fma(dl, wj[b][h], bep[b][h]);
#pragma unroll
            for (int a = 0; a < P1; ++a) {
              alp[a][h] = f2fma(dl, ui[a], alp[a][h]);
#pragma unroll
              for (int b = 0; b < P2; ++b) gap[a][b][h] = f2fma(ui[a], wj[b][h], gap[a][b][h]);
            }
          }
        }
      }
    } else {
      for (int c4 = 0; c4 < dpad; c4 += 4) {
        const float4 xr = *reinterpret_cast<const float4*>(rbase + c4);
        float4 ur[P1 > 0 ? P1 : 1];
#pragma unroll
        for (int a = 0; a < P1; ++a) ur[a] = *reinterpret_cast<const float4*>(rbase + (1 + a) * dpad + c4);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float4 xj4 = *reinterpret_cast<const float4*>(cs + (c4 + k) * TJ + 4 * lane);
          const float2 xj[2] = {make_float2(xj4.x, xj4.y), make_float2(xj4.z, xj4.w)};
          const float2 xi = f2bc(k == 0 ? xr.x : k == 1 ? xr.y : k == 2 ? xr.z : xr.w);
          float2 ui[P1 > 0 ? P1 : 1];
#pragma unroll
          for (int a = 0; a < P1; ++a) ui[a] = f2bc(k == 0 ? ur[a].x : k == 1 ? ur[a].y : k == 2 ? ur[a].z : ur[a].w);
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const float2 dl = f2sub(xi, xj[h]);
            r2p[h] = f2fma(dl, dl, r2p[h]);
#pragma unroll
            for (int a = 0; a < P1; ++a) alp[a][h] = f2fma(dl, ui[a], alp[a][h]);
          }
        }
      }
    }
    // unpack (register renaming only)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      r2[2 * h] = r2p[h].x; r2[2 * h + 1] = r2p[h].y;
#pragma unroll
      for (int a = 0; a < P1; ++a) { al[a][2 * h] = alp[a][h].x; al[a][2 * h + 1] = alp[a][h].y; }
      if constexpr (!canon) {
#pragma unroll
        for (int b = 0; b < P2; ++b) { be[b][2 * h] = bep[b][h].x; be[b][2 * h + 1] = bep[b][h].y; }
#pragma unroll
        for (int a = 0; a < P1; ++a)
#pragma unroll
          for (int b = 0; b < P2; ++b) { ga[a][b][2 * h] = gap[a][b][h].x; ga[a][b][2 * h + 1] = gap[a][b][h].y; }
      }
    }
    if constexpr (canon) {
#pragma unroll
      for (int b = 0; b < P2; ++b)
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          be[b][q] = csg[b][q] * (rbase[cix[b][q]] - xjc[b][q]);                   // D . w  with w = +-e_idx
#pragma unroll
          for (int a = 0; a < P1; ++a) ga[a][b][q] = csg[b][q] * rbase[(1 + a) * dpad + cix[b][q]];   // u . w
        }
    }

    float kk[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) kk[q] = os * expf(-0.5f * r2[q] * il2);
#pragma unroll
    for (int a = 0; a < Q1; ++a) {
      float o[4 * Q2];                                     // this lane's 4*Q2 consecutive floats of output row (gi, a)
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const bool dg = (diag_add != 0.f) && (gi == j0 + 4 * lane + q);
        if (a == 0) {
          o[q * Q2] = kk[q] + (dg ? diag_add : 0.f);
#pragma unroll
          for (int b = 0; b < P2; ++b) o[q * Q2 + 1 + b] = kk[q] * be[b][q] * il2;
        } else {
          const float aa = al[a > 0 ? a - 1 : 0][q] * il2;
          o[q * Q2] = -kk[q] * aa;
#pragma unroll
          for (int b = 0; b < P2; ++b)
            o[q * Q2 + 1 + b] = kk[q] * (ga[a > 0 ? a - 1 : 0][b][q] * il2 - aa * be[b][q] * il2) +
                                ((dg && a - 1 == b) ? diag_add : 0.f);
        }
      }
      __syncwarp();
#pragma unroll
      for (int v = 0; v < Q2; ++v)
        *reinterpret_cast<float4*>(mystrip + lane * 4 * Q2 + 4 * v) = make_float4(o[4 * v], o[4 * v + 1], o[4 * v + 2], o[4 * v + 3]);
      __syncwarp();
      if constexpr (OUT == 2) {
        __half* hrow = Kh + (int64_t)(gi * Q1 + a) * ldkh + (int64_t)j0 * Q2;
        __half* lrow = Kl + (int64_t)(gi * Q1 + a) * ldkh + (int64_t)j0 * Q2;
#pragma unroll
        for (int v = 0; v < Q2; ++v) {
          const int col = v * 128 + 4 * lane;
          const float4 t = *reinterpret_cast<const float4*>(mystrip + col);
          const float tv[4] = {t.x * hs, t.y * hs, t.z * hs, t.w * hs};
          __half h[4], l[4];
#pragma unroll
          for (int z = 0; z < 4; ++z) {
            h[z] = __float2half_rn(tv[z]);
            l[z] = __float2half_rn(tv[z] - __half2float(h[z]));
          }
          if (vec_ok && col + 3 < cols) {
            if (stream_stores) {
              __stcs(reinterpret_cast<uint2*>(hrow + col), *reinterpret_cast<const uint2*>(h));
              __stcs(reinterpret_cast<uint2*>(lrow + col), *reinterpret_cast<const uint2*>(l));
            } else {
              *reinterpret_cast<uint2*>(hrow + col) = *reinterpret_cast<const uint2*>(h);
              *reinterpret_cast<uint2*>(lrow + col) = *reinterpret_cast<const uint2*>(l);
            }
          } else {
            for (int z = 0; z < 4; ++z)
              if (col + z < cols) {
                hrow[col + z] = h[z];
                lrow[col + z] = l[z];
              }
          }
        }
        continue;
      }
      float* grow = K + (int64_t)(gi * Q1 + a) * ldk + (int64_t)j0 * Q2;
      float* lrow = WITH_LO ? Klo + (int64_t)(gi * Q1 + a) * ldk + (int64_t)j0 * Q2 : nullptr;   // same leading dimension
#pragma unroll
      for (int v = 0; v < Q2; ++v) {
        const int col = v * 128 + 4 * lane;
        const float4 t = *reinterpret_cast<const float4*>(mystrip + col);
        if (vec_ok && col + 3 < cols && (!WITH_LO || (reinterpret_cast<uintptr_t>(Klo) & 15) == 0)) {
          if (stream_stores) __stcs(reinterpret_cast<float4*>(grow + col), t);
          else *reinterpret_cast<float4*>(grow + col) = t;
          if constexpr (WITH_LO) {
            const float4 tl = make_float4(tf32_lo_part(t.x), tf32_lo_part(t.y), tf32_lo_part(t.z), tf32_lo_part(t.w));
            if (stream_stores) __stcs(reinterpret_cast<float4*>(lrow + col), tl);
            else *reinterpret_cast<float4*>(lrow + col) = tl;
          }
        } else {
          const float tv[4] = {t.x, t.y, t.z, t.w};
          for (int z = 0; z < 4; ++z)
            if (col + z < cols) {
              grow[col + z] = tv[z];
              if constexpr (WITH_LO) lrow[col + z] = tf32_lo_part(tv[z]);
            }
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------- forward (runtime p)
// Fallback for p1 or p2 > DSVGP_MAXP_FAST (e.g. the full-gradient strategy with large d): one thread per
// point pair, directions read through L1/L2.  Correct for any p <= DSVGP_MAXP; not tuned.
template <typename T, typename TK>
__global__ void __launch_bounds__(128)
kdir_fwd_generic(const T* __restrict__ x1, const TK* __restrict__ u1, int n1, int p1, const T* __restrict__ x2,
                 const TK* __restrict__ w2, int n2, int p2, int d, const double* __restrict__ hyp, int use_os,
                 TK diag_add, TK* __restrict__ K, int64_t ldk) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
  if (j >= n2 || i >= n1) return;
  TK al[DSVGP_MAXP], be[DSVGP_MAXP];
  const TK ell = (TK)hyp[0], os = use_os ? (TK)hyp[1] : TK(1), il2 = TK(1) / (ell * ell);
  TK r2 = 0;
  for (int a = 0; a < p1; ++a) al[a] = 0;
  for (int b = 0; b < p2; ++b) be[b] = 0;
  for (int c = 0; c < d; ++c) {
    const TK dl = (TK)x1[(int64_t)i * d + c] - (TK)x2[(int64_t)j * d + c];
    r2 += dl * dl;
    for (int a = 0; a < p1; ++a) al[a] += dl * u1[(int64_t)(i * p1 + a) * d + c];
    for (int b = 0; b < p2; ++b) be[b] += dl * w2[(int64_t)(j * p2 + b) * d + c];
  }
  const TK k = os * dexp<TK>(TK(-0.5) * r2 * il2);
  const bool dg = (diag_add != TK(0)) && (i == j);
  TK* Kb = K + (int64_t)i * (p1 + 1) * ldk + (int64_t)j * (p2 + 1);
  Kb[0] = k + (dg ? diag_add : TK(0));
  for (int b = 0; b < p2; ++b) Kb[1 + b] = k * be[b] * il2;
  for (int a = 0; a < p1; ++a) {
    TK* Ka = Kb + (int64_t)(1 + a) * ldk;
    Ka[0] = -k * al[a] * il2;
    for (int b = 0; b < p2; ++b) {
      TK g = 0;
      for (int c = 0; c < d; ++c) g += u1[(int64_t)(i * p1 + a) * d + c] * w2[(int64_t)(j * p2 + b) * d + c];
      Ka[1 + b] = k * (g * il2 - al[a] * il2 * be[b] * il2) + ((dg && a == b) ? diag_add : TK(0));
    }
  }
}

// ------------------------------------------------------------------------------------------ diag=True branch
// RBFKernelDirectionalGrad.py:110-119: [1, 1/l^2, ..., 1/l^2] per point (times outputscale under ScaleKernel).
template <typename TK>
__global__ void kdir_diag_kernel(int n, int p, const double* __restrict__ hyp, int use_os, TK* __restrict__ out) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (int64_t)n * (p + 1)) return;
  const double ell = hyp[0], os = use_os ? hyp[1] : 1.0;
  out[e] = (TK)((e % (p + 1)) == 0 ? os : os / (ell * ell));
}

// --------------------------------------------------------------------------------------- backward (blocked)
// grid = (column chunks, row tiles).  Per column tile of TJ points:
//   phase A  one thread per point pair recomputes k, alpha, beta, gamma and turns the upstream block
//            g = dK[i*,j*] into the coefficient block Cf such that
//              dx1_i  = sum_j Cf[(i,0),(j,:)] . [x2_j; w_j*]  + x1_i * E0_i + sum_a u_ia * Ea_ia
//              du_ia  = sum_j Cf[(i,a),(j,:)] . [x2_j; w_j*]  + x1_i * Ea_ia
//   phase B  the small GEMM Cf (TI*Q1 x TJ*Q2) x Y (TJ*Q2 x d) accumulated in registers across column tiles.
// Partials per column chunk go to a workspace and are summed (deterministically) by kdir_bwd_reduce.
constexpr int BWD_TI = 16, BWD_TJ = 32, BWD_MAXACC = 16;

template <typename TK> __host__ __device__ constexpr int bwd_ldy(int d) { return d | 1; }

template <typename TK, int P1, int P2>
size_t bwd_smem_bytes(int d) {
  const int ldy = d | 1;
  return sizeof(TK) * (size_t)(BWD_TI * d + BWD_TI * P1 * d + BWD_TJ * (P2 + 1) * ldy +
                               BWD_TI * (P1 + 1) * (BWD_TJ * (P2 + 1) + 1) + BWD_TI * (P1 + 1)) + 64 * sizeof(double);
}

template <typename T, typename TK, int P1, int P2>
__global__ void __launch_bounds__(256)
kdir_bwd_blocked(const T* __restrict__ x1, const TK* __restrict__ u1, int n1, const T* __restrict__ x2,
                 const TK* __restrict__ w2, int n2, int d, const double* __restrict__ hyp, int use_os,
                 const TK* __restrict__ dK, int64_t lddk, int dk_trans, int chunk_pts,
                 TK* __restrict__ part, double* __restrict__ part_sc) {
  constexpr int TI = BWD_TI, TJ = BWD_TJ, Q1 = P1 + 1, Q2 = P2 + 1, LDC = TJ * Q2 + 1, RP = TI / 8;
  const int ldy = d | 1;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* red = reinterpret_cast<double*>(smem_raw);            // [64] reduction scratch
  TK* x1s = reinterpret_cast<TK*>(red + 64);                    // [TI][d]
  TK* u1s = x1s + TI * d;                                       // [TI*P1][d]
  TK* Ys = u1s + TI * P1 * d;                                   // [TJ*Q2][ldy]   row (j,0)=x2_j, (j,b)=w_jb
  TK* Cf = Ys + TJ * Q2 * ldy;                                  // [TI*Q1][LDC]
  TK* rowsum = Cf + TI * Q1 * LDC;                              // [TI*Q1]

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int i0 = blockIdx.y * TI;
  const int jbeg = blockIdx.x * chunk_pts, jend = min(n2, jbeg + chunk_pts);
  const TK ell = (TK)hyp[0], os = use_os ? (TK)hyp[1] : TK(1), il2 = TK(1) / (ell * ell);

  for (int e = tid; e < TI * d; e += 256) {
    const int i = e / d;
    x1s[e] = (i0 + i < n1) ? (TK)x1[(int64_t)i0 * d + e] : TK(0);
  }
  for (int e = tid; e < TI * P1 * d; e += 256) {
    const int ia = e / d;
    u1s[e] = (i0 * P1 + ia < n1 * P1) ? u1[(int64_t)i0 * P1 * d + e] : TK(0);
  }
  for (int e = tid; e < TI * Q1; e += 256) rowsum[e] = 0;

  const int nout = TI * Q1 * d;
  TK acc[BWD_MAXACC];
#pragma unroll
  for (int q = 0; q < BWD_MAXACC; ++q) acc[q] = 0;
  double s_ell = 0, s_os = 0;

  for (int j0 = jbeg; j0 < jend; j0 += TJ) {
    __syncthreads();
    // stage Y = [x2_j; w_j1..w_jP2] rows and the upstream tile
    for (int e = tid; e < TJ * d; e += 256) {
      const int j = e / d, c = e % d;
      Ys[(j * Q2) * ldy + c] = (j0 + j < jend) ? (TK)x2[(int64_t)(j0 + j) * d + c] : TK(0);
    }
    for (int e = tid; e < TJ * P2 * d; e += 256) {
      const int jb = e / d, c = e % d, j = jb / (P2 > 0 ? P2 : 1), b = jb % (P2 > 0 ? P2 : 1);
      Ys[(j * Q2 + 1 + b) * ldy + c] = (j0 + j < jend) ? w2[(int64_t)((j0 + j) * P2 + b) * d + c] : TK(0);
    }
    {
      const int rows = min(TI * Q1, (n1 - i0) * Q1), cols = min(TJ * Q2, (jend - j0) * Q2);
      if (!dk_trans) {
        for (int e = tid; e < TI * Q1 * TJ * Q2; e += 256) {
          const int rr = e / (TJ * Q2), cc = e % (TJ * Q2);
          Cf[rr * LDC + cc] = (rr < rows && cc < cols)
                                  ? dK[(int64_t)(i0 * Q1 + rr) * lddk + (int64_t)j0 * Q2 + cc] : TK(0);
        }
      } else {
        for (int e = tid; e < TI * Q1 * TJ * Q2; e += 256) {
          const int cc = e / (TI * Q1), rr = e % (TI * Q1);
          Cf[rr * LDC + cc] = (rr < rows && cc < cols)
                                  ? dK[(int64_t)((int64_t)j0 * Q2 + cc) * lddk + (i0 * Q1 + rr)] : TK(0);
        }
      }
    }
    __syncthreads();
    // ---- phase A
#pragma unroll
    for (int r = 0; r < RP; ++r) {
      const int i = warp + 8 * r;
      TK r2 = 0, al[P1 > 0 ? P1 : 1], be[P2 > 0 ? P2 : 1], ga[P1 > 0 ? P1 : 1][P2 > 0 ? P2 : 1];
#pragma unroll
      for (int a = 0; a < P1; ++a) al[a] = 0;
#pragma unroll
      for (int b = 0; b < P2; ++b) be[b] = 0;
#pragma unroll
      for (int a = 0; a < P1; ++a)
#pragma unroll
        for (int b = 0; b < P2; ++b) ga[a][b] = 0;
      const TK* yj = Ys + (lane * Q2) * ldy;
      for (int c = 0; c < d; ++c) {
        const TK dl = x1s[i * d + c] - yj[c];
        r2 += dl * dl;
        TK wj[P2 > 0 ? P2 : 1];
#pragma unroll
        for (int b = 0; b < P2; ++b) {
          wj[b] = yj[(1 + b) * ldy + c];
          be[b] += dl * wj[b];
        }
#pragma unroll
        for (int a = 0; a < P1; ++a) {
          const TK ui = u1s[(i * P1 + a) * d + c];
          al[a] += dl * ui;
#pragma unroll
          for (int b = 0; b < P2; ++b) ga[a][b] += ui * wj[b];
        }
      }
#pragma unroll
      for (int a = 0; a < P1; ++a) al[a] *= il2;
#pragma unroll
      for (int b = 0; b < P2; ++b) be[b] *= il2;
      const TK k = os * dexp<TK>(TK(-0.5) * r2 * il2);
      TK* cf = Cf + (i * Q1) * LDC + lane * Q2;
      const TK g00 = cf[0];
      TK q = g00, sdd = 0;           // q = dL/dk ; sdd = sum(dalpha*alpha + dbeta*beta + dgamma*gamma)
      TK dbe[P2 > 0 ? P2 : 1], dal[P1 > 0 ? P1 : 1];
#pragma unroll
      for (int b = 0; b < P2; ++b) {
        dbe[b] = cf[1 + b];
        q += cf[1 + b] * be[b];
      }
#pragma unroll
      for (int a = 0; a < P1; ++a) {
        const TK ga0 = cf[(1 + a) * LDC];
        dal[a] = -ga0;
        q -= ga0 * al[a];
#pragma unroll
        for (int b = 0; b < P2; ++b) {
          const TK gab = cf[(1 + a) * LDC + 1 + b];
          const TK gam = ga[a][b] * il2;
          q += gab * (gam - al[a] * be[b]);
          dal[a] -= gab * be[b];
          dbe[b] -= gab * al[a];
          sdd += k * gab * gam;
          cf[(1 + a) * LDC + 1 + b] = k * gab * il2;       // dgamma / l^2 : multiplies w_jb in du_ia
        }
      }
      const TK e0 = -q * k * il2;
      cf[0] = -e0;
      TK rs0 = e0;
#pragma unroll
      for (int b = 0; b < P2; ++b) {
        const TK db = k * dbe[b];
        sdd += db * be[b];
        cf[1 + b] = db * il2;
      }
      rs0 = warp_sum(rs0);
      if (lane == 0) rowsum[i * Q1] += rs0;
#pragma unroll
      for (int a = 0; a < P1; ++a) {
        const TK da = k * dal[a];
        sdd += da * al[a];
        const TK ea = da * il2;
        cf[(1 + a) * LDC] = -ea;
        const TK rsa = warp_sum(ea);
        if (lane == 0) rowsum[i * Q1 + 1 + a] += rsa;
      }
      s_ell += (double)(q * k * r2 * il2 / ell - TK(2) * sdd / ell);
      s_os += (double)(q * k / os);
    }
    __syncthreads();
    // ---- phase B: acc[(row,c)] += sum_jb Cf[row][jb] * Ys[jb][c]
#pragma unroll
    for (int qd = 0; qd < BWD_MAXACC; ++qd) {
      const int o = tid + 256 * qd;
      if (o < nout) {
        const int row = o / d, c = o % d;
        const TK* cr = Cf + row * LDC;
        TK s = 0;
#pragma unroll 4
        for (int jb = 0; jb < TJ * Q2; ++jb) s += cr[jb] * Ys[jb * ldy + c];
        acc[qd] += s;
      }
    }
  }
  __syncthreads();
  TK* pout = part + ((int64_t)blockIdx.x * n1 * Q1 + (int64_t)i0 * Q1) * d;
#pragma unroll
  for (int qd = 0; qd < BWD_MAXACC; ++qd) {
    const int o = tid + 256 * qd;
    if (o < nout) {
      const int row = o / d, c = o % d, i = row / Q1, a = row % Q1;
      if (i0 + i < n1) {
        TK v = acc[qd] + x1s[i * d + c] * rowsum[row];
        if (a == 0) {
#pragma unroll
          for (int aa = 0; aa < P1; ++aa) v += u1s[(i * P1 + aa) * d + c] * rowsum[i * Q1 + 1 + aa];
        }
        pout[(int64_t)row * d + c] = v;
      }
    }
  }
  const double t_ell = block_sum<double, 256>(s_ell, red);
  const double t_os = block_sum<double, 256>(s_os, red + 32);
  if (tid == 0) {
    const int64_t b = (int64_t)blockIdx.y * gridDim.x + blockIdx.x;
    part_sc[2 * b] = t_ell;
    part_sc[2 * b + 1] = t_os;
  }
}

// ---------------------------------------------------------------------------------- backward (fp32, vectorised)
// Same thread mapping as kdir_fwd_v4 (a lane owns 4 consecutive column points, a CTA keeps one 128-point column tile
// resident and sweeps 64 row points over it, one per warp per pass).  Per row point the lane recomputes its 4 kernel
// blocks, reads the matching 4*(P2+1)-float segments of the upstream rows straight from global memory (contiguous per
// warp), forms the coefficients of d/dx1_i and d/du_ia and accumulates them over the coordinates; a transposing
// butterfly (31 shuffles per 32 values) sums the 32 lanes, and the warp writes ONE partial row per (column tile, row
// point).  kdir_bwd_reduce_rows sums the partials over column tiles (deterministic) and applies the normalisation chain.
template <int NV>
__device__ __forceinline__ void warp_transpose_sum(float (&v)[NV], int lane) {
  // NV = 32: on return lane l holds sum over lanes of v[l] in v[0]
  static_assert(NV == 32, "butterfly works on 32 values");
#pragma unroll
  for (int w = 16; w >= 1; w >>= 1) {
    const bool up = (lane & w) != 0;
#pragma unroll
    for (int i = 0; i < w; ++i) {
      const float send = up ? v[i] : v[i + w];
      const float keep = up ? v[i + w] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, w);
    }
  }
}

// VPL = column points per lane: 4 (a warp spans 128 column points; ~250 registers, one CTA per SM) or 2 (64 column points per
// warp and per CTA tile; half the per-lane arrays, two CTAs = 16 warps per SM -- the kernel is issue-bound on dependent FMA
// chains, ncu: 49 % issue-active with 2 warps per scheduler, so the extra warps are what it needs).
// (+ the staged upstream rows: per warp, two buffers of (P1+1) row segments of 32*VPL*(P2+1) floats -- see the kernel)
template <int P1, int P2, int DP, int VPL>
size_t bwd_v4_smem_bytes() {
  return sizeof(float) * (size_t)(V4_TIB * (P1 + 1) * DP + (P2 + 1) * DP * 32 * VPL + 8 * 2 * (P1 + 1) * 32 * VPL * (P2 + 1)) +
         64 * sizeof(double);
}

// 16- / 8-byte asynchronous global -> shared copies (the upstream block of the NEXT row point is fetched while this one is processed)
template <int BYTES> __device__ __forceinline__ void cp_async_g2s(float* smem_dst, const float* gsrc) {
  const uint32_t dst = (uint32_t)__cvta_generic_to_shared(smem_dst);
  if constexpr (BYTES == 16)
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(dst), "l"(gsrc) : "memory");
  else
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(dst), "l"(gsrc) : "memory");
}

template <int VPL> __device__ __forceinline__ void ld_vpl(const float* p, float (&o)[VPL]) {
  if constexpr (VPL == 4) {
    const float4 t = *reinterpret_cast<const float4*>(p);
    o[0] = t.x; o[1] = t.y; o[2] = t.z; o[3] = t.w;
  } else {
    const float2 t = *reinterpret_cast<const float2*>(p);
    o[0] = t.x; o[1] = t.y;
  }
}

template <int P1, int P2, int DP, int VPL>
__global__ void __launch_bounds__(256, VPL == 4 ? 1 : 2)
kdir_bwd_v4(const float* __restrict__ x1, const float* __restrict__ u1, int n1, const float* __restrict__ x2,
            const float* __restrict__ w2, int n2, int d, const double* __restrict__ hyp, int use_os,
            const float* __restrict__ dK, int64_t lddk, float* __restrict__ part, double* __restrict__ part_sc) {
  constexpr int Q1 = P1 + 1, Q2 = P2 + 1, TJ = 32 * VPL, TIB = V4_TIB, NV = Q1 * DP, NG = (NV + 31) / 32;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* red = reinterpret_cast<double*>(smem_raw);       // [64]
  float* rs = reinterpret_cast<float*>(red + 64);          // [TIB][Q1][DP]
  float* cs = rs + TIB * Q1 * DP;                          // [Q2][DP][TJ]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int i0 = blockIdx.y * TIB, j0 = blockIdx.x * TJ;
  float* gsw = cs + Q2 * DP * TJ + warp * (2 * Q1 * TJ * Q2);   // this warp's [2][Q1][TJ * Q2] staged upstream rows

  // Both tiles arrive through 4-byte cp.async with zero fill: with one CTA per SM nothing hides this prologue, and as a loop
  // of dependent global loads (8 + 15 round trips per thread) it was a quarter of the CTA's life (ncu source page).  Now every
  // element is in flight at once, together with the first row point's upstream rows.
  for (int e = tid; e < TIB * Q1 * DP; e += 256) {
    const int cc = e % DP, ia = e / DP, i = ia / Q1, a = ia % Q1;
    const bool ok = i0 + i < n1 && cc < d;
    const float* src = !ok ? x1 : (a == 0) ? x1 + (int64_t)(i0 + i) * d + cc : u1 + (int64_t)((i0 + i) * P1 + a - 1) * d + cc;
    cp_async4_zfill(rs + e, src, ok);
  }
  {
    const int j = tid & (TJ - 1);
    for (int row = tid / TJ; row < Q2 * DP; row += 256 / TJ) {
      const int b = row / DP, cc = row % DP;
      const bool ok = j0 + j < n2 && cc < d;
      const float* src = !ok ? x2 : (b == 0) ? x2 + (int64_t)(j0 + j) * d + cc : w2 + (int64_t)((j0 + j) * P2 + b - 1) * d + cc;
      cp_async4_zfill(cs + row * TJ + j, src, ok);
    }
  }
  asm volatile("cp.async.commit_group;\n" ::: "memory");

  const float ell = (float)hyp[0], os = use_os ? (float)hyp[1] : 1.f;
  const float il2 = 1.f / (ell * ell), iell = 1.f / ell;
  const bool vec_ok = ((lddk & 3) == 0) && ((reinterpret_cast<uintptr_t>(dK) & 15) == 0);
  const int cols = min(TJ * Q2, (n2 - j0) * Q2);
  double s_ell = 0.0, s_os = 0.0;
  // The upstream rows of a row point are the only large read of the kernel and both warps of a scheduler used to wait for them at
  // the same place of the iteration (ncu: long-scoreboard was the top stall).  For whole, aligned column tiles every lane now
  // fetches ITS OWN segments of the next row point with cp.async while the current one is processed (no cross-lane hand-over:
  // cp.async.wait_group is all the synchronisation there is); ragged / unaligned tiles keep the direct loads.
  constexpr int VWS = VPL == 4 ? 4 : 2, NPIECES = VPL * Q2 / VWS;
  const bool staged = vec_ok && cols == TJ * Q2;           // CTA-uniform
  auto prefetch = [&](int itn) {
    const int gin = i0 + itn * 8 + warp;
    if (itn < TIB / 8 && gin < n1) {
      float* dst = gsw + (itn & 1) * (Q1 * TJ * Q2) + lane * VPL * Q2;
#pragma unroll
      for (int a = 0; a < Q1; ++a) {
        const float* grow = dK + (int64_t)(gin * Q1 + a) * lddk + (int64_t)j0 * Q2 + lane * VPL * Q2;
#pragma unroll
        for (int v = 0; v < NPIECES; ++v) cp_async_g2s<VWS * 4>(dst + a * (TJ * Q2) + VWS * v, grow + VWS * v);
      }
    }
    asm volatile("cp.async.commit_group;\n" ::: "memory");  // (possibly empty: the group count stays uniform)
  };
  if (staged) {
    prefetch(0);
    asm volatile("cp.async.wait_group 1;\n" ::: "memory");   // the tiles (the upstream rows may still be in flight)
  } else {
    asm volatile("cp.async.wait_group 0;\n" ::: "memory");
  }
  __syncthreads();

  for (int it = 0; it < TIB / 8; ++it) {
    const int il = it * 8 + warp, gi = i0 + il;
    if (gi >= n1) break;                                   // warp-uniform
    if (staged) prefetch(it + 1);
    const float* rbase = rs + (il * Q1) * DP;
    // ---- recompute the 4 kernel blocks of this lane
    float r2[VPL], al[P1 > 0 ? P1 : 1][VPL], be[P2 > 0 ? P2 : 1][VPL], ga[P1 > 0 ? P1 : 1][P2 > 0 ? P2 : 1][VPL];
#pragma unroll
    for (int q = 0; q < VPL; ++q) {
      r2[q] = 0.f;
#pragma unroll
      for (int a = 0; a < P1; ++a) al[a][q] = 0.f;
#pragma unroll
      for (int b = 0; b < P2; ++b) be[b][q] = 0.f;
#pragma unroll
      for (int a = 0; a < P1; ++a)
#pragma unroll
        for (int b = 0; b < P2; ++b) ga[a][b][q] = 0.f;
    }
    {
      // dot products on packed pairs (FFMA2): pair h = this lane's column points 2h, 2h + 1
      constexpr int NH = VPL / 2;
      float2 r2p[NH], alp[P1 > 0 ? P1 : 1][NH], bep[P2 > 0 ? P2 : 1][NH], gap[P1 > 0 ? P1 : 1][P2 > 0 ? P2 : 1][NH];
#pragma unroll
      for (int h = 0; h < NH; ++h) {
        r2p[h] = make_float2(0.f, 0.f);
#pragma unroll
        for (int a = 0; a < P1; ++a) alp[a][h] = make_float2(0.f, 0.f);
#pragma unroll
        for (int b = 0; b < P2; ++b) bep[b][h] = make_float2(0.f, 0.f);
#pragma unroll
        for (int a = 0; a < P1; ++a)
#pragma unroll
          for (int b = 0; b < P2; ++b) gap[a][b][h] = make_float2(0.f, 0.f);
      }
#pragma unroll
      for (int c = 0; c < DP; ++c) {
        float xj[VPL], wj[P2 > 0 ? P2 : 1][VPL];
        ld_vpl<VPL>(cs + c * TJ + VPL * lane, xj);
#pragma unroll
        for (int b = 0; b < P2; ++b) ld_vpl<VPL>(cs + ((1 + b) * DP + c) * TJ + VPL * lane, wj[b]);
        const float2 xi = f2bc(rbase[c]);
        float2 ui[P1 > 0 ? P1 : 1];
#pragma unroll
        for (int a = 0; a < P1; ++a) ui[a] = f2bc(rbase[(1 + a) * DP + c]);
#pragma unroll
        for (int h = 0; h < NH; ++h) {
          const float2 dl = f2sub(xi, make_float2(xj[2 * h], xj[2 * h + 1]));
          r2p[h] = f2fma(dl, dl, r2p[h]);
#pragma unroll
          for (int b = 0; b < P2; ++b) bep[b][h] = f2fma(dl, make_float2(wj[b][2 * h], wj[b][2 * h + 1]), bep[b][h]);
#pragma unroll
          for (int a = 0; a < P1; ++a) {
            alp[a][h] = f2fma(dl, ui[a], alp[a][h]);
#pragma unroll
            for (int b = 0; b < P2; ++b) gap[a][b][h] = f2fma(ui[a], make_float2(wj[b][2 * h], wj[b][2 * h + 1]), gap[a][b][h]);
          }
        }
      }
#pragma unroll
      for (int h = 0; h < NH; ++h) {                      // unpack (register renaming only)
        r2[2 * h] = r2p[h].x; r2[2 * h + 1] = r2p[h].y;
#pragma unroll
        for (int a = 0; a < P1; ++a) { al[a][2 * h] = alp[a][h].x; al[a][2 * h + 1] = alp[a][h].y; }
#pragma unroll
        for (int b = 0; b < P2; ++b) { be[b][2 * h] = bep[b][h].x; be[b][2 * h + 1] = bep[b][h].y; }
#pragma unroll
        for (int a = 0; a < P1; ++a)
#pragma unroll
          for (int b = 0; b < P2; ++b) { ga[a][b][2 * h] = gap[a][b][h].x; ga[a][b][2 * h + 1] = gap[a][b][h].y; }
      }
    }
    // ---- upstream blocks: row (gi, a) holds this lane's 4*Q2 consecutive floats
    // (VPL * Q2 consecutive floats per lane: float4 pieces when VPL = 4, float2 pieces when VPL = 2 -- 8-byte aligned for any Q2)
    constexpr int VW = VPL == 4 ? 4 : 2, NPIECE = VPL * Q2 / VW;
    static_assert((VPL * Q2) % VW == 0, "upstream segment must split into whole vector pieces");
    float g[Q1][VPL * Q2];
    if (staged) {
      asm volatile("cp.async.wait_group 1;\n" ::: "memory");
      const float* src = gsw + (it & 1) * (Q1 * TJ * Q2) + lane * VPL * Q2;
#pragma unroll
      for (int a = 0; a < Q1; ++a)
#pragma unroll
        for (int v = 0; v < NPIECE; ++v) {
          if constexpr (VW == 4) {
            const float4 t = *reinterpret_cast<const float4*>(src + a * (TJ * Q2) + 4 * v);
            g[a][4 * v] = t.x; g[a][4 * v + 1] = t.y; g[a][4 * v + 2] = t.z; g[a][4 * v + 3] = t.w;
          } else {
            const float2 t = *reinterpret_cast<const float2*>(src + a * (TJ * Q2) + 2 * v);
            g[a][2 * v] = t.x; g[a][2 * v + 1] = t.y;
          }
        }
    } else
#pragma unroll
    for (int a = 0; a < Q1; ++a) {
      const float* grow = dK + (int64_t)(gi * Q1 + a) * lddk + (int64_t)j0 * Q2 + lane * VPL * Q2;
#pragma unroll
      for (int v = 0; v < NPIECE; ++v) {
        const int col = lane * VPL * Q2 + VW * v;
        if (vec_ok && col + VW - 1 < cols) {
          if constexpr (VW == 4) {
            const float4 t = *reinterpret_cast<const float4*>(grow + 4 * v);
            g[a][4 * v] = t.x; g[a][4 * v + 1] = t.y; g[a][4 * v + 2] = t.z; g[a][4 * v + 3] = t.w;
          } else {
            const float2 t = *reinterpret_cast<const float2*>(grow + 2 * v);
            g[a][2 * v] = t.x; g[a][2 * v + 1] = t.y;
          }
        } else {
#pragma unroll
          for (int z = 0; z < VW; ++z) g[a][VW * v + z] = (col + z < cols) ? grow[VW * v + z] : 0.f;
        }
      }
    }
    // ---- coefficients per pair
    float e0[VPL], ea[P1 > 0 ? P1 : 1][VPL], eb[P2 > 0 ? P2 : 1][VPL], hab[P1 > 0 ? P1 : 1][P2 > 0 ? P2 : 1][VPL];
#pragma unroll
    for (int q = 0; q < VPL; ++q) {
      const float k = os * expf(-0.5f * r2[q] * il2);
      float as[P1 > 0 ? P1 : 1], bs[P2 > 0 ? P2 : 1];
#pragma unroll
      for (int a = 0; a < P1; ++a) as[a] = al[a][q] * il2;
#pragma unroll
      for (int b = 0; b < P2; ++b) bs[b] = be[b][q] * il2;
      float qk = g[0][q * Q2], sdd = 0.f;
      float dbs[P2 > 0 ? P2 : 1], das[P1 > 0 ? P1 : 1];
#pragma unroll
      for (int b = 0; b < P2; ++b) {
        dbs[b] = g[0][q * Q2 + 1 + b];
        qk += dbs[b] * bs[b];
      }
#pragma unroll
      for (int a = 0; a < P1; ++a) {
        const float ga0 = g[1 + (a < P1 ? a : 0)][q * Q2];
        das[a] = -ga0;
        qk -= ga0 * as[a];
#pragma unroll
        for (int b = 0; b < P2; ++b) {
          const float gab = g[1 + (a < P1 ? a : 0)][q * Q2 + 1 + b];
          const float gam = ga[a][b][q] * il2;
          qk += gab * (gam - as[a] * bs[b]);
          das[a] -= gab * bs[b];
          dbs[b] -= gab * as[a];
          sdd += k * gab * gam;
          hab[a][b][q] = k * gab * il2;
        }
      }
      e0[q] = -qk * k * il2;
#pragma unroll
      for (int b = 0; b < P2; ++b) {
        sdd += k * dbs[b] * bs[b];
        eb[b][q] = k * dbs[b] * il2;
      }
#pragma unroll
      for (int a = 0; a < P1; ++a) {
        sdd += k * das[a] * as[a];
        ea[a][q] = k * das[a] * il2;
      }
      s_ell += (double)(qk * k * r2[q] * il2 * iell - 2.f * sdd * iell);
      s_os += (double)(qk * k / os);
    }
    // ---- accumulate d/dx1_i and d/du_ia over this lane's 4 pairs
    float acc[NV];
#pragma unroll
    for (int f = 0; f < NV; ++f) acc[f] = 0.f;
    {
      constexpr int NH = VPL / 2;
      // the coefficients as packed pairs (register renaming), then FFMA2 over the coordinates; the two halves of an accumulator
      // are added once per coordinate
      float2 e0p[NH], eap[P1 > 0 ? P1 : 1][NH], ebp[P2 > 0 ? P2 : 1][NH], habp[P1 > 0 ? P1 : 1][P2 > 0 ? P2 : 1][NH];
#pragma unroll
      for (int h = 0; h < NH; ++h) {
        e0p[h] = make_float2(e0[2 * h], e0[2 * h + 1]);
#pragma unroll
        for (int a = 0; a < P1; ++a) eap[a][h] = make_float2(ea[a][2 * h], ea[a][2 * h + 1]);
#pragma unroll
        for (int b = 0; b < P2; ++b) ebp[b][h] = make_float2(eb[b][2 * h], eb[b][2 * h + 1]);
#pragma unroll
        for (int a = 0; a < P1; ++a)
#pragma unroll
          for (int b = 0; b < P2; ++b) habp[a][b][h] = make_float2(hab[a][b][2 * h], hab[a][b][2 * h + 1]);
      }
#pragma unroll
      for (int c = 0; c < DP; ++c) {
        float xj[VPL], wj[P2 > 0 ? P2 : 1][VPL];
        ld_vpl<VPL>(cs + c * TJ + VPL * lane, xj);
#pragma unroll
        for (int b = 0; b < P2; ++b) ld_vpl<VPL>(cs + ((1 + b) * DP + c) * TJ + VPL * lane, wj[b]);
        const float2 xi = f2bc(rbase[c]);
        float2 ui[P1 > 0 ? P1 : 1];
#pragma unroll
        for (int a = 0; a < P1; ++a) ui[a] = f2bc(rbase[(1 + a) * DP + c]);
        float2 gx = make_float2(0.f, 0.f), gu[P1 > 0 ? P1 : 1];
#pragma unroll
        for (int a = 0; a < P1; ++a) gu[a] = make_float2(0.f, 0.f);
#pragma unroll
        for (int h = 0; h < NH; ++h) {
          const float2 dl = f2sub(xi, make_float2(xj[2 * h], xj[2 * h + 1]));
          gx = f2fma(e0p[h], dl, gx);
#pragma unroll
          for (int b = 0; b < P2; ++b) gx = f2fma(ebp[b][h], make_float2(wj[b][2 * h], wj[b][2 * h + 1]), gx);
#pragma unroll
          for (int a = 0; a < P1; ++a) {
            gx = f2fma(eap[a][h], ui[a], gx);
            gu[a] = f2fma(eap[a][h], dl, gu[a]);
#pragma unroll
            for (int b = 0; b < P2; ++b) gu[a] = f2fma(habp[a][b][h], make_float2(wj[b][2 * h], wj[b][2 * h + 1]), gu[a]);
          }
        }
        acc[c] = gx.x + gx.y;
#pragma unroll
        for (int a = 0; a < P1; ++a) acc[(1 + a) * DP + c] = gu[a].x + gu[a].y;
      }
    }
    // ---- sum over the 32 lanes, one partial row per (column tile, row point)
    float* prow = part + ((int64_t)blockIdx.x * n1 * Q1 + (int64_t)gi * Q1) * d;
    constexpr int NFULL = NV / 32, REM = NV % 32;       // whole groups of 32 values: transposing butterfly; a short remainder: plain sums
#pragma unroll
    for (int grp = 0; grp < NFULL + (REM > 8 ? 1 : 0); ++grp) {
      float v[32];
#pragma unroll
      for (int f = 0; f < 32; ++f) v[f] = (grp * 32 + f < NV) ? acc[(grp * 32 + f < NV) ? grp * 32 + f : 0] : 0.f;
      warp_transpose_sum<32>(v, lane);
      const int f = grp * 32 + lane;                        // flattened (a', c) with pitch DP
      if (f < NV) {
        const int a = f / DP, c = f % DP;
        if (c < d) prow[a * d + c] = v[0];
      }
    }
    if constexpr (REM > 0 && REM <= 8) {
      float mine = 0.f;
#pragma unroll
      for (int r = 0; r < REM; ++r) {
        const float sr = warp_sum(acc[NFULL * 32 + r]);
        if (lane == r) mine = sr;
      }
      const int f = NFULL * 32 + lane;
      if (lane < REM) {
        const int a = f / DP, c = f % DP;
        if (c < d) prow[a * d + c] = mine;
      }
    }
  }
  const double t_ell = block_sum<double, 256>(s_ell, red);
  const double t_os = block_sum<double, 256>(s_os, red + 32);
  if (tid == 0) {
    const int64_t b = (int64_t)blockIdx.y * gridDim.x + blockIdx.x;
    part_sc[2 * b] = t_ell;
    part_sc[2 * b + 1] = t_os;
  }
}

// ------------------------------------------------------------------------- backward, data side (fp32, vectorised)
// d/dx2_j and d/dw_jb of sum(dK * K(x1, x2)) -- the gradient w.r.t. the data points and data-side directions of K_zx.  With
// D = x1_i - x2_j and the coefficients e0, ea, eb, hab of kdir_bwd_v4 (which give d/dx1_i = sum_j e0 D + eb w_jb + ea u_ia):
//   d/dx2_j  = -sum_i (e0 D + sum_b eb w_jb + sum_a ea u_ia)        (x2 enters through -D only)
//   d/dw_jb  =  sum_i (eb D + sum_a hab u_ia)
// One thread per column (data) point, COLS_TJ consecutive points per CTA; the CTA sweeps a chunk of row (inducing) points,
// staged COLS_RT at a time in shared memory and read as broadcasts.  Each thread reads its own Q2 consecutive floats of every
// upstream row (a warp: 32 * Q2 * 4 contiguous bytes), so dK is read once and coalesced and K is recomputed.  The thread's
// column operands and its (1 + P2) * DP sums stay in registers; one fp64 partial per (row chunk, column point) goes to the
// workspace and kdir_bwd_reduce_rows adds the chunks in a fixed order (deterministic, no atomics) and applies the
// normalisation chain of w.  A separate kernel rather than a second output of kdir_bwd_v4, which already needs ~250 registers.
constexpr int COLS_TJ = 256, COLS_RT = 32, COLS_CTAS = 148 * 4;

// row chunks of the data-side kernel: about COLS_CTAS CTAs in all, at least 8 row points per chunk
__host__ __device__ inline int cols_num_chunks(int n1, int n2) {
  const int nct = (n2 + COLS_TJ - 1) / COLS_TJ, maxch = (n1 + 7) / 8;
  int want = (COLS_CTAS + nct - 1) / nct;
  if (want > maxch) want = maxch;
  if (want < 1) want = 1;
  const int pts = (n1 + want - 1) / want;
  return (n1 + pts - 1) / pts;
}

template <int P1, int P2, int DP>
__global__ void __launch_bounds__(COLS_TJ, 1)
kdir_bwd_cols_v4(const float* __restrict__ x1, const float* __restrict__ u1, int n1, const float* __restrict__ x2,
                 const float* __restrict__ w2, int n2, int d, const double* __restrict__ hyp, int use_os,
                 const float* __restrict__ dK, int64_t lddk, int chunk_pts, double* __restrict__ part) {
  constexpr int Q1 = P1 + 1, Q2 = P2 + 1, PA = P1 > 0 ? P1 : 1, PB = P2 > 0 ? P2 : 1;
  __shared__ __align__(16) float rs[COLS_RT * Q1 * DP];   // [row point][Q1][DP]: x1_i then u_i1..u_iP1
  const int tid = threadIdx.x, j = blockIdx.x * COLS_TJ + tid;
  const bool act = j < n2;
  const int ibeg = blockIdx.y * chunk_pts, iend = min(n1, ibeg + chunk_pts);

  float xj[DP], wj[PB][DP], sx[DP], sw[PB][DP];
#pragma unroll
  for (int c = 0; c < DP; ++c) {
    xj[c] = (act && c < d) ? x2[(int64_t)j * d + c] : 0.f;
    sx[c] = 0.f;
#pragma unroll
    for (int b = 0; b < P2; ++b) {
      wj[b][c] = (act && c < d) ? w2[((int64_t)j * P2 + b) * d + c] : 0.f;
      sw[b][c] = 0.f;
    }
  }
  const float ell = (float)hyp[0], os = use_os ? (float)hyp[1] : 1.f;
  const float il2 = 1.f / (ell * ell);
  const float* gcol = dK + (act ? (int64_t)j * Q2 : 0);
  auto load_g = [&](int gi, float (&g)[Q1][Q2]) {
#pragma unroll
    for (int a = 0; a < Q1; ++a)
#pragma unroll
      for (int b = 0; b < Q2; ++b) g[a][b] = act ? gcol[(int64_t)(gi * Q1 + a) * lddk + b] : 0.f;
  };

  for (int i0 = ibeg; i0 < iend; i0 += COLS_RT) {
    const int nr = min(COLS_RT, iend - i0);
    __syncthreads();
    for (int e = tid; e < COLS_RT * Q1 * DP; e += COLS_TJ) {
      const int cc = e % DP, ia = e / DP, i = ia / Q1, a = ia % Q1;
      const bool ok = i < nr && cc < d;
      rs[e] = !ok ? 0.f : (a == 0) ? x1[(int64_t)(i0 + i) * d + cc] : u1[((int64_t)(i0 + i) * P1 + a - 1) * d + cc];
    }
    __syncthreads();
    float g[Q1][Q2], gn[Q1][Q2];
    load_g(i0, g);
    for (int il = 0; il < nr; ++il) {
      load_g(min(i0 + il + 1, iend - 1), gn);             // the next row point's upstream block, in flight during this one
      const float* rb = rs + il * Q1 * DP;
      // ---- recompute r2 = |D|^2, alpha = D.u, beta = D.w, gamma = u.w
      float r2 = 0.f, al[PA], be[PB], ga[PA][PB];
#pragma unroll
      for (int a = 0; a < P1; ++a) al[a] = 0.f;
#pragma unroll
      for (int b = 0; b < P2; ++b) be[b] = 0.f;
#pragma unroll
      for (int a = 0; a < P1; ++a)
#pragma unroll
        for (int b = 0; b < P2; ++b) ga[a][b] = 0.f;
#pragma unroll
      for (int c4 = 0; c4 < DP; c4 += 4) {
        const float4 xr = *reinterpret_cast<const float4*>(rb + c4);
        float4 ur[PA];
#pragma unroll
        for (int a = 0; a < P1; ++a) ur[a] = *reinterpret_cast<const float4*>(rb + (1 + a) * DP + c4);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int c = c4 + k;
          const float dl = (k == 0 ? xr.x : k == 1 ? xr.y : k == 2 ? xr.z : xr.w) - xj[c];
          r2 = fmaf(dl, dl, r2);
#pragma unroll
          for (int b = 0; b < P2; ++b) be[b] = fmaf(dl, wj[b][c], be[b]);
#pragma unroll
          for (int a = 0; a < P1; ++a) {
            const float ui = k == 0 ? ur[a].x : k == 1 ? ur[a].y : k == 2 ? ur[a].z : ur[a].w;
            al[a] = fmaf(dl, ui, al[a]);
#pragma unroll
            for (int b = 0; b < P2; ++b) ga[a][b] = fmaf(ui, wj[b][c], ga[a][b]);
          }
        }
      }
      // ---- coefficients (as in kdir_bwd_v4)
      const float k = os * expf(-0.5f * r2 * il2);
      float as[PA], bs[PB], das[PA], dbs[PB], hab[PA][PB];
#pragma unroll
      for (int a = 0; a < P1; ++a) as[a] = al[a] * il2;
#pragma unroll
      for (int b = 0; b < P2; ++b) bs[b] = be[b] * il2;
      float qk = g[0][0];
#pragma unroll
      for (int b = 0; b < P2; ++b) {
        dbs[b] = g[0][1 + b];
        qk += dbs[b] * bs[b];
      }
#pragma unroll
      for (int a = 0; a < P1; ++a) {
        const float ga0 = g[1 + (a < P1 ? a : 0)][0];
        das[a] = -ga0;
        qk -= ga0 * as[a];
#pragma unroll
        for (int b = 0; b < P2; ++b) {
          const float gab = g[1 + (a < P1 ? a : 0)][1 + b];
          qk += gab * (ga[a][b] * il2 - as[a] * bs[b]);
          das[a] -= gab * bs[b];
          dbs[b] -= gab * as[a];
          hab[a][b] = k * gab * il2;
        }
      }
      const float e0 = -qk * k * il2;
      float ea[PA], eb[PB];
#pragma unroll
      for (int a = 0; a < P1; ++a) ea[a] = k * das[a] * il2;
#pragma unroll
      for (int b = 0; b < P2; ++b) eb[b] = k * dbs[b] * il2;
      // ---- accumulate over this row point
#pragma unroll
      for (int c4 = 0; c4 < DP; c4 += 4) {
        const float4 xr = *reinterpret_cast<const float4*>(rb + c4);
        float4 ur[PA];
#pragma unroll
        for (int a = 0; a < P1; ++a) ur[a] = *reinterpret_cast<const float4*>(rb + (1 + a) * DP + c4);
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          const int c = c4 + kk;
          const float dl = (kk == 0 ? xr.x : kk == 1 ? xr.y : kk == 2 ? xr.z : xr.w) - xj[c];
          float tx = e0 * dl;
#pragma unroll
          for (int b = 0; b < P2; ++b) tx = fmaf(eb[b], wj[b][c], tx);
          float tw[PB];
#pragma unroll
          for (int b = 0; b < P2; ++b) tw[b] = eb[b] * dl;
#pragma unroll
          for (int a = 0; a < P1; ++a) {
            const float ui = kk == 0 ? ur[a].x : kk == 1 ? ur[a].y : kk == 2 ? ur[a].z : ur[a].w;
            tx = fmaf(ea[a], ui, tx);
#pragma unroll
            for (int b = 0; b < P2; ++b) tw[b] = fmaf(hab[a][b], ui, tw[b]);
          }
          sx[c] -= tx;
#pragma unroll
          for (int b = 0; b < P2; ++b) sw[b][c] += tw[b];
        }
      }
#pragma unroll
      for (int a = 0; a < Q1; ++a)
#pragma unroll
        for (int b = 0; b < Q2; ++b) g[a][b] = gn[a][b];
    }
  }
  if (!act) return;
  double* prow = part + ((int64_t)blockIdx.y * n2 * Q2 + (int64_t)j * Q2) * d;   // rows (j, 0..P2) of kdir_bwd_reduce_rows
#pragma unroll
  for (int c = 0; c < DP; ++c)
    if (c < d) {
      prow[c] = (double)sx[c];
#pragma unroll
      for (int b = 0; b < P2; ++b) prow[(1 + b) * d + c] = (double)sw[b][c];
    }
}

// ------------------------------------------------------------------------------------ backward (runtime p)
// One thread per point pair, atomics into double accumulators.  Any p <= DSVGP_MAXP; not tuned.
template <typename T, typename TK>
__global__ void __launch_bounds__(128)
kdir_bwd_generic(const T* __restrict__ x1, const TK* __restrict__ u1, int n1, int p1, const T* __restrict__ x2,
                 const TK* __restrict__ w2, int n2, int p2, int d, const double* __restrict__ hyp, int use_os,
                 const TK* __restrict__ dK, int64_t lddk, int dk_trans, double* __restrict__ gx /*[n1][d]*/,
                 double* __restrict__ gu /*[n1*p1][d]*/, double* __restrict__ gsc /*[2]*/) {
  // Every thread of a CTA works on the SAME row point i (and 128 consecutive column points): contributions are summed over
  // the warp before they reach memory -- one atomic per warp and value instead of 128 colliding ones per CTA (measured at
  // p = d = 5: 0.64 -> see scratch/grad_p_time.py).  Threads past the last column point run on a clamped j with k = 0.
  const int jraw = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
  const bool act = jraw < n2;
  const int j = act ? jraw : n2 - 1;
  const bool lead = (threadIdx.x & 31) == 0;
  double s_ell = 0, s_os = 0;
  if (i < n1) {
    TK al[DSVGP_MAXP], be[DSVGP_MAXP];
    const TK ell = (TK)hyp[0], os = use_os ? (TK)hyp[1] : TK(1), il2 = TK(1) / (ell * ell);
    TK r2 = 0;
    for (int a = 0; a < p1; ++a) al[a] = 0;
    for (int b = 0; b < p2; ++b) be[b] = 0;
    for (int c = 0; c < d; ++c) {
      const TK dl = (TK)x1[(int64_t)i * d + c] - (TK)x2[(int64_t)j * d + c];
      r2 += dl * dl;
      for (int a = 0; a < p1; ++a) al[a] += dl * u1[(int64_t)(i * p1 + a) * d + c];
      for (int b = 0; b < p2; ++b) be[b] += dl * w2[(int64_t)(j * p2 + b) * d + c];
    }
    for (int a = 0; a < p1; ++a) al[a] *= il2;
    for (int b = 0; b < p2; ++b) be[b] *= il2;
    const TK k = act ? os * dexp<TK>(TK(-0.5) * r2 * il2) : TK(0);
    auto G = [&](int a, int b) -> TK {
      const int64_t r = (int64_t)i * (p1 + 1) + a, c = (int64_t)j * (p2 + 1) + b;
      return dk_trans ? dK[c * lddk + r] : dK[r * lddk + c];
    };
    TK q = G(0, 0), sdd = 0;
    for (int b = 0; b < p2; ++b) q += G(0, 1 + b) * be[b];
    for (int a = 0; a < p1; ++a) q -= G(1 + a, 0) * al[a];
    // pass 1 over (a,b): gamma-dependent terms
    for (int a = 0; a < p1; ++a)
      for (int b = 0; b < p2; ++b) {
        TK g = 0;
        for (int c = 0; c < d; ++c) g += u1[(int64_t)(i * p1 + a) * d + c] * w2[(int64_t)(j * p2 + b) * d + c];
        g *= il2;
        const TK gab = G(1 + a, 1 + b);
        q += gab * (g - al[a] * be[b]);
        sdd += k * gab * g;
      }
    const TK e0 = -q * k * il2;
    for (int c = 0; c < d; ++c) {
      const TK dl = (TK)x1[(int64_t)i * d + c] - (TK)x2[(int64_t)j * d + c];
      TK gxc = e0 * dl;
      for (int b = 0; b < p2; ++b) {
        TK db = G(0, 1 + b);
        for (int a = 0; a < p1; ++a) db -= G(1 + a, 1 + b) * al[a];
        gxc += k * db * il2 * w2[(int64_t)(j * p2 + b) * d + c];
      }
      for (int a = 0; a < p1; ++a) {
        TK da = -G(1 + a, 0);
        TK guc = 0;
        for (int b = 0; b < p2; ++b) {
          da -= G(1 + a, 1 + b) * be[b];
          guc += k * G(1 + a, 1 + b) * il2 * w2[(int64_t)(j * p2 + b) * d + c];
        }
        const TK ea = k * da * il2;
        gxc += ea * u1[(int64_t)(i * p1 + a) * d + c];
        guc += ea * dl;
        guc = warp_sum(guc);
        if (lead) atomicAdd(&gu[(int64_t)(i * p1 + a) * d + c], (double)guc);
      }
      gxc = warp_sum(gxc);
      if (lead) atomicAdd(&gx[(int64_t)i * d + c], (double)gxc);
    }
    for (int b = 0; b < p2; ++b) {
      TK db = G(0, 1 + b);
      for (int a = 0; a < p1; ++a) db -= G(1 + a, 1 + b) * al[a];
      sdd += k * db * be[b];
    }
    for (int a = 0; a < p1; ++a) {
      TK da = -G(1 + a, 0);
      for (int b = 0; b < p2; ++b) da -= G(1 + a, 1 + b) * be[b];
      sdd += k * da * al[a];
    }
    s_ell = (double)(q * k * r2 * il2 / ell - TK(2) * sdd / ell);
    s_os = (double)(q * k / os);
  }
  __shared__ double red[64];
  const double t_ell = block_sum<double, 128>(s_ell, red);
  const double t_os = block_sum<double, 128>(s_os, red + 32);
  if (threadIdx.x == 0) {
    atomicAdd(&gsc[0], t_ell);
    atomicAdd(&gsc[1], t_os);
  }
}

// One warp per output row (i,a'): sums the column-chunk partials (TP: fp32 or fp64), applies the chain rule of the row
// normalisation (RBFKernelDirectionalGrad.py:57) for direction rows, and ACCUMULATES scale*grad into the
// double gradient buffers gx (n1,d) / gv (n1*p1,d).
template <typename TP, typename TK>
__global__ void kdir_bwd_reduce_rows(const TP* __restrict__ part, int nchunk, int n1, int p1, int d,
                                     const TK* __restrict__ u1, const TK* __restrict__ inv_norm, double scale,
                                     double* __restrict__ gx, double* __restrict__ gv) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  const int Q1 = p1 + 1;
  if (row >= n1 * Q1) return;
  const int i = row / Q1, a = row % Q1;
  if (a == 0) {
    if (!gx) return;
    for (int c = lane; c < d; c += 32) {
      double s = 0;
      for (int ch = 0; ch < nchunk; ++ch) s += (double)part[((int64_t)ch * n1 * Q1 + row) * d + c];
      gx[(int64_t)i * d + c] += scale * s;
    }
  } else {
    if (!gv) return;
    const int64_t vr = (int64_t)i * p1 + (a - 1);
    double dot = 0;
    for (int c = lane; c < d; c += 32) {
      double s = 0;
      for (int ch = 0; ch < nchunk; ++ch) s += (double)part[((int64_t)ch * n1 * Q1 + row) * d + c];
      dot += s * (double)u1[vr * d + c];
    }
    dot = warp_sum(dot);
    const double inv = (double)inv_norm[vr];
    for (int c = lane; c < d; c += 32) {
      double s = 0;
      for (int ch = 0; ch < nchunk; ++ch) s += (double)part[((int64_t)ch * n1 * Q1 + row) * d + c];
      gv[vr * d + c] += scale * (s - (double)u1[vr * d + c] * dot) * inv;
    }
  }
}

// generic path: gu holds gradients w.r.t. the NORMALISED directions; apply the chain rule into gv
template <typename TK>
__global__ void kdir_bwd_chain_generic(const double* __restrict__ gxt, const double* __restrict__ gut, int n1,
                                       int p1, int d, const TK* __restrict__ u1, const TK* __restrict__ inv_norm,
                                       double scale, double* __restrict__ gx, double* __restrict__ gv) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row < n1) {
    if (gx)
      for (int c = lane; c < d; c += 32) gx[(int64_t)row * d + c] += scale * gxt[(int64_t)row * d + c];
  } else if (row < n1 + n1 * p1) {
    if (!gv) return;
    const int64_t vr = row - n1;
    double dot = 0;
    for (int c = lane; c < d; c += 32) dot += gut[vr * d + c] * (double)u1[vr * d + c];
    dot = warp_sum(dot);
    const double inv = (double)inv_norm[vr];
    for (int c = lane; c < d; c += 32)
      gv[vr * d + c] += scale * (gut[vr * d + c] - (double)u1[vr * d + c] * dot) * inv;
  }
}

__global__ void kdir_bwd_reduce_scalars(const double* __restrict__ part_sc, int nblocks, double* __restrict__ gsc) {
  __shared__ double red[64];
  double a = 0, b = 0;
  for (int e = threadIdx.x; e < nblocks; e += 256) {
    a += part_sc[2 * e];
    b += part_sc[2 * e + 1];
  }
  a = block_sum<double, 256>(a, red);
  b = block_sum<double, 256>(b, red + 32);
  if (threadIdx.x == 0) {
    gsc[0] += a;
    gsc[1] += b;
  }
}

// ================================================================================================ host side
template <typename T, typename TK>
int normalize_dirs(const T* v, int rows, int d, TK* vhat, TK* inv_norm, cudaStream_t st, int* cidx, int* canon_flag) {
  if (rows <= 0) return DSVGP_OK;
  normalize_dirs_kernel<T, TK><<<ceil_div(rows, 8), 256, 0, st>>>(v, rows, d, vhat, inv_norm, cidx, canon_flag);
  CHECK_LAUNCH();
  return DSVGP_OK;
}

template <typename T, typename TK, int P1, int P2>
static int launch_fwd_blocked(const T* x1, const TK* u1, int n1, const T* x2, const TK* w2, int n2, int d,
                              const double* hyp, int use_os, double diag_add, TK* K, int64_t ldk, cudaStream_t st) {
  constexpr size_t smem = fwd_smem_bytes<TK, P1, P2>();
  auto kern = kdir_fwd_blocked<T, TK, P1, P2>;
  if (smem > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  dim3 grid(ceil_div(n2, FWD_TJ), ceil_div(n1, FwdTile<TK>::TI));
  kern<<<grid, 256, smem, st>>>(x1, u1, n1, x2, w2, n2, d, hyp, use_os, (TK)diag_add, K, ldk);
  CHECK_LAUNCH();
  return DSVGP_OK;
}

template <int P1, int P2>
static int launch_fwd_v4(const float* x1, const float* u1, int n1, const float* x2, const float* w2, const int* cidx2,
                         const int* canon_flag, int n2, int d, const double* hyp, int use_os, double diag_add, float* K,
                         int64_t ldk, float* Klo, cudaStream_t st, __half* Kh = nullptr, __half* Kl = nullptr,
                         int64_t ldkh = 0, const float* hscale = nullptr) {
  int tib = g_fwd_tib;
  if (tib <= 0) tib = ((int64_t)ceil_div(n2, V4_TJ) * ceil_div(n1, V4_TIB) < 1024) ? V4_TIB / 2 : V4_TIB;
  const int64_t out_bytes = (int64_t)n1 * (P1 + 1) * n2 * (P2 + 1) * 4 * (Klo ? 2 : 1);
  const int stream_stores = g_fwd_stream_stores == 2 ? (out_bytes > (int64_t)(64 << 20)) : g_fwd_stream_stores;
  const size_t smem = fwd_v4_smem_bytes<P1, P2>((d + 3) & ~3, tib);
  dim3 grid(ceil_div(n2, V4_TJ), ceil_div(n1, tib));
  auto gen = Kh ? kdir_fwd_v4<P1, P2, 2, 0> : Klo ? kdir_fwd_v4<P1, P2, 1, 0> : kdir_fwd_v4<P1, P2, 0, 0>;
  if (smem > 48 * 1024) cudaFuncSetAttribute(gen, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  gen<<<grid, 256, smem, st>>>(x1, u1, n1, x2, w2, cidx2, canon_flag, n2, d, hyp, use_os, (float)diag_add, K, ldk, Klo, tib,
                               stream_stores, Kh, Kl, ldkh, hscale);
  CHECK_LAUNCH();
  if constexpr (P2 > 0) {                   // (no canonical variant without column-side directions: not even compiled)
    if (cidx2 && canon_flag) {
      auto can = Kh ? kdir_fwd_v4<P1, P2, 2, 1> : Klo ? kdir_fwd_v4<P1, P2, 1, 1> : kdir_fwd_v4<P1, P2, 0, 1>;
      if (smem > 48 * 1024) cudaFuncSetAttribute(can, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      can<<<grid, 256, smem, st>>>(x1, u1, n1, x2, w2, cidx2, canon_flag, n2, d, hyp, use_os, (float)diag_add, K, ldk, Klo, tib,
                                   stream_stores, Kh, Kl, ldkh, hscale);
      CHECK_LAUNCH();
    }
  }
  return Kh ? 2 : Klo ? 1 : DSVGP_OK;       // 1: the lo companion was written too; 2: only the half split was written
}

template <typename T, typename TK>
int kdir_fwd(const T* x1, const TK* u1, int n1, int p1, const T* x2, const TK* w2, int n2, int p2, int d,
             const double* hyp, int use_os, double diag_add, TK* K, int64_t ldk, cudaStream_t st, const int* cidx2,
             const int* canon_flag, TK* Klo, void* Kh, void* Kl, int64_t ldkh, const float* hscale) {
  if (n1 <= 0 || n2 <= 0) return DSVGP_OK;
  if (p1 < 0 || p2 < 0 || p1 > DSVGP_MAXP || p2 > DSVGP_MAXP || d <= 0) return DSVGP_ERR_ARG;
  if constexpr (sizeof(T) == 4 && sizeof(TK) == 4) {
    // wide enough for 128-point column tiles, and the resident tiles fit in shared memory
    const int dpad = (d + 3) & ~3;
    const size_t need = sizeof(float) * (size_t)(V4_TIB * (p1 + 1) * dpad + (p2 + 1) * dpad * V4_TJ + 8 * V4_TJ * (p2 + 1));
    if (n2 >= 512 && need <= 200 * 1024) {
#define V4_CASE(A, B)                                                                                          \
  if (p1 == A && p2 == B)                                                                                      \
    return launch_fwd_v4<A, B>(x1, u1, n1, x2, w2, cidx2, canon_flag, n2, d, hyp, use_os, diag_add, K, ldk, Klo, st,          \
                               static_cast<__half*>(Kh), static_cast<__half*>(Kl), ldkh, hscale);
      V4_CASE(0, 0) V4_CASE(1, 1) V4_CASE(2, 2) V4_CASE(3, 3) V4_CASE(1, 0) V4_CASE(2, 0) V4_CASE(3, 0)
#undef V4_CASE
    }
  }
#define FWD_CASE(A, B)                                                                                         \
  if (p1 == A && p2 == B)                                                                                      \
    return launch_fwd_blocked<T, TK, A, B>(x1, u1, n1, x2, w2, n2, d, hyp, use_os, diag_add, K, ldk, st);
  FWD_CASE(0, 0) FWD_CASE(1, 1) FWD_CASE(2, 2) FWD_CASE(3, 3) FWD_CASE(1, 0) FWD_CASE(2, 0) FWD_CASE(3, 0)
#undef FWD_CASE
  dim3 grid(ceil_div(n2, 128), n1);
  kdir_fwd_generic<T, TK><<<grid, 128, 0, st>>>(x1, u1, n1, p1, x2, w2, n2, p2, d, hyp, use_os, (TK)diag_add, K, ldk);
  CHECK_LAUNCH();
  return DSVGP_OK;
}

template <typename TK>
int kdir_diag(int n, int p, const double* hyp, int use_os, TK* out, cudaStream_t st) {
  const int64_t tot = (int64_t)n * (p + 1);
  if (tot <= 0) return DSVGP_OK;
  kdir_diag_kernel<TK><<<(unsigned)ceil_div64(tot, 256), 256, 0, st>>>(n, p, hyp, use_os, out);
  CHECK_LAUNCH();
  return DSVGP_OK;
}

// workspace (bytes) the backward needs for an (n1,p1) x (n2,p2) call
// (p1 = p2 = 0, the plain RBF kernel of the SVGP baseline, has the same d <= 20 limit: an exact DP = 60 instantiation for the
//  rover shape spills 0.8 KB per thread at either VPL (-Xptxas -v: 255 / 128 registers), so d > 20 stays on the blocked kernel)
bool bwd_v4_ok(int n1, int p1, int n2, int p2, int d) {
  return d <= 20 && n2 >= 512 &&
         ((p1 == 0 && p2 == 0) || (p1 == 1 && p2 == 1) || (p1 == 2 && p2 == 2) || (p1 == 1 && p2 == 0) || (p1 == 2 && p2 == 0));
}

template <typename TK>
size_t kdir_bwd_workspace(int n1, int p1, int n2, int p2, int d) {
  if (sizeof(TK) == 4 && bwd_v4_ok(n1, p1, n2, p2, d)) {
    const size_t nt = ceil_div(n2, 64), nrc = ceil_div(n1, 64);      // (64-point column tiles: the VPL = 2 variant; 128 needs half)
    const size_t v4 = sizeof(float) * nt * n1 * (p1 + 1) * d + sizeof(double) * 2 * nt * nrc + 512;
    const int rt0 = ceil_div(n1, BWD_TI), nch0 = bwd_num_chunks(n1, n2);
    const size_t old = sizeof(float) * (size_t)nch0 * n1 * (p1 + 1) * d + sizeof(double) * 2 * (size_t)rt0 * nch0 + 256;
    return v4 > old ? v4 : old;
  }
  const bool fast = (p1 <= DSVGP_MAXP_FAST && (p2 == p1 || p2 == 0) && BWD_TI * (p1 + 1) * d <= 256 * BWD_MAXACC);
  if (!fast) return sizeof(double) * ((size_t)n1 * d + (size_t)n1 * p1 * d) + 256;
  const int rt = ceil_div(n1, BWD_TI);
  int nchunk = bwd_num_chunks(n1, n2);
  return sizeof(TK) * (size_t)nchunk * n1 * (p1 + 1) * d + sizeof(double) * 2 * (size_t)rt * nchunk + 256;
}

int bwd_num_chunks(int n1, int n2) {
  const int rt = ceil_div(n1, BWD_TI);
  const int tiles = ceil_div(n2, BWD_TJ);
  int want = ceil_div(148 * 4, rt);            // ~4 CTAs per SM across the grid
  if (want < 1) want = 1;
  if (want > tiles) want = tiles;
  const int tiles_per_chunk = ceil_div(tiles, want);
  return ceil_div(tiles, tiles_per_chunk);
}

template <typename T, typename TK, int P1, int P2>
static int launch_bwd_blocked(const T* x1, const TK* u1, const TK* inv1, int n1, const T* x2, const TK* w2, int n2,
                              int d, const double* hyp, int use_os, const TK* dK, int64_t lddk, int dk_trans,
                              double scale, double* gx, double* gv, double* gsc, void* ws, cudaStream_t st) {
  const int rt = ceil_div(n1, BWD_TI);
  const int nchunk = bwd_num_chunks(n1, n2);
  const int tiles = ceil_div(n2, BWD_TJ);
  const int chunk_pts = ceil_div(tiles, nchunk) * BWD_TJ;
  TK* part = reinterpret_cast<TK*>(ws);
  size_t part_bytes = round_up64(sizeof(TK) * (size_t)nchunk * n1 * (P1 + 1) * d, 16);
  double* part_sc = reinterpret_cast<double*>(reinterpret_cast<unsigned char*>(ws) + part_bytes);
  const size_t smem = bwd_smem_bytes<TK, P1, P2>(d);
  if (smem > 227 * 1024) return DSVGP_ERR_ARG;
  auto kern = kdir_bwd_blocked<T, TK, P1, P2>;
  if (smem > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  dim3 grid(nchunk, rt);
  kern<<<grid, 256, smem, st>>>(x1, u1, n1, x2, w2, n2, d, hyp, use_os, dK, lddk, dk_trans, chunk_pts, part, part_sc);
  CHECK_LAUNCH();
  kdir_bwd_reduce_rows<TK, TK><<<ceil_div(n1 * (P1 + 1), 8), 256, 0, st>>>(part, nchunk, n1, P1, d, u1, inv1, scale, gx, gv);
  CHECK_LAUNCH();
  if (gsc) {
    kdir_bwd_reduce_scalars<<<1, 256, 0, st>>>(part_sc, rt * nchunk, gsc);
    CHECK_LAUNCH();
  }
  return DSVGP_OK;
}

// Accumulates  scale * dL/dx1 into gx (n1,d),  scale * dL/dv1 into gv (n1*p1,d)  (either may be null) and the
// UNSCALED dL/d ell, dL/d outputscale into gsc[0], gsc[1] (may be null).  All three are double buffers.
template <typename T, typename TK>
int kdir_bwd(const T* x1, const TK* u1, const TK* inv1, int n1, int p1, const T* x2, const TK* w2, int n2, int p2,
             int d, const double* hyp, int use_os, const TK* dK, int64_t lddk, int dk_trans, double scale,
             double* gx, double* gv, double* gsc, void* ws, size_t ws_bytes, cudaStream_t st) {
  if (n1 <= 0 || n2 <= 0) return DSVGP_OK;
  if (p1 < 0 || p2 < 0 || p1 > DSVGP_MAXP || p2 > DSVGP_MAXP || d <= 0) return DSVGP_ERR_ARG;
  if (ws_bytes < kdir_bwd_workspace<TK>(n1, p1, n2, p2, d)) return DSVGP_ERR_WORKSPACE;
  if constexpr (sizeof(T) == 4 && sizeof(TK) == 4) {
    if (bwd_v4_ok(n1, p1, n2, p2, d) && !dk_trans) {
      const int vpl = g_bwd_vpl;
      const int nt = ceil_div(n2, 32 * vpl), nrc = ceil_div(n1, V4_TIB);
      float* part = reinterpret_cast<float*>(ws);
      const size_t part_bytes = round_up64(sizeof(float) * (size_t)nt * n1 * (p1 + 1) * d, 16);
      double* part_sc = reinterpret_cast<double*>(reinterpret_cast<unsigned char*>(ws) + part_bytes);
      // coordinates padded to a multiple of 4, except for the shapes of the shipped workloads, which get an exact instantiation
      // (d = 10: 10 instead of 12 coordinate steps in both FMA phases and one 30-value butterfly; d = 18: 18 instead of 20)
      const int DPr = ((d == 10 && (p1 == 2 || p1 == 0)) || (d == 18 && p2 == 0)) ? d : (d + 3) & ~3;
      dim3 grid(nt, nrc);
      int launched = 0;
#define BV4V(A, B, DPV, VPLV)                                                                                  \
  if (!launched && p1 == A && p2 == B && DPr == DPV && vpl == VPLV) {                                          \
    const size_t smem = bwd_v4_smem_bytes<A, B, DPV, VPLV>();                                                  \
    auto kern = kdir_bwd_v4<A, B, DPV, VPLV>;                                                                  \
    if (smem > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);  \
    kern<<<grid, 256, smem, st>>>(x1, u1, n1, x2, w2, n2, d, hyp, use_os, dK, lddk, part, part_sc);            \
    launched = 1;                                                                                              \
  }
#define BV4(A, B, DPV) BV4V(A, B, DPV, 4) BV4V(A, B, DPV, 2)
#define BV4_ALL(A, B) BV4(A, B, 4) BV4(A, B, 8) BV4(A, B, 12) BV4(A, B, 16)
      BV4_ALL(1, 1) BV4_ALL(2, 2) BV4_ALL(1, 0) BV4_ALL(2, 0)
      BV4(2, 0, 20) BV4(1, 0, 20)                            // d = 17..20 without data-side directions (uci_dfree-shaped, d = 18)
      BV4(2, 2, 10) BV4(2, 0, 10) BV4(2, 0, 18) BV4(1, 0, 18)
      BV4_ALL(0, 0) BV4(0, 0, 20) BV4(0, 0, 10) BV4(0, 0, 18)                 // value-only kernel (SVGP baseline)
#undef BV4_ALL
#undef BV4
#undef BV4V
      if (launched) {
        CHECK_LAUNCH();
        kdir_bwd_reduce_rows<float, float><<<ceil_div(n1 * (p1 + 1), 8), 256, 0, st>>>(part, nt, n1, p1, d, u1, inv1, scale, gx, gv);
        CHECK_LAUNCH();
        if (gsc) {
          kdir_bwd_reduce_scalars<<<1, 256, 0, st>>>(part_sc, nt * nrc, gsc);
          CHECK_LAUNCH();
        }
        return DSVGP_OK;
      }
    }
  }
  const bool fast = (p1 <= DSVGP_MAXP_FAST && (p2 == p1 || p2 == 0) && BWD_TI * (p1 + 1) * d <= 256 * BWD_MAXACC);
  if (fast) {
#define BWD_CASE(A, B)                                                                                         \
  if (p1 == A && p2 == B)                                                                                      \
    return launch_bwd_blocked<T, TK, A, B>(x1, u1, inv1, n1, x2, w2, n2, d, hyp, use_os, dK, lddk, dk_trans,  \
                                           scale, gx, gv, gsc, ws, st);
    BWD_CASE(0, 0) BWD_CASE(1, 1) BWD_CASE(2, 2) BWD_CASE(3, 3) BWD_CASE(1, 0) BWD_CASE(2, 0) BWD_CASE(3, 0)
#undef BWD_CASE
  }
  double* gxt = reinterpret_cast<double*>(ws);
  double* gut = gxt + (size_t)n1 * d;
  cudaMemsetAsync(ws, 0, sizeof(double) * ((size_t)n1 * d + (size_t)n1 * p1 * d + 2), st);
  double* gsc_t = gsc ? gsc : gut + (size_t)n1 * p1 * d;   // scalars accumulate directly (or into scratch)
  dim3 grid(ceil_div(n2, 128), n1);
  kdir_bwd_generic<T, TK><<<grid, 128, 0, st>>>(x1, u1, n1, p1, x2, w2, n2, p2, d, hyp, use_os, dK, lddk, dk_trans,
                                                gxt, gut, gsc_t);
  CHECK_LAUNCH();
  kdir_bwd_chain_generic<TK><<<ceil_div(n1 * (p1 + 1), 8), 256, 0, st>>>(gxt, gut, n1, p1, d, u1, inv1, scale, gx, gv);
  CHECK_LAUNCH();
  return DSVGP_OK;
}

// workspace (bytes) of kdir_bwd_cols: the fp64 chunk partials of the vectorised kernel, or what the blocked kernel needs for
// the swapped problem (data side as the first argument, dK read transposed)
template <typename TK>
size_t kdir_bwd_cols_workspace(int n1, int p1, int n2, int p2, int d) {
  const size_t blocked = kdir_bwd_workspace<TK>(n2, p2, n1, p1, d);
  if (sizeof(TK) == 4 && bwd_v4_ok(n1, p1, n2, p2, d)) {
    const size_t v4 = sizeof(double) * (size_t)cols_num_chunks(n1, n2) * n2 * (p2 + 1) * d + 256;
    return v4 > blocked ? v4 : blocked;
  }
  return blocked;
}

// Accumulates scale * dL/dx2 into gx (n2,d) and scale * dL/dv2 into gv (n2*p2,d) (either may be null; double buffers) for
// dL = sum(dK * K(x1, x2)).  Returns 1 when the vectorised fp32 kernel ran, 0 when the blocked kernel did (dk_trans = 1 on the
// swapped problem: every shape and dtype, reading dK strided).
template <typename T, typename TK>
int kdir_bwd_cols(const T* x1, const TK* u1, int n1, int p1, const T* x2, const TK* w2, const TK* inv2, int n2, int p2, int d,
                  const double* hyp, int use_os, const TK* dK, int64_t lddk, double scale, double* gx, double* gv, void* ws,
                  size_t ws_bytes, cudaStream_t st) {
  if (n1 <= 0 || n2 <= 0) return DSVGP_OK;
  if (p1 < 0 || p2 < 0 || p1 > DSVGP_MAXP || p2 > DSVGP_MAXP || d <= 0) return DSVGP_ERR_ARG;
  if (ws_bytes < kdir_bwd_cols_workspace<TK>(n1, p1, n2, p2, d)) return DSVGP_ERR_WORKSPACE;
  if constexpr (sizeof(T) == 4 && sizeof(TK) == 4) {
    if (bwd_v4_ok(n1, p1, n2, p2, d)) {
      const int nchunk = cols_num_chunks(n1, n2), chunk_pts = ceil_div(n1, nchunk);
      const int DPr = (d + 3) & ~3;
      double* part = reinterpret_cast<double*>(ws);
      dim3 grid(ceil_div(n2, COLS_TJ), nchunk);
      int launched = 0;
#define BCOL(A, B, DPV)                                                                                        \
  if (!launched && p1 == A && p2 == B && DPr == DPV) {                                                         \
    kdir_bwd_cols_v4<A, B, DPV><<<grid, COLS_TJ, 0, st>>>(x1, u1, n1, x2, w2, n2, d, hyp, use_os, dK, lddk,    \
                                                         chunk_pts, part);                                     \
    launched = 1;                                                                                              \
  }
#define BCOL_ALL(A, B) BCOL(A, B, 4) BCOL(A, B, 8) BCOL(A, B, 12) BCOL(A, B, 16)
      BCOL_ALL(0, 0) BCOL_ALL(1, 1) BCOL_ALL(2, 2) BCOL_ALL(1, 0) BCOL_ALL(2, 0)
      BCOL(0, 0, 20) BCOL(1, 1, 20) BCOL(2, 2, 20) BCOL(1, 0, 20) BCOL(2, 0, 20)
#undef BCOL_ALL
#undef BCOL
      if (launched) {
        CHECK_LAUNCH();
        kdir_bwd_reduce_rows<double, float><<<ceil_div(n2 * (p2 + 1), 8), 256, 0, st>>>(part, nchunk, n2, p2, d, w2, inv2, scale,
                                                                                         gx, gv);
        CHECK_LAUNCH();
        return 1;
      }
    }
  }
  return kdir_bwd<T, TK>(x2, w2, inv2, n2, p2, x1, u1, n1, p1, d, hyp, use_os, dK, lddk, 1, scale, gx, gv, nullptr, ws, ws_bytes,
                         st);
}

// explicit instantiations: (T, TK) in {(f32,f32), (f64,f64), (f32,f64)}
#define INST(T, TK)                                                                                             \
  template int normalize_dirs<T, TK>(const T*, int, int, TK*, TK*, cudaStream_t, int*, int*);                               \
  template int kdir_fwd<T, TK>(const T*, const TK*, int, int, const T*, const TK*, int, int, int, const double*, \
                               int, double, TK*, int64_t, cudaStream_t, const int*, const int*, TK*, void*, void*,  \
                               int64_t, const float*);                                                          \
  template int kdir_bwd<T, TK>(const T*, const TK*, const TK*, int, int, const T*, const TK*, int, int, int,    \
                               const double*, int, const TK*, int64_t, int, double, double*, double*, double*,  \
                               void*, size_t, cudaStream_t);
INST(float, float)
INST(double, double)
INST(float, double)
#undef INST
template int kdir_diag<float>(int, int, const double*, int, float*, cudaStream_t);
template int kdir_diag<double>(int, int, const double*, int, double*, cudaStream_t);
template size_t kdir_bwd_workspace<float>(int, int, int, int, int);
template size_t kdir_bwd_workspace<double>(int, int, int, int, int);
template size_t kdir_bwd_cols_workspace<float>(int, int, int, int, int);
template size_t kdir_bwd_cols_workspace<double>(int, int, int, int, int);
template int kdir_bwd_cols<float, float>(const float*, const float*, int, int, const float*, const float*, const float*, int, int,
                                         int, const double*, int, const float*, int64_t, double, double*, double*, void*, size_t,
                                         cudaStream_t);
template int kdir_bwd_cols<double, double>(const double*, const double*, int, int, const double*, const double*, const double*,
                                           int, int, int, const double*, int, const double*, int64_t, double, double*, double*,
                                           void*, size_t, cudaStream_t);

}  // namespace dsvgp
