// Solve + predict + accuracy for the mixed-precision path: the TF32 Cholesky factor of chol_tc.cu is used as a
// preconditioner and the solution is refined in fp64 against the EXACT operator, applied straight from the
// integer cross-products (no fp64 copy of A is ever formed):
//
//   (A alpha)_a = lambda alpha_a + (2/den) [ N^2 (C alpha)_a - N s_a (sum alpha) - N (s . alpha) + Q (sum alpha) ]
//
// with C, s, S, Q the integers of scale.cu / DESIGN.md §1 and den = 2 N S - Q.  Iteration:
//   alpha <- M^-1 y;  repeat { r = y - A alpha;  d = M^-1 r;  alpha += d } until the predicted remaining error
//   max|d| * (observed contraction) <= 1e-8 max|alpha|   (typically 2 sweeps; at most 6)
// where M^-1 = (L L^T)^-1 by blocked substitution (fp32 factor, fp64 accumulation).  Then
//   pred_v = (G_vt alpha)_v from the integer rows of the validation animals, fitness = |pearson(y_v, pred_v)|.
// Same reference lines as solve.cu (tblup/evaluator.py:282-286, :311-314).  One CTA per (individual, row set);
// HBM-bound: per sweep the factor is streamed twice (fp32) and the lower triangle of C twice (int32).
#include "tb_internal.h"
#include <cuda_fp16.h>
#include <type_traits>

namespace {

constexpr int NB = TB_NB;
constexpr int ST = 512;
constexpr int MAX_SWEEPS = 5;
constexpr int MIXED_SMEM_NTP = 4096;  // up to this many (padded) training animals alpha stays in shared memory
constexpr double REL_TOL = 1e-8;
     // stop when the PREDICTED remaining error is below 1e-8 of the solution
                                     // (fitness bar of BASELINE.json: 1e-6 absolute)

__device__ __forceinline__ double warp_sum(double v) {
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_max(double v) {
  for (int o = 16; o; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ double block_sum(double v, double* red) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
  for (int i = 0; i < ST / 32; ++i) t += red[i];
  return t;
}
__device__ double block_max(double v, double* red) {
  v = warp_max(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
  for (int i = 0; i < ST / 32; ++i) t = fmax(t, red[i]);
  return t;
}

__device__ __forceinline__ double dot4(const float4 l, const double* z) {
  const double2 z0 = *reinterpret_cast<const double2*>(z), z1 = *reinterpret_cast<const double2*>(z + 2);
  return (double)l.x * z0.x + (double)l.y * z0.y + (double)l.z * z1.x + (double)l.w * z1.y;
}
__device__ __forceinline__ double dot4i(const int4 c, const double* z) {
  const double2 z0 = *reinterpret_cast<const double2*>(z), z1 = *reinterpret_cast<const double2*>(z + 2);
  return (double)c.x * z0.x + (double)c.y * z0.y + (double)c.z * z1.x + (double)c.w * z1.y;
}

// exact conversion of a non-negative integer below 2^32 without the (slow) I2F pipe: 2^52 + x is representable, so
// placing x in the low mantissa word and subtracting 2^52 costs one fp64 add
__device__ __forceinline__ double u2d(uint32_t x) { return __hiloint2double(0x43300000, (int)x) - 4503599627370496.0; }

// four rows of eight int16 cross-products against the same eight fp64 entries z (read from shared memory ONCE for
// the four rows: ncu showed the LSU 82 % busy on these reads when every row fetched its own copy; a lane-rotated,
// bank-conflict-free read order was tried and lost to the extra selects)
__device__ __forceinline__ void fma4x8s(double (&d)[4], const uint4 v0, const uint4 v1, const uint4 v2, const uint4 v3,
                                        const double* z) {
  const uint32_t w0[4] = {v0.x, v0.y, v0.z, v0.w}, w1[4] = {v1.x, v1.y, v1.z, v1.w};
  const uint32_t w2[4] = {v2.x, v2.y, v2.z, v2.w}, w3[4] = {v3.x, v3.y, v3.z, v3.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const double2 zz = *reinterpret_cast<const double2*>(z + 2 * j);
    d[0] += u2d(w0[j] & 0xffffu) * zz.x + u2d(w0[j] >> 16) * zz.y;
    d[1] += u2d(w1[j] & 0xffffu) * zz.x + u2d(w1[j] >> 16) * zz.y;
    d[2] += u2d(w2[j] & 0xffffu) * zz.x + u2d(w2[j] >> 16) * zz.y;
    d[3] += u2d(w3[j] & 0xffffu) * zz.x + u2d(w3[j] >> 16) * zz.y;
  }
}

// eight int16 cross-products (non-negative) against eight fp64 entries
__device__ __forceinline__ double dot8s(const uint4 c, const double* z) {
  const double2 z0 = *reinterpret_cast<const double2*>(z), z1 = *reinterpret_cast<const double2*>(z + 2);
  const double2 z2 = *reinterpret_cast<const double2*>(z + 4), z3 = *reinterpret_cast<const double2*>(z + 6);
  return (u2d(c.x & 0xffffu) * z0.x + u2d(c.x >> 16) * z0.y) + (u2d(c.y & 0xffffu) * z1.x + u2d(c.y >> 16) * z1.y) +
         (u2d(c.z & 0xffffu) * z2.x + u2d(c.z >> 16) * z2.y) + (u2d(c.w & 0xffffu) * z3.x + u2d(c.w >> 16) * z3.y);
}

__device__ __forceinline__ double dot8h(const uint4 l, const double* z) {
  const float2 f0 = __half22float2(*reinterpret_cast<const __half2*>(&l.x));
  const float2 f1 = __half22float2(*reinterpret_cast<const __half2*>(&l.y));
  const float2 f2 = __half22float2(*reinterpret_cast<const __half2*>(&l.z));
  const float2 f3 = __half22float2(*reinterpret_cast<const __half2*>(&l.w));
  const double2 z0 = *reinterpret_cast<const double2*>(z), z1 = *reinterpret_cast<const double2*>(z + 2);
  const double2 z2 = *reinterpret_cast<const double2*>(z + 4), z3 = *reinterpret_cast<const double2*>(z + 6);
  return ((double)f0.x * z0.x + (double)f0.y * z0.y) + ((double)f1.x * z1.x + (double)f1.y * z1.y) +
         ((double)f2.x * z2.x + (double)f2.y * z2.y) + ((double)f3.x * z3.x + (double)f3.y * z3.y);
}

// Cross-products of the held-out animals (universe positions h0 .. h0 + gap - 1, the hole of the training set) with the
// solution: out[v] = sum_b C(h0 + v, U(b)) alpha_b.  Training animals before the hole lie in the row of the held-out
// animal (four rows per warp), those after it in its COLUMN of the lower triangle (the column pass of sym_matvec16
// restricted to the hole's columns; no diagonal is crossed).
__device__ void hole_predict16(const int16_t* __restrict__ C, int rpad, int n_t, int h0, int gap, const double* alpha,
                               double* out, double* part2) {
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n_v = gap;
  for (int v = 4 * warp; v < n_v; v += 4 * (ST / 32)) {          // gap is a multiple of 8
    const uint4* row = reinterpret_cast<const uint4*>(C + (size_t)(h0 + v) * rpad);
    const size_t rs = rpad / 8;
    double d[4] = {0.0, 0.0, 0.0, 0.0};
    for (int c = lane; c < (h0 >> 3); c += 32) fma4x8s(d, row[c], row[rs + c], row[2 * rs + c], row[3 * rs + c], alpha + 8 * c);
#pragma unroll
    for (int rr = 0; rr < 4; ++rr) {
      const double t = warp_sum(d[rr]);
      if (lane == 0) out[v + rr] = t;
    }
  }
  __syncthreads();
  const int cgl = lane & 7, rsub = lane >> 3, cblk = warp & 7, rsup = warp >> 3;
  const int rg = rsup * 4 + rsub;
  for (int v0 = 0; v0 < n_v; v0 += 512) {
    const int cv = v0 + 64 * cblk + 8 * cgl;
    double acc[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[e] = 0.0;
    auto add8 = [&](const uint4 v, const double w) {
      acc[0] += u2d(v.x & 0xffffu) * w;
      acc[1] += u2d(v.x >> 16) * w;
      acc[2] += u2d(v.y & 0xffffu) * w;
      acc[3] += u2d(v.y >> 16) * w;
      acc[4] += u2d(v.z & 0xffffu) * w;
      acc[5] += u2d(v.z >> 16) * w;
      acc[6] += u2d(v.w & 0xffffu) * w;
      acc[7] += u2d(v.w >> 16) * w;
    };
    if (cv < n_v) {
      const int16_t* colp = C + h0 + cv;
      int b = h0 + rg;                                           // compact rows h0 .. n_t-1 = universe rows + gap
      for (; b + 24 < n_t; b += 32) {
        const uint4 x0 = *reinterpret_cast<const uint4*>(colp + (size_t)(b + gap) * rpad);
        const uint4 x1 = *reinterpret_cast<const uint4*>(colp + (size_t)(b + 8 + gap) * rpad);
        const uint4 x2 = *reinterpret_cast<const uint4*>(colp + (size_t)(b + 16 + gap) * rpad);
        const uint4 x3 = *reinterpret_cast<const uint4*>(colp + (size_t)(b + 24 + gap) * rpad);
        add8(x0, alpha[b]);
        add8(x1, alpha[b + 8]);
        add8(x2, alpha[b + 16]);
        add8(x3, alpha[b + 24]);
      }
      for (; b < n_t; b += 8) add8(*reinterpret_cast<const uint4*>(colp + (size_t)(b + gap) * rpad), alpha[b]);
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      acc[e] += __shfl_xor_sync(0xffffffffu, acc[e], 8);
      acc[e] += __shfl_xor_sync(0xffffffffu, acc[e], 16);
    }
    if (rsub == 0) {
      double* pr = part2 + rsup * 512 + 64 * cblk + 8 * cgl;
#pragma unroll
      for (int e = 0; e < 8; ++e) pr[e] = acc[e];
    }
    __syncthreads();
    const int v = v0 + tid;
    if (v < n_v) out[v] += part2[tid] + part2[512 + tid];
    __syncthreads();
  }
}


// ---- two CTAs per matrix (small batches) --------------------------------------------------------------------------
// With fewer matrices than CTA slots (strong scaling: 125 genomes per GPU; config 4: 53 matrices per wave) one CTA per
// matrix leaves most of the machine idle and the kernel runs at the latency of ONE CTA's byte stream.  CL = 2 runs a
// cluster of two CTAs per matrix: each streams half of every block step of the triangular solves, half of the work units
// of the symmetric mat-vec and half of the validation rows; the 64 partial sums of a step (or the fixed-point partial
// vector of a mat-vec) are read from the partner's shared memory after a cluster barrier.  Everything else is computed
// redundantly -- and identically, since every cross-CTA sum is one commutative addition -- by both CTAs, so they take
// the same branches and meet at the same barriers.
template <int CL>
__device__ __forceinline__ void team_sync() {
  if (CL > 1) {
    // CTA barrier first: the cluster barrier is issued from inline PTX, so the compiler does not know that the warps
    // must have reconverged (callers sit right behind `if (lane == 0)` blocks); the non-.aligned forms tolerate the rest
    __syncwarp();
    __syncthreads();
    asm volatile("barrier.cluster.arrive.release;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire;" ::: "memory");
  } else {
    __syncthreads();
  }
}
__device__ __forceinline__ uint32_t peer_addr(const void* p, uint32_t peer) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"((uint32_t)__cvta_generic_to_shared(p)), "r"(peer));
  return r;
}
__device__ __forceinline__ float ld_peer_f32(const float* p, uint32_t peer) {
  float v;
  asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(peer_addr(p, peer)) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long ld_peer_u64(const unsigned long long* p, uint32_t peer) {
  unsigned long long v;
  asm volatile("ld.shared::cluster.u64 %0, [%1];" : "=l"(v) : "r"(peer_addr(p, peer)) : "memory");
  return v;
}

// ---- fp32 application of the preconditioner -----------------------------------------------------------------------
// wf <- (L L^T)^-1 wf in place, entirely in fp32 (fp16 factor widened pairwise, FFMA accumulation).  The factor is a
// 10-bit preconditioner (it contracts the error ~300x per sweep); applying it with fp32 rounding (~1e-6 relative)
// changes nothing about what the refinement converges to -- the residual is formed in fp64 from the exact integers --
// and frees the fp64 / conversion pipes and half of the shared-memory reads of the solution vector (r01 ncu: XU 33 %,
// fp64 26 %, LSU wavefronts 66 % busy with one fp64 value per factor entry).
__device__ __forceinline__ float dot8hf(const uint4 l, const float4 z0, const float4 z1) {
  const float2 f0 = __half22float2(*reinterpret_cast<const __half2*>(&l.x));
  const float2 f1 = __half22float2(*reinterpret_cast<const __half2*>(&l.y));
  const float2 f2 = __half22float2(*reinterpret_cast<const __half2*>(&l.z));
  const float2 f3 = __half22float2(*reinterpret_cast<const __half2*>(&l.w));
  return ((f0.x * z0.x + f0.y * z0.y) + (f1.x * z0.z + f1.y * z0.w)) + ((f2.x * z1.x + f2.y * z1.y) + (f3.x * z1.z + f3.y * z1.w));
}
__device__ __forceinline__ float warp_sumf(float v) {
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// xp: [2][NB] exchange buffer (CL = 2), crank: this CTA's rank in its cluster
// U: column groups per lane and loop trip in the forward sweep (2 for the large-matrix instantiations, which run one
// CTA per SM with 128 registers: eight 16-byte loads in flight per lane instead of four)
template <int CL, int U>
__device__ void apply_minv_f32(const __half* __restrict__ L, const float* __restrict__ Linv, int ntp, float* wf,
                               float* rvec, float* part, float* xp, int crank) {
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int nb = ntp / NB;
  int par = 0;
  for (int b = 0; b < nb; ++b) {                      // forward: L z = wf
    const int kc = b * NB;
    {
      const uint4* r0 = reinterpret_cast<const uint4*>(L + (size_t)(kc + 4 * warp) * ntp);
      const size_t rs = ntp / 8;
      float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
      for (int c = lane + 32 * crank; c < kc / 8; c += 32 * CL * U) {
        uint4 l[U][4];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int cu = c + 32 * CL * u;
          if (cu < kc / 8) {
            l[u][0] = r0[cu];
            l[u][1] = r0[rs + cu];
            l[u][2] = r0[2 * rs + cu];
            l[u][3] = r0[3 * rs + cu];
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int cu = c + 32 * CL * u;
          if (cu < kc / 8) {
            const float4 z0 = *reinterpret_cast<const float4*>(wf + 8 * cu), z1 = *reinterpret_cast<const float4*>(wf + 8 * cu + 4);
            s0 += dot8hf(l[u][0], z0, z1);
            s1 += dot8hf(l[u][1], z0, z1);
            s2 += dot8hf(l[u][2], z0, z1);
            s3 += dot8hf(l[u][3], z0, z1);
          }
        }
      }
      s0 = warp_sumf(s0);
      s1 = warp_sumf(s1);
      s2 = warp_sumf(s2);
      s3 = warp_sumf(s3);
      if (CL > 1) {
        if (lane == 0) {
          float* x = xp + par * NB + 4 * warp;
          x[0] = s0;
          x[1] = s1;
          x[2] = s2;
          x[3] = s3;
        }
        team_sync<CL>();
        if (tid < NB) rvec[tid] = wf[kc + tid] - (xp[par * NB + tid] + ld_peer_f32(xp + par * NB + tid, crank ^ 1));
        par ^= 1;
      } else if (lane == 0) {
        rvec[4 * warp + 0] = wf[kc + 4 * warp + 0] - s0;
        rvec[4 * warp + 1] = wf[kc + 4 * warp + 1] - s1;
        rvec[4 * warp + 2] = wf[kc + 4 * warp + 2] - s2;
        rvec[4 * warp + 3] = wf[kc + 4 * warp + 3] - s3;
      }
    }
    __syncthreads();
    {
      const int i = tid >> 3, sub = tid & 7;
      const float4* li = reinterpret_cast<const float4*>(Linv + ((size_t)kc + i) * NB + sub * 8);
      const float4 a0 = li[0], a1 = li[1];
      const float4 z0 = *reinterpret_cast<const float4*>(rvec + sub * 8), z1 = *reinterpret_cast<const float4*>(rvec + sub * 8 + 4);
      float sv = (a0.x * z0.x + a0.y * z0.y) + (a0.z * z0.z + a0.w * z0.w) + (a1.x * z1.x + a1.y * z1.y) + (a1.z * z1.z + a1.w * z1.w);
      sv += __shfl_xor_sync(0xffffffffu, sv, 1);
      sv += __shfl_xor_sync(0xffffffffu, sv, 2);
      sv += __shfl_xor_sync(0xffffffffu, sv, 4);
      if (sub == 0) wf[kc + i] = sv;
    }
    __syncthreads();
  }
  for (int b = nb - 1; b >= 0; --b) {                 // backward: L^T d = z
    const int kc = b * NB;
    {
      const int cq = tid & 7, rg = tid >> 3;           // thread = 8 consecutive columns x one of 64 row groups
      float a[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) a[e] = 0.f;
      const __half* base = L + kc + 8 * cq;
      auto acc8 = [&](const uint4 l, const float w) {
        const float2 f0 = __half22float2(*reinterpret_cast<const __half2*>(&l.x));
        const float2 f1 = __half22float2(*reinterpret_cast<const __half2*>(&l.y));
        const float2 f2 = __half22float2(*reinterpret_cast<const __half2*>(&l.z));
        const float2 f3 = __half22float2(*reinterpret_cast<const __half2*>(&l.w));
        a[0] = fmaf(f0.x, w, a[0]);
        a[1] = fmaf(f0.y, w, a[1]);
        a[2] = fmaf(f1.x, w, a[2]);
        a[3] = fmaf(f1.y, w, a[3]);
        a[4] = fmaf(f2.x, w, a[4]);
        a[5] = fmaf(f2.y, w, a[5]);
        a[6] = fmaf(f3.x, w, a[6]);
        a[7] = fmaf(f3.y, w, a[7]);
      };
      // rows kc + 64 + rg + 64 j below the block; with CL = 2 CTA r takes the 64-row groups j = r (mod 2)
      int i = kc + NB + rg + 64 * crank;
      constexpr int RS = 64 * CL;
      for (; i + 7 * RS < ntp; i += 8 * RS) {          // eight independent 16-byte loads in flight
        uint4 l[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) l[u] = *reinterpret_cast<const uint4*>(base + (size_t)(i + RS * u) * ntp);
#pragma unroll
        for (int u = 0; u < 8; ++u) acc8(l[u], wf[i + RS * u]);
      }
      for (; i < ntp; i += RS) acc8(*reinterpret_cast<const uint4*>(base + (size_t)i * ntp), wf[i]);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        a[e] += __shfl_xor_sync(0xffffffffu, a[e], 8);
        a[e] += __shfl_xor_sync(0xffffffffu, a[e], 16);
      }
      if (lane < 8) {
        float* pr = part + warp * NB + 8 * cq;
        *reinterpret_cast<float4*>(pr) = make_float4(a[0], a[1], a[2], a[3]);
        *reinterpret_cast<float4*>(pr + 4) = make_float4(a[4], a[5], a[6], a[7]);
      }
    }
    __syncthreads();
    if (CL > 1) {
      if (tid < NB) {
        float sv = 0.f;
#pragma unroll
        for (int gI = 0; gI < ST / 32; ++gI) sv += part[gI * NB + tid];
        xp[par * NB + tid] = sv;
      }
      team_sync<CL>();
      if (tid < NB) rvec[tid] = wf[kc + tid] - (xp[par * NB + tid] + ld_peer_f32(xp + par * NB + tid, crank ^ 1));
      par ^= 1;
    } else if (tid < NB) {
      float sv = 0.f;
#pragma unroll
      for (int gI = 0; gI < ST / 32; ++gI) sv += part[gI * NB + tid];
      rvec[tid] = wf[kc + tid] - sv;
    }
    __syncthreads();
    {
      const int i = tid & 63, grp = tid >> 6;
      const float* li = Linv + (size_t)kc * NB;
      float sv = 0.f;
#pragma unroll
      for (int pp = 0; pp < 8; ++pp) {
        const int q = grp * 8 + pp;
        sv = fmaf(li[q * NB + i], rvec[q], sv);
      }
      part[grp * NB + i] = sv;
    }
    __syncthreads();
    if (tid < NB) {
      float sv = 0.f;
#pragma unroll
      for (int gI = 0; gI < 8; ++gI) sv += part[gI * NB + tid];
      wf[kc + tid] = sv;
    }
    __syncthreads();
  }
}

// ---- symmetric mat-vec in ONE pass over the lower triangle --------------------------------------------------------
// out[a] = (C alpha)_a for contiguous training animals from int16 cross-products.  Every 16-byte load of C feeds BOTH
// the row dot product (out[r] += C[r][c] alpha[c]) and the column update (out[c] += C[r][c] alpha[r]), so the
// triangle crosses HBM once per sweep instead of twice (r01: "by rows, then by columns").
// Work unit = 128 rows x one 128-column strip, taken by a warp from a shared counter (largest strips first).  A lane
// owns 4 consecutive columns of the strip (8-byte loads, eight rows in flight): their alpha entries and the 8 column accumulators stay in registers down
// the unit; the row partials of four rows are reduced across the warp by a transposing butterfly (6 shuffles per four
// rows) and added to out[] with shared-memory atomics, as are the column sums at the end of the unit (about 40
// warp-level atomics per 16 K entries of C).  The same "prefix with one aligned hole" index mapping as before.
template <bool HOLE, typename CT, int CL, bool WIDE_REGS>
__device__ void sym_matvec16_1p(const CT* __restrict__ C, int rpad, int n_t, int h0, int gap, const double* alpha,
                                double amax, int cmax, double* out, int* counter, int crank) {
  constexpr bool W16 = sizeof(CT) == 2;              // int16 cross-products (8-byte loads of 4) or int32 (16-byte loads of 4)
  const int tid = threadIdx.x, lane = tid & 31;
  auto U = [&](int i) { return HOLE ? i + (i >= h0 ? gap : 0) : i; };   // compact index -> universe position
  // The partial sums of many warps meet in out[]: they are accumulated as 64-bit FIXED-POINT integers, so the result
  // does not depend on the order in which the warps arrive (bit-identical from run to run and for any wave size).
  // |sum_b C_ab alpha_b| <= 4 k n_t amax =: bound < 2^ex; one quantum = 2^(ex - 62) <= bound 2^-61 -- finer than the
  // rounding of the fp64 dot product it replaces (~ n_t 2^-53 of the same bound).
  unsigned long long* outq = reinterpret_cast<unsigned long long*>(out);
  const double bound = (double)cmax * (double)n_t * fmax(amax, 1e-290);   // C_ab <= 4 k
  const int ex = ((__double2hiint(bound) >> 20) & 0x7ff) - 1022;
  const double scale = __hiloint2double((62 - ex + 1023) << 20, 0), inv_scale = __hiloint2double((ex - 62 + 1023) << 20, 0);
  for (int a = tid; a < n_t; a += ST) outq[a] = 0ull;
  if (tid == 0) *counter = 0;
  __syncthreads();
  constexpr int SW = 128, RU = 128;                  // strip width (4 columns per lane), rows per unit
  const int n_strips = (n_t + SW - 1) / SW;
  int total = 0;
  for (int s = 0; s < n_strips; ++s) total += (n_t - SW * s + RU - 1) / RU;
  for (;;) {
    int u = 0;
    if (lane == 0) u = atomicAdd(counter, 1);
    u = __shfl_sync(0xffffffffu, u, 0) * CL + crank;  // CL = 2: the partner CTA takes the other units
    if (u >= total) break;
    int s = 0;
    for (;; ++s) {
      const int cnt = (n_t - SW * s + RU - 1) / RU;
      if (u < cnt) break;
      u -= cnt;
    }
    const int c0 = SW * s + 4 * lane;                // this lane's first column (compact index)
    const int r0 = SW * s + RU * u, r1 = min(n_t, r0 + RU);
    const bool col_ok = c0 < n_t;                     // n_t is a multiple of 4: a lane's four columns are all in or all out
    double ac[4], al[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      ac[e] = 0.0;
      al[e] = col_ok ? alpha[c0 + e] : 0.0;
    }
    const CT* colp = C + U(c0);
    const bool diag_unit = u == 0;                    // SW == RU: only a strip's first unit reaches its diagonal
    constexpr int RB = (W16 || WIDE_REGS) ? 8 : 4;    // rows in flight per lane (64 bytes of loads; 128 with 128 registers)
    for (int r = r0; r < r1; r += RB) {               // n_t % 4 == 0
      uint4 v[RB];                                    // int16: .x, .y hold the four entries; int32: all four words
#pragma unroll
      for (int q = 0; q < RB; ++q) {
        v[q] = make_uint4(0u, 0u, 0u, 0u);
        if (col_ok && r + q < r1 && (!diag_unit || c0 <= r + q)) {
          if (W16) {
            const uint2 t2 = *reinterpret_cast<const uint2*>(colp + (size_t)U(r + q) * rpad);
            v[q].x = t2.x;
            v[q].y = t2.y;
          } else {
            v[q] = *reinterpret_cast<const uint4*>(colp + (size_t)U(r + q) * rpad);
          }
        }
      }
#pragma unroll
      for (int h = 0; h < RB / 4; ++h) {
        if (r + 4 * h >= r1) break;
        double p[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int rr = r + 4 * h + q;
          const double ar = alpha[rr];
          const uint4 vv = v[4 * h + q];
          const double cc[4] = {W16 ? u2d(vv.x & 0xffffu) : u2d(vv.x), W16 ? u2d(vv.x >> 16) : u2d(vv.y),
                                W16 ? u2d(vv.y & 0xffffu) : u2d(vv.z), W16 ? u2d(vv.y >> 16) : u2d(vv.w)};
          double pr = 0.0;
          if (!diag_unit || c0 + 3 < rr) {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              pr += cc[e] * al[e];
              ac[e] += cc[e] * ar;
            }
          } else if (c0 <= rr) {                      // the 4-column group that holds the diagonal of row rr
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              if (c0 + e <= rr) pr += cc[e] * al[e];   // the diagonal entry counts once (in the row part)
              if (c0 + e < rr) ac[e] += cc[e] * ar;
            }
          }
          p[q] = pr;
        }
        // transposing butterfly: afterwards lane 8 q (q = 0..3) holds the sum over the warp of p[q]
        const bool hi16 = lane & 16, hi8 = lane & 8;
        double x0 = hi16 ? p[2] : p[0], x1 = hi16 ? p[3] : p[1];
        const double s0 = hi16 ? p[0] : p[2], s1 = hi16 ? p[1] : p[3];
        x0 += __shfl_xor_sync(0xffffffffu, s0, 16);
        x1 += __shfl_xor_sync(0xffffffffu, s1, 16);
        double yv = hi8 ? x1 : x0;
        const double sy = hi8 ? x0 : x1;
        yv += __shfl_xor_sync(0xffffffffu, sy, 8);
        yv += __shfl_xor_sync(0xffffffffu, yv, 4);
        yv += __shfl_xor_sync(0xffffffffu, yv, 2);
        yv += __shfl_xor_sync(0xffffffffu, yv, 1);
        if ((lane & 7) == 0)
          atomicAdd(outq + r + 4 * h + 2 * (lane >> 4) + ((lane >> 3) & 1), (unsigned long long)__double2ll_rn(yv * scale));
        __syncwarp();      // the 64-bit shared atomic is a CAS spin loop: bring the lanes back together (see below)
      }
    }
    if (col_ok) {
#pragma unroll
      for (int e = 0; e < 4; ++e) atomicAdd(outq + c0 + e, (unsigned long long)__double2ll_rn(ac[e] * scale));
    }
    __syncwarp();
  }
  // MEASURED (r02): without this reconvergence a warp that ran the CAS-loop atomics above stayed split, reached the
  // block barriers below in pieces and ended up one barrier behind the others -- with a single work unit (n_t <= 128)
  // the triangular solves then read a stale partial sum of that warp (fp64 fallback on every small matrix), and the
  // cluster barrier of the two-CTA variant dead-locked.
  __syncwarp();
  if (CL > 1) {
    // own + partner's partial vector (integers: the order does not matter); the partner reads ours at the same time,
    // so nothing is overwritten before both have read a chunk
    for (int base = 0; base < n_t; base += 8 * ST) {
      team_sync<CL>();
      double v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int a = base + j * ST + tid;
        v[j] = a < n_t ? (double)(long long)(outq[a] + ld_peer_u64(outq + a, crank ^ 1)) * inv_scale : 0.0;
      }
      team_sync<CL>();
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int a = base + j * ST + tid;
        if (a < n_t) out[a] = v[j];
      }
    }
    __syncthreads();
    return;
  }
  __syncthreads();
  for (int a = tid; a < n_t; a += ST) out[a] = (double)(long long)outq[a] * inv_scale;
  __syncthreads();
}

// (C alpha)_a over the training animals into work[a]; CONTIG: training animal b sits at universe position b.
// CT: element type of the stored cross-products (int32_t, or int16_t in C16 mode).
template <bool CONTIG, bool HOLE, typename CT, int CL, bool WIDE_REGS>
__device__ void sym_matvec(const CT* __restrict__ C, int rpad, int n_t, int h0, int gap, const int* tp,
                           const double* alpha, double amax, int cmax, double* work, double* part2, int crank) {
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if constexpr (CONTIG) {
    // one pass over the triangle for both storage widths (HOLE only occurs with the int16 layout)
    sym_matvec16_1p<HOLE, CT, CL, WIDE_REGS>(C, rpad, n_t, h0, gap, alpha, amax, cmax, work, reinterpret_cast<int*>(part2), crank);
  } else {
    for (int a = warp; a < n_t; a += ST / 32) {
      const int pa = tp[a];
      double d0 = 0.0, d1 = 0.0;
      int b = lane;
      for (; b + 32 <= a; b += 64) {
        const int p0 = tp[b], p1 = tp[b + 32];
        const int c0 = C[(size_t)(pa > p0 ? pa : p0) * rpad + (pa > p0 ? p0 : pa)];
        const int c1 = C[(size_t)(pa > p1 ? pa : p1) * rpad + (pa > p1 ? p1 : pa)];
        d0 += (double)c0 * alpha[b];
        d1 += (double)c1 * alpha[b + 32];
      }
      for (; b <= a; b += 32) {
        const int p0 = tp[b];
        d0 += (double)C[(size_t)(pa > p0 ? pa : p0) * rpad + (pa > p0 ? p0 : pa)] * alpha[b];
      }
      const double d = warp_sum(d0 + d1);
      if (lane == 0) work[a] = d;
    }
    __syncthreads();
    for (int a0 = 0; a0 < n_t; a0 += ST) {
      const int a = a0 + tid;
      if (a < n_t) {
        const int pa = tp[a];
        double d0 = 0.0, d1 = 0.0, d2 = 0.0, d3 = 0.0;
        int b = a + 1;
        for (; b + 3 < n_t; b += 4) {
          const int p0 = tp[b], p1 = tp[b + 1], p2 = tp[b + 2], p3 = tp[b + 3];
          const int c0 = C[(size_t)(pa > p0 ? pa : p0) * rpad + (pa > p0 ? p0 : pa)];
          const int c1 = C[(size_t)(pa > p1 ? pa : p1) * rpad + (pa > p1 ? p1 : pa)];
          const int c2 = C[(size_t)(pa > p2 ? pa : p2) * rpad + (pa > p2 ? p2 : pa)];
          const int c3 = C[(size_t)(pa > p3 ? pa : p3) * rpad + (pa > p3 ? p3 : pa)];
          d0 += (double)c0 * alpha[b];
          d1 += (double)c1 * alpha[b + 1];
          d2 += (double)c2 * alpha[b + 2];
          d3 += (double)c3 * alpha[b + 3];
        }
        for (; b < n_t; ++b) {
          const int p0 = tp[b];
          d0 += (double)C[(size_t)(pa > p0 ? pa : p0) * rpad + (pa > p0 ? p0 : pa)] * alpha[b];
        }
        work[a] += (d0 + d1) + (d2 + d3);
      }
    }
    __syncthreads();
  }
}

template <bool CONTIG, bool BIG, bool C16, bool HOLE, int CL>
__global__ void __launch_bounds__(ST, BIG ? 1 : 2) solve_mixed_kernel(const TbSolveMixedJob* __restrict__ jobs) {
  static_assert(CL == 1 || CONTIG, "two CTAs per matrix only with the contiguous kernels");
  using CT = typename std::conditional<C16, int16_t, int32_t>::type;
  extern __shared__ double msm[];
  const TbSolveMixedJob jb = jobs[blockIdx.x / CL];
  int crank = 0;
  if (CL > 1) {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    crank = (int)r;
  }
  const int ntp = jb.ntp, n_t = jb.n_t, n_v = jb.n_v, rpad = jb.rpad;
  // small matrices keep alpha and the position table in shared memory; beyond MIXED_SMEM_NTP rows alpha lives in
  // the job's global output vector and the positions are read from the row set (both stay L1/L2 resident)
  // (BIG is a template parameter so that each instantiation knows the address space of alpha / tp statically)
  constexpr bool big = BIG;
  double* work = msm;                // [ntp]   (C alpha) / residual in fp64
  double* part2 = work + ntp;        // [4][512] scratch of the column passes (its first word: work counter)
  double* red = part2 + 4 * 512;     // [ST/32]
  double* alpha;                     // [ntp]
  const int* tp;                     // [n_t]
  int* tp_w = nullptr;
  float* wf;                         // [ntp]   right-hand side / result of the fp32 preconditioner application
  if constexpr (BIG) {
    alpha = jb.alpha;
    tp = jb.tpos;
    wf = reinterpret_cast<float*>(red + ST / 32);
  } else {
    alpha = red + ST / 32;
    tp_w = reinterpret_cast<int*>(alpha + ntp);
    tp = tp_w;
    wf = reinterpret_cast<float*>(tp_w + ntp);
  }
  float* rvec = wf + ntp;            // [NB]
  float* part = rvec + NB;           // [ST/32][NB]
  float* xp = part + (ST / 32) * NB; // [2][NB] partial sums offered to the partner CTA (CL = 2)
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const double Nd = (double)jb.N, Sd = (double)jb.SQ[0], Qd = (double)jb.SQ[1];
  const double coef = 2.0 / (2.0 * Nd * Sd - Qd);
  const CT* C = reinterpret_cast<const CT*>(jb.C);

  for (int a = tid; a < ntp; a += ST) {
    if (tp_w) tp_w[a] = a < n_t ? jb.tpos[a] : 0;
    wf[a] = (float)jb.y_t[a];
  }
  __syncthreads();
  apply_minv_f32<CL, BIG ? 2 : 1>(static_cast<const __half*>(jb.L16), jb.Linv32, ntp, wf, rvec, part, xp, crank);
  // (BIG: alpha is the job's global vector -- with CL = 2 both CTAs store the same values, then meet at a barrier)
  for (int a = tid; a < ntp; a += ST) alpha[a] = (double)wf[a];
  if (BIG) team_sync<CL>();
  else __syncthreads();

  int sweeps = 0;
  bool solved = false;               // refinement reached the tolerance (else the host re-runs the job in fp64)
  double sa = 0.0, ssa = 0.0, prev_dmax = 1e300;
  for (;;) {
    double l0 = 0.0, l1 = 0.0, l2 = 0.0;
    for (int a = tid; a < n_t; a += ST) {
      l0 += alpha[a];
      l1 += (double)jb.s[tp[a]] * alpha[a];
      l2 = fmax(l2, fabs(alpha[a]) < 1e300 ? fabs(alpha[a]) : __longlong_as_double(0x7ff0000000000000LL));
    }
    sa = block_sum(l0, red);
    ssa = block_sum(l1, red);
    const double amax_now = block_max(l2, red);
    if (sweeps == MAX_SWEEPS) break;
    if (!(amax_now < 1e300)) break;                     // non-finite first solve (overflowing factor): leave it to fp64
    sym_matvec<CONTIG, HOLE, CT, CL, BIG>(C, rpad, n_t, jb.hole0, jb.gap, tp, alpha, amax_now, jb.cmax, work, part2, crank);   // work[a] = (C alpha)_a
    for (int a = tid; a < ntp; a += ST) {
      double rr = 0.0;
      if (a < n_t) {
        const double Aa = jb.lambda * alpha[a] +
                          coef * (Nd * Nd * work[a] - Nd * (double)jb.s[tp[a]] * sa - Nd * ssa + Qd * sa);
        rr = jb.y_t[a] - Aa;
      }
      wf[a] = (float)rr;
    }
    __syncthreads();
    apply_minv_f32<CL, BIG ? 2 : 1>(static_cast<const __half*>(jb.L16), jb.Linv32, ntp, wf, rvec, part, xp, crank);
    double dmax = 0.0, amax = 0.0;
    const double INF = __longlong_as_double(0x7ff0000000000000LL);
    if (BIG && CL > 1) {
      // alpha is ONE global vector shared by the pair: both CTAs read it to form the same maxima, then one of them updates
      for (int a = tid; a < ntp; a += ST) {
        const double d = (double)wf[a];
        const double v = alpha[a] + d;
        dmax = fmax(dmax, fabs(d) < 1e300 ? fabs(d) : INF);
        amax = fmax(amax, fabs(v) < 1e300 ? fabs(v) : INF);
      }
      team_sync<CL>();
      if (crank == 0)
        for (int a = tid; a < ntp; a += ST) alpha[a] = alpha[a] + (double)wf[a];
      team_sync<CL>();
    } else {
      for (int a = tid; a < ntp; a += ST) {
        const double d = (double)wf[a];
        const double v = alpha[a] + d;
        alpha[a] = v;
        // fmax drops NaN operands: map anything non-finite to +inf so that it cannot pass for "converged"
        dmax = fmax(dmax, fabs(d) < 1e300 ? fabs(d) : INF);
        amax = fmax(amax, fabs(v) < 1e300 ? fabs(v) : INF);
      }
    }
    dmax = block_max(dmax, red);
    amax = block_max(amax, red);
    ++sweeps;
    // the correction just applied was the previous error; the error now left is about dmax * rho with
    // rho = dmax / prev_dmax the observed contraction (first sweep: assume rho <= 0.05, the TF32 factor
    // contracts by 1e-2 .. 1e-3 for cond(A) up to a few hundred)
    const double rho = sweeps == 1 ? 0.05 : fmin(1.0, dmax / prev_dmax);
    const bool finite = dmax < 1e300 && amax < 1e300;   // an overflowing fp16 factor / Inf from apply_minv: not solved
    if (!finite) break;                                 // solved stays false: the host re-runs the job in fp64
    const bool converged = dmax * rho <= REL_TOL * amax;
    // corrections no longer shrink: either the rounding floor of the residual (then they are tiny) or a factor too
    // poor to precondition (ill-conditioned matrix: lambda -> 0) -- only the first counts as solved
    const bool stalled = sweeps > 1 && dmax > 0.5 * prev_dmax;
    prev_dmax = dmax;
    if (converged || stalled) {
      solved = converged || dmax <= 1e-7 * amax;
      double m0 = 0.0, m1 = 0.0;
      for (int a = tid; a < n_t; a += ST) {
        m0 += alpha[a];
        m1 += (double)jb.s[tp[a]] * alpha[a];
      }
      sa = block_sum(m0, red);
      ssa = block_sum(m1, red);
      break;
    }
  }
  if (!big && crank == 0)
    for (int a = tid; a < ntp; a += ST) jb.alpha[a] = alpha[a];
  // diagnostics: sweeps in the low byte, + 256 when the refinement did not reach the tolerance, + 512 on a pivot failure
  if (tid == 0 && crank == 0 && jb.sweeps) *jb.sweeps = sweeps | (solved ? 0 : 256) | (*jb.status != 0 ? 512 : 0);
  if (tid == 0 && crank == 0 && jb.fail && (!solved || *jb.status != 0)) *jb.fail = 1;

  // ---- predictions on the validation animals
  if constexpr (CONTIG && C16) {
    // four validation rows per warp share every alpha piece (see sym_matvec16); rows at/after n_t are plain rows of C
      if (HOLE && jb.gap > 0 && jb.valid_in_hole) {
      // k-fold cross-validation: the validation animals are exactly the hole of the training set
      __syncthreads();
      if (crank == 0) {                                 // (not split over the pair: a tenth of a sweep's bytes)
        hole_predict16(reinterpret_cast<const int16_t*>(C), rpad, n_t, jb.hole0, jb.gap, alpha, work, part2);
        for (int v = tid; v < n_v; v += ST)
          jb.pred[v] = coef * (Nd * Nd * work[v] - Nd * (double)jb.s[jb.hole0 + v] * sa - Nd * ssa + Qd * sa);
      }
    } else
    for (int v0i = 4 * (warp + (ST / 32) * crank); v0i < n_v; v0i += 4 * (ST / 32) * CL) {
      int pv[4];
      bool fast = true;
#pragma unroll
      for (int rr = 0; rr < 4; ++rr) {
        pv[rr] = jb.vpos[min(v0i + rr, n_v - 1)];
        fast = fast && pv[rr] >= n_t && (!HOLE || jb.gap == 0);
      }
      double d[4] = {0.0, 0.0, 0.0, 0.0};
      if (fast) {
        const uint4* r0 = reinterpret_cast<const uint4*>(C + (size_t)pv[0] * rpad);
        const uint4* r1 = reinterpret_cast<const uint4*>(C + (size_t)pv[1] * rpad);
        const uint4* r2 = reinterpret_cast<const uint4*>(C + (size_t)pv[2] * rpad);
        const uint4* r3 = reinterpret_cast<const uint4*>(C + (size_t)pv[3] * rpad);
        const int n8 = n_t / 8;
        for (int c = lane; c < n8; c += 32) fma4x8s(d, r0[c], r1[c], r2[c], r3[c], alpha + 8 * c);
        for (int b = 8 * n8 + lane; b < n_t; b += 32) {
          const double z = alpha[b];
#pragma unroll
          for (int rr = 0; rr < 4; ++rr) d[rr] += (double)C[(size_t)pv[rr] * rpad + b] * z;
        }
      } else {
        for (int b = lane; b < n_t; b += 32) {
          const int p0 = tp[b];
          const double z = alpha[b];
#pragma unroll
          for (int rr = 0; rr < 4; ++rr)
            d[rr] += (double)C[(size_t)(pv[rr] > p0 ? pv[rr] : p0) * rpad + (pv[rr] > p0 ? p0 : pv[rr])] * z;
        }
      }
#pragma unroll
      for (int rr = 0; rr < 4; ++rr) {
        const double t = warp_sum(d[rr]);
        if (lane == 0 && v0i + rr < n_v)
          jb.pred[v0i + rr] = coef * (Nd * Nd * t - Nd * (double)jb.s[pv[rr]] * sa - Nd * ssa + Qd * sa);
      }
    }
  } else {
  for (int v = warp + (ST / 32) * crank; v < n_v; v += (ST / 32) * CL) {
    const int pv = jb.vpos[v];
    double d0 = 0.0, d1 = 0.0, d2 = 0.0, d3 = 0.0;
    if (CONTIG && !C16 && pv >= n_t) {
      const int4* row = reinterpret_cast<const int4*>(C + (size_t)pv * rpad);
      const int n4 = n_t / 4;
      int c = lane;
      for (; c + 96 < n4; c += 128) {
        const int4 v0 = row[c], v1 = row[c + 32], v2 = row[c + 64], v3 = row[c + 96];
        d0 += dot4i(v0, alpha + 4 * c);
        d1 += dot4i(v1, alpha + 4 * (c + 32));
        d2 += dot4i(v2, alpha + 4 * (c + 64));
        d3 += dot4i(v3, alpha + 4 * (c + 96));
      }
      for (; c < n4; c += 32) d0 += dot4i(row[c], alpha + 4 * c);
      for (int b = 4 * n4 + lane; b < n_t; b += 32) d1 += (double)C[(size_t)pv * rpad + b] * alpha[b];
    } else {
      int b = lane;
      for (; b + 32 < n_t; b += 64) {
        const int p0 = tp[b], p1 = tp[b + 32];
        const int c0 = C[(size_t)(pv > p0 ? pv : p0) * rpad + (pv > p0 ? p0 : pv)];
        const int c1 = C[(size_t)(pv > p1 ? pv : p1) * rpad + (pv > p1 ? p1 : pv)];
        d0 += (double)c0 * alpha[b];
        d1 += (double)c1 * alpha[b + 32];
      }
      for (; b < n_t; b += 32) {
        const int p0 = tp[b];
        d0 += (double)C[(size_t)(pv > p0 ? pv : p0) * rpad + (pv > p0 ? p0 : pv)] * alpha[b];
      }
    }
    const double d = warp_sum((d0 + d1) + (d2 + d3));
    if (lane == 0) jb.pred[v] = coef * (Nd * Nd * d - Nd * (double)jb.s[pv] * sa - Nd * ssa + Qd * sa);
  }
  }
  team_sync<CL>();                    // (CL = 2: the partner's half of the predictions is visible in global memory)
  if (crank != 0) return;             // the accuracy is one CTA's work; nothing of this CTA is read remotely any more

  double sy = 0.0, sp = 0.0;
  for (int v = tid; v < n_v; v += ST) {
    sy += jb.y_v[v];
    sp += jb.pred[v];
  }
  const double my = block_sum(sy, red) / n_v;
  const double mp = block_sum(sp, red) / n_v;
  double sxy = 0.0, sxx = 0.0, syy = 0.0;
  for (int v = tid; v < n_v; v += ST) {
    const double dy = jb.y_v[v] - my, dp = jb.pred[v] - mp;
    sxy += dy * dp;
    sxx += dy * dy;
    syy += dp * dp;
  }
  sxy = block_sum(sxy, red);
  sxx = block_sum(sxx, red);
  syy = block_sum(syy, red);
  if (tid == 0) {
    double r;
    if (*jb.status != 0 || !(sxx > 0.0) || !(syy > 0.0)) {
      r = __longlong_as_double(0x7ff8000000000000LL);
    } else {
      r = sxy / (sqrt(sxx) * sqrt(syy));
      r = (fabs(r) < 1e300) ? fabs(fmax(fmin(r, 1.0), -1.0)) : __longlong_as_double(0x7ff8000000000000LL);
    }
    *jb.fitness = r;
  }
}

// fp32 copy of A = G_tt + lambda I (lower triangle, identity padding) for the tensor-core factorisation.
// Block = 64 rows x 128 columns; a thread owns 4 consecutive columns (one 16-byte load of C, one 16-byte store) of
// 8 rows, so the per-column setup (positions, column terms) is amortised over 8 rows and the 8 row loads are
// independent.  (The exact operator lives in solve_mixed_kernel; this matrix only feeds the 10-bit preconditioner.)
constexpr int S32_ROWS = 64;
template <bool C16>
__global__ void __launch_bounds__(256) scale32_kernel(const TbScaleJob* __restrict__ jobs, float* __restrict__ L32,
                                                      int ntp_all) {
  const TbScaleJob jb = jobs[blockIdx.z];
  const int ntp = jb.ntp, n_t = jb.n_t, rpad = jb.rpad;
  const int r0 = blockIdx.y * S32_ROWS, c0 = blockIdx.x * 128;
  if (r0 >= ntp || c0 >= ntp || c0 > r0 + S32_ROWS - 1) return;
  const int c = c0 + (threadIdx.x & 31) * 4;
  if (c >= ntp) return;
  // same evaluation as the fused Gram epilogue (gram_tc.cu): coefficients from the exact integers in fp64, rounded
  // once; the fp32 combination below only handles O(1) quantities and no 64-bit integer -> float conversion
  const long long N = jb.N, S = jb.SQ[0], Q = jb.SQ[1];
  const double inv_d = 2.0 / (double)(2 * N * S - Q);
  const float scale = (float)(inv_d * (double)(N * N)), lam = (float)jb.lambda;
  int pc[4];
  float sc[4];
  bool creal[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    creal[i] = c + i < n_t;
    pc[i] = creal[i] ? jb.tpos[c + i] : 0;
    sc[i] = creal[i] ? (float)(inv_d * (double)(Q - N * jb.s[pc[i]])) : 0.f;
  }
  const bool run = creal[3] && pc[1] == pc[0] + 1 && pc[2] == pc[0] + 2 && pc[3] == pc[0] + 3 && (pc[0] & 3) == 0;
  float* out_base = L32 + (size_t)blockIdx.z * ntp_all * ntp_all;
  const int rbase = r0 + (threadIdx.x >> 5);
  // phase 1: positions, row terms and the integer cross-products of the 8 rows (independent loads)
  int pr[8];
  float sr[8];
  int4 cv[8];
#pragma unroll
  for (int h = 0; h < 8; ++h) {
    const int r = rbase + 8 * h;
    pr[h] = (r < n_t) ? jb.tpos[r] : -1;
  }
#pragma unroll
  for (int h = 0; h < 8; ++h) {
    const int r = rbase + 8 * h;
    sr[h] = 0.f;
    cv[h] = make_int4(0, 0, 0, 0);
    if (pr[h] >= 0 && c <= r) {
      sr[h] = (float)(inv_d * (double)(-N * jb.s[pr[h]]));
      if (run && pc[3] < pr[h]) {
        if (C16) {
          const uint2 u = *reinterpret_cast<const uint2*>(reinterpret_cast<const int16_t*>(jb.C) + (size_t)pr[h] * rpad + pc[0]);
          cv[h] = make_int4((int)(u.x & 0xffffu), (int)(u.x >> 16), (int)(u.y & 0xffffu), (int)(u.y >> 16));
        } else {
          cv[h] = *reinterpret_cast<const int4*>(jb.C + (size_t)pr[h] * rpad + pc[0]);
        }
      } else {
        int t[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int hi = pr[h] > pc[i] ? pr[h] : pc[i], lo = pr[h] > pc[i] ? pc[i] : pr[h];
          t[i] = !creal[i] ? 0
                 : C16 ? (int)reinterpret_cast<const int16_t*>(jb.C)[(size_t)hi * rpad + lo]
                       : jb.C[(size_t)hi * rpad + lo];
        }
        cv[h] = make_int4(t[0], t[1], t[2], t[3]);
      }
    }
  }
  // phase 2: arithmetic and stores
#pragma unroll
  for (int h = 0; h < 8; ++h) {
    const int r = rbase + 8 * h;
    if (r >= ntp || c > r) continue;
    float out[4];
    if (r >= n_t) {
#pragma unroll
      for (int i = 0; i < 4; ++i) out[i] = (r == c + i) ? 1.f : 0.f;
    } else {
      const int cvv[4] = {cv[h].x, cv[h].y, cv[h].z, cv[h].w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float g = 0.f;
        if (creal[i]) {
          // cross-products are below 2^23: 0x4b000000 | c is the float 2^23 + c
          const float cf = __uint_as_float(0x4b000000u | (unsigned)cvv[i]) - 8388608.f;
          g = fmaf(cf, scale, sr[h] + sc[i]);
          if (r == c + i) g += lam;
        }
        out[i] = g;
      }
    }
    *reinterpret_cast<float4*>(out_base + (size_t)r * ntp_all + c) = make_float4(out[0], out[1], out[2], out[3]);
  }
}

// Row / column terms and coefficients of the scaled matrix for the Cholesky update's epilogue (see TbFromC): the same
// fp64-from-exact-integers coefficients, rounded once, that scale32_kernel and the old fused Gram epilogue used.
__global__ void fuse_terms_kernel(const TbScaleJob* __restrict__ jobs, int ntp, float* __restrict__ terms,
                                  TbFuseCoef* __restrict__ coef) {
  const TbScaleJob jb = jobs[blockIdx.y];
  const long long N = jb.N, S = jb.SQ[0], Q = jb.SQ[1];
  const double inv_d = 2.0 / (double)(2 * N * S - Q);
  const int a = blockIdx.x * blockDim.x + threadIdx.x;
  if (a == 0)
    coef[blockIdx.y] = TbFuseCoef{(float)(inv_d * (double)(N * N)), (float)jb.lambda, jb.n_t, jb.hole0, jb.gap, jb.cw};
  if (a >= ntp) return;
  float rt = 0.f, ct = 0.f;
  if (a < jb.n_t) {
    const long long sa = jb.s[jb.tpos[a]];
    rt = (float)(inv_d * (double)(-N * sa));
    ct = (float)(inv_d * (double)(Q - N * sa));
  }
  terms[(size_t)blockIdx.y * 2 * ntp + a] = rt;
  terms[(size_t)blockIdx.y * 2 * ntp + ntp + a] = ct;
}

int g_solve_mixed_smem_max = 0;

}  // namespace

void tb_solve_mixed_set_debug(int) {}

static inline int solve_mixed_smem_bytes(int ntp) {
  const int fixed = (ntp + 4 * 512 + ST / 32) * (int)sizeof(double) + (ntp + NB + (ST / 32) * NB + 2 * NB) * (int)sizeof(float);
  return ntp > MIXED_SMEM_NTP ? fixed : fixed + ntp * (int)(sizeof(double) + sizeof(int));
}

cudaError_t tb_solve_mixed_init() {
  g_solve_mixed_smem_max = 220 * 1024;
  cudaError_t e = cudaSuccess;
  auto set = [&](const void* fn) {
    if (e == cudaSuccess) e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, g_solve_mixed_smem_max);
  };
  set((const void*)solve_mixed_kernel<true, false, false, false, 1>);
  set((const void*)solve_mixed_kernel<false, false, false, false, 1>);
  set((const void*)solve_mixed_kernel<true, true, false, false, 1>);
  set((const void*)solve_mixed_kernel<false, true, false, false, 1>);
  set((const void*)solve_mixed_kernel<true, false, true, false, 1>);
  set((const void*)solve_mixed_kernel<false, false, true, false, 1>);
  set((const void*)solve_mixed_kernel<true, true, true, false, 1>);
  set((const void*)solve_mixed_kernel<false, true, true, false, 1>);
  set((const void*)solve_mixed_kernel<true, false, true, true, 1>);
  set((const void*)solve_mixed_kernel<true, true, true, true, 1>);
  set((const void*)solve_mixed_kernel<true, false, false, false, 2>);
  set((const void*)solve_mixed_kernel<true, true, false, false, 2>);
  set((const void*)solve_mixed_kernel<true, false, true, false, 2>);
  set((const void*)solve_mixed_kernel<true, true, true, false, 2>);
  set((const void*)solve_mixed_kernel<true, false, true, true, 2>);
  set((const void*)solve_mixed_kernel<true, true, true, true, 2>);
  return e;
}

bool tb_solve_mixed_fits(int ntp) { return solve_mixed_smem_bytes(ntp) <= 220 * 1024; }

// contiguous != 0: every job's training animal b sits at universe position b and n_t is a multiple of 4
// (vectorised symmetric mat-vec); otherwise positions are looked up per element.
// hole != 0 (with contiguous and c16): some row set is contiguous with one aligned hole (see TbRowSet).
cudaError_t tb_launch_solve_mixed(const TbSolveMixedJob* d_jobs, int n_jobs, int ntp, int contiguous, int c16, int hole,
                                  cudaStream_t st, int n_sm, int pair_mode, int* variant) {
  const int smem = solve_mixed_smem_bytes(ntp);
  if (smem > g_solve_mixed_smem_max) return cudaErrorInvalidConfiguration;
  const bool big = ntp > MIXED_SMEM_NTP;
  // two CTAs per matrix when the batch would leave more than half of the CTA slots empty (pair_mode: 0 never, 1 auto,
  // 2 always); contiguous kernels only
  const int slots = n_sm * ((smem + 1024) * 2 <= 228 * 1024 ? 2 : 1);
  const bool pair = contiguous && pair_mode != 0 && (pair_mode == 2 || 2 * n_jobs <= slots);
  // the instantiation launched below, as the TB_SOLVE_* bits of tb_get_info "last_solve"
  if (variant)
    *variant = (contiguous ? 1 : 0) | (big ? 2 : 0) | (c16 ? 4 : 0) | (hole && contiguous && c16 ? 8 : 0) | (pair ? 16 : 0);
  if (pair) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * n_jobs);
    cfg.blockDim = dim3(ST);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    if (hole && c16) {
      if (big) return cudaLaunchKernelEx(&cfg, solve_mixed_kernel<true, true, true, true, 2>, d_jobs);
      return cudaLaunchKernelEx(&cfg, solve_mixed_kernel<true, false, true, true, 2>, d_jobs);
    }
    if (c16) {
      if (big) return cudaLaunchKernelEx(&cfg, solve_mixed_kernel<true, true, true, false, 2>, d_jobs);
      return cudaLaunchKernelEx(&cfg, solve_mixed_kernel<true, false, true, false, 2>, d_jobs);
    }
    if (big) return cudaLaunchKernelEx(&cfg, solve_mixed_kernel<true, true, false, false, 2>, d_jobs);
    return cudaLaunchKernelEx(&cfg, solve_mixed_kernel<true, false, false, false, 2>, d_jobs);
  }
  if (hole && contiguous && c16) {
    if (big) solve_mixed_kernel<true, true, true, true, 1><<<n_jobs, ST, smem, st>>>(d_jobs);
    else solve_mixed_kernel<true, false, true, true, 1><<<n_jobs, ST, smem, st>>>(d_jobs);
    return cudaGetLastError();
  }
  const int which = (contiguous ? 4 : 0) | (big ? 2 : 0) | (c16 ? 1 : 0);
  switch (which) {
    case 0: solve_mixed_kernel<false, false, false, false, 1><<<n_jobs, ST, smem, st>>>(d_jobs); break;
    case 1: solve_mixed_kernel<false, false, true, false, 1><<<n_jobs, ST, smem, st>>>(d_jobs); break;
    case 2: solve_mixed_kernel<false, true, false, false, 1><<<n_jobs, ST, smem, st>>>(d_jobs); break;
    case 3: solve_mixed_kernel<false, true, true, false, 1><<<n_jobs, ST, smem, st>>>(d_jobs); break;
    case 4: solve_mixed_kernel<true, false, false, false, 1><<<n_jobs, ST, smem, st>>>(d_jobs); break;
    case 5: solve_mixed_kernel<true, false, true, false, 1><<<n_jobs, ST, smem, st>>>(d_jobs); break;
    case 6: solve_mixed_kernel<true, true, false, false, 1><<<n_jobs, ST, smem, st>>>(d_jobs); break;
    default: solve_mixed_kernel<true, true, true, false, 1><<<n_jobs, ST, smem, st>>>(d_jobs); break;
  }
  return cudaGetLastError();
}

cudaError_t tb_launch_fuse_terms(const TbScaleJob* d_jobs, int n_jobs, int ntp, float* terms, TbFuseCoef* coef,
                                 cudaStream_t st) {
  dim3 grid((ntp + 255) / 256, n_jobs);
  fuse_terms_kernel<<<grid, 256, 0, st>>>(d_jobs, ntp, terms, coef);
  return cudaGetLastError();
}

cudaError_t tb_launch_scale32(const TbScaleJob* d_jobs, int n_jobs, int ntp, float* L32, int c16, cudaStream_t st,
                              int col_end) {
  const int cols = col_end > 0 && col_end < ntp ? col_end : ntp;
  dim3 grid((cols + 127) / 128, (ntp + S32_ROWS - 1) / S32_ROWS, n_jobs);
  if (c16) scale32_kernel<true><<<grid, 256, 0, st>>>(d_jobs, L32, ntp);
  else scale32_kernel<false><<<grid, 256, 0, st>>>(d_jobs, L32, ntp);
  return cudaGetLastError();
}
