// Mixed-precision batched Cholesky on the 5th-generation tensor cores.
//
// The factorisation of A = G_tt + lambda I only has to be good enough to precondition: solve.cu refines the
// solution against the exact integer cross-products in fp64 until the correction vanishes (cond(A) <= ~150,
// so a TF32 factor contracts the error by > 100x per sweep; see DESIGN.md §3).  That moves the n^3/3 flops of
// tblup/evaluator.py:282 from the FP64 pipe (37 TFLOP/s) to tcgen05.mma.kind::tf32 (~1.1 PFLOP/s nominal).
//
// Storage: one fp32 matrix per (individual, row set), L32[job][ntp][ntp] (lower triangle meaningful), plus the
// fp32 inverses of the 64 x 64 diagonal blocks.  Two-level left-looking schedule, all jobs in lock-step:
//   outer block column J (256 wide):  T[:, J] -= L[:, 0:J] L[J, 0:J]^T          tf32_gemm  N = 256, K = 256 J
//   inner block column i (64 wide):   T[:, i] -= L[:, J0:i] L[i, J0:i]^T        tf32_gemm  N = 64,  K <= 192
//                                     L[i][i] = chol(T[i][i]), Linv_i           chol_diag32_kernel (fp64 math)
//                                     L[:, i] = T[:, i] Linv_i^T                tf32_gemm  N = 64,  K = 64
// The wide outer update keeps DRAM traffic at n^3/(6*256) words per matrix (a 64-wide left-looking sweep would be
// HBM-bound) and gives the MMA its most efficient shape (M128 x N256); the narrow inner steps touch only the
// 256-wide panel.
//
// tf32_gemm_kernel is the Gram kernel's structure (gram_tc.cu) with fp32 operands: persistent CTAs, warp 0 = TMA
// producer (SWIZZLE_128B boxes of 32 floats x 64 rows, 4-stage ring), warp 1 = single-thread MMA issuer
// (tcgen05.mma.cta_group::1.kind::tf32, M = 128, N = 64..256, K = 8 per instruction, fp32 accumulators in TMEM,
// double-buffered), warps 2-5 = epilogue (tcgen05.ld -> read-modify-write of the fp32 tile in global memory).
#include "tb_internal.h"
#include "tb_ptx.cuh"
#include <cuda_fp16.h>

namespace {

using namespace tbptx;

constexpr int NB = TB_NB;            // 64
constexpr int TBM = 128;             // tile rows
constexpr int TBK = 32;              // floats per k-block (one 128-byte swizzle span)
constexpr int BOX_ROWS = 64;         // TMA box: 32 floats x 64 rows = 8 KiB
constexpr int BOX_BYTES = BOX_ROWS * TBK * 4;
constexpr int MAX_N = 256;
constexpr int TSTAGES = 4;
constexpr int TA_BYTES = TBM * TBK * 4;          // 16 KiB
constexpr int TB_BYTES_MAX = MAX_N * TBK * 4;    // 32 KiB
constexpr int TSTAGE_BYTES = TA_BYTES + TB_BYTES_MAX;
constexpr int TACC = 2;
// epilogue warps (template parameter EW): 8 or 16 -- EW / 4 warps per TMEM lane quarter share the columns of a tile
constexpr int t_threads(int ew) { return 64 + 32 * ew; }
constexpr int HBK = 64;              // halves per k-block when the operands are fp16 (same 128-byte span)
// ring + alignment slack + barriers + per-warp transposition buffers (coalescing epilogue stores)
constexpr int t_smem(int ew) { return TSTAGES * TSTAGE_BYTES + 1024 + 256 + ew * 2048; }

struct GemmParams {
  int n_jobs;
  int ntp;           // rows (= columns) of every job's matrix; also rows per job in tensor map A
  int row0;          // first output row
  int row_end;       // one past the last output row (<= ntp)
  int n_mtiles;      // ceil((row_end - row0) / 128)
  int a_col0;        // K range of the A operand: columns [a_col0, a_col0 + K)
  int K;             // multiple of 32
  int b_row0;        // first row of the B operand inside its job
  int b_col0;        // first column of the B operand
  int b_rows_per_job;
  int c_col0;        // first output column (in L32)
  int N;             // output columns: 64, 128, 192 or 256
  int mode;          // 0: C -= A B^T   1: C = A B^T rounded to TF32 (final L entries)
  int skip32;        // mode 1 only: do not write the fp32 copy (nothing reads these entries of L32 again)
  float* L32;
  __half* L16;       // optional half-precision copy of the final factor entries (read by the solve)
  int from_c;        // mode 0 only: the matrix entries come from the integer cross-products (TbFromC), not from L32
  int t16;           // mode 0 only: tiles BELOW the 256-row diagonal block (m-tile >= 2) are written as halves into L16 (where
                     // the wide panel GEMM reads them and writes the final factor entries in place), not as fp32 into L32
  int f16ops;        // mode 1 only: both operands are fp16 (A from L16 in place, B the fp16 inverse of the diagonal block)
  TbFromC fc;
};

struct TBarriers {
  uint64_t full[TSTAGES];
  uint64_t empty[TSTAGES];
  uint64_t acc_full[TACC];
  uint64_t acc_empty[TACC];
  uint32_t tmem_base;
};

__host__ __device__ constexpr uint32_t umma_idesc_tf32(int m, int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<uint32_t>(n >> 3) << 17) |
         (static_cast<uint32_t>(m >> 4) << 24);
}

__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// fp16 operands, fp32 accumulation: the factor is rounded to 10 mantissa bits anyway, so its half-precision copy
// carries the same values at half the bytes and the MMA runs at twice the TF32 rate.
__host__ __device__ constexpr uint32_t umma_idesc_f16(int m, int n) {
  return (1u << 4) | (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(m >> 4) << 24);
}

__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

__device__ __forceinline__ float round_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}

// A cross-product as a float.  Integers below 2^23: 0x4b000000 | c is the float 2^23 + c (no converter pipe); one byte
// permute per int16 half of a word.
__device__ __forceinline__ float c_from_i16(uint32_t w, bool hi) {
  return __uint_as_float(__byte_perm(w, 0x4b000000u, hi ? 0x7432 : 0x7410)) - 8388608.f;
}
__device__ __forceinline__ float c_from_i32(uint32_t w) { return __uint_as_float(0x4b000000u | w) - 8388608.f; }

// SRC: where update mode reads the entries it modifies -- 0: the fp32 matrix L32, 1: int16 cross-products, 2: int32
// cross-products (TbFromC: the scaled matrix is formed on the fly)
template <bool F16, int SRC, int EW>
__global__ void __launch_bounds__(t_threads(EW), 1)
tf32_gemm_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                 const __grid_constant__ GemmParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  TBarriers* bars = reinterpret_cast<TBarriers*>(smem + TSTAGES * TSTAGE_BYTES);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_items = p.n_jobs * p.n_mtiles;
  constexpr int KB_ELEMS = F16 ? HBK : TBK;       // elements per 128-byte k-block
  const int nkb = p.K / KB_ELEMS;
  const int n_bbox = p.N / BOX_ROWS;
  const uint32_t stage_tx = TA_BYTES + n_bbox * BOX_BYTES;

  if (warp == 0 && lane == 0) {
    prefetch_tensormap(&tmap_a);
    prefetch_tensormap(&tmap_b);
    for (int s = 0; s < TSTAGES; ++s) {
      mbar_init(&bars->full[s], 1);
      mbar_init(&bars->empty[s], 1);
    }
    for (int s = 0; s < TACC; ++s) {
      mbar_init(&bars->acc_full[s], 1);
      mbar_init(&bars->acc_empty[s], EW);
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<TACC * MAX_N>(&bars->tmem_base);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = bars->tmem_base;

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
        const int job = item / p.n_mtiles, mt = item - job * p.n_mtiles;
        const int row_a = job * p.ntp + p.row0 + mt * TBM;
        const int row_b = job * p.b_rows_per_job + p.b_row0;
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&bars->empty[stage], phase ^ 1);
          uint8_t* sa = smem + stage * TSTAGE_BYTES;
          mbar_arrive_expect_tx(&bars->full[stage], stage_tx);
          tma_load_2d(sa, &tmap_a, &bars->full[stage], p.a_col0 + kb * KB_ELEMS, row_a);
          tma_load_2d(sa + BOX_BYTES, &tmap_a, &bars->full[stage], p.a_col0 + kb * KB_ELEMS, row_a + BOX_ROWS);
          for (int b = 0; b < n_bbox; ++b)
            tma_load_2d(sa + TA_BYTES + b * BOX_BYTES, &tmap_b, &bars->full[stage], p.b_col0 + kb * KB_ELEMS,
                        row_b + b * BOX_ROWS);
          if (++stage == TSTAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && nkb > 0) {       // (K = 0: block column 0 formed from the cross-products alone, no product to subtract)
      const uint32_t idesc = F16 ? umma_idesc_f16(TBM, p.N) : umma_idesc_tf32(TBM, p.N);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
        mbar_wait(&bars->acc_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * MAX_N;
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&bars->full[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * TSTAGE_BYTES);
          const uint64_t adesc = umma_desc_k_sw128(sa);
          const uint64_t bdesc = umma_desc_k_sw128(sa + TA_BYTES);
#pragma unroll
          for (int k = 0; k < 4; ++k) {          // four 32-byte K slices per 128-byte span (8 floats / 16 halves)
            if (F16) umma_f16(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0);
            else umma_tf32(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0);
          }
          umma_commit(&bars->empty[stage]);
          if (++stage == TSTAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        umma_commit(&bars->acc_full[acc]);
        if (++acc == TACC) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
    }
  } else {
    // Epilogue: warp w reads TMEM lanes 32 (w & 3) .. +31 (one accumulator row per thread); the EW / 4 warps of a lane
    // quarter take the 32-column chunks of the tile round-robin (chunk g, g + CG, ...).  In update mode the C values a
    // thread will modify do not depend on the MMA, so all of its loads are issued BEFORE it waits for the accumulator:
    // the read latency hides behind the tile's own MMA instead of serialising chunk by chunk.
    // The first block columns of a factorisation are bound by THIS code, not by the operand stream (the K = 0 launch
    // runs at what the epilogue alone sustains); sixteen warps instead of eight double the latency cover, and the
    // per-entry work is what the common case needs: the diagonal (+ lambda) and the padding rows are patched in
    // warp-uniform side branches instead of being tested per entry.
    constexpr int CG = EW / 4;                                  // column groups
    constexpr int MAXI = 8 / CG;                                // chunks per warp at N = 256
    constexpr int CVN = SRC == 1 ? 4 : 8;                       // 16-byte loads per chunk and thread
    const int q = warp & 3, g = (warp - 2) >> 2;
    const uint32_t stg = smem_u32(smem + TSTAGES * TSTAGE_BYTES + 256) + (warp - 2) * 2048;
    const int nchunks = p.N / 32;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
      const int job = item / p.n_mtiles, mt = item - job * p.n_mtiles;
      const int r = p.row0 + mt * TBM + q * 32 + lane;          // row inside the job's matrix
      const int r_hi = p.row0 + mt * TBM + TBM - 1;
      const float* crow = p.L32 + ((size_t)job * p.ntp + (r < p.row_end ? r : 0)) * p.ntp + p.c_col0;
      float4 cv[MAXI][CVN];
      float f_scale = 0.f, f_lam = 0.f, f_rt = 0.f;
      int f_nt = 0, f_h0 = 0, f_gap = 0;
      const float* f_ct = nullptr;
      if (SRC != 0) {
        // the entries of A this thread needs, as integer cross-products (8 or 16 bytes per 4 entries instead of a
        // read of an fp32 matrix somebody had to write): cv holds the RAW bits until the accumulator is there
        const TbFuseCoef cf = p.fc.coef[job];
        f_scale = cf.scale;
        f_lam = cf.lam;
        f_nt = cf.n_t;
        f_rt = p.fc.terms[(size_t)job * 2 * p.ntp + (r < p.row_end ? r : 0)];
        f_ct = p.fc.terms + (size_t)job * 2 * p.ntp + p.ntp + p.c_col0;
        // compact index -> panel row / column: a + (a >= hole0 ? gap : 0); hole0 and gap are multiples of 8, so an
        // 8-column group never straddles the hole (plain prefix: hole0 = n_t, gap = 0)
        const int rr = r < cf.n_t ? r + (r >= cf.hole0 ? cf.gap : 0) : 0;
        const size_t rowoff = ((size_t)cf.cw * p.fc.rpad + rr) * p.fc.rpad;
        f_h0 = cf.hole0;
        f_gap = cf.gap;
#pragma unroll
        for (int i = 0; i < MAXI; ++i) {
          const int ch = g + CG * i;
          if (ch < nchunks && p.c_col0 + ch * 32 <= r_hi && r < p.row_end) {
            if (SRC == 1) {
#pragma unroll
              for (int j = 0; j < 4; ++j) {                      // 8 columns per 16-byte load
                const int b = p.c_col0 + ch * 32 + 8 * j;
                const int ub = b + ((b >= f_h0 && b < f_nt) ? f_gap : 0);
                const uint4 u = *reinterpret_cast<const uint4*>(static_cast<const int16_t*>(p.fc.C) + rowoff + ub);
                cv[i][j] = make_float4(__uint_as_float(u.x), __uint_as_float(u.y), __uint_as_float(u.z), __uint_as_float(u.w));
              }
            } else {
#pragma unroll
              for (int j = 0; j < CVN; ++j) {                    // 4 columns per 16-byte load
                const int b = p.c_col0 + ch * 32 + 4 * j;
                const int ub = b + ((b >= f_h0 && b < f_nt) ? f_gap : 0);
                cv[i][j] = *reinterpret_cast<const float4*>(static_cast<const int32_t*>(p.fc.C) + rowoff + ub);
              }
            }
          }
        }
      } else if (p.mode == 0) {
#pragma unroll
        for (int i = 0; i < MAXI; ++i) {
          const int ch = g + CG * i;
          if (ch < nchunks && p.c_col0 + ch * 32 <= r_hi && r < p.row_end) {
            const float4* src = reinterpret_cast<const float4*>(crow + ch * 32);
#pragma unroll
            for (int j = 0; j < CVN; ++j) cv[i][j] = src[j];
          }
        }
      }
      const bool has_acc = nkb > 0;
      if (has_acc) {
        mbar_wait(&bars->acc_full[acc], acc_phase);
        tc_fence_after();
      }
      // stores go through the per-warp staging buffer (tb_ptx.cuh): 8 rows x 64 contiguous bytes per instruction
      const int rw0 = p.row0 + mt * TBM + q * 32;               // first row of this warp
      const bool tile16 = p.mode == 0 && p.t16 && mt >= 2;      // (tile-uniform) block-column entries kept as halves
      const int rl = lane >> 2, gl = 4 * (lane & 3);
#pragma unroll
      for (int i = 0; i < MAXI; ++i) {
        const int ch = g + CG * i;
        const int b0 = p.c_col0 + ch * 32;
        if (ch >= nchunks || b0 > r_hi) continue;                // beyond N, or strictly above the diagonal
        uint32_t v[32];
        if (has_acc) {
          tmem_ld_32x32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * MAX_N + ch * 32, v);
          tmem_ld_wait();
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = 0u;
        }
        uint32_t o[32];
        if (SRC != 0) {
          // A_rb = scale C_rb + rowterm_r + colterm_b (+ lambda on the diagonal; identity on the padding rows), T = A - acc
          const bool pad_warp = rw0 + 32 > f_nt;                 // (warp-uniform) some rows of this warp are padding
          const bool real_row = r < f_nt;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 ct = *reinterpret_cast<const float4*>(f_ct + ch * 32 + 4 * j);
            float cx[4];
            if (SRC == 1) {
              const float4 raw = cv[i][j >> 1];
              const uint32_t w0 = (j & 1) ? __float_as_uint(raw.z) : __float_as_uint(raw.x);
              const uint32_t w1 = (j & 1) ? __float_as_uint(raw.w) : __float_as_uint(raw.y);
              cx[0] = c_from_i16(w0, false);
              cx[1] = c_from_i16(w0, true);
              cx[2] = c_from_i16(w1, false);
              cx[3] = c_from_i16(w1, true);
            } else {
              const float4 raw = cv[i][SRC == 1 ? 0 : j];
              cx[0] = c_from_i32(__float_as_uint(raw.x));
              cx[1] = c_from_i32(__float_as_uint(raw.y));
              cx[2] = c_from_i32(__float_as_uint(raw.z));
              cx[3] = c_from_i32(__float_as_uint(raw.w));
            }
            const float ctv[4] = {ct.x, ct.y, ct.z, ct.w};
            if (pad_warp) {
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const float a = real_row ? fmaf(cx[e], f_scale, f_rt + ctv[e]) : (b0 + 4 * j + e == r ? 1.f : 0.f);
                o[4 * j + e] = __float_as_uint(a - __uint_as_float(v[4 * j + e]));
              }
            } else {
#pragma unroll
              for (int e = 0; e < 4; ++e)
                o[4 * j + e] = __float_as_uint(fmaf(cx[e], f_scale, f_rt + ctv[e]) - __uint_as_float(v[4 * j + e]));
            }
          }
          if (b0 < rw0 + 32 && b0 + 32 > rw0) {                  // (warp-uniform) the chunk holds diagonal entries
            if (real_row) {
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (b0 + j == r) o[j] = __float_as_uint(__uint_as_float(o[j]) + f_lam);
            }
          }
        } else if (p.mode == 0) {
#pragma unroll
          for (int j = 0; j < CVN; ++j) {
            o[4 * j] = __float_as_uint(cv[i][j].x - __uint_as_float(v[4 * j]));
            o[4 * j + 1] = __float_as_uint(cv[i][j].y - __uint_as_float(v[4 * j + 1]));
            o[4 * j + 2] = __float_as_uint(cv[i][j].z - __uint_as_float(v[4 * j + 2]));
            o[4 * j + 3] = __float_as_uint(cv[i][j].w - __uint_as_float(v[4 * j + 3]));
          }
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) o[j] = __float_as_uint(round_tf32(__uint_as_float(v[j])));
        }
        if (!(p.mode != 0 && p.skip32) && !tile16) {
          float* wbase = p.L32 + ((size_t)job * p.ntp + rw0) * p.ntp + b0;
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            stage_write16(stg, lane, o + 16 * h);
            __syncwarp();
#pragma unroll
            for (int it = 0; it < 4; ++it) {
              const uint4 u = stage_read16(stg, lane, it);
              if (rw0 + 8 * it + rl < p.row_end)
                *reinterpret_cast<uint4*>(wbase + (size_t)(8 * it + rl) * p.ntp + 16 * h + gl) = u;
            }
            __syncwarp();
          }
        }
        if ((p.mode != 0 && p.L16) || tile16) {
          uint32_t hv[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const __half2 hh = __floats2half2_rn(__uint_as_float(o[2 * j]), __uint_as_float(o[2 * j + 1]));
            hv[j] = *reinterpret_cast<const uint32_t*>(&hh);
          }
          __half* hbase = p.L16 + ((size_t)job * p.ntp + rw0) * p.ntp + b0;
          stage_write16(stg, lane, hv);
          __syncwarp();
#pragma unroll
          for (int it = 0; it < 4; ++it) {
            const uint4 u = stage_read16(stg, lane, it);
            if (rw0 + 8 * it + rl < p.row_end)
              *reinterpret_cast<uint4*>(hbase + (size_t)(8 * it + rl) * p.ntp + 2 * gl) = u;
          }
          __syncwarp();
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0 && has_acc) mbar_arrive(&bars->acc_empty[acc]);
      if (++acc == TACC) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<TACC * MAX_N>(tmem_base);
  }
}

// The rows below the 256-row diagonal block of a wide block column formed from the cross-products, finished in ONE
// launch (option panel_fused).  Per 128 x 256 tile:
//   phase 1  T = A - L[:, 0:c0] L[J, 0:c0]^T   the outer update and its epilogue; T, rounded to halves, goes into a
//                                              shared-memory tile laid out as the K-major SWIZZLE_128B MMA operand
//   phase 2  L = T X^T                         X = the fp16 inverse of the diagonal block (K = 256); the rounded factor
//                                              entries go back into the same buffer and leave by TMA store into L16
// Same operands, MMA shapes and K order as the update (t16) + wide panel GEMM (f16ops) pair, so the factor is
// bit-identical; T no longer makes a round trip through L16 (2 + 2 bytes per entry) and the panel launch is gone.
// Shared memory: a 3-stage ring (144 KB; phase 2 only fills the B slots) + the 64 KB T tile.  Both TMEM accumulators
// are used: phase 2 of tile k reuses tile k's accumulator once phase 1's epilogue has drained it, and the MMA warp
// issues phase 1 of tile k + 1 BEFORE phase 2 of tile k, so the tensor pipe runs the long product while the epilogue
// stages T (the epilogue, which reads the cross-products, is the longer of the two).
constexpr int FSTAGES = 3;
constexpr int FT_KB_BYTES = TBM * 128;              // one 64-half k-block of the T tile
constexpr int FT_BYTES = 4 * FT_KB_BYTES;           // 64 KiB
constexpr int F_SMEM = FSTAGES * TSTAGE_BYTES + FT_BYTES + 1024 + 256;

struct FBarriers {
  uint64_t full[FSTAGES];
  uint64_t empty[FSTAGES];
  uint64_t p1_full[TACC];      // phase 1 product of the tile in accumulator a complete
  uint64_t p2_full[TACC];      // phase 2 product complete (the T tile has been read)
  uint64_t acc_empty[TACC];
  uint64_t t_full;             // the T tile is in shared memory
  uint32_t tmem_base;
};
static_assert(sizeof(FBarriers) <= 256, "barrier block");

template <int SRC, int EW>
__global__ void __launch_bounds__(t_threads(EW), 1)
panel_fused_kernel(const __grid_constant__ CUtensorMap tmap_l, const __grid_constant__ CUtensorMap tmap_x,
                   const __grid_constant__ GemmParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* tbuf = smem + FSTAGES * TSTAGE_BYTES;
  FBarriers* bars = reinterpret_cast<FBarriers*>(tbuf + FT_BYTES);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_items = p.n_jobs * p.n_mtiles;
  const int nkb1 = p.K / HBK;                       // phase 1 k-blocks (0 for block column 0: T is A itself)
  constexpr int NKB2 = 256 / HBK;
  const int n_my = blockIdx.x < n_items ? (n_items - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

  if (warp == 0 && lane == 0) {
    prefetch_tensormap(&tmap_l);
    prefetch_tensormap(&tmap_x);
    for (int s = 0; s < FSTAGES; ++s) {
      mbar_init(&bars->full[s], 1);
      mbar_init(&bars->empty[s], 1);
    }
    for (int s = 0; s < TACC; ++s) {
      mbar_init(&bars->p1_full[s], 1);
      mbar_init(&bars->p2_full[s], 1);
      mbar_init(&bars->acc_empty[s], EW);
    }
    mbar_init(&bars->t_full, EW);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<TACC * MAX_N>(&bars->tmem_base);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = bars->tmem_base;

  // ring order, shared by the producer and the MMA issuer: P1(0), then P1(k + 1), P2(k) for k = 0, 1, ...
  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      auto next = [&]() {
        if (++stage == FSTAGES) {
          stage = 0;
          phase ^= 1;
        }
      };
      auto load_p1 = [&](int k) {
        const int item = blockIdx.x + k * gridDim.x;
        const int job = item / p.n_mtiles, mt = item - job * p.n_mtiles;
        const int row_a = job * p.ntp + p.row0 + mt * TBM, row_b = job * p.ntp + p.c_col0;
        for (int kb = 0; kb < nkb1; ++kb) {
          mbar_wait(&bars->empty[stage], phase ^ 1);
          uint8_t* sa = smem + stage * TSTAGE_BYTES;
          mbar_arrive_expect_tx(&bars->full[stage], TA_BYTES + 4 * BOX_BYTES);
          tma_load_2d(sa, &tmap_l, &bars->full[stage], kb * HBK, row_a);
          tma_load_2d(sa + BOX_BYTES, &tmap_l, &bars->full[stage], kb * HBK, row_a + BOX_ROWS);
          for (int b = 0; b < 4; ++b)
            tma_load_2d(sa + TA_BYTES + b * BOX_BYTES, &tmap_l, &bars->full[stage], kb * HBK, row_b + b * BOX_ROWS);
          next();
        }
      };
      auto load_p2 = [&](int k) {
        const int job = (blockIdx.x + k * gridDim.x) / p.n_mtiles;
        for (int kb = 0; kb < NKB2; ++kb) {
          mbar_wait(&bars->empty[stage], phase ^ 1);
          uint8_t* sb = smem + stage * TSTAGE_BYTES + TA_BYTES;
          mbar_arrive_expect_tx(&bars->full[stage], 4 * BOX_BYTES);
          for (int b = 0; b < 4; ++b)
            tma_load_2d(sb + b * BOX_BYTES, &tmap_x, &bars->full[stage], kb * HBK, job * 256 + b * BOX_ROWS);
          next();
        }
      };
      if (n_my > 0) load_p1(0);
      for (int k = 0; k < n_my; ++k) {
        if (k + 1 < n_my) load_p1(k + 1);
        load_p2(k);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = umma_idesc_f16(TBM, 256);
      int stage = 0;
      uint32_t phase = 0;
      auto kblock = [&](uint32_t tmem_d, uint32_t sa, int kb) {
        mbar_wait(&bars->full[stage], phase);
        tc_fence_after();
        const uint64_t adesc = umma_desc_k_sw128(sa);
        const uint64_t bdesc = umma_desc_k_sw128(smem_u32(smem + stage * TSTAGE_BYTES + TA_BYTES));
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_f16(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0);
        umma_commit(&bars->empty[stage]);
        if (++stage == FSTAGES) {
          stage = 0;
          phase ^= 1;
        }
      };
      auto claim = [&](int k) {                     // first use of tile k's accumulator
        mbar_wait(&bars->acc_empty[k & 1], ((k >> 1) & 1) ^ 1);
        tc_fence_after();
      };
      auto p1 = [&](int k) {
        claim(k);
        const uint32_t tmem_d = tmem_base + (k & 1) * MAX_N;
        for (int kb = 0; kb < nkb1; ++kb) kblock(tmem_d, smem_u32(smem + stage * TSTAGE_BYTES), kb);
        umma_commit(&bars->p1_full[k & 1]);
      };
      if (n_my > 0 && nkb1 > 0) p1(0);
      for (int k = 0; k < n_my; ++k) {
        if (k + 1 < n_my && nkb1 > 0) p1(k + 1);
        if (nkb1 == 0) claim(k);
        mbar_wait(&bars->t_full, k & 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + (k & 1) * MAX_N;
        for (int kb = 0; kb < NKB2; ++kb) kblock(tmem_d, smem_u32(tbuf + kb * FT_KB_BYTES), kb);
        umma_commit(&bars->p2_full[k & 1]);
      }
    }
  } else {
    // Epilogue: thread = one row of the tile (TMEM lane quarter q = warp & 3), the EW / 4 warps of a quarter take its
    // 32-column chunks round-robin as in tf32_gemm_kernel, in units of 16 columns.  The cross-products of PF units are
    // in flight ahead of their use -- the first ones of the NEXT tile while phase 2 of this one runs -- as many as the
    // register budget allows without spilling (96 registers per thread at EW = 16, 168 at EW = 8).
    constexpr int CG = EW / 4;
    constexpr int NU = 2 * (8 / CG);                              // 16-column units per thread and tile
    constexpr int CVU = SRC == 1 ? 2 : 4;                         // 16-byte loads per unit
    constexpr int PF = SRC == 1 ? NU : 2;                         // int16: the whole tile; int32: two units
    const int q = warp & 3, g = (warp - 2) >> 2;
    const int tr = q * 32 + lane;                                 // tile row of this thread
    const uint32_t tsm = smem_u32(tbuf) + tr * 128;
    const bool storer = warp == 2 && lane == 0;
    const bool has_acc = nkb1 > 0;
    uint4 cv[NU][CVU];
    size_t rowoff = 0;                                            // cross-product row of the tile whose units load next
    int l_h0 = 0, l_gap = 0, l_nt = 0;
    // (rows past the job's end are padding rows, r >= n_t: they read panel row 0, so every load is in bounds and
    // needs no branch)
    auto tile_src = [&](int item) {
      const int job = item / p.n_mtiles, mt = item - job * p.n_mtiles;
      const int r = p.row0 + mt * TBM + tr;
      const TbFuseCoef cf = p.fc.coef[job];
      const int rr = r < cf.n_t ? r + (r >= cf.hole0 ? cf.gap : 0) : 0;
      rowoff = ((size_t)cf.cw * p.fc.rpad + rr) * p.fc.rpad;
      l_h0 = cf.hole0;
      l_gap = cf.gap;
      l_nt = cf.n_t;
    };
    auto load_unit = [&](uint4 (&dst)[CVU], int u) {
      const int b = p.c_col0 + (g + CG * (u >> 1)) * 32 + 16 * (u & 1);
#pragma unroll
      for (int j = 0; j < CVU; ++j) {
        const int bj = b + (SRC == 1 ? 8 : 4) * j;              // (8-column groups never straddle the hole)
        const int ub = bj + ((bj >= l_h0 && bj < l_nt) ? l_gap : 0);
        dst[j] = SRC == 1 ? *reinterpret_cast<const uint4*>(static_cast<const int16_t*>(p.fc.C) + rowoff + ub)
                          : *reinterpret_cast<const uint4*>(static_cast<const int32_t*>(p.fc.C) + rowoff + ub);
      }
    };
    // 16 halves of this thread's row (tile columns col .. col + 15) into the T tile, swizzled as a TMA load would place them
    auto put_t = [&](int col, const uint32_t (&h)[8]) {
      const uint32_t base = tsm + (col >> 6) * FT_KB_BYTES;
      const int c16 = (col & 63) >> 3;
#pragma unroll
      for (int s = 0; s < 2; ++s)
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(base + (((c16 + s) ^ (tr & 7)) << 4)),
                     "r"(h[4 * s]), "r"(h[4 * s + 1]), "r"(h[4 * s + 2]), "r"(h[4 * s + 3])
                     : "memory");
    };
    auto epi_sync = [&]() { asm volatile("bar.sync 1, %0;" ::"n"(EW * 32) : "memory"); };

    if (n_my > 0) {
      tile_src(blockIdx.x);
#pragma unroll
      for (int u = 0; u < PF; ++u) load_unit(cv[u], u);
    }
    for (int k = 0; k < n_my; ++k) {
      const int item = blockIdx.x + k * gridDim.x;
      const int job = item / p.n_mtiles, mt = item - job * p.n_mtiles;
      const int a = k & 1;
      const uint32_t par = (k >> 1) & 1;
      const int r = p.row0 + mt * TBM + tr;
      const int rw0 = p.row0 + mt * TBM + q * 32;
      const TbFuseCoef cf = p.fc.coef[job];
      const float f_scale = cf.scale;
      const float f_rt = p.fc.terms[(size_t)job * 2 * p.ntp + (r < p.row_end ? r : 0)];
      const float* f_ct = p.fc.terms + (size_t)job * 2 * p.ntp + p.ntp + p.c_col0;
      const bool pad_warp = rw0 + 32 > cf.n_t;                   // (warp-uniform) some rows of this warp are padding
      const bool real_row = r < cf.n_t;
      const uint32_t tacc = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + a * MAX_N;
      if (has_acc) {
        mbar_wait(&bars->p1_full[a], par);
        tc_fence_after();
      }
      if (storer) bulk_wait_group_read0();                        // the previous tile's store has read the buffer
      epi_sync();
      // phase 1 epilogue: T = A - acc (every entry lies below the diagonal: no lambda; padding rows are zero)
#pragma unroll
      for (int u = 0; u < NU; ++u) {
        if (u + PF < NU) load_unit(cv[u + PF], u + PF);
        const int col = (g + CG * (u >> 1)) * 32 + 16 * (u & 1);   // tile column
        uint32_t v[16];
        if (has_acc) {
          tmem_ld_32x16(tacc + col, v);
          tmem_ld_wait();
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = 0u;
        }
        float o[16];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 ct = *reinterpret_cast<const float4*>(f_ct + col + 4 * j);
          const float ctv[4] = {ct.x, ct.y, ct.z, ct.w};
          float cx[4];
          if (SRC == 1) {
            const uint4 raw = cv[u][j >> 1];
            const uint32_t w0 = (j & 1) ? raw.z : raw.x, w1 = (j & 1) ? raw.w : raw.y;
            cx[0] = c_from_i16(w0, false);
            cx[1] = c_from_i16(w0, true);
            cx[2] = c_from_i16(w1, false);
            cx[3] = c_from_i16(w1, true);
          } else {
            const uint4 raw = cv[u][SRC == 1 ? 0 : j];
            cx[0] = c_from_i32(raw.x);
            cx[1] = c_from_i32(raw.y);
            cx[2] = c_from_i32(raw.z);
            cx[3] = c_from_i32(raw.w);
          }
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float av = (!pad_warp || real_row) ? fmaf(cx[e], f_scale, f_rt + ctv[e]) : 0.f;
            o[4 * j + e] = av - __uint_as_float(v[4 * j + e]);
          }
        }
        uint32_t h[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const __half2 hh = __floats2half2_rn(o[2 * j], o[2 * j + 1]);
          h[j] = *reinterpret_cast<const uint32_t*>(&hh);
        }
        put_t(col, h);
      }
      tc_fence_before();
      fence_proxy_async_smem();                                   // T is read by the MMA (async proxy)
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars->t_full);
      // the next tile's first cross-products travel while phase 2 runs
      if (k + 1 < n_my) {
        tile_src(item + gridDim.x);
#pragma unroll
        for (int u = 0; u < PF; ++u) load_unit(cv[u], u);
      }
      mbar_wait(&bars->p2_full[a], par);
      tc_fence_after();
      // phase 2 epilogue: the final factor entries, rounded as the panel GEMM rounds them (TF32, then half)
#pragma unroll
      for (int u = 0; u < NU; ++u) {
        const int col = (g + CG * (u >> 1)) * 32 + 16 * (u & 1);
        uint32_t v[16];
        tmem_ld_32x16(tacc + col, v);
        tmem_ld_wait();
        uint32_t h[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const __half2 hh = __floats2half2_rn(round_tf32(__uint_as_float(v[2 * j])), round_tf32(__uint_as_float(v[2 * j + 1])));
          h[j] = *reinterpret_cast<const uint32_t*>(&hh);
        }
        put_t(col, h);
      }
      tc_fence_before();
      fence_proxy_async_smem();                                   // the tile is read by the TMA store (async proxy)
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars->acc_empty[a]);
      epi_sync();
      if (storer) {
        // ntp is a multiple of 64: a 64-row box lies wholly inside or wholly outside the job's rows
        const int row_t = p.row0 + mt * TBM;
#pragma unroll
        for (int hb = 0; hb < 2; ++hb) {
          if (row_t + hb * BOX_ROWS >= p.row_end) continue;
#pragma unroll
          for (int kb = 0; kb < 4; ++kb)
            tma_store_2d(&tmap_l, tbuf + kb * FT_KB_BYTES + hb * BOX_BYTES, p.c_col0 + kb * HBK,
                         job * p.ntp + row_t + hb * BOX_ROWS);
        }
        bulk_commit_group();
      }
    }
    if (storer) bulk_wait_group0();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<TACC * MAX_N>(tmem_base);
  }
}

// Diagonal block of the fp32 matrix (64 x 64): Cholesky factor + its inverse, in fp32 -- the factor is rounded to TF32
// (10 mantissa bits) on the way out, so fp32 math is ample.  The rounded factor is the one that gets inverted and
// stored, so the tensor-core operand truncation is a no-op and the triangular solves in solve_mixed.cu use exactly
// the operator the factorisation built.
// Recursive 2 x 2 blocking with WARP-LEVEL 32 x 32 kernels: a warp holds a 32 x 32 block one row (or column) per lane
// in registers and exchanges pivot columns by shuffle, so the 64 dependent steps of the factorisation need no
// block-wide barrier and ~5x fewer issued instructions than the previous thread-per-quarter-row scheme (the launch
// was issue-bound: 97 us for 1 000 blocks).
//   L11 = chol(A11)                      warp 0
//   L21 = A21 L11^-T,  X11 = L11^-1      warps 1, 2
//   A22 -= L21 L21^T                     all
//   L22 = chol(A22)                      warp 0
//   X22 = L22^-1,  P = L21 X11           warp 3, others
//   X21 = -X22 P                         all
constexpr int DLD = NB + 1;

// a[c] = A[lane][c] (c <= lane valid) -> L[lane][c]; returns false on a non-positive pivot
__device__ __forceinline__ bool warp_potrf32(float (&a)[32]) {
  bool ok = true;
#pragma unroll
  for (int c = 0; c < 32; ++c) {
    const float d = __shfl_sync(0xffffffffu, a[c], c);
    ok = ok && d > 0.f;
    const float l = a[c] * rsqrtf(d);                     // L[lane][c] for lane >= c
    a[c] = l;
#pragma unroll
    for (int cc = c + 1; cc < 32; ++cc) a[cc] = fmaf(-l, __shfl_sync(0xffffffffu, l, cc), a[cc]);
  }
  return ok;
}
// row `lane` of B solved against the lower factor L (shared memory, leading dimension DLD): x L^T = b, in place
__device__ __forceinline__ void warp_trsm32(float (&b)[32], const float* L) {
#pragma unroll
  for (int c = 0; c < 32; ++c) {
    float s = b[c];
#pragma unroll
    for (int p = 0; p < c; ++p) s = fmaf(-b[p], L[c * DLD + p], s);
    b[c] = s / L[c * DLD + c];
  }
}
// column `lane` of X = L^-1: x[r] (zero for r < lane)
__device__ __forceinline__ void warp_trinv32(float (&x)[32], const float* L, int lane) {
#pragma unroll
  for (int r = 0; r < 32; ++r) {
    float s = r == lane ? 1.f : 0.f;
#pragma unroll
    for (int p = 0; p < r; ++p) s = fmaf(-L[r * DLD + p], x[p], s);
    x[r] = r >= lane ? s / L[r * DLD + r] : 0.f;
  }
}

// 128 threads and 29 KiB of shared memory per block: SEVEN blocks per SM, so 1 000 matrices are one wave (the version
// with 256 threads / 37 KiB ran four per SM = two waves, with one warp of eight busy in the serial phases).
constexpr int DT = 128;                                   // threads that work on one 64 x 64 diagonal block
constexpr int XLD = 33;
constexpr int DIAG_SCRATCH = NB * DLD + 3 * 32 * XLD;     // floats: Ls, X11, X22, X21

// barrier of the DT threads that run diag64_body: the whole block (stand-alone kernel) or named barrier 1 (fused chain,
// where the other warps of the block wait at barrier 0)
template <bool NAMED>
__device__ __forceinline__ void diag_sync() {
  if (NAMED) asm volatile("bar.sync 1, 128;" ::: "memory");
  else __syncthreads();
}

// Ls [64][DLD]: in = the block (lower triangle meaningful), out = its factor rounded to TF32 (upper-left / lower-right
// triangles zeroed; the UPPER-RIGHT quadrant is scratch and holds garbage).  X11 / X22 / X21 [32][XLD]: quadrants of
// the inverse of the factor (not yet rounded).  Called by DT threads (tid 0 .. DT-1) after a barrier that made Ls
// visible; ends with a diag_sync.  Returns false (to every thread of warp 0 only) on a non-positive pivot.
template <bool NAMED>
__device__ __forceinline__ bool diag64_body(float* Ls, float* X11, float* X22, float* X21, int tid) {
  float* Ps = Ls + 32;                                    // P = L21 X11 lives in the (unused) upper-right quadrant, stride DLD
  const int warp = tid >> 5, lane = tid & 31;
  bool ok = true;
  float a[32];
  if (warp == 0) {                                        // L11
#pragma unroll
    for (int c = 0; c < 32; ++c) a[c] = Ls[lane * DLD + c];
    ok = warp_potrf32(a);
#pragma unroll
    for (int c = 0; c < 32; ++c) Ls[lane * DLD + c] = c <= lane ? round_tf32(a[c]) : 0.f;
  }
  diag_sync<NAMED>();
  if (warp == 1) {                                        // L21 = A21 L11^-T
#pragma unroll
    for (int c = 0; c < 32; ++c) a[c] = Ls[(32 + lane) * DLD + c];
    warp_trsm32(a, Ls);
#pragma unroll
    for (int c = 0; c < 32; ++c) Ls[(32 + lane) * DLD + c] = round_tf32(a[c]);
  } else if (warp == 2) {                                 // X11 = L11^-1
    warp_trinv32(a, Ls, lane);
#pragma unroll
    for (int r = 0; r < 32; ++r) X11[r * XLD + lane] = a[r];
  }
  diag_sync<NAMED>();
  {                                                       // A22 -= L21 L21^T (lower part), 8 entries per thread
    const int r = tid >> 2, c0 = (tid & 3) * 8;
    if (c0 <= r) {
      float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      for (int p = 0; p < 32; ++p) {
        const float lr = Ls[(32 + r) * DLD + p];
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] = fmaf(lr, Ls[(32 + c0 + j) * DLD + p], acc[j]);
      }
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (c0 + j <= r) Ls[(32 + r) * DLD + 32 + c0 + j] -= acc[j];
    }
  }
  diag_sync<NAMED>();
  if (warp == 0) {                                        // L22
#pragma unroll
    for (int c = 0; c < 32; ++c) a[c] = Ls[(32 + lane) * DLD + 32 + c];
    ok = warp_potrf32(a) && ok;
#pragma unroll
    for (int c = 0; c < 32; ++c) Ls[(32 + lane) * DLD + 32 + c] = c <= lane ? round_tf32(a[c]) : 0.f;
  } else {                                                // P = L21 X11, meanwhile (96 threads, 32 x 32 outputs)
    for (int e = tid - 32; e < 32 * 32; e += DT - 32) {
      const int r = e >> 5, c = e & 31;
      float s = 0.f;
      for (int p = c; p < 32; ++p) s = fmaf(Ls[(32 + r) * DLD + p], X11[p * XLD + c], s);   // X11 is lower triangular
      Ps[r * DLD + c] = s;
    }
  }
  diag_sync<NAMED>();
  if (warp == 3) {                                        // X22 = L22^-1
    warp_trinv32(a, Ls + 32 * DLD + 32, lane);
#pragma unroll
    for (int r = 0; r < 32; ++r) X22[r * XLD + lane] = a[r];
  }
  diag_sync<NAMED>();
  {                                                       // X21 = -X22 P
    const int r = tid >> 2, c0 = (tid & 3) * 8;
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int p = 0; p <= r; ++p) {                        // X22 is lower triangular
      const float xr = X22[r * XLD + p];
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] = fmaf(xr, Ps[p * DLD + c0 + j], acc[j]);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) X21[r * XLD + c0 + j] = -acc[j];
  }
  diag_sync<NAMED>();
  return ok;
}
// entries of the results of diag64_body: the factor (zero above the diagonal) and its inverse
__device__ __forceinline__ float diag_l(const float* Ls, int rr, int c) {
  return (rr < 32 && c >= 32) ? 0.f : Ls[rr * DLD + c];
}
__device__ __forceinline__ float diag_x(const float* X11, const float* X22, const float* X21, int rr, int c) {
  return rr < 32 ? (c < 32 ? X11[rr * XLD + c] : 0.f) : (c < 32 ? X21[(rr - 32) * XLD + c] : X22[(rr - 32) * XLD + c - 32]);
}

__global__ void __launch_bounds__(DT) chol_diag32_kernel(float* __restrict__ L32, float* __restrict__ Linv32,
                                                         __half* __restrict__ L16, int* __restrict__ status, int ntp,
                                                         int jb) {
  __shared__ float sc[DIAG_SCRATCH];
  float* Ls = sc;
  float* X11 = Ls + NB * DLD;
  float* X22 = X11 + 32 * XLD;
  float* X21 = X22 + 32 * XLD;
  const int job = blockIdx.x;
  float* D = L32 + ((size_t)job * ntp + (size_t)jb * NB) * ntp + jb * NB;
  const int tid = threadIdx.x;
  for (int e = tid; e < NB * 16; e += DT) {               // coalesced rows, 16 bytes per thread
    const int r = e >> 4, c4 = (e & 15) * 4;
    const float4 v = *reinterpret_cast<const float4*>(D + (size_t)r * ntp + c4);
    Ls[r * DLD + c4] = v.x;
    Ls[r * DLD + c4 + 1] = v.y;
    Ls[r * DLD + c4 + 2] = v.z;
    Ls[r * DLD + c4 + 3] = v.w;
  }
  __syncthreads();
  const bool ok = diag64_body<false>(Ls, X11, X22, X21, tid);
  if (!ok && tid < 32) status[job] = 1;                   // (warp 0 holds the verdict)
  float* Li = Linv32 + ((size_t)job * ntp + (size_t)jb * NB) * NB;
  for (int e = tid; e < NB * NB; e += DT) {
    const int rr = e >> 6, c = e & 63;
    const float l = diag_l(Ls, rr, c);
    D[(size_t)rr * ntp + c] = l;
    if (L16) L16[((size_t)job * ntp + (size_t)jb * NB + rr) * ntp + jb * NB + c] = __float2half_rn(l);
    Li[e] = round_tf32(diag_x(X11, X22, X21, rr, c));
  }
}

// Inverse of the 256 x 256 lower-triangular diagonal block of the factor, from its 64 x 64 blocks and the inverses of
// its four diagonal blocks (chol_diag32_kernel):   X_bb = Linv_b,   X_ib = -Linv_i * sum_{k=b}^{i-1} L_ik X_kb  (i > b).
// With X = L_JJ^-1 the whole panel below the diagonal block is ONE tensor-core GEMM, L[:, J] = T[:, J] X^T (K = 256),
// instead of four narrow triangular-solve / update rounds over all rows.  One CTA per job; the 64^3 block products
// run on mma.sync m16n8k8 TF32 (every operand is already rounded to TF32; X is rounded on the way out).
constexpr int XS_LD = 72, AS_LD = 68;     // smem strides: conflict-free B[k][n] and A[m][k] fragment loads
constexpr int TRINV_SMEM = (4 * 64 * XS_LD + 64 * AS_LD + 64 * XS_LD) * 4;

__device__ __forceinline__ void mma_tf32_16x8x8(float (&c)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile(
      "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
      "{%0, %1, %2, %3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

// acc[nt] (16 x 8 fragments, nt = 0..3) += As[64][AS_LD] (rows 16 (warp & 3) ..) * Bs[64][BLD] (cols 32 (warp >> 2) ..)
template <int BLD = XS_LD>
__device__ __forceinline__ void block_mma(float (&acc)[4][4], const float* As, const float* Bs, int warp, int lane) {
  constexpr int XS_LD = BLD;
  const int g = lane >> 2, t = lane & 3;
  const float* a_base = As + (16 * (warp & 3) + g) * AS_LD + t;
  const float* b_base = Bs + t * XS_LD + 32 * (warp >> 2) + g;
#pragma unroll
  for (int k = 0; k < 64; k += 8) {
    uint32_t a[4];
    a[0] = __float_as_uint(a_base[k]);
    a[1] = __float_as_uint(a_base[8 * AS_LD + k]);
    a[2] = __float_as_uint(a_base[k + 4]);
    a[3] = __float_as_uint(a_base[8 * AS_LD + k + 4]);
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      uint32_t b[2];
      b[0] = __float_as_uint(b_base[k * XS_LD + 8 * nt]);
      b[1] = __float_as_uint(b_base[(k + 4) * XS_LD + 8 * nt]);
      mma_tf32_16x8x8(acc[nt], a, b);
    }
  }
}

// X16 (nullable): the inverse goes out as halves [job][256][256] instead of the fp32 Linv256 (its entries are rounded to
// 10 mantissa bits either way); the wide panel GEMM then runs on fp16 operands.
__global__ void __launch_bounds__(256) trinv256_kernel(const float* __restrict__ L32, const float* __restrict__ Linv32,
                                                       float* __restrict__ Linv256, __half* __restrict__ X16, int ntp,
                                                       int c0) {
  extern __shared__ float tsm[];
  float* Xs = tsm;                       // [4][64][XS_LD]  X_kb of the current block column b
  float* As = Xs + 4 * 64 * XS_LD;       // [64][AS_LD]     left operand
  float* Ss = As + 64 * AS_LD;           // [64][XS_LD]     sum_k L_ik X_kb
  const int job = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const float* Lj = L32 + ((size_t)job * ntp + c0) * ntp + c0;
  const float* Dj = Linv32 + ((size_t)job * ntp + c0) * NB;
  float* Out = Linv256 + (size_t)job * 256 * 256;
  __half* Out16 = X16 ? X16 + (size_t)job * 256 * 256 : nullptr;
  const int g = lane >> 2, t = lane & 3;
  const int frow = 16 * (warp & 3) + g, fcol = 32 * (warp >> 2) + 2 * t;    // this thread's fragment origin
  auto put4 = [&](size_t off, const float4 v) {                            // entries off .. off + 3 of this job's inverse
    if (Out16) {
      const __half2 a = __floats2half2_rn(v.x, v.y), b = __floats2half2_rn(v.z, v.w);
      *reinterpret_cast<uint2*>(Out16 + off) =
          make_uint2(*reinterpret_cast<const uint32_t*>(&a), *reinterpret_cast<const uint32_t*>(&b));
    } else {
      *reinterpret_cast<float4*>(Out + off) = v;
    }
  };
  auto put2 = [&](size_t off, const float2 v) {
    if (Out16) *reinterpret_cast<__half2*>(Out16 + off) = __floats2half2_rn(v.x, v.y);
    else *reinterpret_cast<float2*>(Out + off) = v;
  };

  // 64 x 64 block, row stride ld_src, into smem with row stride ld_dst (16-byte loads, coalesced rows)
  auto load_block = [&](const float* src, size_t ld_src, float* dst, int ld_dst) {
    for (int e = tid; e < 64 * 16; e += 256) {
      const int r = e >> 4, c4 = (e & 15) * 4;
      const float4 v = *reinterpret_cast<const float4*>(src + (size_t)r * ld_src + c4);
      *reinterpret_cast<float4*>(dst + r * ld_dst + c4) = v;
    }
  };
  // per block column b: zero blocks above the diagonal, X_bb = Linv_b
  auto column_setup = [&](int b) {
    for (int i = 0; i < b; ++i)
      for (int e = tid; e < 64 * 16; e += 256)
        put4((size_t)(64 * i + (e >> 4)) * 256 + 64 * b + (e & 15) * 4, make_float4(0.f, 0.f, 0.f, 0.f));
    load_block(Dj + (size_t)b * 64 * NB, NB, Xs + b * 64 * XS_LD, XS_LD);
    __syncthreads();
    for (int e = tid; e < 64 * 16; e += 256) {
      const int r = e >> 4, c4 = (e & 15) * 4;
      put4((size_t)(64 * b + r) * 256 + 64 * b + c4, *reinterpret_cast<const float4*>(Xs + b * 64 * XS_LD + r * XS_LD + c4));
    }
  };
  // The left operands form a fixed sequence (b, i, k): L_ik for k = b .. i-1, then Linv_i (written k = i), for
  // i = b+1 .. 3, b = 0 .. 2.  Each one is fetched into registers while the previous product runs, so the global-load
  // latency (the launch was bound by it: 16 dependent load -> barrier -> mma rounds) hides behind the tensor work.
  auto operand = [&](int b, int i, int k, const float*& src, size_t& ld) {
    if (k < i) {
      src = Lj + (size_t)(64 * i) * ntp + 64 * k;
      ld = (size_t)ntp;
    } else {
      src = Dj + (size_t)i * 64 * NB;
      ld = NB;
    }
  };
  float4 pre[4];
  auto fetch = [&](int b, int i, int k) {
    const float* src;
    size_t ld;
    operand(b, i, k, src, ld);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int e = tid + 256 * u;
      pre[u] = *reinterpret_cast<const float4*>(src + (size_t)(e >> 4) * ld + (e & 15) * 4);
    }
  };
  auto deposit = [&]() {
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int e = tid + 256 * u;
      *reinterpret_cast<float4*>(As + (e >> 4) * AS_LD + (e & 15) * 4) = pre[u];
    }
  };
  int b = 0, i = 1, k = 0;
  fetch(b, i, k);
  float acc[4][4];
  for (;;) {
    if (i == b + 1 && k == b) column_setup(b);           // first operand of block column b
    deposit();
    __syncthreads();
    int nb = b, ni = i, nk = k + 1;                       // successor in the sequence
    if (nk > i) {
      ni = i + 1;
      nk = b;
      if (ni > 3) {
        nb = b + 1;
        ni = nb + 1;
        nk = nb;
      }
    }
    const bool more = nb < 3;
    if (more) fetch(nb, ni, nk);
    if (k == b) {
#pragma unroll
      for (int nt = 0; nt < 4; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) acc[nt][e] = 0.f;
    }
    if (k < i) {
      block_mma(acc, As, Xs + k * 64 * XS_LD, warp, lane);
      if (k == i - 1) {                                   // S = sum_k L_ik X_kb complete: becomes the right operand
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
          *reinterpret_cast<float2*>(Ss + frow * XS_LD + fcol + 8 * nt) = make_float2(round_tf32(acc[nt][0]), round_tf32(acc[nt][1]));
          *reinterpret_cast<float2*>(Ss + (frow + 8) * XS_LD + fcol + 8 * nt) = make_float2(round_tf32(acc[nt][2]), round_tf32(acc[nt][3]));
        }
      }
    } else {                                              // X_ib = -Linv_i S
      float acc2[4][4];
#pragma unroll
      for (int nt = 0; nt < 4; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) acc2[nt][e] = 0.f;
      block_mma(acc2, As, Ss, warp, lane);
      float* Xi = Xs + i * 64 * XS_LD;
      const size_t oi = (size_t)(64 * i) * 256 + 64 * b;
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        const float2 lo = make_float2(round_tf32(-acc2[nt][0]), round_tf32(-acc2[nt][1]));
        const float2 hi = make_float2(round_tf32(-acc2[nt][2]), round_tf32(-acc2[nt][3]));
        *reinterpret_cast<float2*>(Xi + frow * XS_LD + fcol + 8 * nt) = lo;
        *reinterpret_cast<float2*>(Xi + (frow + 8) * XS_LD + fcol + 8 * nt) = hi;
        put2(oi + (size_t)frow * 256 + fcol + 8 * nt, lo);
        put2(oi + (size_t)(frow + 8) * 256 + fcol + 8 * nt, hi);
      }
    }
    __syncthreads();
    if (!more) break;
    b = nb;
    i = ni;
    k = nk;
  }
  column_setup(3);
}

// acc (16 x 8 fragments, nt = 0..3) += As[64][AS_LD] * Bt[64][AS_LD]^T: both operands row-major [row][k]
__device__ __forceinline__ void block_mma_nt(float (&acc)[4][4], const float* As, const float* Bt, int warp, int lane) {
  const int g = lane >> 2, t = lane & 3;
  const float* a_base = As + (16 * (warp & 3) + g) * AS_LD + t;
  const float* b_base = Bt + (32 * (warp >> 2) + g) * AS_LD + t;
#pragma unroll
  for (int k = 0; k < 64; k += 8) {
    uint32_t a[4];
    a[0] = __float_as_uint(a_base[k]);
    a[1] = __float_as_uint(a_base[8 * AS_LD + k]);
    a[2] = __float_as_uint(a_base[k + 4]);
    a[3] = __float_as_uint(a_base[8 * AS_LD + k + 4]);
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      uint32_t b[2];
      b[0] = __float_as_uint(b_base[8 * nt * AS_LD + k]);
      b[1] = __float_as_uint(b_base[8 * nt * AS_LD + k + 4]);
      mma_tf32_16x8x8(acc[nt], a, b);
    }
  }
}

// The narrow work of one inner step b inside the (up to) 256-row diagonal block, one CTA per job, after
// chol_diag32_kernel(b):   L_ib = T_ib Linv_b^T for the blocks below (i > b), written as the fp32 / fp16 factor, and the
// left-looking update of the NEXT block column, T_ij -= sum_{k <= b} L_ik L_jk^T (j = b + 1, i >= j).
// Sixteen 64^3 products per diagonal block on mma.sync instead of six persistent tcgen05 launches whose fixed cost
// (TMEM allocation, pipeline fill) dwarfed the 2 000 small tiles they covered.
__global__ void __launch_bounds__(256) chol_narrow_kernel(float* __restrict__ L32, __half* __restrict__ L16,
                                                          const float* __restrict__ Linv32, int ntp, int c0, int b,
                                                          int nbk) {
  __shared__ float As[64 * AS_LD];
  __shared__ float Bs[64 * AS_LD];
  const int job = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  float* base = L32 + ((size_t)job * ntp + c0) * ntp + c0;
  __half* base16 = L16 ? L16 + ((size_t)job * ntp + c0) * ntp + c0 : nullptr;
  const int g = lane >> 2, t = lane & 3;
  const int frow = 16 * (warp & 3) + g, fcol = 32 * (warp >> 2) + 2 * t;
  auto load_block = [&](const float* src, size_t ld_src, float* dst) {
    for (int e = tid; e < 64 * 16; e += 256) {
      const int r = e >> 4, c4 = (e & 15) * 4;
      *reinterpret_cast<float4*>(dst + r * AS_LD + c4) = *reinterpret_cast<const float4*>(src + (size_t)r * ld_src + c4);
    }
  };
  float acc[4][4];
  auto clear = [&]() {
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[nt][e] = 0.f;
  };
  // (i) triangular solves of block column b
  load_block(Linv32 + ((size_t)job * ntp + c0 + 64 * b) * NB, NB, Bs);
  for (int i = b + 1; i < nbk; ++i) {
    float* blk = base + (size_t)(64 * i) * ntp + 64 * b;
    load_block(blk, ntp, As);
    __syncthreads();
    clear();
    block_mma_nt(acc, As, Bs, warp, lane);
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      const float2 lo = make_float2(round_tf32(acc[nt][0]), round_tf32(acc[nt][1]));
      const float2 hi = make_float2(round_tf32(acc[nt][2]), round_tf32(acc[nt][3]));
      *reinterpret_cast<float2*>(blk + (size_t)frow * ntp + fcol + 8 * nt) = lo;
      *reinterpret_cast<float2*>(blk + (size_t)(frow + 8) * ntp + fcol + 8 * nt) = hi;
      if (base16) {
        __half* h = base16 + (size_t)(64 * i) * ntp + 64 * b;
        *reinterpret_cast<__half2*>(h + (size_t)frow * ntp + fcol + 8 * nt) = __floats2half2_rn(lo.x, lo.y);
        *reinterpret_cast<__half2*>(h + (size_t)(frow + 8) * ntp + fcol + 8 * nt) = __floats2half2_rn(hi.x, hi.y);
      }
    }
    __syncthreads();                 // the block just written is read again below; As is reused
  }
  // (ii) update of block column j = b + 1 with every finished column of the diagonal block
  const int j = b + 1;
  if (j >= nbk) return;
  for (int i = j; i < nbk; ++i) {
    clear();
    for (int k = 0; k <= b; ++k) {
      load_block(base + (size_t)(64 * i) * ntp + 64 * k, ntp, As);
      load_block(base + (size_t)(64 * j) * ntp + 64 * k, ntp, Bs);
      __syncthreads();
      block_mma_nt(acc, As, Bs, warp, lane);
      __syncthreads();
    }
    float* blk = base + (size_t)(64 * i) * ntp + 64 * j;
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      float2* p0 = reinterpret_cast<float2*>(blk + (size_t)frow * ntp + fcol + 8 * nt);
      float2* p1 = reinterpret_cast<float2*>(blk + (size_t)(frow + 8) * ntp + fcol + 8 * nt);
      float2 v0 = *p0, v1 = *p1;
      v0.x -= acc[nt][0];
      v0.y -= acc[nt][1];
      v1.x -= acc[nt][2];
      v1.y -= acc[nt][3];
      *p0 = v0;
      *p1 = v1;
    }
  }
}

// The whole diagonal-block chain of one block column in ONE kernel, for small batches (n_jobs <= ~ SM count: strong
// scaling at 125 genomes per GPU, config 4's waves).  There the eight launches per block column (diag32 x 4,
// narrow x 3 ...) are pure dependent latency: every stage re-loads its operands from global memory behind a kernel
// boundary.  Here one CTA per job keeps the lower triangle of the (up to) 256 x 256 block in shared memory (ten
// 64 x 64 blocks, 174 KB) and walks the same stages -- the device code of chol_diag32_kernel and chol_narrow_kernel on
// shared-memory operands, same order of operations, bit-identical results.  The slot of a diagonal block receives the
// inverse of its factor once it is known (the right operand of the solves below it).  trinv256_kernel follows as before.
constexpr int CH_BLK = 64 * AS_LD;                        // floats per block slot
constexpr int CHAIN_SMEM = 13 * CH_BLK * 4;               // ten blocks + three for the inverse (they overlap the diagonal scratch)
static_assert(DIAG_SCRATCH <= 3 * CH_BLK, "diagonal scratch must fit into the inverse's buffers");
__device__ __forceinline__ int ch_slot(int i, int j) { return (i * (i + 1) / 2 + j) * CH_BLK; }   // i >= j

__global__ void __launch_bounds__(256, 1) chol_chain256_kernel(float* __restrict__ L32, float* __restrict__ Linv32,
                                                               __half* __restrict__ L16, int* __restrict__ status,
                                                               float* __restrict__ X32, __half* __restrict__ X16,
                                                               int ntp, int c0, int nbk) {
  extern __shared__ float csm[];
  float* S = csm;
  float* Ls = S + 10 * CH_BLK;
  float* X11 = Ls + NB * DLD;
  float* X22 = X11 + 32 * XLD;
  float* X21 = X22 + 32 * XLD;
  const int job = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  float* base = L32 + ((size_t)job * ntp + c0) * ntp + c0;
  __half* base16 = L16 ? L16 + ((size_t)job * ntp + c0) * ntp + c0 : nullptr;
  const int g = lane >> 2, t = lane & 3;
  const int frow = 16 * (warp & 3) + g, fcol = 32 * (warp >> 2) + 2 * t;
  for (int i = 0; i < nbk; ++i)
    for (int j = 0; j <= i; ++j) {
      float* dst = S + ch_slot(i, j);
      const float* src = base + (size_t)(64 * i) * ntp + 64 * j;
      for (int e = tid; e < 64 * 16; e += 256) {
        const int r = e >> 4, c4 = (e & 15) * 4;
        *reinterpret_cast<float4*>(dst + r * AS_LD + c4) = *reinterpret_cast<const float4*>(src + (size_t)r * ntp + c4);
      }
    }
  __syncthreads();
  float acc[4][4];
  auto clear = [&]() {
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[nt][e] = 0.f;
  };
  for (int b = 0; b < nbk; ++b) {
    float* Sbb = S + ch_slot(b, b);
    for (int e = tid; e < NB * NB; e += 256) Ls[(e >> 6) * DLD + (e & 63)] = Sbb[(e >> 6) * AS_LD + (e & 63)];
    __syncthreads();
    if (tid < DT) {
      const bool ok = diag64_body<true>(Ls, X11, X22, X21, tid);
      if (!ok && tid < 32) status[job] = 1;
    }
    __syncthreads();
    float* Li = Linv32 + ((size_t)job * ntp + c0 + 64 * b) * NB;
    for (int e = tid; e < NB * NB; e += 256) {
      const int rr = e >> 6, c = e & 63;
      const float l = diag_l(Ls, rr, c);
      base[(size_t)(64 * b + rr) * ntp + 64 * b + c] = l;
      if (base16) base16[(size_t)(64 * b + rr) * ntp + 64 * b + c] = __float2half_rn(l);
      const float x = round_tf32(diag_x(X11, X22, X21, rr, c));
      Li[e] = x;
      Sbb[rr * AS_LD + c] = x;
    }
    __syncthreads();
    if (b + 1 >= nbk) break;
    // (i) triangular solves of block column b: L_ib = T_ib Linv_b^T
    for (int i = b + 1; i < nbk; ++i) {
      float* Sib = S + ch_slot(i, b);
      clear();
      block_mma_nt(acc, Sib, Sbb, warp, lane);
      __syncthreads();                 // every warp has read Sib before anybody replaces it
      float* blk = base + (size_t)(64 * i) * ntp + 64 * b;
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        const float2 lo = make_float2(round_tf32(acc[nt][0]), round_tf32(acc[nt][1]));
        const float2 hi = make_float2(round_tf32(acc[nt][2]), round_tf32(acc[nt][3]));
        *reinterpret_cast<float2*>(Sib + frow * AS_LD + fcol + 8 * nt) = lo;
        *reinterpret_cast<float2*>(Sib + (frow + 8) * AS_LD + fcol + 8 * nt) = hi;
        *reinterpret_cast<float2*>(blk + (size_t)frow * ntp + fcol + 8 * nt) = lo;
        *reinterpret_cast<float2*>(blk + (size_t)(frow + 8) * ntp + fcol + 8 * nt) = hi;
        if (base16) {
          __half* h = base16 + (size_t)(64 * i) * ntp + 64 * b;
          *reinterpret_cast<__half2*>(h + (size_t)frow * ntp + fcol + 8 * nt) = __floats2half2_rn(lo.x, lo.y);
          *reinterpret_cast<__half2*>(h + (size_t)(frow + 8) * ntp + fcol + 8 * nt) = __floats2half2_rn(hi.x, hi.y);
        }
      }
    }
    __syncthreads();
    // (ii) left-looking update of block column j = b + 1 with every finished column of the diagonal block
    const int j = b + 1;
    for (int i = j; i < nbk; ++i) {
      clear();
      for (int k = 0; k <= b; ++k) block_mma_nt(acc, S + ch_slot(i, k), S + ch_slot(j, k), warp, lane);
      float* Sij = S + ch_slot(i, j);  // (nobody reads column j during this phase: fragments are private)
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        float2* p0 = reinterpret_cast<float2*>(Sij + frow * AS_LD + fcol + 8 * nt);
        float2* p1 = reinterpret_cast<float2*>(Sij + (frow + 8) * AS_LD + fcol + 8 * nt);
        float2 v0 = *p0, v1 = *p1;
        v0.x -= acc[nt][0];
        v0.y -= acc[nt][1];
        v1.x -= acc[nt][2];
        v1.y -= acc[nt][3];
        *p0 = v0;
        *p1 = v1;
      }
    }
    __syncthreads();
  }
  if (X32 == nullptr && X16 == nullptr) return;
  // Inverse of the 256 x 256 factor (trinv256_kernel's recurrence in the same order, operands already in shared memory:
  // off-diagonal slots hold L_ik, diagonal slots Linv_i):  X_bb = Linv_b,  X_ib = -Linv_i sum_{k=b}^{i-1} L_ik X_kb.
  float* Out = X32 ? X32 + (size_t)job * 256 * 256 : nullptr;
  __half* Out16 = X16 ? X16 + (size_t)job * 256 * 256 : nullptr;
  auto put4 = [&](size_t off, const float4 v) {
    if (Out16) {
      const __half2 a = __floats2half2_rn(v.x, v.y), b = __floats2half2_rn(v.z, v.w);
      *reinterpret_cast<uint2*>(Out16 + off) =
          make_uint2(*reinterpret_cast<const uint32_t*>(&a), *reinterpret_cast<const uint32_t*>(&b));
    } else {
      *reinterpret_cast<float4*>(Out + off) = v;
    }
  };
  auto put2 = [&](size_t off, const float2 v) {
    if (Out16) *reinterpret_cast<__half2*>(Out16 + off) = __floats2half2_rn(v.x, v.y);
    else *reinterpret_cast<float2*>(Out + off) = v;
  };
  float* Ss = S + 10 * CH_BLK;         // (the diagonal scratch is free now)
  float* XA = Ss + CH_BLK;             // X_{b+1, b}
  float* XB = XA + CH_BLK;             // X_{b+2, b}
  for (int b = 0; b < 4; ++b) {
    for (int i = 0; i < b; ++i)
      for (int e = tid; e < 64 * 16; e += 256)
        put4((size_t)(64 * i + (e >> 4)) * 256 + 64 * b + (e & 15) * 4, make_float4(0.f, 0.f, 0.f, 0.f));
    const float* Xbb = S + ch_slot(b, b);
    for (int e = tid; e < 64 * 16; e += 256) {
      const int r = e >> 4, c4 = (e & 15) * 4;
      put4((size_t)(64 * b + r) * 256 + 64 * b + c4, *reinterpret_cast<const float4*>(Xbb + r * AS_LD + c4));
    }
  }
  for (int b = 0; b < 3; ++b) {
    for (int i = b + 1; i < 4; ++i) {
      clear();
      for (int k = b; k < i; ++k)
        block_mma<AS_LD>(acc, S + ch_slot(i, k), k == b ? S + ch_slot(b, b) : (k == b + 1 ? XA : XB), warp, lane);
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        *reinterpret_cast<float2*>(Ss + frow * AS_LD + fcol + 8 * nt) = make_float2(round_tf32(acc[nt][0]), round_tf32(acc[nt][1]));
        *reinterpret_cast<float2*>(Ss + (frow + 8) * AS_LD + fcol + 8 * nt) = make_float2(round_tf32(acc[nt][2]), round_tf32(acc[nt][3]));
      }
      __syncthreads();
      clear();
      block_mma<AS_LD>(acc, S + ch_slot(i, i), Ss, warp, lane);
      float* Xi = i == b + 1 ? XA : (i == b + 2 ? XB : nullptr);
      const size_t oi = (size_t)(64 * i) * 256 + 64 * b;
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        const float2 lo = make_float2(round_tf32(-acc[nt][0]), round_tf32(-acc[nt][1]));
        const float2 hi = make_float2(round_tf32(-acc[nt][2]), round_tf32(-acc[nt][3]));
        if (Xi) {
          *reinterpret_cast<float2*>(Xi + frow * AS_LD + fcol + 8 * nt) = lo;
          *reinterpret_cast<float2*>(Xi + (frow + 8) * AS_LD + fcol + 8 * nt) = hi;
        }
        put2(oi + (size_t)frow * 256 + fcol + 8 * nt, lo);
        put2(oi + (size_t)(frow + 8) * 256 + fcol + 8 * nt, hi);
      }
      __syncthreads();
    }
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn g_encode32 = nullptr;
constexpr int DIAG32_SMEM = 0;

cudaError_t encode_f32(CUtensorMap* tm, const float* base, size_t cols, size_t rows, std::string* err) {
  const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)cols * sizeof(float)};
  const cuuint32_t box[2] = {(cuuint32_t)TBK, (cuuint32_t)BOX_ROWS};
  const cuuint32_t estr[2] = {1, 1};
  CUresult r = g_encode32(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    if (err) *err = "cuTensorMapEncodeTiled(f32) failed with CUresult " + std::to_string((int)r);
    return cudaErrorInvalidValue;
  }
  return cudaSuccess;
}

cudaError_t encode_f16(CUtensorMap* tm, const __half* base, size_t cols, size_t rows, std::string* err) {
  const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)cols * sizeof(__half)};
  const cuuint32_t box[2] = {(cuuint32_t)HBK, (cuuint32_t)BOX_ROWS};
  const cuuint32_t estr[2] = {1, 1};
  CUresult r = g_encode32(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<__half*>(base), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    if (err) *err = "cuTensorMapEncodeTiled(f16) failed with CUresult " + std::to_string((int)r);
    return cudaErrorInvalidValue;
  }
  return cudaSuccess;
}

}  // namespace

cudaError_t tb_chol_tc_init() {
  if (!g_encode32) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess) return e;
    if (!fn || qres != cudaDriverEntryPointSuccess) return cudaErrorNotSupported;
    g_encode32 = reinterpret_cast<EncodeTiledFn>(fn);
  }
  cudaError_t e = cudaFuncSetAttribute(trinv256_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TRINV_SMEM);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(chol_chain256_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, CHAIN_SMEM);
  if (e != cudaSuccess) return e;
#define TB_GEMM_ATTR(F, S, W)                                                                                       \
  e = cudaFuncSetAttribute(tf32_gemm_kernel<F, S, W>, cudaFuncAttributeMaxDynamicSharedMemorySize, t_smem(W)); \
  if (e != cudaSuccess) return e;
  TB_GEMM_ATTR(false, 0, 8) TB_GEMM_ATTR(true, 0, 8) TB_GEMM_ATTR(true, 1, 8) TB_GEMM_ATTR(true, 2, 8)
  TB_GEMM_ATTR(false, 0, 16) TB_GEMM_ATTR(true, 0, 16) TB_GEMM_ATTR(true, 1, 16) TB_GEMM_ATTR(true, 2, 16)
#undef TB_GEMM_ATTR
#define TB_FUSED_ATTR(S, W)                                                                                   \
  e = cudaFuncSetAttribute(panel_fused_kernel<S, W>, cudaFuncAttributeMaxDynamicSharedMemorySize, F_SMEM); \
  if (e != cudaSuccess) return e;
  TB_FUSED_ATTR(1, 8) TB_FUSED_ATTR(2, 8) TB_FUSED_ATTR(1, 16)
#undef TB_FUSED_ATTR
  return cudaSuccess;
}

// Factor every job's fp32 matrix in place.  L32: [n_jobs * ntp + 128 slack rows][ntp]; Linv32: [n_jobs * ntp][64].
// L16 (optional): [n_jobs * ntp][ntp] halves, receives a half-precision copy of the factor.
// launches[0] / launches[1] receive the number of GEMM / diagonal-block kernel launches.
cudaError_t tb_chol_tc_factor(float* L32, float* Linv32, void* L16, float* Linv256, int* status, int n_jobs, int ntp,
                              int n_sm, cudaStream_t st, int* launches, std::string* err,
                              void (*mark)(void*, int, int), void* mark_ctx, const TbFromC* from_c, int t16, int epi_warps,
                              int chain_fused_jobs, int panel_fused) {
  const bool chain_inverse = chain_fused_jobs >= 0;      // (negative: fused chain for -n jobs without the inverse; A/B)
  if (chain_fused_jobs < 0) chain_fused_jobs = -chain_fused_jobs;
  CUtensorMap tm_l, tm_inv, tm_inv256;
  cudaError_t e = encode_f32(&tm_l, L32, (size_t)ntp, (size_t)n_jobs * ntp + 128, err);
  if (e != cudaSuccess) return e;
  e = encode_f32(&tm_inv, Linv32, (size_t)NB, (size_t)n_jobs * ntp, err);
  if (e != cudaSuccess) return e;
  CUtensorMap tm_x16;
  if (Linv256) {
    e = encode_f32(&tm_inv256, Linv256, 256, (size_t)n_jobs * 256, err);
    if (e != cudaSuccess) return e;
    // the same scratch viewed as halves (first half of the allocation): fp16 inverses of the 256-wide diagonal blocks
    e = encode_f16(&tm_x16, reinterpret_cast<const __half*>(Linv256), 256, (size_t)n_jobs * 256, err);
    if (e != cudaSuccess) return e;
  }
  // updates (C -= A B^T with both operands finished columns of L) stream the half-precision copy of the factor
  const bool upd16 = L16 != nullptr;
  CUtensorMap tm_l16;
  if (upd16) {
    e = encode_f16(&tm_l16, static_cast<const __half*>(L16), (size_t)ntp, (size_t)n_jobs * ntp, err);
    if (e != cudaSuccess) return e;
  }
  auto gemm = [&](const CUtensorMap& tb, GemmParams p) -> cudaError_t {
    p.n_jobs = n_jobs;
    p.ntp = ntp;
    p.L32 = L32;
    p.L16 = static_cast<__half*>(L16);
    if (p.row_end <= 0 || p.row_end > ntp) p.row_end = ntp;
    p.n_mtiles = (p.row_end - p.row0 + TBM - 1) / TBM;
    if (p.n_mtiles <= 0 || (p.K <= 0 && !p.from_c)) return cudaSuccess;
    const int items = n_jobs * p.n_mtiles;
    const int grid = items < n_sm ? items : n_sm;
    // variant: 0 = fp32 operands, 1 = fp16 operands / fp32 entries, 2 = fp16 / int16 cross-products, 3 = fp16 / int32
    int variant = 0;
    const CUtensorMap* ta = &tm_l;
    const CUtensorMap* tbb = &tb;
    if (p.mode != 0 && p.f16ops) { variant = 1; ta = &tm_l16; }
    else if (p.mode == 0 && upd16) { variant = p.from_c ? (p.fc.c16 ? 2 : 3) : 1; ta = &tm_l16; tbb = &tm_l16; }
#define TB_GEMM_LAUNCH(F, S, W) tf32_gemm_kernel<F, S, W><<<grid, t_threads(W), t_smem(W), st>>>(*ta, *tbb, p)
    if (epi_warps == 16) {
      if (variant == 0) TB_GEMM_LAUNCH(false, 0, 16);
      else if (variant == 1) TB_GEMM_LAUNCH(true, 0, 16);
      else if (variant == 2) TB_GEMM_LAUNCH(true, 1, 16);
      else TB_GEMM_LAUNCH(true, 2, 16);
    } else {
      if (variant == 0) TB_GEMM_LAUNCH(false, 0, 8);
      else if (variant == 1) TB_GEMM_LAUNCH(true, 0, 8);
      else if (variant == 2) TB_GEMM_LAUNCH(true, 1, 8);
      else TB_GEMM_LAUNCH(true, 2, 8);
    }
#undef TB_GEMM_LAUNCH
    launches[0]++;
    return cudaGetLastError();
  };
  const int OB = 256;
  for (int c0 = 0; c0 < ntp; c0 += OB) {
    const int w = (ntp - c0) < OB ? (ntp - c0) : OB;
    // With the inverse of the whole diagonal block the rows below it need ONE GEMM (K = 256) instead of four narrow
    // update / triangular-solve rounds; the narrow rounds then only cover the 256 rows of the diagonal block itself.
    const bool wide = Linv256 != nullptr && w == OB && c0 + w < ntp;
    // ... and when this block column is formed from the cross-products, its rows below the diagonal block never exist
    // in fp32: the update writes them as halves into L16, the panel GEMM (fp16 operands) replaces them in place by the
    // factor entries -- 2 + 2 bytes per entry instead of 4 + 4
    const bool col16 = wide && t16 && upd16 && from_c && !(c0 == 0 && from_c->skip_blk0);
    // ... and those rows can be finished by one launch after the diagonal chain (panel_fused_kernel): the update before
    // the chain then only covers the diagonal block
    const bool fused = col16 && panel_fused;
    if (c0 > 0 || (from_c && upd16 && !from_c->skip_blk0)) {
      // (block column 0 with from_c: K = 0, the launch only forms the block column from the cross-products)
      if (mark) mark(mark_ctx, 0, 0);
      GemmParams p{};
      p.row0 = c0; p.a_col0 = 0; p.K = c0; p.b_row0 = c0; p.b_col0 = 0; p.b_rows_per_job = ntp; p.c_col0 = c0;
      p.N = w; p.mode = 0;
      if (fused) p.row_end = c0 + w;
      if (from_c && upd16) {                       // this launch is the first touch of block column c0: form it from C
        p.from_c = 1;
        p.fc = *from_c;
        p.t16 = col16 ? 1 : 0;
      }
      if ((e = gemm(tm_l, p)) != cudaSuccess) return e;
      if (mark) mark(mark_ctx, 0, 1);
    }
    if (mark) mark(mark_ctx, 1, 0);
    const int narrow_end = wide ? c0 + w : ntp;
    bool chain_has_inverse = false;      // the fused chain kernel also wrote the inverse of the diagonal block
    if (Linv256 != nullptr && narrow_end == c0 + w) {
      // the narrow rounds only cover the diagonal block itself: potrf + inverse per 64-block, then one small
      // mma.sync kernel per step for the solves below it and the update of the next block column
      const int nbk = w / NB;
      if (n_jobs <= chain_fused_jobs) {
        // small batch: the whole chain of this block column in one launch, one CTA per job
        chol_chain256_kernel<<<n_jobs, 256, CHAIN_SMEM, st>>>(
            L32, Linv32, static_cast<__half*>(L16), status, wide && chain_inverse && !col16 ? Linv256 : nullptr,
            wide && chain_inverse && col16 ? reinterpret_cast<__half*>(Linv256) : nullptr, ntp, c0, nbk);
        chain_has_inverse = wide && chain_inverse;
        launches[1]++;
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
      } else
      for (int b = 0; b < nbk; ++b) {
        chol_diag32_kernel<<<n_jobs, DT, DIAG32_SMEM, st>>>(L32, Linv32, static_cast<__half*>(L16), status, ntp,
                                                             (c0 + b * NB) / NB);
        launches[1]++;
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        if (b + 1 < nbk) {
          chol_narrow_kernel<<<n_jobs, 256, 0, st>>>(L32, static_cast<__half*>(L16), Linv32, ntp, c0, b, nbk);
          launches[1]++;
          if ((e = cudaGetLastError()) != cudaSuccess) return e;
        }
      }
    } else
    for (int cc = c0; cc < c0 + w; cc += NB) {
      if (cc > c0) {
        GemmParams p{};
        p.row0 = cc; p.row_end = narrow_end; p.a_col0 = c0; p.K = cc - c0; p.b_row0 = cc; p.b_col0 = c0;
        p.b_rows_per_job = ntp; p.c_col0 = cc; p.N = NB; p.mode = 0;
        if ((e = gemm(tm_l, p)) != cudaSuccess) return e;
      }
      chol_diag32_kernel<<<n_jobs, DT, DIAG32_SMEM, st>>>(L32, Linv32, static_cast<__half*>(L16), status, ntp, cc / NB);
      launches[1]++;
      if ((e = cudaGetLastError()) != cudaSuccess) return e;
      if (cc + NB < narrow_end) {
        GemmParams p{};
        p.row0 = cc + NB; p.row_end = narrow_end; p.a_col0 = cc; p.K = NB; p.b_row0 = cc; p.b_col0 = 0;
        p.b_rows_per_job = ntp; p.c_col0 = cc; p.N = NB; p.mode = 1;
        if ((e = gemm(tm_inv, p)) != cudaSuccess) return e;
      }
    }
    if (wide && !chain_has_inverse) {
      trinv256_kernel<<<n_jobs, 256, TRINV_SMEM, st>>>(L32, Linv32, Linv256,
                                                       col16 ? reinterpret_cast<__half*>(Linv256) : nullptr, ntp, c0);
      launches[1]++;
      if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    if (wide && !fused) {
      GemmParams p{};
      p.row0 = c0 + w; p.a_col0 = c0; p.K = w; p.b_row0 = 0; p.b_col0 = 0; p.b_rows_per_job = 256; p.c_col0 = c0;
      p.N = w; p.mode = 1;
      // rows below the diagonal block: later steps read them only through the fp16 copy (updates, solve sweeps)
      p.skip32 = upd16 ? 1 : 0;
      p.f16ops = col16 ? 1 : 0;
      if ((e = gemm(col16 ? tm_x16 : tm_inv256, p)) != cudaSuccess) return e;
    }
    if (mark) mark(mark_ctx, 1, 1);
    if (fused) {
      // timed as chol_update: it is the update of these rows (plus the panel product that used to be its own launch)
      if (mark) mark(mark_ctx, 0, 0);
      GemmParams p{};
      p.n_jobs = n_jobs; p.ntp = ntp; p.L32 = L32; p.L16 = static_cast<__half*>(L16);
      p.row0 = c0 + w; p.row_end = ntp; p.n_mtiles = (ntp - p.row0 + TBM - 1) / TBM;
      p.K = c0; p.c_col0 = c0; p.N = w; p.from_c = 1; p.fc = *from_c;
      const int items = n_jobs * p.n_mtiles;
      const int grid = items < n_sm ? items : n_sm;
#define TB_FUSED_LAUNCH(S, W) panel_fused_kernel<S, W><<<grid, t_threads(W), F_SMEM, st>>>(tm_l16, tm_x16, p)
      // (int32 cross-products: eight epilogue warps -- at sixteen, 96 registers per thread do not hold a prefetched unit)
      if (!from_c->c16) TB_FUSED_LAUNCH(2, 8);
      else if (epi_warps == 16) TB_FUSED_LAUNCH(1, 16);
      else TB_FUSED_LAUNCH(1, 8);
#undef TB_FUSED_LAUNCH
      launches[0]++;
      if ((e = cudaGetLastError()) != cudaSuccess) return e;
      if (mark) mark(mark_ctx, 0, 1);
    }
  }
  return cudaSuccess;
}
