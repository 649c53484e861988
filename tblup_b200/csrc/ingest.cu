// Genotype ingest: animal-major int8 rows (host order already permuted into "universe" order) or SNP-major 2-bit
// packed rows (file order, permuted here) -> SNP-major device matrix, kept as int8 dosages or re-packed to 2 bits
// per dosage; plus per-marker dosage sums over a set of animals.
// HBM-bound byte work; runs once per data set / per row set, never in the per-generation loop.
//
// Replaces the per-worker `np.load(data_path)` of tblup/evaluator.py:215 and the column means of
// tblup/utils.py:14 and tblup/evaluator.py:304 (kept as exact integer sums).
#include "tb_internal.h"

namespace {

// rows: [n_rows][m] (m contiguous).  x: [m][ldn], writes x[j][pos0 + r].
// Row tiles stride by gridDim.y: a chunk of more than 65 535 x 64 animals (few markers) needs no second launch.
__global__ void transpose_rows_kernel(const int8_t* __restrict__ rows, int n_rows, int m, int8_t* __restrict__ x,
                                      int ldn, int pos0) {
  __shared__ int8_t tile[64][65];
  const int j0 = blockIdx.x * 64;
  const int tx = threadIdx.x, ty = threadIdx.y;  // 64 x 4
  for (int r0 = blockIdx.y * 64; r0 < n_rows; r0 += gridDim.y * 64) {
    for (int rr = ty; rr < 64; rr += 4) {
      int r = r0 + rr, j = j0 + tx;
      tile[rr][tx] = (r < n_rows && j < m) ? rows[(size_t)r * m + j] : (int8_t)0;
    }
    __syncthreads();
    for (int jj = ty; jj < 64; jj += 4) {
      int j = j0 + jj, r = r0 + tx;
      if (j < m && r < n_rows) x[(size_t)j * ldn + pos0 + r] = tile[tx][jj];
    }
    __syncthreads();
  }
}

// One warp per marker: colsum[j] = sum_i x[j][pos[i]].
__global__ void colsum_kernel(const int8_t* __restrict__ x, int ldn, int m, const int* __restrict__ pos, int n_pos,
                              int* __restrict__ colsum) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= m) return;
  const int8_t* row = x + (size_t)warp * ldn;
  int acc = 0;
  for (int i = lane; i < n_pos; i += 32) acc += row[pos[i]];
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) colsum[warp] = acc;
}

// 2-bit packed storage (four animals per byte, animal 4q + i in bits 2i..2i+1, the bit order of a PLINK .bed row):
// x2[j][q] packs x[j][4q .. 4q+3].  ldn is a multiple of 128, so every row is whole words.
__global__ void pack2_kernel(const int8_t* __restrict__ x, size_t n_words, uint8_t* __restrict__ x2) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < n_words; q += stride) {
    const uint32_t w = reinterpret_cast<const uint32_t*>(x)[q];
    x2[q] = (uint8_t)((w & 3u) | ((w >> 6) & 0xcu) | ((w >> 12) & 0x30u) | ((w >> 18) & 0xc0u));
  }
}

// rows2: [n_rows][stride] packed markers of a chunk, animals in FILE order; x[j0 + r][p] = code of animal perm[p].
// Code 3 is not a dosage: counted in *bad (the caller rejects the data set).  Markers stride by gridDim.y: a chunk is
// up to 256 MiB of rows, which for fewer than ~16 400 animals is more markers than gridDim.y can hold.
__global__ void unpack2_perm_kernel(const uint8_t* __restrict__ rows2, int n_rows, int stride, const int* __restrict__ perm,
                                    int n, int8_t* __restrict__ x, int ldn, int j0, int* __restrict__ bad) {
  int local_bad = 0;
  for (int r = blockIdx.y; r < n_rows; r += gridDim.y) {
    const uint8_t* src = rows2 + (size_t)r * stride;
    int8_t* dst = x + (size_t)(j0 + r) * ldn;
    for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < n; p += gridDim.x * blockDim.x) {
      const int a = perm[p];
      const int code = (src[a >> 2] >> (2 * (a & 3))) & 3;
      local_bad |= code == 3;
      dst[p] = (int8_t)code;
    }
  }
  if (local_bad) atomicAdd(bad, 1);
}

__global__ void colsum2_kernel(const uint8_t* __restrict__ x2, int ld4, int m, const int* __restrict__ pos, int n_pos,
                               int* __restrict__ colsum) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= m) return;
  const uint8_t* row = x2 + (size_t)warp * ld4;
  int acc = 0;
  for (int i = lane; i < n_pos; i += 32) {
    const int p = pos[i];
    acc += (row[p >> 2] >> (2 * (p & 3))) & 3;
  }
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) colsum[warp] = acc;
}

// Per-marker statistics over a list of animals with one weight each (the GWAS-style scan of the top-SNPs seeder,
// tblup/seeder.py:144-160,202-210 -> sklearn f_regression): one warp per marker,
//   sx[j] = sum_i x_ij,   sxx[j] = sum_i x_ij^2   (exact integers),   sxw[j] = sum_i x_ij w_i   (fp64, fixed order).
// HBM-bound: every marker row of the resident matrix is read once.
__global__ void marker_stats_kernel(TbGeno g, int m, const int* __restrict__ pos, const double* __restrict__ w, int n_pos,
                                    double* __restrict__ sx, double* __restrict__ sxx, double* __restrict__ sxw) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= m) return;
  int a1 = 0, a2 = 0;
  double aw = 0.0;
  if (g.x2) {
    const uint8_t* row = g.x2 + (size_t)warp * g.ld4;
    for (int i = lane; i < n_pos; i += 32) {
      const int p = pos[i];
      const int v = (row[p >> 2] >> (2 * (p & 3))) & 3;
      a1 += v;
      a2 += v * v;
      aw += (double)v * w[i];
    }
  } else {
    const int8_t* row = g.x + (size_t)warp * g.ldn;
    for (int i = lane; i < n_pos; i += 32) {
      const int v = row[pos[i]];
      a1 += v;
      a2 += v * v;
      aw += (double)v * w[i];
    }
  }
  for (int o = 16; o; o >>= 1) {
    a1 += __shfl_xor_sync(0xffffffffu, a1, o);
    a2 += __shfl_xor_sync(0xffffffffu, a2, o);
    aw += __shfl_xor_sync(0xffffffffu, aw, o);
  }
  if (lane == 0) {
    sx[warp] = (double)a1;
    sxx[warp] = (double)a2;
    sxw[warp] = aw;
  }
}

}  // namespace

cudaError_t tb_launch_pack2(const int8_t* d_x, int ldn, int m, uint8_t* d_x2, cudaStream_t st) {
  const size_t n_words = (size_t)m * (ldn / 4);
  const int blocks = (int)std::min<size_t>((n_words + 255) / 256, 148 * 16);
  pack2_kernel<<<blocks, 256, 0, st>>>(d_x, n_words, d_x2);
  return cudaGetLastError();
}

cudaError_t tb_launch_unpack2_perm(const uint8_t* d_rows2, int n_rows, int stride, const int* d_perm, int n,
                                   int8_t* d_x, int ldn, int j0, int* d_bad, cudaStream_t st) {
  dim3 grid((n + 1023) / 1024 > 8 ? 8 : (n + 1023) / 1024, std::min(n_rows, 65535));
  unpack2_perm_kernel<<<grid, 256, 0, st>>>(d_rows2, n_rows, stride, d_perm, n, d_x, ldn, j0, d_bad);
  return cudaGetLastError();
}

cudaError_t tb_launch_transpose_rows(const int8_t* d_rows, int n_rows, int m, int8_t* d_x, int ldn, int pos0,
                                     cudaStream_t st) {
  dim3 grid((m + 63) / 64, std::min((n_rows + 63) / 64, 65535)), block(64, 4);
  transpose_rows_kernel<<<grid, block, 0, st>>>(d_rows, n_rows, m, d_x, ldn, pos0);
  return cudaGetLastError();
}

cudaError_t tb_launch_colsum(const TbGeno& g, int m, const int* d_pos, int n_pos, int* d_colsum, cudaStream_t st) {
  const int warps_per_block = 8;
  if (g.x2) {
    colsum2_kernel<<<(m + warps_per_block - 1) / warps_per_block, warps_per_block * 32, 0, st>>>(g.x2, g.ld4, m, d_pos,
                                                                                                n_pos, d_colsum);
    return cudaGetLastError();
  }
  const int8_t* d_x = g.x;
  const int ldn = g.ldn;
  colsum_kernel<<<(m + warps_per_block - 1) / warps_per_block, warps_per_block * 32, 0, st>>>(d_x, ldn, m, d_pos,
                                                                                             n_pos, d_colsum);
  return cudaGetLastError();
}

cudaError_t tb_launch_marker_stats(const TbGeno& g, int m, const int* d_pos, const double* d_w, int n_pos, double* d_sx,
                                   double* d_sxx, double* d_sxw, cudaStream_t st) {
  const int warps_per_block = 8;
  marker_stats_kernel<<<(m + warps_per_block - 1) / warps_per_block, warps_per_block * 32, 0, st>>>(g, m, d_pos, d_w, n_pos,
                                                                                                   d_sx, d_sxx, d_sxw);
  return cudaGetLastError();
}
