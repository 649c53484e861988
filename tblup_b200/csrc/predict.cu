// Panel models: the marker effects behind a genome's fitness, and breeding values of any animal from them.
//
// The fitness path solves (G_TT + lambda I) alpha = y_T for every (genome, row set) and keeps only the Pearson r of
// the validation predictions.  The model behind it is linear in the listed markers j_1..j_k (duplicates count twice):
//
//   c_q  = colsum_q / N                          centre 2p of listed marker q over the N frequency animals
//   d    = (2 N S - Q) / (2 N^2)                 S = sum_q colsum_q, Q = sum_q colsum_q^2  (= 2 sum p (1 - p))
//   b_q  = (sum_{a in T} x_{a,j_q} alpha_a - c_q sum_{a in T} alpha_a) / d
//   yhat_b = b0 + sum_q (x_{b,j_q} - c_q) b_q     b0 = 0 (gblup), mean(y_T) (snp_blup)
//
// since G = (X - c)(X - c)^T / d: G_{bT} alpha = sum_q (x_{b,q} - c_q) [(X_T - c)^T alpha]_q / d.  For the snp_blup
// branch b and b0 are exactly sklearn's Ridge(alpha = lambda d) coef_ / intercept_ on X_T - c (the dual solution).
//
// Kernels (both storages of the resident matrix, TbGeno):
//   fit_prep_kernel         one CTA per genome: sum alpha over T (fixed-order tree), S and Q (exact int64) -> d
//   marker_effects_kernel   (genome, block of 64 listed markers): one dot product of a marker row over T with alpha
//   predict_effects_kernel  (tile of 512 targets, genome, marker split): sum_q (x - c_q) b_q for four targets a thread
//   predict_finish_kernel   b0 + the marker splits, in split order
// No atomics; every sum runs in a fixed order that depends on the shapes only, so results are bit-identical between
// the int8 and 2-bit storages and from run to run.  A thread always handles four consecutive list entries (training
// animals or targets); when their positions are four aligned consecutive universe columns -- prefix row sets, targets
// listed in universe order -- the four dosages come from ONE load (a 32-bit word of int8 dosages, or one byte of
// 2-bit codes), else from four.  The values, and their order of summation, are the same either way.
//
// Work and bytes per genome: k n_t dosage products for the effects, k n_targets for the predictions, one fp64 add each
// (plus a 3-way select on the integer pipe).  A warp reads 32 B (packed) or 128 B (int8) of a marker row per 128
// list entries.  At 5 000 x 50 000 the packed matrix (62.5 MB) stays in L2; at 20 000 x 500 000 (2.5 GB) each genome
// streams k rows over T / the targets from HBM: k n_t / 4 bytes (packed) for the effects, k n / 4 for the predictions.
// At both sizes the fp64 adds are the larger floor.  The kernels reach 4-7 % of it (DESIGN.md §3e has the measured
// numbers).
#include "tb_internal.h"
#include "../../include/tblup_b200.h"

#include <cmath>

namespace {

constexpr int EFF_WARPS = 8;      // warps per CTA of marker_effects_kernel
constexpr int EFF_MPW = 8;        // listed markers per warp (their dot products share the alpha / position loads)
constexpr int EFF_MARKERS = EFF_WARPS * EFF_MPW;
constexpr int PRED_THREADS = 128;
constexpr int PRED_TILE = 4 * PRED_THREADS;   // targets per CTA
constexpr int PRED_CHUNK = 128;               // listed markers staged in shared memory at a time

struct FitGenome {
  const int* colsum;     // d_colsum_all (gblup) or the row set's d_colsum_train (snp_blup)
  long long N;           // animals behind the frequencies
  double asum;           // sum_{a in T} alpha_a            (fit_prep_kernel)
  double d;              // (2 N S - Q) / (2 N^2)           (fit_prep_kernel)
};

// the four positions are four aligned consecutive universe columns: their dosages sit in one word / one byte
__device__ __forceinline__ bool is_run(int4 p) {
  return p.y == p.x + 1 && p.z == p.x + 2 && p.w == p.x + 3 && (p.x & 3) == 0;
}

// four dosages of marker row j at universe positions p (x, y, z, w), as four bytes of one word (RUN: is_run(p))
template <bool PACKED, bool RUN>
__device__ __forceinline__ uint32_t load4(const TbGeno& g, int j, int4 p) {
  if constexpr (PACKED) {
    const uint8_t* row = g.x2 + (size_t)j * g.ld4;
    if constexpr (RUN) {
      const uint32_t b = __ldg(row + (p.x >> 2));
      return (b & 3u) | ((b >> 2) & 3u) << 8 | ((b >> 4) & 3u) << 16 | (b >> 6) << 24;
    }
    auto code = [&](int q) { return (uint32_t)(__ldg(row + (q >> 2)) >> (2 * (q & 3))) & 3u; };
    return code(p.x) | code(p.y) << 8 | code(p.z) << 16 | code(p.w) << 24;
  } else {
    const uint8_t* row = reinterpret_cast<const uint8_t*>(g.x) + (size_t)j * g.ldn;
    if constexpr (RUN) return __ldg(reinterpret_cast<const uint32_t*>(row + p.x));
    return (uint32_t)__ldg(row + p.x) | (uint32_t)__ldg(row + p.y) << 8 | (uint32_t)__ldg(row + p.z) << 16 |
           (uint32_t)__ldg(row + p.w) << 24;
  }
}

// v0, v1 or v2 for a dosage code 0, 1 or 2, by bit masks: no branch (a ?: chain compiles to divergent branches)
__device__ __forceinline__ double pick(uint32_t code, double v0, double v1, double v2) {
  const long long m1 = -(long long)(code & 1u), m2 = -(long long)(code >> 1), m0 = ~(m1 | m2);
  return __longlong_as_double((__double_as_longlong(v0) & m0) | (__double_as_longlong(v1) & m1) |
                              (__double_as_longlong(v2) & m2));
}
__device__ __forceinline__ double pick0(uint32_t code, double v1, double v2) {      // v0 = +0.0
  const long long m1 = -(long long)(code & 1u), m2 = -(long long)(code >> 1);
  return __longlong_as_double((__double_as_longlong(v1) & m1) | (__double_as_longlong(v2) & m2));
}

// fixed-order block reductions (blockDim.x = 256)
__device__ double block_sum_d(double v, double* red) {
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  double s = 0.0;
  for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red[w];
  return s;
}
__device__ long long block_sum_ll(long long v, long long* red) {
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  long long s = 0;
  for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red[w];
  return s;
}

__global__ void __launch_bounds__(256) fit_prep_kernel(FitGenome* __restrict__ gen, const int* __restrict__ idx,
                                                       const long long* __restrict__ off, const double* __restrict__ alpha,
                                                       int n_t, int ntp) {
  __shared__ double redd[8];
  __shared__ long long redl[8];
  const int g = blockIdx.x;
  const double* al = alpha + (size_t)g * ntp;
  double a = 0.0;
  for (int i = threadIdx.x; i < n_t; i += blockDim.x) a += al[i];
  const double asum = block_sum_d(a, redd);
  const int* cs = gen[g].colsum;
  long long s = 0, q = 0;
  for (long long t = off[g] + threadIdx.x; t < off[g + 1]; t += blockDim.x) {
    const long long v = cs[idx[t]];
    s += v;
    q += v * v;
  }
  const long long S = block_sum_ll(s, redl);
  const long long Q = block_sum_ll(q, redl);
  if (threadIdx.x == 0) {
    const long long N = gen[g].N;
    gen[g].asum = asum;
    gen[g].d = (double)(2 * N * S - Q) / (2.0 * (double)N * (double)N);
  }
}

// beta[off[g] + q] and centre[off[g] + q] for every listed marker q of genome g = blockIdx.y.
// tp: [ntp] universe positions of the training animals (zero beyond n_t), alpha: [P][ntp]
template <bool PACKED>
__global__ void __launch_bounds__(EFF_WARPS * 32, 2) marker_effects_kernel(
    TbGeno geno, const int* __restrict__ idx, const long long* __restrict__ off, const int* __restrict__ tp,
    const double* __restrict__ alpha, int n_t, int ntp, const FitGenome* __restrict__ gen, double* __restrict__ beta,
    double* __restrict__ centre) {
  const int g = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long o = off[g];
  const int k = (int)(off[g + 1] - o);
  const int q0 = blockIdx.x * EFF_MARKERS + warp * EFF_MPW;
  if (q0 >= k) return;
  int j[EFF_MPW];
#pragma unroll
  for (int u = 0; u < EFF_MPW; ++u) j[u] = idx[o + min(q0 + u, k - 1)];
  const double* al = alpha + (size_t)g * ntp;
  double acc[EFF_MPW];
#pragma unroll
  for (int u = 0; u < EFF_MPW; ++u) acc[u] = 0.0;
  for (int i0 = 4 * lane; i0 < n_t; i0 += 128) {
    const int4 p = *reinterpret_cast<const int4*>(tp + i0);
    const double2 x01 = *reinterpret_cast<const double2*>(al + i0);
    const double2 x23 = *reinterpret_cast<const double2*>(al + i0 + 2);
    const double a0 = x01.x, a1 = i0 + 1 < n_t ? x01.y : 0.0, a2 = i0 + 2 < n_t ? x23.x : 0.0,
                 a3 = i0 + 3 < n_t ? x23.y : 0.0;
    const double d0 = a0 + a0, d1 = a1 + a1, d2 = a2 + a2, d3 = a3 + a3;
    uint32_t w[EFF_MPW];
    if (is_run(p)) {
#pragma unroll
      for (int u = 0; u < EFF_MPW; ++u) w[u] = load4<PACKED, true>(geno, j[u], p);
    } else {
#pragma unroll
      for (int u = 0; u < EFF_MPW; ++u) w[u] = load4<PACKED, false>(geno, j[u], p);
    }
#pragma unroll
    for (int u = 0; u < EFF_MPW; ++u) {
      acc[u] += pick0(w[u] & 0xffu, a0, d0);
      acc[u] += pick0((w[u] >> 8) & 0xffu, a1, d1);
      acc[u] += pick0((w[u] >> 16) & 0xffu, a2, d2);
      acc[u] += pick0(w[u] >> 24, a3, d3);
    }
  }
#pragma unroll
  for (int u = 0; u < EFF_MPW; ++u)
    for (int s = 16; s; s >>= 1) acc[u] += __shfl_xor_sync(0xffffffffu, acc[u], s);
  if (lane < EFF_MPW && q0 + lane < k) {
    double dot = acc[0];
#pragma unroll
    for (int u = 1; u < EFF_MPW; ++u) dot = lane == u ? acc[u] : dot;
    const FitGenome fg = gen[g];
    int jj = j[0];
#pragma unroll
    for (int u = 1; u < EFF_MPW; ++u) jj = lane == u ? j[u] : jj;
    const double c = (double)fg.colsum[jj] / (double)fg.N;
    beta[o + q0 + lane] = (dot - c * fg.asum) / fg.d;
    centre[o + q0 + lane] = c;
  }
}

// partial[s][g][b] (or out[g][b] when there is one split) = sum over the markers of split s of (x_{b,j_q} - c_q) b_q,
// for the targets of tile blockIdx.x; pos: [n_pad] universe positions of the targets (zero beyond n_targets)
template <bool PACKED>
__global__ void __launch_bounds__(PRED_THREADS) predict_effects_kernel(
    TbGeno geno, const int* __restrict__ idx, const long long* __restrict__ off, const double* __restrict__ centre,
    const double* __restrict__ beta, const double* __restrict__ b0, const int* __restrict__ pos, int n_targets,
    int n_pad, int n_split, double* __restrict__ partial, double* __restrict__ out) {
  __shared__ int sj[PRED_CHUNK];
  __shared__ double st[3][PRED_CHUNK];
  const int g = blockIdx.y, split = blockIdx.z;
  const long long o = off[g];
  const int k = (int)(off[g + 1] - o);
  const int per = (k + n_split - 1) / n_split;
  const int qa = min(k, split * per), qb = min(k, qa + per);
  const int b = blockIdx.x * PRED_TILE + 4 * threadIdx.x;
  const int4 p = b < n_pad ? *reinterpret_cast<const int4*>(pos + b) : make_int4(0, 0, 0, 0);
  const bool run = is_run(p);
  double y0 = 0.0, y1 = 0.0, y2 = 0.0, y3 = 0.0;
  auto step = [&](uint32_t w, int t) {
    const double v0 = st[0][t], v1 = st[1][t], v2 = st[2][t];
    y0 += pick(w & 0xffu, v0, v1, v2);
    y1 += pick((w >> 8) & 0xffu, v0, v1, v2);
    y2 += pick((w >> 16) & 0xffu, v0, v1, v2);
    y3 += pick(w >> 24, v0, v1, v2);
  };
  for (int q = qa; q < qb; q += PRED_CHUNK) {
    const int nq = min(PRED_CHUNK, qb - q);
    __syncthreads();
    for (int t = threadIdx.x; t < nq; t += PRED_THREADS) {
      const double c = centre[o + q + t], e = beta[o + q + t];
      sj[t] = idx[o + q + t];
      st[0][t] = (0.0 - c) * e;
      st[1][t] = (1.0 - c) * e;
      st[2][t] = (2.0 - c) * e;
    }
    __syncthreads();
    if (run) {
#pragma unroll 4
      for (int t = 0; t < nq; ++t) step(load4<PACKED, true>(geno, sj[t], p), t);
    } else {
#pragma unroll 4
      for (int t = 0; t < nq; ++t) step(load4<PACKED, false>(geno, sj[t], p), t);
    }
  }
  const double y[4] = {y0, y1, y2, y3};
  for (int r = 0; r < 4; ++r) {
    if (b + r >= n_targets) break;
    if (n_split == 1) out[(size_t)g * n_targets + b + r] = b0[g] + y[r];
    else partial[((size_t)split * gridDim.y + g) * n_targets + b + r] = y[r];
  }
}

__global__ void predict_finish_kernel(const double* __restrict__ partial, const double* __restrict__ b0, int P,
                                      int n_targets, int n_split, double* __restrict__ out) {
  const size_t total = (size_t)P * n_targets;
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
    double acc = 0.0;
    for (int s = 0; s < n_split; ++s) acc += partial[(size_t)s * total + e];
    out[e] = b0[e / n_targets] + acc;
  }
}

int pfail(TbCtx* c, const std::string& msg, int code = -1) {
  c->err = msg;
  return code;
}

// device buffers of one call, freed on every exit path
struct Buffers {
  std::vector<void*> p;
  template <typename T>
  cudaError_t take(T** out, size_t n) {
    void* q = nullptr;
    cudaError_t e = cudaMalloc(&q, std::max<size_t>(n, 1) * sizeof(T));
    if (e == cudaSuccess) p.push_back(q);
    *out = static_cast<T*>(q);
    return e;
  }
  ~Buffers() {
    for (void* q : p) cudaFree(q);
  }
};

// marker splits of the prediction: enough CTAs to fill the GPU several times over (HBM-bound shapes need the bytes in
// flight), never fewer than 256 markers a split.  Depends on the shapes only, so results do not depend on the device.
int pred_splits(int P, int n_targets, long long kmax) {
  const long long ctas = (long long)P * ((n_targets + PRED_TILE - 1) / PRED_TILE);
  long long s = (8 * 148 + ctas - 1) / ctas;
  s = std::min<long long>(s, (kmax + 255) / 256);
  return (int)std::max<long long>(1, std::min<long long>(s, 64));
}

}  // namespace

extern "C" {

int tb_fit_effects(tb_ctx* c, int slot, double h2, int mode_rule, double* effects_out, double* centre_out,
                   double* intercept_out, double* fitness_out) {
  if (!c) return -1;
  if (!effects_out || !centre_out || !intercept_out) return pfail(c, "tb_fit_effects: null output");
  if (c->P <= 0) return pfail(c, "tb_fit_effects: no genomes staged");
  if (slot < 0 || slot >= TB_MAX_SLOTS || !c->slots[slot].valid)
    return pfail(c, "tb_fit_effects: row set " + std::to_string(slot) + " is not defined");
  if (mode_rule < 0 || mode_rule > 2) return pfail(c, "tb_fit_effects: bad mode_rule");
  if (c->stop_after >= 0) return pfail(c, "tb_fit_effects: the stop_after debug option is set");
  for (int i = 0; i < c->P; ++i)
    if (c->h_off[i + 1] <= c->h_off[i]) return pfail(c, "tb_fit_effects: empty genome at position " + std::to_string(i));
  TB_CUDA(c, cudaSetDevice(c->device));
  const TbRowSet& rs = c->slots[slot];
  const int P = c->P, n_t = rs.n_t, ntp = rs.ntp;
  const size_t total = (size_t)c->h_off[P];
  cudaStream_t st = c->stream;
  Buffers buf;
  double *d_alpha = nullptr, *d_fit = nullptr, *d_beta = nullptr, *d_centre = nullptr;
  int* d_tp = nullptr;
  long long* d_off = nullptr;
  FitGenome* d_gen = nullptr;
  TB_CUDA(c, buf.take(&d_alpha, (size_t)P * ntp));
  TB_CUDA(c, buf.take(&d_fit, (size_t)P));
  TB_CUDA(c, buf.take(&d_beta, total));
  TB_CUDA(c, buf.take(&d_centre, total));
  TB_CUDA(c, buf.take(&d_tp, (size_t)ntp));
  TB_CUDA(c, buf.take(&d_off, (size_t)P + 1));
  TB_CUDA(c, buf.take(&d_gen, (size_t)P));
  std::vector<FitGenome> h_gen(P);
  for (int i = 0; i < P; ++i) {
    const long long k = c->h_off[i + 1] - c->h_off[i];
    const bool gblup = mode_rule == TB_MODE_GBLUP || (mode_rule == TB_MODE_AUTO && k > c->n);
    h_gen[i] = FitGenome{gblup ? c->d_colsum_all : rs.d_colsum_train, gblup ? (long long)c->n : (long long)n_t, 0.0, 0.0};
    intercept_out[i] = gblup ? 0.0 : rs.yt_mean;
  }
  // the solve, exactly as tb_eval_staged runs it for this row set, keeping every genome's alpha
  if (int rc = tb_internal_eval_alpha(c, slot, h2, mode_rule, d_fit, d_alpha)) {
    cudaStreamSynchronize(st);
    tb_internal_collect_spans(c);
    return rc;
  }
  TB_CUDA(c, cudaMemsetAsync(d_tp, 0, (size_t)ntp * sizeof(int), st));
  TB_CUDA(c, cudaMemcpyAsync(d_tp, rs.d_tpos, (size_t)n_t * sizeof(int), cudaMemcpyDeviceToDevice, st));
  TB_CUDA(c, cudaMemcpyAsync(d_off, c->h_off.data(), (size_t)(P + 1) * sizeof(long long), cudaMemcpyHostToDevice, st));
  TB_CUDA(c, cudaMemcpyAsync(d_gen, h_gen.data(), (size_t)P * sizeof(FitGenome), cudaMemcpyHostToDevice, st));
  fit_prep_kernel<<<P, 256, 0, st>>>(d_gen, c->d_idx, d_off, d_alpha, n_t, ntp);
  TB_CUDA(c, cudaGetLastError());
  long long kmax = 0;
  for (int i = 0; i < P; ++i) kmax = std::max(kmax, c->h_off[i + 1] - c->h_off[i]);
  const dim3 grid((unsigned)((kmax + EFF_MARKERS - 1) / EFF_MARKERS), (unsigned)P);
  if (c->d_x2)
    marker_effects_kernel<true><<<grid, EFF_WARPS * 32, 0, st>>>(c->geno(), c->d_idx, d_off, d_tp, d_alpha, n_t, ntp,
                                                                  d_gen, d_beta, d_centre);
  else
    marker_effects_kernel<false><<<grid, EFF_WARPS * 32, 0, st>>>(c->geno(), c->d_idx, d_off, d_tp, d_alpha, n_t, ntp,
                                                                   d_gen, d_beta, d_centre);
  TB_CUDA(c, cudaGetLastError());
  c->launches += 2;
  TB_CUDA(c, cudaMemcpyAsync(effects_out, d_beta, total * sizeof(double), cudaMemcpyDeviceToHost, st));
  TB_CUDA(c, cudaMemcpyAsync(centre_out, d_centre, total * sizeof(double), cudaMemcpyDeviceToHost, st));
  if (fitness_out) TB_CUDA(c, cudaMemcpyAsync(fitness_out, d_fit, (size_t)P * sizeof(double), cudaMemcpyDeviceToHost, st));
  const cudaError_t se = cudaStreamSynchronize(st);
  tb_internal_collect_spans(c);
  if (se != cudaSuccess) return pfail(c, std::string("tb_fit_effects: device execution failed: ") + cudaGetErrorString(se), -2);
  return 0;
}

int tb_predict_effects(tb_ctx* c, const int32_t* idx_flat, const int64_t* idx_off, int P, const double* centre,
                       const double* effects, const double* intercept, const int32_t* animals, int n_animals,
                       double* out) {
  if (!c) return -1;
  if (!idx_flat || !idx_off || !centre || !effects || !intercept || !animals || !out || P <= 0 || n_animals <= 0)
    return pfail(c, "tb_predict_effects: null or empty argument");
  if (idx_off[0] != 0) return pfail(c, "tb_predict_effects: idx_off[0] must be 0");
  long long kmax = 0;
  for (int i = 0; i < P; ++i) {
    if (idx_off[i + 1] <= idx_off[i]) return pfail(c, "tb_predict_effects: empty genome at position " + std::to_string(i));
    kmax = std::max<long long>(kmax, idx_off[i + 1] - idx_off[i]);
  }
  if (kmax > 0x7fffffffLL) return pfail(c, "tb_predict_effects: genome too long");
  const size_t total = (size_t)idx_off[P];
  for (size_t q = 0; q < total; ++q)
    if (idx_flat[q] < 0 || idx_flat[q] >= c->m)
      return pfail(c, "tb_predict_effects: marker index " + std::to_string(idx_flat[q]) + " out of range [0, " +
                          std::to_string(c->m) + ")");
  const int n_pad = tb_round_up(n_animals, 4);
  std::vector<int> pos(n_pad, 0);
  for (int i = 0; i < n_animals; ++i) {
    if (animals[i] < 0 || animals[i] >= c->n)
      return pfail(c, "tb_predict_effects: animal index " + std::to_string(animals[i]) + " out of range [0, " +
                          std::to_string(c->n) + ")");
    pos[i] = c->pos_of[animals[i]];
  }
  TB_CUDA(c, cudaSetDevice(c->device));
  cudaStream_t st = c->stream;
  const int n_split = pred_splits(P, n_animals, kmax);
  Buffers buf;
  int *d_idx = nullptr, *d_pos = nullptr;
  long long* d_off = nullptr;
  double *d_centre = nullptr, *d_beta = nullptr, *d_b0 = nullptr, *d_out = nullptr, *d_part = nullptr;
  TB_CUDA(c, buf.take(&d_idx, total));
  TB_CUDA(c, buf.take(&d_off, (size_t)P + 1));
  TB_CUDA(c, buf.take(&d_centre, total));
  TB_CUDA(c, buf.take(&d_beta, total));
  TB_CUDA(c, buf.take(&d_b0, (size_t)P));
  TB_CUDA(c, buf.take(&d_pos, (size_t)n_pad));
  TB_CUDA(c, buf.take(&d_out, (size_t)P * n_animals));
  if (n_split > 1) TB_CUDA(c, buf.take(&d_part, (size_t)n_split * P * n_animals));
  TB_CUDA(c, cudaMemcpyAsync(d_idx, idx_flat, total * sizeof(int), cudaMemcpyHostToDevice, st));
  TB_CUDA(c, cudaMemcpyAsync(d_off, idx_off, (size_t)(P + 1) * sizeof(long long), cudaMemcpyHostToDevice, st));
  TB_CUDA(c, cudaMemcpyAsync(d_centre, centre, total * sizeof(double), cudaMemcpyHostToDevice, st));
  TB_CUDA(c, cudaMemcpyAsync(d_beta, effects, total * sizeof(double), cudaMemcpyHostToDevice, st));
  TB_CUDA(c, cudaMemcpyAsync(d_b0, intercept, (size_t)P * sizeof(double), cudaMemcpyHostToDevice, st));
  TB_CUDA(c, cudaMemcpyAsync(d_pos, pos.data(), (size_t)n_pad * sizeof(int), cudaMemcpyHostToDevice, st));
  const dim3 grid((unsigned)((n_animals + PRED_TILE - 1) / PRED_TILE), (unsigned)P, (unsigned)n_split);
  if (c->d_x2)
    predict_effects_kernel<true><<<grid, PRED_THREADS, 0, st>>>(c->geno(), d_idx, d_off, d_centre, d_beta, d_b0, d_pos,
                                                                n_animals, n_pad, n_split, d_part, d_out);
  else
    predict_effects_kernel<false><<<grid, PRED_THREADS, 0, st>>>(c->geno(), d_idx, d_off, d_centre, d_beta, d_b0, d_pos,
                                                                 n_animals, n_pad, n_split, d_part, d_out);
  TB_CUDA(c, cudaGetLastError());
  c->launches += 1;
  if (n_split > 1) {
    predict_finish_kernel<<<4 * 148, 256, 0, st>>>(d_part, d_b0, P, n_animals, n_split, d_out);
    TB_CUDA(c, cudaGetLastError());
    c->launches += 1;
  }
  TB_CUDA(c, cudaMemcpyAsync(out, d_out, (size_t)P * n_animals * sizeof(double), cudaMemcpyDeviceToHost, st));
  const cudaError_t se = cudaStreamSynchronize(st);
  if (se != cudaSuccess) return pfail(c, std::string("tb_predict_effects: device execution failed: ") + cudaGetErrorString(se), -2);
  return 0;
}

}  // extern "C"
