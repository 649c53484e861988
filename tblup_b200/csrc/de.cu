// On-device differential-evolution step on random-key individuals (SURVEY.md §8f row F1, north_star (e)):
// the P x m key matrix lives in HBM, so genomes never round-trip to the host between generations.
//
//   evolve   child_i = where(cross_i, a + F (b - c), parent_i), optional clip      tblup/evolver.py:63-83,104-157
//   decode   genome_i = indices of the `length` largest keys                          tblup/individual.py:155-156
//   evaluate (the fitness pipeline of api.cu on the decoded lists, already on the device)
//   select   child replaces parent iff strictly fitter, NaN never wins               tblup/selector.py:18-34
//
// The random draws (three distinct parents != i, one forced crossover position, the U(0,1) crossover mask) can be
// supplied by the host -- that is how the parity tests replay the reference's own Mersenne-Twister draws bit for
// bit -- or generated on the device from a counter-based hash (production mode; a different but equally valid
// random stream, see DESIGN.md).  All kernels are HBM-bound byte/word movers.
#include "tb_internal.h"
#include "../../include/tblup_b200.h"

namespace {

__device__ __forceinline__ unsigned long long mix64(unsigned long long z) {
  z += 0x9E3779B97F4A7C15ULL;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
  return z ^ (z >> 31);
}
__device__ __forceinline__ double u01(unsigned long long seed, unsigned long long ctr) {
  return (double)(mix64(seed ^ mix64(ctr)) >> 11) * (1.0 / 9007199254740992.0);
}

__global__ void de_init_keys_kernel(double* __restrict__ keys, size_t total, unsigned long long seed) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < total) keys[i] = u01(seed, i);
}

// device-side parent picks: three distinct indices, all different from i (exclusive_randrange, tblup/utils.py:21-36)
__global__ void de_pick_kernel(int* __restrict__ abc, int* __restrict__ fixed, int P, int m, unsigned long long seed) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P) return;
  unsigned long long ctr = (unsigned long long)i << 20;
  int pick[3];
  for (int t = 0; t < 3; ++t) {
    for (;;) {
      const int r = (int)(mix64(seed ^ mix64(ctr++)) % (unsigned long long)P);
      bool clash = r == i;
      for (int q = 0; q < t; ++q) clash |= r == pick[q];
      if (!clash) {
        pick[t] = r;
        break;
      }
    }
  }
  abc[3 * i] = pick[0];
  abc[3 * i + 1] = pick[1];
  abc[3 * i + 2] = pick[2];
  fixed[i] = (int)(mix64(seed ^ mix64(ctr)) % (unsigned long long)m);
}

// mask: optional [P][m] bytes (1 = take the mutant); when null the mask is drawn on the device.
__global__ void __launch_bounds__(256) de_evolve_kernel(const double* __restrict__ keys, double* __restrict__ child,
                                                        const int* __restrict__ abc, const int* __restrict__ fixed,
                                                        const unsigned char* __restrict__ mask, int m, double F,
                                                        double CR, int clip, unsigned long long seed) {
  const int i = blockIdx.y;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= m) return;
  const size_t row = (size_t)i * m;
  bool cross;
  if (mask)
    cross = mask[row + j] != 0;
  else
    cross = u01(seed, 0x4000000000000000ULL + row + j) < CR;
  cross = cross || j == fixed[i];
  double v = keys[row + j];
  if (cross) {
    const double ka = keys[(size_t)abc[3 * i] * m + j], kb = keys[(size_t)abc[3 * i + 1] * m + j],
                 kc = keys[(size_t)abc[3 * i + 2] * m + j];
    v = __dadd_rn(ka, __dmul_rn(F, __dsub_rn(kb, kc)));   // numpy's a + mi * (b - c): three roundings, no fma
  }
  // np.clip(v, 0, m - 1): NaN and -0.0 pass through unchanged (fmin / fmax would turn a NaN into a bound)
  if (clip) {
    const double hi = (double)(m - 1);
    v = v < 0.0 ? 0.0 : v;
    v = v > hi ? hi : v;
  }
  child[row + j] = v;
}

// Order-preserving map of a key to an unsigned integer, in numpy's sort order: -0.0 and +0.0 are one value, and every
// NaN (either sign, any payload) is one value above +inf.  Keys numpy holds equal therefore map to one integer, and
// the decode's tie rule (lowest index first) covers them all.
__device__ __forceinline__ unsigned long long sortable(double d) {
  unsigned long long b = (unsigned long long)__double_as_longlong(d);
  b = d != d ? 0x7FF8000000000000ULL : d == 0.0 ? 0ULL : b;
  return (b >> 63) ? ~b : (b | 0x8000000000000000ULL);
}

// One CTA per individual: exact k-th largest key by MSD radix select (8 bits per pass), then an order-preserving
// compaction of the indices whose key is above the threshold (ties at the threshold: lowest indices first).
__global__ void __launch_bounds__(1024) de_decode_kernel(const double* __restrict__ keys, int m, int k,
                                                         int* __restrict__ idx_out, int out_stride) {
  __shared__ unsigned int hist[256];
  __shared__ unsigned long long s_prefix;
  __shared__ unsigned int s_rank, s_base, s_tie_base;
  __shared__ unsigned int wsum[32][2];
  const double* row = keys + (size_t)blockIdx.x * m;
  int* out = idx_out + (size_t)blockIdx.x * out_stride;      // lists out_stride >= k apart
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) {
    s_prefix = 0;
    s_rank = (unsigned int)(m - k);   // rank (ascending, 0-based) of the k-th largest key
  }
  __syncthreads();
  for (int pass = 0; pass < 8; ++pass) {
    const int shift = 56 - 8 * pass;
    if (tid < 256) hist[tid] = 0;
    __syncthreads();
    const unsigned long long prefix = s_prefix;
    for (int j = tid; j < m; j += 1024) {
      const unsigned long long u = sortable(row[j]);
      if (pass == 0 || (u >> (shift + 8)) == prefix) atomicAdd(&hist[(u >> shift) & 255], 1u);
    }
    __syncthreads();
    if (tid == 0) {
      unsigned int r = s_rank, acc = 0;
      int b = 0;
      for (; b < 256; ++b) {
        if (acc + hist[b] > r) break;
        acc += hist[b];
      }
      s_rank = r - acc;
      s_prefix = (prefix << 8) | (unsigned long long)b;
    }
    __syncthreads();
  }
  const unsigned long long T = s_prefix;          // sortable value of the k-th largest key
  // count keys strictly above T
  unsigned int gt = 0;
  for (int j = tid; j < m; j += 1024) gt += sortable(row[j]) > T;
  for (int o = 16; o; o >>= 1) gt += __shfl_xor_sync(0xffffffffu, gt, o);
  if (lane == 0) wsum[warp][0] = gt;
  __syncthreads();
  if (tid == 0) {
    unsigned int t = 0;
    for (int w = 0; w < 32; ++w) t += wsum[w][0];
    s_base = 0;
    s_tie_base = 0;
    s_rank = (unsigned int)k - t;                 // how many keys equal to T are taken
  }
  __syncthreads();
  const unsigned int ties_wanted = s_rank;
  for (int j0 = 0; j0 < m; j0 += 1024) {
    const int j = j0 + tid;
    bool above = false, tie = false;
    if (j < m) {
      const unsigned long long u = sortable(row[j]);
      above = u > T;
      tie = u == T;
    }
    const unsigned int ma = __ballot_sync(0xffffffffu, above), mt = __ballot_sync(0xffffffffu, tie);
    if (lane == 0) {
      wsum[warp][0] = __popc(ma);
      wsum[warp][1] = __popc(mt);
    }
    __syncthreads();
    unsigned int pa = 0, pt = 0, ta = 0, tt = 0;
    for (int w = 0; w < 32; ++w) {
      if (w < warp) {
        pa += wsum[w][0];
        pt += wsum[w][1];
      }
      ta += wsum[w][0];
      tt += wsum[w][1];
    }
    const unsigned int lt_mask = (1u << lane) - 1u;
    const unsigned int tie_rank = s_tie_base + pt + __popc(mt & lt_mask);        // this tie's index among all ties
    const bool take = above || (tie && tie_rank < ties_wanted);
    // output position: everything taken before me, in index order
    const unsigned int ties_before = min(s_tie_base + pt + __popc(mt & lt_mask), ties_wanted) - min(s_tie_base, ties_wanted);
    const unsigned int pos = s_base + pa + __popc(ma & lt_mask) + ties_before;
    if (take) out[pos] = j;
    __syncthreads();
    if (tid == 0) {
      const unsigned int old_tie = s_tie_base;
      s_tie_base = old_tie + tt;
      s_base += ta + (min(old_tie + tt, ties_wanted) - min(old_tie, ties_wanted));
    }
    __syncthreads();
  }
}

// ---- SNP removal on the device (tblup/evaluator.py:589-633) -------------------------------------------------------
// banned[j] = 1 for every marker removed so far.  The fitness of an individual is computed on
// setdiff1d(genome, removed) (evaluator.py:617), its testing accuracy on union1d(genome, removed) (:627-633).

// rows: [P][stride] decoded genomes (`len_in` entries each).  Keeps the entries that are not banned, in order,
// in place; lens[i] = how many are left.
__global__ void __launch_bounds__(1024) de_filter_banned_kernel(int* __restrict__ rows, int stride, int len_in,
                                                                const unsigned char* __restrict__ banned,
                                                                int* __restrict__ lens) {
  __shared__ unsigned int wsum[32];
  __shared__ unsigned int s_base;
  int* row = rows + (size_t)blockIdx.x * stride;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_base = 0;
  __syncthreads();
  for (int j0 = 0; j0 < len_in; j0 += 1024) {
    const int j = j0 + tid;
    int v = -1;
    bool keep = false;
    if (j < len_in) {
      v = row[j];
      keep = banned[v] == 0;
    }
    const unsigned int mk = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) wsum[warp] = __popc(mk);
    __syncthreads();                               // every read of this chunk is done before any write below
    unsigned int before = 0, total = 0;
    for (int w = 0; w < 32; ++w) {
      if (w < warp) before += wsum[w];
      total += wsum[w];
    }
    const unsigned int pos = s_base + before + __popc(mk & ((1u << lane) - 1u));
    if (keep) row[pos] = v;                        // pos <= j: never overtakes an unread entry of a later chunk
    __syncthreads();
    if (tid == 0) s_base += total;
    __syncthreads();
  }
  if (tid == 0) lens[blockIdx.x] = (int)s_base;
}

// rows: [P][stride], the first k entries hold the decoded genome.  Appends every banned marker that is not already in
// the genome (membership through a bitmap in shared memory): rows[i] = union(genome_i, removed), lens[i] = its size.
__global__ void __launch_bounds__(1024) de_union_banned_kernel(int* __restrict__ rows, int stride, int k, int m,
                                                               const int* __restrict__ banned_list, int n_banned,
                                                               int* __restrict__ lens) {
  extern __shared__ unsigned int member[];         // m bits
  __shared__ unsigned int wsum[32];
  __shared__ unsigned int s_base;
  int* row = rows + (size_t)blockIdx.x * stride;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int q = tid; q < (m + 31) / 32; q += 1024) member[q] = 0;
  if (tid == 0) s_base = (unsigned int)k;
  __syncthreads();
  for (int j = tid; j < k; j += 1024) atomicOr(&member[row[j] >> 5], 1u << (row[j] & 31));
  __syncthreads();
  for (int j0 = 0; j0 < n_banned; j0 += 1024) {
    const int j = j0 + tid;
    int v = -1;
    bool add = false;
    if (j < n_banned) {
      v = banned_list[j];
      add = ((member[v >> 5] >> (v & 31)) & 1u) == 0;
    }
    const unsigned int mk = __ballot_sync(0xffffffffu, add);
    if (lane == 0) wsum[warp] = __popc(mk);
    __syncthreads();
    unsigned int before = 0, total = 0;
    for (int w = 0; w < 32; ++w) {
      if (w < warp) before += wsum[w];
      total += wsum[w];
    }
    if (add) row[s_base + before + __popc(mk & ((1u << lane) - 1u))] = v;
    __syncthreads();
    if (tid == 0) s_base += total;
    __syncthreads();
  }
  if (tid == 0) lens[blockIdx.x] = (int)s_base;
}

// flat[off[i] + j] = rows[i][j], j < off[i+1] - off[i]  (ragged lists behind one another, what the pipeline reads)
__global__ void de_pack_rows_kernel(const int* __restrict__ rows, int stride, const long long* __restrict__ off,
                                    int* __restrict__ flat) {
  const int i = blockIdx.y;
  const long long o0 = off[i];
  const int len = (int)(off[i + 1] - o0);
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < len; j += gridDim.x * blockDim.x)
    flat[o0 + j] = rows[(size_t)i * stride + j];
}

__global__ void de_set_flags_kernel(unsigned char* __restrict__ banned, const int* __restrict__ list, int n) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < n) banned[list[j]] = 1;
}

// an individual whose every marker is banned is not evaluated: its fitness is 0.0 (evaluator.py:617-619)
__global__ void de_zero_empty_kernel(double* __restrict__ fit, const int* __restrict__ lens, int P) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < P && lens[i] == 0) fit[i] = 0.0;
}

__global__ void de_mean_kernel(const double* __restrict__ f, int n_slots, int P, double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P) return;
  double s = 0.0;
  for (int q = 0; q < n_slots; ++q) s += f[(size_t)i * n_slots + q];
  out[i] = n_slots > 1 ? s / n_slots : s;
}

__global__ void __launch_bounds__(256) de_select_kernel(double* __restrict__ keys, const double* __restrict__ child,
                                                        double* __restrict__ fit, const double* __restrict__ child_fit,
                                                        int m, int* __restrict__ take) {
  const int i = blockIdx.y;
  const bool better = child_fit[i] > fit[i];      // false for NaN on either side, as in the reference
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (better && j < m) keys[(size_t)i * m + j] = child[(size_t)i * m + j];
  if (j == 0 && take) take[i] = better ? 1 : 0;
}

__global__ void de_commit_fitness_kernel(double* __restrict__ fit, const double* __restrict__ child_fit,
                                         const int* __restrict__ take, int P) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < P && take[i]) fit[i] = child_fit[i];
}

int de_fail(TbCtx* c, const std::string& msg, int code = -1) {
  c->err = msg;
  return code;
}

void de_free(TbCtx* c) {
  cudaFree(c->de.keys);
  cudaFree(c->de.child);
  cudaFree(c->de.fit);
  cudaFree(c->de.child_fit);
  cudaFree(c->de.raw_fit);
  cudaFree(c->de.abc);
  cudaFree(c->de.fixed);
  cudaFree(c->de.take);
  cudaFree(c->de.mask);
  cudaFree(c->de.banned);
  cudaFree(c->de.banned_list);
  cudaFree(c->de.rows);
  cudaFree(c->de.lens);
  cudaFree(c->de.d_off);
  c->de = TbCtx::DeState();
}

int de_ensure_idx(TbCtx* c, size_t total) {
  if (total > c->idx_cap) {
    TB_CUDA(c, cudaStreamSynchronize(c->stream));
    cudaFree(c->d_idx);
    c->d_idx = nullptr;
    c->idx_cap = 0;
    TB_CUDA(c, cudaMalloc(&c->d_idx, total * sizeof(int)));
    c->idx_cap = total;
  }
  return 0;
}

int de_ensure_rows(TbCtx* c, int stride) {
  auto& d = c->de;
  if ((size_t)d.P * stride > d.rows_cap) {
    TB_CUDA(c, cudaStreamSynchronize(c->stream));
    cudaFree(d.rows);
    d.rows = nullptr;
    TB_CUDA(c, cudaMalloc(&d.rows, (size_t)d.P * stride * sizeof(int)));
    d.rows_cap = (size_t)d.P * stride;
  }
  if (!d.lens) TB_CUDA(c, cudaMalloc(&d.lens, (size_t)d.P * sizeof(int)));
  if (!d.d_off) TB_CUDA(c, cudaMalloc(&d.d_off, (size_t)(d.P + 1) * sizeof(long long)));
  return 0;
}

// rows [P][stride] with lens on the device -> the context's staged ragged batch (c->d_idx, c->h_off, c->P).
// Only the P lengths visit the host (the offsets the wave scheduler plans with); an empty list is staged as one
// arbitrary marker and its fitness overwritten afterwards (h_lens tells which).
int de_stage_rows(TbCtx* c, int stride, std::vector<int>& h_lens, int count = -1) {
  auto& d = c->de;
  if (count < 0) count = d.P;
  h_lens.resize(count);
  TB_CUDA(c, cudaMemcpyAsync(h_lens.data(), d.lens, (size_t)count * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  TB_CUDA(c, cudaStreamSynchronize(c->stream));
  c->h_off.resize(count + 1);
  c->h_off[0] = 0;
  for (int i = 0; i < count; ++i) c->h_off[i + 1] = c->h_off[i] + std::max(h_lens[i], 1);
  c->P = count;
  if (int rc = de_ensure_idx(c, (size_t)c->h_off[count])) return rc;
  TB_CUDA(c, cudaMemcpyAsync(d.d_off, c->h_off.data(), (size_t)(count + 1) * sizeof(long long), cudaMemcpyHostToDevice,
                             c->stream));
  dim3 grid((unsigned)std::min(64, (stride + 255) / 256), count);
  de_pack_rows_kernel<<<grid, 256, 0, c->stream>>>(d.rows, stride, d.d_off, c->d_idx);
  TB_CUDA(c, cudaGetLastError());
  c->launches += 1;
  return 0;
}

int de_ensure_raw(TbCtx* c, int n_slots) {
  auto& d = c->de;
  if ((size_t)d.P * n_slots > d.raw_cap) {
    TB_CUDA(c, cudaStreamSynchronize(c->stream));
    cudaFree(d.raw_fit);
    d.raw_fit = nullptr;
    TB_CUDA(c, cudaMalloc(&d.raw_fit, (size_t)d.P * n_slots * sizeof(double)));
    d.raw_cap = (size_t)d.P * n_slots;
  }
  return 0;
}

// decode `src` keys into the context's staged-genome buffer (minus the banned markers, if any) and evaluate them;
// result (mean over slots) -> dst
// [first, first + count) of the individuals whose keys are in `src` (P x m): decode, drop banned markers, evaluate;
// the mean over the row sets goes to dst[first ...].  count = P scores everybody; a smaller range is one rank's shard
// of a population whose keys are replicated on every GPU.
int de_decode_and_eval(TbCtx* c, const double* src, const int32_t* slots, int n_slots, double h2, int mode,
                       double* dst, int first = 0, int count = -1) {
  auto& d = c->de;
  if (count < 0) count = d.P - first;
  if (count <= 0) return 0;
  src += (size_t)first * c->m;
  dst += first;
  std::vector<int> h_lens;
  if (d.n_banned == 0) {
    if (int rc = de_ensure_idx(c, (size_t)count * d.k)) return rc;
    de_decode_kernel<<<count, 1024, 0, c->stream>>>(src, c->m, d.k, c->d_idx, d.k);
    TB_CUDA(c, cudaGetLastError());
    c->launches += 1;
    c->h_off.resize(count + 1);
    for (int i = 0; i <= count; ++i) c->h_off[i] = (long long)i * d.k;
    c->P = count;
  } else {
    if (int rc = de_ensure_rows(c, d.k)) return rc;
    de_decode_kernel<<<count, 1024, 0, c->stream>>>(src, c->m, d.k, d.rows, d.k);
    TB_CUDA(c, cudaGetLastError());
    de_filter_banned_kernel<<<count, 1024, 0, c->stream>>>(d.rows, d.k, d.k, d.banned, d.lens);
    TB_CUDA(c, cudaGetLastError());
    c->launches += 2;
    if (int rc = de_stage_rows(c, d.k, h_lens, count)) return rc;
  }
  if (int rc = de_ensure_raw(c, n_slots)) return rc;
  int rc = tb_internal_eval_device(c, slots, n_slots, h2, mode, d.raw_fit);
  if (rc) return rc;
  de_mean_kernel<<<(count + 255) / 256, 256, 0, c->stream>>>(d.raw_fit, n_slots, count, dst);
  TB_CUDA(c, cudaGetLastError());
  c->launches += 1;
  if (d.n_banned) {
    de_zero_empty_kernel<<<(count + 255) / 256, 256, 0, c->stream>>>(dst, d.lens, count);
    TB_CUDA(c, cudaGetLastError());
    c->launches += 1;
  }
  return 0;
}

// banned flags -> ascending list on the device + count
int de_refresh_banned_list(TbCtx* c) {
  auto& d = c->de;
  std::vector<unsigned char> flags(c->m);
  TB_CUDA(c, cudaMemcpy(flags.data(), d.banned, (size_t)c->m, cudaMemcpyDeviceToHost));
  std::vector<int> list;
  for (int j = 0; j < c->m; ++j)
    if (flags[j]) list.push_back(j);
  d.n_banned = (int)list.size();
  if (!d.banned_list) TB_CUDA(c, cudaMalloc(&d.banned_list, (size_t)c->m * sizeof(int)));
  if (d.n_banned)
    TB_CUDA(c, cudaMemcpy(d.banned_list, list.data(), list.size() * sizeof(int), cudaMemcpyHostToDevice));
  return 0;
}

int de_ensure_banned(TbCtx* c) {
  auto& d = c->de;
  if (!d.banned) {
    TB_CUDA(c, cudaMalloc(&d.banned, (size_t)c->m));
    TB_CUDA(c, cudaMemset(d.banned, 0, (size_t)c->m));
  }
  return 0;
}

}  // namespace

void tb_de_release(TbCtx* c) { de_free(c); }

extern "C" {

int tb_de_init(tb_ctx* c, int P, int length, const double* keys_host, uint64_t seed) {
  if (!c) return -1;
  if (P < 4) return de_fail(c, "tb_de_init: DE/rand/1 needs at least 4 individuals");
  if (length < 1 || length > c->m) return de_fail(c, "tb_de_init: genome length must be in [1, markers]");
  TB_CUDA(c, cudaSetDevice(c->device));
  TB_CUDA(c, cudaStreamSynchronize(c->stream));
  de_free(c);
  auto& d = c->de;
  d.P = P;
  d.k = length;
  const size_t total = (size_t)P * c->m;
  TB_CUDA(c, cudaMalloc(&d.keys, total * sizeof(double)));
  TB_CUDA(c, cudaMalloc(&d.child, total * sizeof(double)));
  TB_CUDA(c, cudaMalloc(&d.fit, P * sizeof(double)));
  TB_CUDA(c, cudaMalloc(&d.child_fit, P * sizeof(double)));
  TB_CUDA(c, cudaMalloc(&d.abc, 3 * P * sizeof(int)));
  TB_CUDA(c, cudaMalloc(&d.fixed, P * sizeof(int)));
  TB_CUDA(c, cudaMalloc(&d.take, P * sizeof(int)));
  if (keys_host) {
    TB_CUDA(c, cudaMemcpyAsync(d.keys, keys_host, total * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  } else {
    de_init_keys_kernel<<<(unsigned)((total + 255) / 256), 256, 0, c->stream>>>(d.keys, total, seed);
    TB_CUDA(c, cudaGetLastError());
    c->launches += 1;
  }
  TB_CUDA(c, cudaStreamSynchronize(c->stream));
  return 0;
}

int tb_de_evaluate(tb_ctx* c, const int32_t* slots, int n_slots, double h2, int mode_rule) {
  if (!c) return -1;
  if (!c->de.keys) return de_fail(c, "tb_de_evaluate: call tb_de_init first");
  TB_CUDA(c, cudaSetDevice(c->device));
  int rc = de_decode_and_eval(c, c->de.keys, slots, n_slots, h2, mode_rule, c->de.fit);
  cudaError_t se = cudaStreamSynchronize(c->stream);
  tb_internal_collect_spans(c);
  if (rc) return rc;
  if (se != cudaSuccess) return de_fail(c, std::string("device execution failed: ") + cudaGetErrorString(se), -2);
  return 0;
}

int tb_de_step_begin(tb_ctx* c, const int32_t* slots, int n_slots, double h2, int mode_rule, double F, double CR,
                     int clip, const int32_t* abc, const int32_t* fixed, const uint8_t* mask, uint64_t seed, int first,
                     int count) {
  if (!c) return -1;
  auto& d = c->de;
  if (!d.keys) return de_fail(c, "tb_de_step: call tb_de_init and tb_de_evaluate first");
  if ((abc == nullptr) != (fixed == nullptr)) return de_fail(c, "tb_de_step: pass both abc and fixed, or neither");
  if (first < 0 || count < 0 || first + count > d.P) return de_fail(c, "tb_de_step_begin: shard out of range");
  TB_CUDA(c, cudaSetDevice(c->device));
  cudaStream_t st = c->stream;
  const int P = d.P, m = c->m;
  if (abc) {
    for (int i = 0; i < P; ++i) {
      const int a = abc[3 * i], b = abc[3 * i + 1], cc = abc[3 * i + 2];
      if (a < 0 || a >= P || b < 0 || b >= P || cc < 0 || cc >= P || fixed[i] < 0 || fixed[i] >= m)
        return de_fail(c, "tb_de_step: parent index or forced position out of range");
    }
    TB_CUDA(c, cudaMemcpyAsync(d.abc, abc, 3 * P * sizeof(int), cudaMemcpyHostToDevice, st));
    TB_CUDA(c, cudaMemcpyAsync(d.fixed, fixed, P * sizeof(int), cudaMemcpyHostToDevice, st));
  } else {
    de_pick_kernel<<<(P + 127) / 128, 128, 0, st>>>(d.abc, d.fixed, P, m, seed);
    TB_CUDA(c, cudaGetLastError());
    c->launches += 1;
  }
  d.drawn = true;
  const unsigned char* d_mask = nullptr;
  if (mask) {
    if (!d.mask) TB_CUDA(c, cudaMalloc(&d.mask, (size_t)P * m));
    TB_CUDA(c, cudaMemcpyAsync(d.mask, mask, (size_t)P * m, cudaMemcpyHostToDevice, st));
    d_mask = d.mask;
  }
  // every rank evolves the WHOLE offspring population from the replicated parents (same draws, same keys: cheap,
  // and no key ever crosses NVLink); only the evaluation is sharded
  dim3 grid((m + 255) / 256, P);
  de_evolve_kernel<<<grid, 256, 0, st>>>(d.keys, d.child, d.abc, d.fixed, d_mask, m, F, CR, clip, seed);
  TB_CUDA(c, cudaGetLastError());
  c->launches += 1;
  int rc = de_decode_and_eval(c, d.child, slots, n_slots, h2, mode_rule, d.child_fit, first, count);
  cudaError_t se = cudaStreamSynchronize(st);
  tb_internal_collect_spans(c);
  if (rc) return rc;
  if (se != cudaSuccess) return de_fail(c, std::string("device execution failed: ") + cudaGetErrorString(se), -2);
  return 0;
}

int tb_de_step_end(tb_ctx* c, int32_t* take_out) {
  if (!c) return -1;
  auto& d = c->de;
  if (!d.keys) return de_fail(c, "tb_de_step_end: no DE state");
  TB_CUDA(c, cudaSetDevice(c->device));
  cudaStream_t st = c->stream;
  const int P = d.P, m = c->m;
  int rc = 0;
  dim3 grid((m + 255) / 256, P);
  de_select_kernel<<<grid, 256, 0, st>>>(d.keys, d.child, d.fit, d.child_fit, m, d.take);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) {
    de_commit_fitness_kernel<<<(P + 255) / 256, 256, 0, st>>>(d.fit, d.child_fit, d.take, P);
    e = cudaGetLastError();
  }
  c->launches += 2;
  if (e != cudaSuccess) rc = de_fail(c, std::string("selection launch: ") + cudaGetErrorString(e), -2);
  if (rc == 0 && take_out) {
    e = cudaMemcpyAsync(take_out, d.take, P * sizeof(int), cudaMemcpyDeviceToHost, st);
    if (e != cudaSuccess) rc = de_fail(c, std::string("D2H take: ") + cudaGetErrorString(e), -2);
  }
  cudaError_t se = cudaStreamSynchronize(st);
  if (rc) return rc;
  if (se != cudaSuccess) return de_fail(c, std::string("device execution failed: ") + cudaGetErrorString(se), -2);
  return 0;
}

int tb_de_step(tb_ctx* c, const int32_t* slots, int n_slots, double h2, int mode_rule, double F, double CR, int clip,
               const int32_t* abc, const int32_t* fixed, const uint8_t* mask, uint64_t seed, int32_t* take_out) {
  if (!c) return -1;
  int rc = tb_de_step_begin(c, slots, n_slots, h2, mode_rule, F, CR, clip, abc, fixed, mask, seed, 0, c->de.P);
  if (rc) return rc;
  return tb_de_step_end(c, take_out);
}

// Device pointers of the population / offspring fitness vectors [P] (what = 0 / 1), for collectives issued by the
// caller between tb_de_step_begin and tb_de_step_end (all-gather of the shards' offspring fitness).
void* tb_de_device_ptr(tb_ctx* c, int what) {
  if (!c || !c->de.keys) return nullptr;
  return what == 0 ? (void*)c->de.fit : what == 1 ? (void*)c->de.child_fit : nullptr;
}

int tb_de_evaluate_shard(tb_ctx* c, const int32_t* slots, int n_slots, double h2, int mode_rule, int first, int count) {
  if (!c) return -1;
  if (!c->de.keys) return de_fail(c, "tb_de_evaluate_shard: call tb_de_init first");
  if (first < 0 || count < 0 || first + count > c->de.P) return de_fail(c, "tb_de_evaluate_shard: shard out of range");
  TB_CUDA(c, cudaSetDevice(c->device));
  int rc = de_decode_and_eval(c, c->de.keys, slots, n_slots, h2, mode_rule, c->de.fit, first, count);
  cudaError_t se = cudaStreamSynchronize(c->stream);
  tb_internal_collect_spans(c);
  if (rc) return rc;
  if (se != cudaSuccess) return de_fail(c, std::string("device execution failed: ") + cudaGetErrorString(se), -2);
  return 0;
}

int tb_de_set_removed(tb_ctx* c, const int32_t* markers, int n) {
  if (!c) return -1;
  auto& d = c->de;
  if (!d.keys) return de_fail(c, "tb_de_set_removed: call tb_de_init first");
  if (n < 0 || (n > 0 && !markers)) return de_fail(c, "tb_de_set_removed: bad argument");
  for (int j = 0; j < n; ++j)
    if (markers[j] < 0 || markers[j] >= c->m) return de_fail(c, "tb_de_set_removed: marker index out of range");
  TB_CUDA(c, cudaSetDevice(c->device));
  TB_CUDA(c, cudaStreamSynchronize(c->stream));
  if (int rc = de_ensure_banned(c)) return rc;
  std::vector<unsigned char> flags(c->m, 0);
  for (int j = 0; j < n; ++j) flags[markers[j]] = 1;
  TB_CUDA(c, cudaMemcpy(d.banned, flags.data(), (size_t)c->m, cudaMemcpyHostToDevice));
  return de_refresh_banned_list(c);
}

int tb_de_ban_genome(tb_ctx* c, int which, int32_t* n_removed_out) {
  if (!c) return -1;
  auto& d = c->de;
  if (!d.keys) return de_fail(c, "tb_de_ban_genome: call tb_de_init first");
  if (which < 0 || which >= d.P) return de_fail(c, "tb_de_ban_genome: individual out of range");
  TB_CUDA(c, cudaSetDevice(c->device));
  if (int rc = de_ensure_banned(c)) return rc;
  int* tmp = nullptr;
  TB_CUDA(c, cudaMalloc(&tmp, (size_t)d.k * sizeof(int)));
  de_decode_kernel<<<1, 1024, 0, c->stream>>>(d.keys + (size_t)which * c->m, c->m, d.k, tmp, d.k);
  de_set_flags_kernel<<<(d.k + 255) / 256, 256, 0, c->stream>>>(d.banned, tmp, d.k);
  cudaError_t e = cudaGetLastError();
  cudaError_t e2 = cudaStreamSynchronize(c->stream);
  cudaFree(tmp);
  c->launches += 2;
  if (e != cudaSuccess || e2 != cudaSuccess) return de_fail(c, "tb_de_ban_genome: device execution failed", -2);
  if (int rc = de_refresh_banned_list(c)) return rc;
  if (n_removed_out) *n_removed_out = d.n_banned;
  return 0;
}

int tb_de_evaluate_testing(tb_ctx* c, int slot, double h2, int mode_rule, double* fitness_out) {
  if (!c) return -1;
  auto& d = c->de;
  if (!d.keys) return de_fail(c, "tb_de_evaluate_testing: call tb_de_init first");
  if (!fitness_out) return de_fail(c, "tb_de_evaluate_testing: null output");
  TB_CUDA(c, cudaSetDevice(c->device));
  const int stride = d.k + d.n_banned;
  const size_t smem = ((size_t)(c->m + 31) / 32) * 4;                                 // membership bitmap, m bits
  if (d.n_banned && smem > 200 * 1024) return de_fail(c, "tb_de_evaluate_testing: marker bitmap exceeds shared memory");
  std::vector<int> h_lens;
  if (int rc = de_ensure_rows(c, stride)) return rc;
  de_decode_kernel<<<d.P, 1024, 0, c->stream>>>(d.keys, c->m, d.k, d.rows, stride);   // room for the removed markers
  TB_CUDA(c, cudaGetLastError());
  c->launches += 1;
  if (d.n_banned) {
    if (smem > 48 * 1024)
      TB_CUDA(c, cudaFuncSetAttribute(de_union_banned_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    de_union_banned_kernel<<<d.P, 1024, smem, c->stream>>>(d.rows, stride, d.k, c->m, d.banned_list, d.n_banned, d.lens);
    TB_CUDA(c, cudaGetLastError());
    c->launches += 1;
    if (int rc = de_stage_rows(c, stride, h_lens)) return rc;
  } else {
    if (int rc = de_ensure_idx(c, (size_t)d.P * d.k)) return rc;
    TB_CUDA(c, cudaMemcpyAsync(c->d_idx, d.rows, (size_t)d.P * d.k * sizeof(int), cudaMemcpyDeviceToDevice, c->stream));
    c->h_off.resize(d.P + 1);
    for (int i = 0; i <= d.P; ++i) c->h_off[i] = (long long)i * d.k;
    c->P = d.P;
  }
  if (int rc = de_ensure_raw(c, 1)) return rc;
  const int32_t slots[1] = {slot};
  int rc = tb_internal_eval_device(c, slots, 1, h2, mode_rule, d.raw_fit);
  cudaError_t ce = cudaSuccess;
  if (rc == 0) ce = cudaMemcpyAsync(fitness_out, d.raw_fit, (size_t)d.P * sizeof(double), cudaMemcpyDeviceToHost, c->stream);
  cudaError_t se = cudaStreamSynchronize(c->stream);
  tb_internal_collect_spans(c);
  if (rc) return rc;
  if (ce != cudaSuccess || se != cudaSuccess) return de_fail(c, "tb_de_evaluate_testing: device execution failed", -2);
  return 0;
}

int tb_de_get(tb_ctx* c, int what, int which, void* out, size_t nbytes) {
  if (!c || !out) return -1;
  auto& d = c->de;
  if (!d.keys) return de_fail(c, "tb_de_get: no DE state");
  TB_CUDA(c, cudaSetDevice(c->device));
  const void* src = nullptr;
  size_t need = 0;
  switch (what) {
    case 0: src = d.fit; need = (size_t)d.P * 8; break;                           // population fitness
    case 1: src = d.child_fit; need = (size_t)d.P * 8; break;                     // last offspring fitness
    case 2: src = d.keys; need = (size_t)d.P * c->m * 8; break;                   // population keys
    case 3: src = d.child; need = (size_t)d.P * c->m * 8; break;                  // last offspring keys
    case 4: {                                                                     // decoded genome of individual `which`
      if (which < 0 || which >= d.P) return de_fail(c, "tb_de_get: individual out of range");
      need = (size_t)d.k * 4;
      if (nbytes < need) return de_fail(c, "tb_de_get: buffer too small");
      int* tmp = nullptr;
      TB_CUDA(c, cudaMalloc(&tmp, need));
      de_decode_kernel<<<1, 1024, 0, c->stream>>>(d.keys + (size_t)which * c->m, c->m, d.k, tmp, d.k);
      cudaError_t e = cudaMemcpyAsync(out, tmp, need, cudaMemcpyDeviceToHost, c->stream);
      cudaError_t e2 = cudaStreamSynchronize(c->stream);
      cudaFree(tmp);
      c->launches += 1;
      if (e != cudaSuccess || e2 != cudaSuccess) return de_fail(c, "tb_de_get: decode failed", -2);
      return 0;
    }
    case 5: {                                                                     // genomes of the last evaluated batch
      // shard-local after tb_de_evaluate_shard / tb_de_step_begin: c->P genomes are staged, not d.P
      if ((int)c->h_off.size() < c->P + 1 || c->P <= 0) return de_fail(c, "tb_de_get: no batch staged");
      src = c->d_idx; need = (size_t)c->h_off[c->P] * 4; break;
    }
    case 6: src = d.banned_list; need = (size_t)d.n_banned * 4; break;            // removed markers, ascending
    case 7: src = d.lens; need = (size_t)std::min(d.P, std::max(c->P, 0)) * 4; break;  // list lengths of the last filtered batch (staged genomes only)
    case 8: {                                                                     // flat lists of the last evaluated batch
      if ((int)c->h_off.size() < c->P + 1 || c->P <= 0) return de_fail(c, "tb_de_get: no batch staged");
      src = c->d_idx; need = (size_t)c->h_off[c->P] * 4; break;
    }
    case 9:                                                                       // parent picks of the last step [P][3]
      if (!d.drawn) return de_fail(c, "tb_de_get: no generation has been evolved yet");
      src = d.abc; need = (size_t)d.P * 3 * 4; break;
    case 10:                                                                      // forced crossover positions [P]
      if (!d.drawn) return de_fail(c, "tb_de_get: no generation has been evolved yet");
      src = d.fixed; need = (size_t)d.P * 4; break;
    default: return de_fail(c, "tb_de_get: unknown item");
  }
  if (nbytes < need) return de_fail(c, "tb_de_get: buffer too small");
  if (need == 0) return 0;
  if (!src) return de_fail(c, "tb_de_get: nothing recorded yet for this item");
  TB_CUDA(c, cudaMemcpy(out, src, need, cudaMemcpyDeviceToHost));
  return 0;
}

}  // extern "C"
