// C-ABI of libtblup_b200 (see include/tblup_b200.h): context lifetime, row sets, genome staging and the
// wave scheduler that drives gather -> centring terms -> tcgen05 Gram -> scale -> batched Cholesky ->
// solve/predict/Pearson for one generation's batch.  Takes over _evaluate() / worker() / blup() of
// tblup/evaluator.py:205-263,380-405.
#include "tb_internal.h"
#include "../../include/tblup_b200.h"

#include <algorithm>
#include <cmath>
#include <chrono>
#include <thread>

namespace {

std::string g_create_err;

struct Arena {
  char* base = nullptr;
  size_t off = 0, cap = 0;
  template <typename T>
  T* take(size_t n) {
    off = (off + 255) & ~size_t(255);
    T* p = reinterpret_cast<T*>(base + off);
    off += n * sizeof(T);
    return p;
  }
};

int fail(TbCtx* c, const std::string& msg, int code = -1) {
  c->err = msg;
  return code;
}

void free_rowset(TbRowSet& r) {
  cudaFree(r.d_tpos);
  cudaFree(r.d_vpos);
  cudaFree(r.d_rowmap);
  cudaFree(r.d_ident);
  cudaFree(r.d_colsum_train);
  cudaFree(r.d_yt_raw);
  cudaFree(r.d_yt_ctr);
  cudaFree(r.d_yv);
  r = TbRowSet();
}

size_t span_begin(TbCtx* c, int stage) {
  if (!c->profile) return 0;
  if (c->ev_used + 2 > c->ev_pool.size()) {
    size_t old = c->ev_pool.size();
    c->ev_pool.resize(old + 256);
    for (size_t i = old; i < c->ev_pool.size(); ++i) cudaEventCreate(&c->ev_pool[i]);
  }
  size_t b = c->ev_used;
  c->ev_used += 2;
  cudaEventRecord(c->ev_pool[b], c->stream);
  c->spans.push_back({stage, b, b + 1});
  return b;
}
void span_end(TbCtx* c, size_t b) {
  if (!c->profile) return;
  cudaEventRecord(c->ev_pool[b + 1], c->stream);
}
void spans_collect(TbCtx* c) {
  if (!c->profile) return;
  for (auto& s : c->spans) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, c->ev_pool[s.b], c->ev_pool[s.e]) == cudaSuccess) c->stage_ms[s.stage] += ms;
  }
  c->spans.clear();
  c->ev_used = 0;
}
inline void count(TbCtx* c, int stage, int n) {
  c->stage_launches[stage] += n;
  c->launches += n;
}

// all tiles (128 x 256) that intersect the lower triangle of [0, rpad)^2 and touch a training row or column.
// Order matters for L2 reuse when one genome's panel is larger than L2 (config 4: 800 MB): the persistent CTAs
// take consecutive list entries, so the list walks super-blocks of 12 x 6 tiles (1 536 x 1 536 entries): the ~148
// tiles in flight then share 12 A row-blocks and 6 B row-blocks instead of streaming one long tile row.
void build_tiles(int rpad, const std::vector<unsigned char>& has_train, std::vector<int>& tiles, int bn = TB_GRAM_BN,
                 bool pairs = false) {
  tiles.clear();
  if (pairs) {
    // items for the paired Gram kernel: row blocks (I, I + 1) x column block J, listed when either tile is needed
    const int nI = rpad / TB_GRAM_BM, nJ = (rpad + bn - 1) / bn;
    auto need = [&](int I, int J) {
      if (I >= nI || J * bn > I * TB_GRAM_BM + TB_GRAM_BM - 1) return false;
      if (has_train.empty() || has_train[I]) return true;
      for (int blk = J * bn / TB_GRAM_BM; blk <= (J * bn + bn - 1) / TB_GRAM_BM; ++blk)
        if (blk < nI && has_train[blk]) return true;
      return false;
    };
    const int SBI = 12, SBJ = 6;
    for (int I0 = 0; I0 < nI; I0 += SBI)
      for (int J0 = 0; J0 < nJ; J0 += SBJ)
        for (int I = I0; I < std::min(nI, I0 + SBI); I += 2)
          for (int J = J0; J < std::min(nJ, J0 + SBJ); ++J)
            if (need(I, J) || need(I + 1, J)) tiles.push_back((I << 16) | J);
    return;
  }
  const int nI = rpad / TB_GRAM_BM, nJ = (rpad + bn - 1) / bn;
  const int SBI = 12, SBJ = 6;
  for (int I0 = 0; I0 < nI; I0 += SBI) {
    for (int J0 = 0; J0 < nJ; J0 += SBJ) {
      for (int I = I0; I < std::min(nI, I0 + SBI); ++I) {
        for (int J = J0; J < std::min(nJ, J0 + SBJ); ++J) {
          if (J * bn > I * TB_GRAM_BM + TB_GRAM_BM - 1) continue;
          bool need = has_train.empty() || has_train[I];
          for (int blk = J * bn / TB_GRAM_BM; blk <= (J * bn + bn - 1) / TB_GRAM_BM && !need; ++blk)
            if (blk < nI && has_train[blk]) need = true;
          if (need) tiles.push_back((I << 16) | J);
        }
      }
    }
  }
}

int ensure_ws(TbCtx* c, size_t bytes) {
  if (bytes <= c->ws_bytes) return 0;
  if (c->ws) cudaFree(c->ws);
  c->ws = nullptr;
  c->ws_bytes = 0;
  TB_CUDA(c, cudaMalloc(&c->ws, bytes));
  c->ws_bytes = bytes;
  return 0;
}

struct MarkCtx {
  TbCtx* c;
  size_t open;
  int n_update = 0;
};
void mark_cb(void* p, int which, int end) {
  MarkCtx* m = static_cast<MarkCtx*>(p);
  if (!end) {
    m->open = span_begin(m->c, which == 0 ? TB_ST_CHOL_UPDATE : TB_ST_CHOL_PANEL);
    if (which == 0) m->n_update++;
  } else {
    span_end(m->c, m->open);
  }
}

int fp64_fallback(TbCtx* c, const int32_t* slots, int n_slots, double h2, int mode_rule, double* d_fit, double* d_alpha);

// d_alpha [P][ntp] (one row set): rows [w0, w0 + Wc) <- the solutions of the wave just solved.  Entry i of a job's
// vector belongs to training animal i of the row set, d_tpos[i], on every layout: the solves index alpha by training
// position and reach the universe row through tpos (prefix, aligned hole) or through the panel permutation, where
// d_ident[i] = i is panel row rowmap[d_tpos[i]] = i.  With one row set the arena places the vectors at one stride.
int copy_alpha(TbCtx* c, double* d_alpha, int w0, int Wc, int ntp) {
  const std::vector<double*>& al = c->dbg.alpha;
  const ptrdiff_t stride = Wc > 1 ? al[1] - al[0] : ntp;
  bool uniform = stride >= ntp;
  for (int w = 1; w < Wc && uniform; ++w) uniform = al[w] - al[w - 1] == stride;
  if (uniform) {
    TB_CUDA(c, cudaMemcpy2DAsync(d_alpha + (size_t)w0 * ntp, (size_t)ntp * sizeof(double), al[0], (size_t)stride * sizeof(double),
                                 (size_t)ntp * sizeof(double), (size_t)Wc, cudaMemcpyDeviceToDevice, c->stream));
    return 0;
  }
  for (int w = 0; w < Wc; ++w)
    TB_CUDA(c, cudaMemcpyAsync(d_alpha + (size_t)(w0 + w) * ntp, al[w], (size_t)ntp * sizeof(double),
                               cudaMemcpyDeviceToDevice, c->stream));
  return 0;
}

struct SlotView {
  const TbRowSet* rs;
  size_t m_elems, linv_elems;
};

// d_alpha (nullable, one row set only): [P][ntp] device destination of every genome's solution (see copy_alpha)
// reml (nullable): the "row sets" are reml->n copies of one row set, one per h2 point of the profile; each job gets its
// own lambda, an fp64 A of ntp x ntp only (no G_vt rows) and reml_kernel instead of the solve (d_fit and h2 unused)
int eval_core(TbCtx* c, const int32_t* slots, int n_slots, double h2, int mode_rule, double* d_fit,
              bool allow_fallback = true, double* d_alpha = nullptr, const TbRemlReq* reml = nullptr) {
  const auto t_host0 = std::chrono::steady_clock::now();
  if (c->P <= 0) return fail(c, "tb_eval_staged: no genomes staged");
  if (n_slots <= 0 || n_slots > TB_MAX_SLOTS) return fail(c, "tb_eval_staged: bad n_slots");
  if (d_alpha && n_slots != 1) return fail(c, "internal: solutions are kept for one row set only");
  if (reml && (d_alpha || reml->n != n_slots)) return fail(c, "internal: bad REML request");
  if (!reml && (!(h2 > 0.0) || !(h2 <= 1.0))) return fail(c, "tb_eval_staged: heritability must be in (0, 1]");
  if (mode_rule < 0 || mode_rule > 2) return fail(c, "tb_eval_staged: bad mode_rule");
  const double lambda = (1.0 - h2) / h2;   // tblup/evaluator.py:277
  std::vector<SlotView> sv(n_slots);
  int rpad = 0, max_ntp = 0, max_rows = 0;
  std::vector<unsigned char> has_train;
  size_t per_ind = 0;
  for (int s = 0; s < n_slots; ++s) {
    if (slots[s] < 0 || slots[s] >= TB_MAX_SLOTS || !c->slots[slots[s]].valid)
      return fail(c, "tb_eval_staged: row set " + std::to_string(slots[s]) + " is not defined");
    const TbRowSet* rs = &c->slots[slots[s]];
    sv[s].rs = rs;
    const int n_v = reml ? 0 : rs->n_v;              // REML forms A only
    sv[s].m_elems = (size_t)(rs->ntp + n_v) * rs->ntp;
    sv[s].linv_elems = (size_t)rs->ntp * TB_NB;
    rpad = std::max(rpad, rs->rpad);
    max_ntp = std::max(max_ntp, rs->ntp);
    max_rows = std::max(max_rows, rs->ntp + n_v);
    if (has_train.size() < rs->has_train.size()) has_train.resize(rs->has_train.size(), 0);
    for (size_t i = 0; i < rs->has_train.size(); ++i) has_train[i] |= rs->has_train[i];
    per_ind += (sv[s].m_elems + sv[s].linv_elems + rs->ntp + n_v) * sizeof(double) + (reml ? sizeof(TbRemlJob) : 0) + 1024;
  }
  has_train.resize(rpad / TB_GRAM_BM, 0);
  const int P = c->P;
  int kmax = 0;
  for (int i = 0; i < P; ++i) {
    const int k = (int)(c->h_off[i + 1] - c->h_off[i]);
    if (k <= 0) return fail(c, "tb_eval_staged: empty genome at position " + std::to_string(i));
    kmax = std::max(kmax, k);
  }
  // E2M1 Gram: needs the packed resident matrix (its gather is written for it); every sum is an integer <= 4 kmax,
  // exact in the fp32 accumulators below 2^24
  const bool fp4 = c->gram_fp4 && c->d_x2 != nullptr && 4LL * kmax < (1LL << 24);
  c->last_fp4 = fp4 ? 1 : 0;
  // a single scattered row set (Monte-Carlo split, unaligned fold, custom splitter): permute the panel rows at gather
  // time -- training animals first, validation animals next -- and everything downstream sees a plain prefix
  if (n_slots > 1 && !reml && c->perm_rows && fp4 && c->precision == 0 && c->stop_after < 0) {
    // Several row sets share one Gram only while each of them can run the contiguous kernels (a prefix, or -- int16
    // layout -- a prefix with one aligned hole).  Otherwise the refinement would fall back to per-element position
    // lookups (measured 14x slower per solve than a whole extra Gram): evaluate the row sets one at a time instead,
    // each as a prefix of its own permuted panel.
    const bool c16_possible = c->narrow_c && 4LL * kmax <= 32767;
    bool split = false;
    for (int s = 0; s < n_slots; ++s) {
      const TbRowSet* rs = sv[s].rs;
      const bool fast = (rs->contiguous && rs->n_t % 4 == 0) || (c16_possible && rs->seg_ok);
      split = split || (!fast && rs->perm_ok);
    }
    if (split) {
      if ((size_t)P > c->split_cap) {
        TB_CUDA(c, cudaStreamSynchronize(c->stream));
        cudaFree(c->d_split);
        c->d_split = nullptr;
        c->split_cap = 0;
        TB_CUDA(c, cudaMalloc(&c->d_split, (size_t)P * sizeof(double)));
        c->split_cap = (size_t)P;
      }
      int fallbacks = 0;
      for (int s = 0; s < n_slots; ++s) {
        if (int rc = eval_core(c, slots + s, 1, h2, mode_rule, c->d_split, allow_fallback)) return rc;
        fallbacks += c->last_fallbacks;
        TB_CUDA(c, cudaMemcpy2DAsync(d_fit + s, (size_t)n_slots * sizeof(double), c->d_split, sizeof(double),
                                     sizeof(double), (size_t)P, cudaMemcpyDeviceToDevice, c->stream));
      }
      c->last_fallbacks = fallbacks;
      c->last_split = 1;
      return 0;
    }
  }
  if (n_slots > 1) c->last_split = 0;
  const bool use_perm = (n_slots == 1 || reml) && c->perm_rows && fp4 && !sv[0].rs->contiguous && sv[0].rs->perm_ok;
  c->last_perm = use_perm ? 1 : 0;
  if (use_perm) {
    const TbRowSet* rs = sv[0].rs;
    rpad = tb_round_up(rs->n_t + rs->n_v, TB_GRAM_BM);
    has_train.assign(rpad / TB_GRAM_BM, 0);
    for (int blk = 0; blk * TB_GRAM_BM < rs->n_t; ++blk) has_train[blk] = 1;
  }
  // the mixed path turns cross-products (<= 4 k) into floats through the 2^23 mantissa trick: 4 kmax < 2^23
  // (REML always runs the fp64 Cholesky: the 10-bit factor would put an error of order n 1e-3 into log|A|)
  bool mixed = !reml && c->precision == 0 && tb_solve_mixed_fits(max_ntp) && 4LL * kmax < (1LL << 23);
  for (int s = 0; s < n_slots; ++s) mixed = mixed && sv[s].rs->ntp == max_ntp;
  c->last_mixed = mixed ? 1 : 0;
  if (allow_fallback) c->last_fallbacks = 0;
  if (mixed) {
    const size_t need = (size_t)P * n_slots;
    if (need > c->fail_cap) {
      TB_CUDA(c, cudaStreamSynchronize(c->stream));
      cudaFree(c->d_fail);
      c->d_fail = nullptr;
      c->fail_cap = 0;
      TB_CUDA(c, cudaMalloc(&c->d_fail, need * sizeof(int)));
      c->fail_cap = need;
    }
    TB_CUDA(c, cudaMemsetAsync(c->d_fail, 0, need * sizeof(int), c->stream));
    per_ind = 0;
    for (int s = 0; s < n_slots; ++s)
      per_ind += (size_t)max_ntp * max_ntp * (sizeof(float) + 2) + (size_t)max_ntp * (TB_NB + 2) * sizeof(float) + 256 +
                 (size_t)256 * 256 * sizeof(float) +
                 (size_t)(max_ntp + sv[s].rs->n_v) * sizeof(double) + 1024;
  }
  // one contiguous row set: the Gram epilogue writes the fp32 matrix itself (no separate scaling pass over C)
  const bool fuse_scale = mixed && n_slots == 1 && (sv[0].rs->contiguous || use_perm) && c->n <= 46340 && c->fuse_scale;
  // the scaled fp32 matrix is not written by a pass of its own when every row set is a prefix of the panel rows or a
  // prefix with one aligned hole (k-fold training sets): the Cholesky updates form it from C block column by block column
  bool from_c_ok = mixed && c->n <= 46340 && c->fuse_scale;
  for (int s = 0; s < n_slots; ++s)
    from_c_ok = from_c_ok && (sv[s].rs->contiguous || (n_slots == 1 && use_perm) || sv[s].rs->seg_ok) && sv[s].rs->n_t % 4 == 0;
  c->last_fused = (fuse_scale || from_c_ok) ? 1 : 0;
  const int kq = fp4 ? TB_GRAM_BK_FP4 : TB_GRAM_BK;      // markers per k-block
  const int kstride_max = tb_round_up(kmax, kq);
  // every cross-product is at most 4 k: int16 storage is exact for the whole batch when 4 kmax <= 32 767
  const bool c16 = mixed && c->narrow_c && 4LL * kmax <= 32767;
  c->last_c16 = c16 ? 1 : 0;
  per_ind += (size_t)rpad * kstride_max + (size_t)rpad * rpad * sizeof(int32_t) +
             (size_t)n_slots * (rpad + 2) * sizeof(long long) + (size_t)n_slots * kstride_max * sizeof(int) + 4096;

  const size_t fixed = (size_t)128 * kstride_max + (size_t)P * n_slots * 512 + (size_t)128 * max_ntp * sizeof(float) + (1 << 20);
  const int want = std::max(1, std::min(c->max_wave > 0 ? std::min(P, c->max_wave) : P, 1024));
  size_t budget;
  if (!c->ws_limit && fixed + per_ind * (size_t)want <= c->ws_bytes) {
    budget = c->ws_bytes;                          // the arena already holds the whole batch: no driver query needed
  } else {
    size_t free_b = 0, total_b = 0;
    TB_CUDA(c, cudaMemGetInfo(&free_b, &total_b));
    budget = c->ws_limit ? c->ws_limit : (size_t)((double)(free_b + c->ws_bytes) * 0.80);
  }
  if (budget < fixed + per_ind) budget = fixed + per_ind;
  long long Wll = (long long)((budget - fixed) / per_ind);
  int W = (int)std::min<long long>(Wll, P);
  if (c->max_wave > 0) W = std::min(W, c->max_wave);
  W = std::max(1, std::min(W, 1024));
  if (reml) W = std::max(1, std::min(W, 65535 / n_slots));   // jobs of a wave index gridDim.y of the Cholesky GEMMs
  c->last_wave = W;
  if (int rc = ensure_ws(c, fixed + per_ind * (size_t)W)) return rc;

  cudaStream_t st = c->stream;
  // tile list + genome offsets (device copies live at the start of the arena)
  std::vector<int> tiles;
  const int gram_pair = (fuse_scale && c->fuse_in_gram) ? 0 : c->gram_pair;     // 0 single CTA, 1 multicast pair, 2 tcgen05 CTA pair
  build_tiles(rpad, has_train, tiles, fp4 ? TB_GRAM_BN_FP4 : TB_GRAM_BN, gram_pair != 0);
  const int n_tiles = (int)tiles.size();

  Arena ar;
  ar.base = (char*)c->ws;
  ar.cap = c->ws_bytes;
  int* d_tiles = ar.take<int>(tiles.size());
  long long* d_off = ar.take<long long>(P + 1);
  TB_CUDA(c, cudaMemcpyAsync(d_tiles, tiles.data(), tiles.size() * sizeof(int), cudaMemcpyHostToDevice, st));
  TB_CUDA(c, cudaMemcpyAsync(d_off, c->h_off.data(), (P + 1) * sizeof(long long), cudaMemcpyHostToDevice, st));
  const size_t arena_mark = ar.off;

  std::vector<TbScaleJob> h_scale;
  std::vector<TbCholJob> h_chol;
  std::vector<TbSolveJob> h_solve;
  std::vector<TbSolveMixedJob> h_msolve;
  std::vector<const int*> h_cs;
  std::vector<int> h_kb;
  std::vector<TbRemlJob> h_reml;

  for (int w0 = 0; w0 < P; w0 += W) {
    const int Wc = std::min(W, P - w0);
    const int n_jobs = Wc * n_slots;
    int kw = 0;
    h_kb.resize(Wc);
    for (int w = 0; w < Wc; ++w) {
      const int k = (int)(c->h_off[w0 + w + 1] - c->h_off[w0 + w]);
      kw = std::max(kw, k);
      h_kb[w] = tb_round_up(k, kq) / kq;
    }
    const int kstride = tb_round_up(kw, kq);             // markers
    const int kstride_b = fp4 ? kstride / 2 : kstride;    // bytes of one panel row

    ar.off = arena_mark;
    int8_t* d_panel = ar.take<int8_t>(((size_t)Wc * rpad + 128) * kstride_b);
    int32_t* d_C = ar.take<int32_t>((size_t)Wc * rpad * rpad);
    long long* d_s = ar.take<long long>((size_t)n_jobs * rpad);
    long long* d_SQ = ar.take<long long>((size_t)n_jobs * 2);
    int* d_csg = ar.take<int>((size_t)n_jobs * kstride);
    int* d_status = ar.take<int>(n_jobs);
    int* d_kb = ar.take<int>(Wc);
    const int** d_cs = ar.take<const int*>(n_jobs);
    TbScaleJob* d_scale = ar.take<TbScaleJob>(n_jobs);
    TbCholJob* d_chol = ar.take<TbCholJob>(n_jobs);
    TbSolveJob* d_solve = ar.take<TbSolveJob>(n_jobs);
    TbSolveMixedJob* d_msolve = ar.take<TbSolveMixedJob>(n_jobs);
    int* d_sweeps = ar.take<int>(n_jobs);
    TbRemlJob* d_reml = reml ? ar.take<TbRemlJob>(n_jobs) : nullptr;
    float* d_L32 = nullptr;
    float* d_Linv32 = nullptr;
    unsigned short* d_L16 = nullptr;
    float* d_Linv256 = nullptr;
    float* d_terms = nullptr;
    TbFuseCoef* d_coef = nullptr;
    if (mixed) {
      if (from_c_ok) {
        d_terms = ar.take<float>((size_t)n_jobs * 2 * max_ntp);
        d_coef = ar.take<TbFuseCoef>(n_jobs);
      }
      if (c->wide_panel) d_Linv256 = ar.take<float>((size_t)n_jobs * 256 * 256);
      d_L32 = ar.take<float>(((size_t)n_jobs * max_ntp + 128) * max_ntp);
      d_Linv32 = ar.take<float>((size_t)n_jobs * max_ntp * TB_NB);
      d_L16 = ar.take<unsigned short>((size_t)n_jobs * max_ntp * max_ntp);
    }

    h_scale.resize(n_jobs);
    h_chol.resize(n_jobs);
    h_solve.resize(n_jobs);
    h_msolve.resize(n_jobs);
    h_cs.resize(n_jobs);
    if (reml) h_reml.resize(n_jobs);
    c->dbg.L32 = d_L32;
    c->dbg.L16 = d_L16;
    c->dbg.Linv32 = d_Linv32;
    c->dbg.sweeps = d_sweeps;
    c->dbg.ntp_all = max_ntp;
    c->dbg.W = Wc;
    c->dbg.n_slots = n_slots;
    c->dbg.rpad = rpad;
    c->dbg.kstride = kstride;
    c->dbg.C = d_C;
    c->dbg.s = d_s;
    c->dbg.SQ = d_SQ;
    c->dbg.M.assign(n_jobs, nullptr);
    c->dbg.alpha.assign(n_jobs, nullptr);
    c->dbg.pred.assign(n_jobs, nullptr);
    c->dbg.ntp.assign(n_jobs, 0);
    c->dbg.n_v.assign(n_jobs, 0);
    // the centring terms depend on the row set only through the frequency animals: when every genome of the wave
    // takes the gblup branch (all-animal frequencies) one set of terms per genome serves all its row sets
    bool wave_all_gblup = true;
    for (int w = 0; w < Wc; ++w) {
      const int k = (int)(c->h_off[w0 + w + 1] - c->h_off[w0 + w]);
      wave_all_gblup = wave_all_gblup && (mode_rule == TB_MODE_GBLUP || (mode_rule == TB_MODE_AUTO && k > c->n));
    }
    // (the REML jobs of a genome all sit on one row set: one set of terms per genome whatever the branch)
    const bool centre_shared = wave_all_gblup || reml;
    const int centre_slots = centre_shared ? 1 : n_slots;
    c->dbg.centre_shared = centre_shared ? 1 : 0;
    for (int w = 0; w < Wc; ++w) {
      const int k = (int)(c->h_off[w0 + w + 1] - c->h_off[w0 + w]);
      const bool gblup = mode_rule == TB_MODE_GBLUP || (mode_rule == TB_MODE_AUTO && k > c->n);
      for (int s = 0; s < n_slots; ++s) {
        const int job = w * n_slots + s;
        const int cjob = centre_shared ? w : job;       // index of this job's centring terms
        const TbRowSet* rs = sv[s].rs;
        const int n_v = reml ? 0 : rs->n_v;
        double* Mj = mixed ? nullptr : ar.take<double>(sv[s].m_elems);
        double* Lj = mixed ? nullptr : ar.take<double>(sv[s].linv_elems);
        double* aj = ar.take<double>(rs->ntp);
        double* pj = ar.take<double>(n_v);
        double lambda_j = lambda;
        if (reml) {
          const double h2j = reml->h2[(size_t)(w0 + w) * reml->ld + reml->s0 + s];
          lambda_j = (1.0 - h2j) / h2j;
          const size_t o = (size_t)(w0 + w) * reml->n_out + reml->s0 + s;
          h_reml[job] = TbRemlJob{Mj, Lj, rs->d_yt_ctr, d_status + job, rs->yt_mean, rs->n_t, rs->ntp,
                                  reml->d_loglik + o, reml->d_sigma_g2 + o, reml->d_mu + o};
        }
        h_cs[cjob] = gblup ? c->d_colsum_all : rs->d_colsum_train;
        TbScaleJob& sj = h_scale[job];
        sj.C = c16 ? reinterpret_cast<const int32_t*>(reinterpret_cast<const int16_t*>(d_C) + (size_t)w * rpad * rpad)
                   : d_C + (size_t)w * rpad * rpad;
        sj.s = d_s + (size_t)cjob * rpad;
        sj.SQ = d_SQ + (size_t)cjob * 2;
        sj.tpos = use_perm ? rs->d_ident : rs->d_tpos;
        sj.vpos = use_perm ? rs->d_ident + rs->n_t : rs->d_vpos;
        sj.M = Mj;
        sj.N = gblup ? c->n : rs->n_t;
        sj.n_t = rs->n_t;
        sj.n_v = n_v;
        sj.ntp = rs->ntp;
        sj.rpad = rpad;
        sj.lambda = lambda_j;
        sj.hole0 = use_perm ? rs->n_t : rs->hole0;
        sj.gap = use_perm ? 0 : rs->gap;
        sj.cw = w;
        TbCholJob& cj = h_chol[job];
        cj.M = Mj;
        cj.Linv = Lj;
        cj.ntp = rs->ntp;
        cj.status = d_status + job;
        TbSolveJob& oj = h_solve[job];
        oj.M = Mj;
        oj.Linv = Lj;
        oj.y_t = gblup ? rs->d_yt_raw : rs->d_yt_ctr;
        oj.y_v = rs->d_yv;
        oj.status = d_status + job;
        oj.alpha = aj;
        oj.pred = pj;
        oj.fitness = d_fit ? d_fit + (size_t)(w0 + w) * n_slots + s : nullptr;
        oj.n_t = rs->n_t;
        oj.n_v = n_v;
        oj.ntp = rs->ntp;
        TbSolveMixedJob& mj = h_msolve[job];
        mj.L32 = d_L32 ? d_L32 + (size_t)job * max_ntp * max_ntp : nullptr;
        mj.L16 = d_L16 ? d_L16 + (size_t)job * max_ntp * max_ntp : nullptr;
        mj.Linv32 = d_Linv32 ? d_Linv32 + (size_t)job * max_ntp * TB_NB : nullptr;
        mj.C = sj.C;
        mj.s = sj.s;
        mj.SQ = sj.SQ;
        mj.tpos = sj.tpos;
        mj.vpos = sj.vpos;
        mj.y_t = oj.y_t;
        mj.y_v = oj.y_v;
        mj.status = d_status + job;
        mj.alpha = aj;
        mj.pred = pj;
        mj.fitness = oj.fitness;
        mj.sweeps = d_sweeps + job;
        mj.fail = mixed ? c->d_fail + (size_t)(w0 + w) * n_slots + s : nullptr;
        mj.N = sj.N;
        mj.n_t = rs->n_t;
        mj.n_v = rs->n_v;
        mj.ntp = rs->ntp;
        mj.rpad = rpad;
        mj.hole0 = use_perm ? rs->n_t : rs->hole0;
        mj.gap = use_perm ? 0 : rs->gap;
        mj.valid_in_hole = (!use_perm && rs->valid_in_hole) ? 1 : 0;
        mj.lambda = lambda;
        mj.cmax = 4 * k;
        c->dbg.M[job] = Mj;
        c->dbg.alpha[job] = aj;
        c->dbg.pred[job] = pj;
        c->dbg.ntp[job] = rs->ntp;
        c->dbg.n_v[job] = n_v;
      }
    }
    if (ar.off > ar.cap) return fail(c, "internal: wave workspace overflow");

    size_t sp = span_begin(c, TB_ST_H2D);
    TB_CUDA(c, cudaMemcpyAsync(d_kb, h_kb.data(), Wc * sizeof(int), cudaMemcpyHostToDevice, st));
    TB_CUDA(c, cudaMemcpyAsync(d_cs, h_cs.data(), n_jobs * sizeof(int*), cudaMemcpyHostToDevice, st));
    TB_CUDA(c, cudaMemcpyAsync(d_scale, h_scale.data(), n_jobs * sizeof(TbScaleJob), cudaMemcpyHostToDevice, st));
    TB_CUDA(c, cudaMemcpyAsync(d_chol, h_chol.data(), n_jobs * sizeof(TbCholJob), cudaMemcpyHostToDevice, st));
    TB_CUDA(c, cudaMemcpyAsync(d_solve, h_solve.data(), n_jobs * sizeof(TbSolveJob), cudaMemcpyHostToDevice, st));
    TB_CUDA(c, cudaMemcpyAsync(d_msolve, h_msolve.data(), n_jobs * sizeof(TbSolveMixedJob), cudaMemcpyHostToDevice, st));
    if (reml) TB_CUDA(c, cudaMemcpyAsync(d_reml, h_reml.data(), n_jobs * sizeof(TbRemlJob), cudaMemcpyHostToDevice, st));
    TB_CUDA(c, cudaMemsetAsync(d_status, 0, n_jobs * sizeof(int), st));
    span_end(c, sp);

    sp = span_begin(c, TB_ST_GATHER);
    if (fp4)
      TB_CUDA(c, tb_launch_gather_fp4(c->geno(), c->d_idx, d_off, w0, Wc, rpad, kstride_b, d_panel, st,
                                      use_perm ? sv[0].rs->d_rowmap : nullptr, use_perm ? sv[0].rs->rows_univ : 0));
    else
      TB_CUDA(c, tb_launch_gather(c->geno(), c->d_idx, d_off, w0, Wc, rpad, kstride, d_panel, st));
    span_end(c, sp);
    count(c, TB_ST_GATHER, 1);
    if (c->stop_after == TB_ST_GATHER) continue;

    sp = span_begin(c, TB_ST_CENTRE);
    TB_CUDA(c, tb_launch_centre_terms(d_panel, rpad, kstride, c->d_idx, d_off, w0, Wc, centre_slots, d_kb, d_cs, d_csg, d_s, d_SQ, st, fp4 ? (c->n <= 32767 ? 2 : 1) : 0));
    span_end(c, sp);
    count(c, TB_ST_CENTRE, 2);
    if (c->stop_after == TB_ST_CENTRE) continue;

    sp = span_begin(c, TB_ST_GRAM);
    {
      std::string e;
      // (the Gram no longer writes the scaled matrix: with fuse_scale the Cholesky updates form it from C on the fly)
      cudaError_t ce = tb_launch_gram_tc(d_panel, Wc, rpad, kstride_b, d_kb, d_tiles, n_tiles, d_C, c->n_sm, st, &e,
                                         (fuse_scale && c->fuse_in_gram) ? d_scale : nullptr, d_L32,
                                         c->gram_experiment ? -c->gram_experiment : max_ntp, c16 ? 1 : 0, fp4 ? 1 : 0, gram_pair);
      if (ce != cudaSuccess) return fail(c, "gram launch: " + (e.empty() ? std::string(cudaGetErrorString(ce)) : e), -2);
    }
    span_end(c, sp);
    count(c, TB_ST_GRAM, 1);
    if (c->stop_after == TB_ST_GRAM) continue;

    if (mixed) {
      const bool from_c = from_c_ok && !(fuse_scale && c->fuse_in_gram) && c->stop_after < 0;
      TbFromC fc{};
      if (!(fuse_scale && c->fuse_in_gram)) {
        sp = span_begin(c, TB_ST_SCALE);
        if (from_c) {
          // every block column (the first one included: a launch with K = 0) is formed inside the update kernel's epilogue
          TB_CUDA(c, tb_launch_fuse_terms(d_scale, n_jobs, max_ntp, d_terms, d_coef, st));
          if (c->blk0_scale32) TB_CUDA(c, tb_launch_scale32(d_scale, n_jobs, max_ntp, d_L32, c16 ? 1 : 0, st, 256));
          count(c, TB_ST_SCALE, c->blk0_scale32 ? 2 : 1);
          fc.skip_blk0 = c->blk0_scale32;
          fc.C = d_C;
          fc.terms = d_terms;
          fc.coef = d_coef;
          fc.rpad = rpad;
          fc.c16 = c16 ? 1 : 0;
        } else {
          TB_CUDA(c, tb_launch_scale32(d_scale, n_jobs, max_ntp, d_L32, c16 ? 1 : 0, st));
          count(c, TB_ST_SCALE, 1);
        }
        span_end(c, sp);
      }
      if (c->stop_after == TB_ST_SCALE) continue;
      {
        int nl[2] = {0, 0};
        std::string e;
        MarkCtx mc{c, 0};
        cudaError_t ce = tb_chol_tc_factor(d_L32, d_Linv32, d_L16, d_Linv256, d_status, n_jobs, max_ntp, c->n_sm, st, nl, &e,
                                           c->profile ? &mark_cb : nullptr, &mc, from_c ? &fc : nullptr, c->t16, c->epi_warps,
                                           (c->chain_fused < 0 ? c->n_sm : c->chain_fused) * (c->chain_inverse ? 1 : -1),
                                           c->panel_fused);
        if (ce != cudaSuccess)
          return fail(c, "tensor-core Cholesky: " + (e.empty() ? std::string(cudaGetErrorString(ce)) : e), -2);
        count(c, TB_ST_CHOL_UPDATE, mc.n_update);
        count(c, TB_ST_CHOL_PANEL, nl[0] + nl[1] - mc.n_update);
      }
      if (c->stop_after == TB_ST_CHOL_UPDATE || c->stop_after == TB_ST_CHOL_PANEL) continue;
      sp = span_begin(c, TB_ST_SOLVE);
      // contiguous kernels: every row set is a prefix of the universe, or (int16 layout) a prefix with one aligned hole
      bool contig = true, hole = false;
      for (int s = 0; s < n_slots; ++s) {
        contig = contig && (((sv[s].rs->contiguous || use_perm) && sv[s].rs->n_t % 4 == 0) || (c16 && sv[s].rs->seg_ok));
        hole = hole || (!use_perm && sv[s].rs->gap > 0);
      }
      TB_CUDA(c, tb_launch_solve_mixed(d_msolve, n_jobs, max_ntp, contig ? 1 : 0, c16 ? 1 : 0, hole ? 1 : 0, st, c->n_sm,
                                       c->solve_pair));
      span_end(c, sp);
      count(c, TB_ST_SOLVE, 1);
      if (d_alpha)
        if (int rc = copy_alpha(c, d_alpha, w0, Wc, max_ntp)) return rc;
      continue;
    }

    sp = span_begin(c, TB_ST_SCALE);
    TB_CUDA(c, tb_launch_scale(d_scale, n_jobs, max_rows, max_ntp, st));
    span_end(c, sp);
    count(c, TB_ST_SCALE, 1);
    if (c->stop_after == TB_ST_SCALE) continue;

    const int nb = max_ntp / TB_NB;
    for (int j = 0; j < nb; ++j) {
      if (j > 0) {
        sp = span_begin(c, TB_ST_CHOL_UPDATE);
        TB_CUDA(c, tb_launch_chol_update(d_chol, n_jobs, max_ntp, j, st));
        span_end(c, sp);
        count(c, TB_ST_CHOL_UPDATE, 1);
      }
      sp = span_begin(c, TB_ST_CHOL_PANEL);
      TB_CUDA(c, tb_launch_chol_diag(d_chol, n_jobs, max_ntp, j, st));
      count(c, TB_ST_CHOL_PANEL, 1);
      if (j + 1 < nb) {
        TB_CUDA(c, tb_launch_chol_panel(d_chol, n_jobs, max_ntp, j, st));
        count(c, TB_ST_CHOL_PANEL, 1);
      }
      span_end(c, sp);
    }
    if (c->stop_after == TB_ST_CHOL_UPDATE || c->stop_after == TB_ST_CHOL_PANEL) continue;

    sp = span_begin(c, TB_ST_SOLVE);
    if (reml) {                                      // log|A|, the forward substitution of [y_T, 1] and the profile
      TB_CUDA(c, tb_launch_reml(d_reml, n_jobs, max_ntp, st));
      span_end(c, sp);
      count(c, TB_ST_SOLVE, 1);
      continue;
    }
    TB_CUDA(c, tb_launch_solve(d_solve, n_jobs, max_ntp, st));
    span_end(c, sp);
    count(c, TB_ST_SOLVE, 1);
    if (d_alpha)
      if (int rc = copy_alpha(c, d_alpha, w0, Wc, max_ntp)) return rc;
  }
  // host time spent issuing the evaluation (everything above is asynchronous): diagnostics, "last_issue_us"
  c->last_issue_us = (long long)std::chrono::duration_cast<std::chrono::microseconds>(
                         std::chrono::steady_clock::now() - t_host0).count();
  if (mixed && allow_fallback && c->stop_after < 0 && !c->no_fallback) return fp64_fallback(c, slots, n_slots, h2, mode_rule, d_fit, d_alpha);
  return 0;
}

// Jobs whose mixed-precision solve gave up (pivot breakdown of the low-precision factor or no convergence of the
// refinement: lambda -> 0, i.e. h2 -> 1, makes A ill-conditioned) are evaluated again with the fp64 Cholesky, which
// is what the reference's fp64 inverse (tblup/evaluator.py:282) can still handle.  One small D2H of the flags per
// evaluation; in the normal case nothing else happens.
int fp64_fallback(TbCtx* c, const int32_t* slots, int n_slots, double h2, int mode_rule, double* d_fit, double* d_alpha) {
  const int P = c->P;
  std::vector<int> h_fail((size_t)P * n_slots);
  TB_CUDA(c, cudaMemcpyAsync(h_fail.data(), c->d_fail, h_fail.size() * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  TB_CUDA(c, cudaStreamSynchronize(c->stream));
  std::vector<int> redo;
  int n_failed = 0;
  for (int i = 0; i < P; ++i) {
    bool any = false;
    for (int s = 0; s < n_slots; ++s) {
      any = any || h_fail[(size_t)i * n_slots + s] != 0;
      n_failed += h_fail[(size_t)i * n_slots + s] != 0;
    }
    if (any) redo.push_back(i);
  }
  if (redo.empty()) return 0;
  spans_collect(c);                                  // the recursive evaluation reuses the event pool
  std::vector<long long> sub_off(redo.size() + 1, 0);
  for (size_t j = 0; j < redo.size(); ++j) sub_off[j + 1] = sub_off[j] + (c->h_off[redo[j] + 1] - c->h_off[redo[j]]);
  int* d_sub = nullptr;
  double* d_subfit = nullptr;
  double* d_subalpha = nullptr;                      // [redo][ntp] solutions of the sub-batch (kept alpha only)
  const int ntp = d_alpha ? c->slots[slots[0]].ntp : 0;
  TB_CUDA(c, cudaMalloc(&d_sub, (size_t)sub_off.back() * sizeof(int)));
  if (cudaMalloc(&d_subfit, redo.size() * n_slots * sizeof(double)) != cudaSuccess ||
      (d_alpha && cudaMalloc(&d_subalpha, redo.size() * ntp * sizeof(double)) != cudaSuccess)) {
    cudaFree(d_sub);
    cudaFree(d_subfit);
    return fail(c, "fp64 fallback: out of memory", -2);
  }
  for (size_t j = 0; j < redo.size(); ++j)
    cudaMemcpyAsync(d_sub + sub_off[j], c->d_idx + c->h_off[redo[j]],
                    (size_t)(sub_off[j + 1] - sub_off[j]) * sizeof(int), cudaMemcpyDeviceToDevice, c->stream);
  // evaluate the sub-batch as the staged batch, in fp64, then put everything back
  std::vector<long long> keep_off;
  keep_off.swap(c->h_off);
  int* keep_idx = c->d_idx;
  const size_t keep_cap = c->idx_cap;
  const int keep_P = c->P, keep_prec = c->precision;
  const int keep_c16 = c->last_c16, keep_fused = c->last_fused, keep_fp4 = c->last_fp4, keep_wave = c->last_wave;
  c->h_off = sub_off;
  c->d_idx = d_sub;
  c->idx_cap = (size_t)sub_off.back();
  c->P = (int)redo.size();
  c->precision = 1;
  int rc = eval_core(c, slots, n_slots, h2, mode_rule, d_subfit, false, d_subalpha);
  c->precision = keep_prec;
  c->P = keep_P;
  c->d_idx = keep_idx;
  c->idx_cap = keep_cap;
  c->h_off.swap(keep_off);
  c->last_mixed = 1;
  c->last_c16 = keep_c16;
  c->last_fused = keep_fused;
  c->last_fp4 = keep_fp4;
  c->last_wave = keep_wave;
  if (rc == 0) {
    for (size_t j = 0; j < redo.size(); ++j)
      for (int s = 0; s < n_slots; ++s)
        if (h_fail[(size_t)redo[j] * n_slots + s])
          cudaMemcpyAsync(d_fit + (size_t)redo[j] * n_slots + s, d_subfit + j * n_slots + s, sizeof(double),
                          cudaMemcpyDeviceToDevice, c->stream);
    if (d_alpha)                                     // one row set: every redone genome failed on it
      for (size_t j = 0; j < redo.size(); ++j)
        cudaMemcpyAsync(d_alpha + (size_t)redo[j] * ntp, d_subalpha + j * ntp, (size_t)ntp * sizeof(double),
                        cudaMemcpyDeviceToDevice, c->stream);
  }
  cudaError_t se = cudaStreamSynchronize(c->stream);
  cudaFree(d_sub);
  cudaFree(d_subfit);
  cudaFree(d_subalpha);
  if (rc) return rc;
  if (se != cudaSuccess) return fail(c, std::string("fp64 fallback: ") + cudaGetErrorString(se), -2);
  c->last_fallbacks = n_failed;
  return 0;
}

}  // namespace

int tb_internal_eval_device(TbCtx* c, const int32_t* slots, int n_slots, double h2, int mode_rule, double* d_fit) {
  return eval_core(c, slots, n_slots, h2, mode_rule, d_fit);
}
int tb_internal_eval_alpha(TbCtx* c, int slot, double h2, int mode_rule, double* d_fit, double* d_alpha) {
  return eval_core(c, &slot, 1, h2, mode_rule, d_fit, true, d_alpha);
}
int tb_internal_eval_reml(TbCtx* c, int slot, int mode_rule, const TbRemlReq* req) {
  if (!req || req->n < 1 || req->n > TB_MAX_SLOTS) return fail(c, "internal: bad REML request");
  const std::vector<int32_t> slots(req->n, slot);
  return eval_core(c, slots.data(), req->n, 0.0, mode_rule, nullptr, false, nullptr, req);
}
void tb_internal_collect_spans(TbCtx* c) { spans_collect(c); }

extern "C" {

int tb_abi_version(void) { return TB_ABI_VERSION; }

const char* tb_last_error(const tb_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }

int tb_create(const int8_t* geno, int n, int m, const double* y, const int32_t* perm, int device, tb_ctx** out) {
  return tb_create_ex(geno, TB_LAYOUT_INT8_ANIMAL_MAJOR, TB_STORE_INT8, n, m, y, perm, device, out);
}

int tb_create_ex(const void* geno_any, int layout, int storage, int n, int m, const double* y, const int32_t* perm,
                 int device, tb_ctx** out) {
  if (!out) return -1;
  *out = nullptr;
  if (!geno_any || n <= 0 || m <= 0) {
    g_create_err = "tb_create: null or empty input";
    return -1;
  }
  if ((layout != TB_LAYOUT_INT8_ANIMAL_MAJOR && layout != TB_LAYOUT_PACKED2_SNP_MAJOR) ||
      (storage != TB_STORE_INT8 && storage != TB_STORE_PACKED2)) {
    g_create_err = "tb_create_ex: unknown layout or storage";
    return -1;
  }
  const int8_t* geno = static_cast<const int8_t*>(geno_any);
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    g_create_err = std::string("tb_create: no CUDA device (") + cudaGetErrorString(e) + "); there is no CPU fallback";
    return -3;
  }
  if (device < 0 || device >= ndev) {
    g_create_err = "tb_create: bad device ordinal";
    return -1;
  }
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  if (prop.major != 10) {
    g_create_err = std::string("tb_create: device '") + prop.name + "' is sm_" + std::to_string(prop.major) +
                   std::to_string(prop.minor) + "; this library is built for sm_100a only";
    return -3;
  }
  TbCtx* c = new TbCtx();
  auto bail = [&](const std::string& msg) {
    g_create_err = msg.empty() ? c->err : msg;
    tb_destroy(c);
    return -2;
  };
  c->device = device;
  c->n = n;
  c->m = m;
  c->ldn = tb_round_up(n, 128);
  c->storage = storage;
  c->n_sm = prop.multiProcessorCount;
  if (cudaSetDevice(device) != cudaSuccess) return bail("cudaSetDevice failed");
  std::vector<int> p(n);
  c->pos_of.assign(n, -1);
  for (int i = 0; i < n; ++i) {
    p[i] = perm ? perm[i] : i;
    if (p[i] < 0 || p[i] >= n || c->pos_of[p[i]] != -1) return bail("tb_create: perm is not a permutation of 0..n-1");
    c->pos_of[p[i]] = i;
  }
  c->has_pheno = y != nullptr;
  c->y_univ.assign(n, 0.0);
  if (y)
    for (int i = 0; i < n; ++i) c->y_univ[i] = y[p[i]];

  auto chk = [&](cudaError_t ce, const char* what) {
    if (ce == cudaSuccess) return false;
    c->err = std::string(what) + ": " + cudaGetErrorString(ce);
    return true;
  };
  if (chk(cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking), "cudaStreamCreate")) return bail("");
  c->stream = c->own_stream;
  if (chk(cudaMalloc(&c->d_x, (size_t)m * c->ldn), "cudaMalloc genotypes")) return bail("");
  if (chk(cudaMemsetAsync(c->d_x, 0, (size_t)m * c->ldn, c->stream), "memset")) return bail("");
  if (chk(cudaMalloc(&c->d_colsum_all, (size_t)m * sizeof(int)), "cudaMalloc colsum")) return bail("");

  bool bad_value = false, cuda_bad = false;
  if (layout == TB_LAYOUT_INT8_ANIMAL_MAJOR) {
    // upload in universe order, transposing chunks of animals to SNP-major on the device
    int chunk = (int)std::max<long long>(64, std::min<long long>(n, ((long long)256 << 20) / m));
    chunk = std::min(chunk, n);
    int8_t *h_stage = nullptr, *d_stage = nullptr;
    if (chk(cudaMallocHost(&h_stage, (size_t)chunk * m), "cudaMallocHost staging")) return bail("");
    if (chk(cudaMalloc(&d_stage, (size_t)chunk * m), "cudaMalloc staging")) {
      cudaFreeHost(h_stage);
      return bail("");
    }
    for (int p0 = 0; p0 < n && !cuda_bad && !bad_value; p0 += chunk) {
      const int rows = std::min(chunk, n - p0);
      // copy + validate the chunk with several host threads (the byte loop was the whole cost of creating a context at
      // config 4's 10 GB; rows are independent)
      const int nt = (int)std::max<size_t>(1, std::min<size_t>(16, std::min<size_t>(std::thread::hardware_concurrency(),
                                                                                  ((size_t)rows * m) >> 22)));
      std::vector<unsigned char> tmax(nt, 0);
      auto work = [&](int t) {
        unsigned char mx = 0;
        for (int r = t; r < rows; r += nt) {
          const int8_t* src = geno + (size_t)p[p0 + r] * m;
          int8_t* dst = h_stage + (size_t)r * m;
          memcpy(dst, src, (size_t)m);
          unsigned char rowmax = 0;
          for (int j = 0; j < m; ++j) rowmax = std::max(rowmax, (unsigned char)src[j]);   // negative values map to >= 128
          mx = std::max(mx, rowmax);
        }
        tmax[t] = mx;
      };
      {
        std::vector<std::thread> th;
        for (int t = 1; t < nt; ++t) th.emplace_back(work, t);
        work(0);
        for (auto& x : th) x.join();
      }
      unsigned char maxv = 0;
      for (int t = 0; t < nt; ++t) maxv = std::max(maxv, tmax[t]);
      if (maxv > 2) {
        bad_value = true;
        break;
      }
      cuda_bad |= chk(cudaMemcpyAsync(d_stage, h_stage, (size_t)rows * m, cudaMemcpyHostToDevice, c->stream), "H2D genotypes");
      cuda_bad |= chk(tb_launch_transpose_rows(d_stage, rows, m, c->d_x, c->ldn, p0, c->stream), "transpose");
      cuda_bad |= chk(cudaStreamSynchronize(c->stream), "sync after transpose");
      c->launches += 1;
    }
    cudaFreeHost(h_stage);
    cudaFree(d_stage);
  } else {
    // SNP-major 2-bit rows in file order (stride = ceil(n / 4) bytes per marker, the layout of a PLINK .bed body
    // with dosage codes): chunks of markers are contiguous, the device expands them and applies the permutation
    const int stride = (n + 3) / 4;
    const uint8_t* packed = static_cast<const uint8_t*>(geno_any);
    int chunk = (int)std::max<long long>(1, std::min<long long>(m, ((long long)256 << 20) / stride));
    uint8_t* d_stage = nullptr;
    int *d_perm = nullptr, *d_bad = nullptr;
    cuda_bad |= chk(cudaMalloc(&d_stage, (size_t)chunk * stride), "cudaMalloc staging");
    cuda_bad |= chk(cudaMalloc(&d_perm, (size_t)n * sizeof(int)), "cudaMalloc perm");
    cuda_bad |= chk(cudaMalloc(&d_bad, sizeof(int)), "cudaMalloc flag");
    if (!cuda_bad) {
      cuda_bad |= chk(cudaMemcpyAsync(d_perm, p.data(), (size_t)n * sizeof(int), cudaMemcpyHostToDevice, c->stream), "H2D perm");
      cuda_bad |= chk(cudaMemsetAsync(d_bad, 0, sizeof(int), c->stream), "memset");
    }
    for (int j0 = 0; j0 < m && !cuda_bad; j0 += chunk) {
      const int rows = std::min(chunk, m - j0);
      cuda_bad |= chk(cudaMemcpyAsync(d_stage, packed + (size_t)j0 * stride, (size_t)rows * stride, cudaMemcpyHostToDevice, c->stream), "H2D packed genotypes");
      cuda_bad |= chk(tb_launch_unpack2_perm(d_stage, rows, stride, d_perm, n, c->d_x, c->ldn, j0, d_bad, c->stream), "unpack");
      cuda_bad |= chk(cudaStreamSynchronize(c->stream), "sync after unpack");
      c->launches += 1;
    }
    if (!cuda_bad) {
      int h_bad = 0;
      cuda_bad |= chk(cudaMemcpy(&h_bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost), "D2H flag");
      bad_value = h_bad != 0;
    }
    cudaFree(d_stage);
    cudaFree(d_perm);
    cudaFree(d_bad);
  }
  if (bad_value) return bail("tb_create: genotype values must be dosages in {0, 1, 2}");
  if (cuda_bad) return bail("");
  {
    std::vector<int> ident(n);
    for (int i = 0; i < n; ++i) ident[i] = i;
    int* d_pos = nullptr;
    if (chk(cudaMalloc(&d_pos, n * sizeof(int)), "cudaMalloc")) return bail("");
    bool b2 = chk(cudaMemcpyAsync(d_pos, ident.data(), n * sizeof(int), cudaMemcpyHostToDevice, c->stream), "H2D");
    b2 |= chk(tb_launch_colsum(c->geno(), m, d_pos, n, c->d_colsum_all, c->stream), "colsum");
    b2 |= chk(cudaStreamSynchronize(c->stream), "sync after colsum");
    cudaFree(d_pos);
    c->launches += 1;
    if (b2) return bail("");
  }
  if (storage == TB_STORE_PACKED2) {
    // keep only the 2-bit copy resident (a quarter of the bytes; the gather expands it on the fly)
    if (chk(cudaMalloc(&c->d_x2, (size_t)m * (c->ldn / 4)), "cudaMalloc packed genotypes")) return bail("");
    bool b2 = chk(tb_launch_pack2(c->d_x, c->ldn, m, c->d_x2, c->stream), "pack");
    b2 |= chk(cudaStreamSynchronize(c->stream), "sync after pack");
    c->launches += 1;
    if (b2) return bail("");
    cudaFree(c->d_x);
    c->d_x = nullptr;
  }
  if (chk(tb_gram_tc_init(), "gram kernel init") || chk(tb_chol_init(), "cholesky kernel init") ||
      chk(tb_solve_init(), "solve kernel init") ||
      chk(tb_chol_tc_init(), "tensor-core cholesky init") || chk(tb_solve_mixed_init(), "mixed solve init") ||
      chk(tb_gather_init(), "gather init") || chk(tb_reml_init(), "reml kernel init"))
    return bail("");
  *out = c;
  return 0;
}

// A second context on another GPU of the box without a second ingest: the resident genotype matrix (already validated,
// permuted, transposed and packed) and the column sums are copied device to device (NVLink / NVSwitch peer copy).
// Row sets are not copied -- the caller defines them with tb_set_rowset as on any context.
int tb_clone(const tb_ctx* src, int device, tb_ctx** out) {
  if (!out) return -1;
  *out = nullptr;
  if (!src) {
    g_create_err = "tb_clone: null source context";
    return -1;
  }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) {
    g_create_err = "tb_clone: bad device ordinal";
    return -1;
  }
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  if (prop.major != 10) {
    g_create_err = "tb_clone: target device is not sm_100";
    return -3;
  }
  cudaSetDevice(src->device);
  cudaStreamSynchronize(src->stream);
  TbCtx* c = new TbCtx();
  auto bail = [&](const std::string& msg) {
    g_create_err = msg.empty() ? c->err : msg;
    tb_destroy(c);
    return -2;
  };
  c->device = device;
  c->n = src->n;
  c->m = src->m;
  c->ldn = src->ldn;
  c->storage = src->storage;
  c->n_sm = prop.multiProcessorCount;
  c->y_univ = src->y_univ;
  c->has_pheno = src->has_pheno;
  c->pos_of = src->pos_of;
  if (cudaSetDevice(device) != cudaSuccess) return bail("cudaSetDevice failed");
  auto chk = [&](cudaError_t ce, const char* what) {
    if (ce == cudaSuccess) return false;
    c->err = std::string(what) + ": " + cudaGetErrorString(ce);
    return true;
  };
  if (device != src->device) {
    int can = 0;
    cudaDeviceCanAccessPeer(&can, device, src->device);
    if (can) {
      cudaError_t pe = cudaDeviceEnablePeerAccess(src->device, 0);
      if (pe != cudaSuccess && pe != cudaErrorPeerAccessAlreadyEnabled) (void)pe;
      cudaGetLastError();     // "already enabled" is not an error
    }
  }
  if (chk(cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking), "cudaStreamCreate")) return bail("");
  c->stream = c->own_stream;
  const size_t bytes = (size_t)c->m * (size_t)(c->storage == TB_STORE_PACKED2 ? c->ldn / 4 : c->ldn);
  void* dst = nullptr;
  if (chk(cudaMalloc(&dst, bytes), "cudaMalloc genotypes")) return bail("");
  const void* from = c->storage == TB_STORE_PACKED2 ? (const void*)src->d_x2 : (const void*)src->d_x;
  if (c->storage == TB_STORE_PACKED2) c->d_x2 = static_cast<uint8_t*>(dst);
  else c->d_x = static_cast<int8_t*>(dst);
  if (chk(cudaMalloc(&c->d_colsum_all, (size_t)c->m * sizeof(int)), "cudaMalloc colsum")) return bail("");
  if (chk(cudaMemcpyPeerAsync(dst, device, from, src->device, bytes, c->stream), "peer copy genotypes")) return bail("");
  if (chk(cudaMemcpyPeerAsync(c->d_colsum_all, device, src->d_colsum_all, src->device, (size_t)c->m * sizeof(int), c->stream),
          "peer copy colsum"))
    return bail("");
  if (chk(cudaStreamSynchronize(c->stream), "peer copy")) return bail("");
  if (chk(tb_gram_tc_init(), "gram kernel init") || chk(tb_chol_init(), "cholesky kernel init") ||
      chk(tb_solve_init(), "solve kernel init") || chk(tb_chol_tc_init(), "tensor-core cholesky init") ||
      chk(tb_solve_mixed_init(), "mixed solve init") || chk(tb_gather_init(), "gather init") ||
      chk(tb_reml_init(), "reml kernel init"))
    return bail("");
  *out = c;
  return 0;
}

int tb_destroy(tb_ctx* c) {
  if (!c) return 0;
  cudaSetDevice(c->device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  for (auto& r : c->slots) free_rowset(r);
  tb_de_release(c);
  for (auto ev : c->ev_pool) cudaEventDestroy(ev);
  cudaFree(c->d_x);
  cudaFree(c->d_x2);
  cudaFree(c->d_colsum_all);
  cudaFree(c->d_idx);
  cudaFree(c->d_fail);
  cudaFree(c->d_fit_out);
  cudaFree(c->d_split);
  cudaFree(c->ws);
  if (c->own_stream) cudaStreamDestroy(c->own_stream);
  delete c;
  return 0;
}

int tb_set_rowset(tb_ctx* c, int slot, const int32_t* train, int n_t, const int32_t* valid, int n_v) {
  if (!c) return -1;
  if (slot < 0 || slot >= TB_MAX_SLOTS) return fail(c, "tb_set_rowset: slot out of range");
  if (!train || !valid || n_t < 2 || n_v < 2) return fail(c, "tb_set_rowset: need at least 2 training and 2 validation animals");
  if (!c->has_pheno) return fail(c, "tb_set_rowset: this context was created without phenotypes");
  TB_CUDA(c, cudaSetDevice(c->device));
  TB_CUDA(c, cudaStreamSynchronize(c->stream));
  TbRowSet& r = c->slots[slot];
  free_rowset(r);
  std::vector<int> tpos(n_t), vpos(n_v);
  int maxpos = 0;
  for (int i = 0; i < n_t; ++i) {
    if (train[i] < 0 || train[i] >= c->n) return fail(c, "tb_set_rowset: training index out of range");
    tpos[i] = c->pos_of[train[i]];
    maxpos = std::max(maxpos, tpos[i]);
  }
  for (int i = 0; i < n_v; ++i) {
    if (valid[i] < 0 || valid[i] >= c->n) return fail(c, "tb_set_rowset: validation index out of range");
    vpos[i] = c->pos_of[valid[i]];
    maxpos = std::max(maxpos, vpos[i]);
  }
  r.n_t = n_t;
  r.n_v = n_v;
  r.ntp = tb_round_up(n_t, TB_NB);
  r.rows = maxpos + 1;
  r.rpad = tb_round_up(r.rows, TB_GRAM_BM);
  r.has_train.assign(r.rpad / TB_GRAM_BM, 0);
  for (int i = 0; i < n_t; ++i) r.has_train[tpos[i] / TB_GRAM_BM] = 1;
  r.contiguous = true;
  for (int i = 0; i < n_t; ++i) r.contiguous = r.contiguous && tpos[i] == i;
  {
    int h0 = 0;
    while (h0 < n_t && tpos[h0] == h0) ++h0;
    r.hole0 = h0;
    r.gap = h0 < n_t ? tpos[h0] - h0 : 0;
    bool ok = h0 == n_t || r.gap > 0;
    for (int i = h0; i < n_t && ok; ++i) ok = tpos[i] == i + r.gap;
    r.seg_ok = ok && h0 % 8 == 0 && r.gap % 8 == 0 && n_t % 8 == 0;
    r.valid_in_hole = r.seg_ok && r.gap > 0 && n_v == r.gap && n_v <= r.ntp;
    for (int i = 0; i < n_v && r.valid_in_hole; ++i) r.valid_in_hole = vpos[i] == h0 + i;
    if (!r.seg_ok) {
      r.hole0 = n_t;
      r.gap = 0;
    }
  }
  std::vector<int> rowmap, ident;
  r.rows_univ = maxpos + 1;
  r.perm_ok = false;
  if (!r.contiguous) {
    // panel-row permutation: training animals first, validation animals next, nobody else
    rowmap.assign(maxpos + 1, -1);
    bool ok = n_t % 4 == 0;
    for (int i = 0; i < n_t && ok; ++i) {
      ok = rowmap[tpos[i]] < 0;
      rowmap[tpos[i]] = i;
    }
    for (int i = 0; i < n_v && ok; ++i) {
      ok = rowmap[vpos[i]] < 0;
      rowmap[vpos[i]] = n_t + i;
    }
    r.perm_ok = ok;
    ident.resize(n_t + n_v);
    for (int i = 0; i < n_t + n_v; ++i) ident[i] = i;
  }
  std::vector<double> yt(r.ntp, 0.0), ytc(r.ntp, 0.0), yv(n_v);
  double mean = 0.0;
  for (int i = 0; i < n_t; ++i) {
    yt[i] = c->y_univ[tpos[i]];
    mean += yt[i];
  }
  mean /= n_t;
  r.yt_mean = mean;
  for (int i = 0; i < n_t; ++i) ytc[i] = yt[i] - mean;
  for (int i = 0; i < n_v; ++i) yv[i] = c->y_univ[vpos[i]];
  TB_CUDA(c, cudaMalloc(&r.d_tpos, n_t * sizeof(int)));
  TB_CUDA(c, cudaMalloc(&r.d_vpos, n_v * sizeof(int)));
  TB_CUDA(c, cudaMalloc(&r.d_colsum_train, (size_t)c->m * sizeof(int)));
  TB_CUDA(c, cudaMalloc(&r.d_yt_raw, r.ntp * sizeof(double)));
  TB_CUDA(c, cudaMalloc(&r.d_yt_ctr, r.ntp * sizeof(double)));
  TB_CUDA(c, cudaMalloc(&r.d_yv, n_v * sizeof(double)));
  if (r.perm_ok) {
    TB_CUDA(c, cudaMalloc(&r.d_rowmap, rowmap.size() * sizeof(int)));
    TB_CUDA(c, cudaMalloc(&r.d_ident, ident.size() * sizeof(int)));
    TB_CUDA(c, cudaMemcpyAsync(r.d_rowmap, rowmap.data(), rowmap.size() * sizeof(int), cudaMemcpyHostToDevice, c->stream));
    TB_CUDA(c, cudaMemcpyAsync(r.d_ident, ident.data(), ident.size() * sizeof(int), cudaMemcpyHostToDevice, c->stream));
  }
  TB_CUDA(c, cudaMemcpyAsync(r.d_tpos, tpos.data(), n_t * sizeof(int), cudaMemcpyHostToDevice, c->stream));
  TB_CUDA(c, cudaMemcpyAsync(r.d_vpos, vpos.data(), n_v * sizeof(int), cudaMemcpyHostToDevice, c->stream));
  TB_CUDA(c, cudaMemcpyAsync(r.d_yt_raw, yt.data(), r.ntp * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  TB_CUDA(c, cudaMemcpyAsync(r.d_yt_ctr, ytc.data(), r.ntp * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  TB_CUDA(c, cudaMemcpyAsync(r.d_yv, yv.data(), n_v * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  TB_CUDA(c, tb_launch_colsum(c->geno(), c->m, r.d_tpos, n_t, r.d_colsum_train, c->stream));
  c->launches += 1;
  TB_CUDA(c, cudaStreamSynchronize(c->stream));
  r.valid = true;
  return 0;
}

int tb_stage_genomes(tb_ctx* c, const int32_t* idx_flat, const int64_t* idx_off, int P) {
  if (!c) return -1;
  if (!idx_flat || !idx_off || P <= 0) return fail(c, "tb_stage_genomes: null or empty batch");
  if (idx_off[0] != 0) return fail(c, "tb_stage_genomes: idx_off[0] must be 0");
  for (int i = 0; i < P; ++i)
    if (idx_off[i + 1] < idx_off[i]) return fail(c, "tb_stage_genomes: offsets must be non-decreasing");
  const size_t total = (size_t)idx_off[P];
  TB_CUDA(c, cudaSetDevice(c->device));
  if (total > c->idx_cap) {
    TB_CUDA(c, cudaStreamSynchronize(c->stream));
    cudaFree(c->d_idx);
    c->d_idx = nullptr;
    c->idx_cap = 0;
    TB_CUDA(c, cudaMalloc(&c->d_idx, std::max<size_t>(total, 1) * sizeof(int)));
    c->idx_cap = total;
  }
  // start the copy first, validate while it is in flight (pinned caller buffers make it truly asynchronous); a bad
  // index invalidates the staged batch before anything can read it
  size_t sp = span_begin(c, TB_ST_H2D);
  TB_CUDA(c, cudaMemcpyAsync(c->d_idx, idx_flat, total * sizeof(int), cudaMemcpyHostToDevice, c->stream));
  span_end(c, sp);
  {
    // branch-free range check (vectorises): any index outside [0, m) sets the flag; the slow path names it
    const unsigned um = (unsigned)c->m;
    auto scan = [&](size_t lo, size_t hi) {
      unsigned b = 0;
      for (size_t q = lo; q < hi; ++q) b |= (unsigned)((unsigned)idx_flat[q] >= um);
      return b;
    };
    unsigned bad = 0;
    if (total >= ((size_t)1 << 20)) {               // a generation's worth of indices: four host threads
      constexpr int NT = 4;
      unsigned part[NT] = {0, 0, 0, 0};
      std::thread th[NT - 1];
      const size_t chunk = (total + NT - 1) / NT;
      for (int t = 1; t < NT; ++t)
        th[t - 1] = std::thread([&, t] { part[t] = scan(std::min(total, t * chunk), std::min(total, (t + 1) * chunk)); });
      part[0] = scan(0, std::min(total, chunk));
      for (int t = 1; t < NT; ++t) th[t - 1].join();
      for (int t = 0; t < NT; ++t) bad |= part[t];
    } else {
      bad = scan(0, total);
    }
    if (bad) {
      cudaStreamSynchronize(c->stream);
      c->P = 0;
      for (size_t q = 0; q < total; ++q)
        if (idx_flat[q] < 0 || idx_flat[q] >= c->m)
          return fail(c, "tb_stage_genomes: marker index " + std::to_string(idx_flat[q]) + " out of range [0, " +
                             std::to_string(c->m) + ")");
    }
  }
  c->h_off.assign(idx_off, idx_off + P + 1);
  c->P = P;
  return 0;
}

int tb_pack_index_lists(const void* const* lists, const int64_t* lens, const int32_t* elem_bytes, int P, int64_t m,
                        int32_t* idx_flat, int64_t* idx_off, int64_t* bad_index) {
  if (!lens || !idx_off || P < 0 || m <= 0 || m > 0x7fffffffLL) return -1;
  idx_off[0] = 0;
  for (int i = 0; i < P; ++i) {
    if (lens[i] < 0 || (lens[i] > 0 && (!lists || !lists[i])) || !elem_bytes || (elem_bytes[i] != 4 && elem_bytes[i] != 8))
      return -1;
    idx_off[i + 1] = idx_off[i] + lens[i];
  }
  const int64_t total = idx_off[P];
  if (total > 0 && !idx_flat) return -1;
  // lists [lo, hi): copy + narrow + wrap; returns the number of the first list with an index out of range (or P)
  auto run = [&](int lo, int hi, int64_t* bad) -> int {
    for (int i = lo; i < hi; ++i) {
      int32_t* dst = idx_flat + idx_off[i];
      const int64_t n = lens[i];
      unsigned flag = 0;
      if (elem_bytes[i] == 8) {
        const int64_t* src = static_cast<const int64_t*>(lists[i]);
        for (int64_t q = 0; q < n; ++q) {
          int64_t v = src[q];
          v += v < 0 ? m : 0;
          flag |= (unsigned)((uint64_t)v >= (uint64_t)m);
          dst[q] = (int32_t)v;
        }
      } else {
        const int32_t* src = static_cast<const int32_t*>(lists[i]);
        for (int64_t q = 0; q < n; ++q) {
          int64_t v = src[q];
          v += v < 0 ? m : 0;
          flag |= (unsigned)((uint64_t)v >= (uint64_t)m);
          dst[q] = (int32_t)v;
        }
      }
      if (flag) {                                   // slow path: name the value
        for (int64_t q = 0; q < n; ++q) {
          const int64_t v = elem_bytes[i] == 8 ? static_cast<const int64_t*>(lists[i])[q]
                                               : (int64_t) static_cast<const int32_t*>(lists[i])[q];
          if (v >= m || v < -m) {
            *bad = v;
            return i;
          }
        }
      }
    }
    return P;
  };
  int first_bad = P;
  int64_t bad_value = 0;
  const int nt = total >= ((int64_t)1 << 20)
                     ? (int)std::max(1u, std::min(8u, std::min((unsigned)P, std::thread::hardware_concurrency())))
                     : 1;
  if (nt > 1) {
    // contiguous groups of lists with about the same number of indices each
    std::vector<int> cut(nt + 1, P);
    cut[0] = 0;
    for (int t = 1, i = 0; t < nt; ++t) {
      while (i < P && idx_off[i] < total * t / nt) ++i;
      cut[t] = i;
    }
    std::vector<int> where(nt, P);
    std::vector<int64_t> what(nt, 0);
    std::vector<std::thread> th;
    for (int t = 1; t < nt; ++t) th.emplace_back([&, t] { where[t] = run(cut[t], cut[t + 1], &what[t]); });
    where[0] = run(cut[0], cut[1], &what[0]);
    for (auto& x : th) x.join();
    for (int t = 0; t < nt; ++t)
      if (where[t] < first_bad) {
        first_bad = where[t];
        bad_value = what[t];
      }
  } else {
    first_bad = run(0, P, &bad_value);
  }
  if (first_bad < P) {
    if (bad_index) *bad_index = bad_value;
    return -3;
  }
  return 0;
}

int tb_eval_staged(tb_ctx* c, const int32_t* slots, int n_slots, double h2, int mode_rule, double* fitness_out,
                   int out_is_device) {
  if (!c) return -1;
  if (!slots || !fitness_out) return fail(c, "tb_eval_staged: null argument");
  TB_CUDA(c, cudaSetDevice(c->device));
  const size_t n_out = (size_t)c->P * (size_t)std::max(n_slots, 0);
  double* d_fit = fitness_out;
  if (!out_is_device) {
    if (n_out > c->fit_cap) {                      // persistent device buffer for the host-output path
      TB_CUDA(c, cudaStreamSynchronize(c->stream));
      cudaFree(c->d_fit_out);
      c->d_fit_out = nullptr;
      c->fit_cap = 0;
      TB_CUDA(c, cudaMalloc(&c->d_fit_out, std::max<size_t>(n_out, 1) * sizeof(double)));
      c->fit_cap = n_out;
    }
    d_fit = c->d_fit_out;
  }
  int rc = eval_core(c, slots, n_slots, h2, mode_rule, d_fit);
  cudaError_t ce = cudaSuccess;
  if (rc == 0 && !out_is_device) {
    size_t sp = span_begin(c, TB_ST_D2H);
    ce = cudaMemcpyAsync(fitness_out, d_fit, n_out * sizeof(double), cudaMemcpyDeviceToHost, c->stream);
    span_end(c, sp);
  }
  cudaError_t se = cudaStreamSynchronize(c->stream);
  spans_collect(c);
  if (rc != 0) return rc;
  if (ce != cudaSuccess) return fail(c, std::string("D2H fitness: ") + cudaGetErrorString(ce), -2);
  if (se != cudaSuccess) return fail(c, std::string("device execution failed: ") + cudaGetErrorString(se), -2);
  return 0;
}

int tb_eval(tb_ctx* c, const int32_t* slots, int n_slots, const int32_t* idx_flat, const int64_t* idx_off, int P,
            double h2, int mode_rule, double* fitness_out) {
  int rc = tb_stage_genomes(c, idx_flat, idx_off, P);
  if (rc) return rc;
  return tb_eval_staged(c, slots, n_slots, h2, mode_rule, fitness_out, 0);
}

int tb_gram_debug(tb_ctx* c, const int32_t* idx, int k, int rows, int impl, int32_t* out) {
  if (!c) return -1;
  if (!idx || !out || k <= 0 || rows <= 0 || rows > c->n) return fail(c, "tb_gram_debug: bad argument");
  for (int q = 0; q < k; ++q)
    if (idx[q] < 0 || idx[q] >= c->m) return fail(c, "tb_gram_debug: marker index out of range");
  TB_CUDA(c, cudaSetDevice(c->device));
  const bool fp4 = impl == 2 || impl == 4 || impl == 6;
  const int pair = (impl == 3 || impl == 4) ? 1 : (impl == 5 || impl == 6) ? 2 : 0;   // clusters of two CTAs: multicast / tcgen05 pair
  if (impl == 6) impl = 4;
  if (fp4 && !c->d_x2) return fail(c, "tb_gram_debug: the fp4 Gram needs packed resident genotypes");
  const int kq = fp4 ? TB_GRAM_BK_FP4 : TB_GRAM_BK;
  const int rpad = tb_round_up(rows, TB_GRAM_BM), kmark = tb_round_up(k, kq);
  const int kstride = fp4 ? kmark / 2 : kmark;          // bytes per panel row
  std::vector<int> tiles;
  build_tiles(rpad, std::vector<unsigned char>(), tiles, fp4 ? TB_GRAM_BN_FP4 : TB_GRAM_BN, pair != 0);
  const long long off[2] = {0, k};
  const int kb = kmark / kq;
  int8_t* d_panel = nullptr;
  int32_t* d_C = nullptr;
  int *d_i = nullptr, *d_t = nullptr, *d_kb = nullptr;
  long long* d_off = nullptr;
  cudaStream_t st = c->stream;
  int rc = 0;
  auto ck = [&](cudaError_t e, const char* what) {
    if (e != cudaSuccess && rc == 0) rc = fail(c, std::string("tb_gram_debug ") + what + ": " + cudaGetErrorString(e), -2);
  };
  ck(cudaMalloc(&d_panel, ((size_t)rpad + 128) * kstride), "malloc");
  ck(cudaMalloc(&d_C, (size_t)rpad * rpad * sizeof(int32_t)), "malloc");
  ck(cudaMalloc(&d_i, k * sizeof(int)), "malloc");
  ck(cudaMalloc(&d_t, tiles.size() * sizeof(int)), "malloc");
  ck(cudaMalloc(&d_kb, sizeof(int)), "malloc");
  ck(cudaMalloc(&d_off, 2 * sizeof(long long)), "malloc");
  if (rc == 0) {
    ck(cudaMemsetAsync(d_C, 0, (size_t)rpad * rpad * sizeof(int32_t), st), "memset");
    ck(cudaMemcpyAsync(d_i, idx, k * sizeof(int), cudaMemcpyHostToDevice, st), "H2D");
    ck(cudaMemcpyAsync(d_t, tiles.data(), tiles.size() * sizeof(int), cudaMemcpyHostToDevice, st), "H2D");
    ck(cudaMemcpyAsync(d_kb, &kb, sizeof(int), cudaMemcpyHostToDevice, st), "H2D");
    ck(cudaMemcpyAsync(d_off, off, sizeof(off), cudaMemcpyHostToDevice, st), "H2D");
    if (fp4) ck(tb_launch_gather_fp4(c->geno(), d_i, d_off, 0, 1, rpad, kstride, d_panel, st), "gather");
    else ck(tb_launch_gather(c->geno(), d_i, d_off, 0, 1, rpad, kstride, d_panel, st), "gather");
    if (impl == 0 || fp4 || pair) {
      std::string e;
      cudaError_t ce = tb_launch_gram_tc(d_panel, 1, rpad, kstride, d_kb, d_t, (int)tiles.size(), d_C, c->n_sm, st, &e,
                                         nullptr, nullptr, 0, 0, fp4 ? 1 : 0, pair);
      if (ce != cudaSuccess && rc == 0) rc = fail(c, "tb_gram_debug gram_tc: " + (e.empty() ? std::string(cudaGetErrorString(ce)) : e), -2);
    } else {
      ck(tb_launch_gram_simt(d_panel, 1, rpad, kstride, d_kb, d_C, st), "gram_simt");
    }
    c->launches += 2;
    std::vector<int32_t> h((size_t)rpad * rpad);
    ck(cudaMemcpyAsync(h.data(), d_C, h.size() * sizeof(int32_t), cudaMemcpyDeviceToHost, st), "D2H");
    ck(cudaStreamSynchronize(st), "execution");
    if (rc == 0) {
      for (int a = 0; a < rows; ++a)
        for (int b = 0; b < rows; ++b) out[(size_t)a * rows + b] = b <= a ? h[(size_t)a * rpad + b] : 0;
    }
  }
  cudaFree(d_panel);
  cudaFree(d_C);
  cudaFree(d_i);
  cudaFree(d_t);
  cudaFree(d_kb);
  cudaFree(d_off);
  return rc;
}

int tb_debug_fetch(tb_ctx* c, int what, int job, void* out, size_t nbytes) {
  if (!c) return -1;
  if (!out) return fail(c, "tb_debug_fetch: null output");
  const auto& d = c->dbg;
  const int n_jobs = d.W * d.n_slots;
  if (n_jobs == 0) return fail(c, "tb_debug_fetch: nothing evaluated yet");
  if (job < 0 || job >= n_jobs) return fail(c, "tb_debug_fetch: job out of range");
  TB_CUDA(c, cudaSetDevice(c->device));
  const void* src = nullptr;
  size_t need = 0;
  int dims[4] = {d.rpad, d.ntp[job], d.n_v[job], d.kstride};
  switch (what) {
    case TB_DBG_C: src = d.C + (size_t)(job / d.n_slots) * d.rpad * d.rpad; need = (size_t)d.rpad * d.rpad * 4; break;
    case TB_DBG_S: src = d.s + (size_t)(d.centre_shared ? job / d.n_slots : job) * d.rpad; need = (size_t)d.rpad * 8; break;
    case TB_DBG_SQ: src = d.SQ + (size_t)(d.centre_shared ? job / d.n_slots : job) * 2; need = 16; break;
    case 7:
      if (!d.L32) return fail(c, "tb_debug_fetch: no fp32 factor (fp64 precision mode)");
      src = d.L32 + (size_t)job * d.ntp_all * d.ntp_all; need = (size_t)d.ntp_all * d.ntp_all * 4; break;
    case 8: src = d.sweeps + job; need = 4; break;
    case TB_DBG_LINV32:
      if (!d.Linv32) return fail(c, "tb_debug_fetch: no diagonal-block inverses (fp64 precision mode)");
      src = d.Linv32 + (size_t)job * d.ntp_all * TB_NB; need = (size_t)d.ntp_all * TB_NB * 4; break;
    case TB_DBG_M:
      if (!d.M[job]) return fail(c, "tb_debug_fetch: [A ; G_vt] is not formed in mixed precision mode");
      src = d.M[job]; need = (size_t)(d.ntp[job] + d.n_v[job]) * d.ntp[job] * 8; break;
    case TB_DBG_ALPHA: src = d.alpha[job]; need = (size_t)d.ntp[job] * 8; break;
    case TB_DBG_PRED: src = d.pred[job]; need = (size_t)d.n_v[job] * 8; break;
    case TB_DBG_DIMS:
      if (nbytes < sizeof(dims)) return fail(c, "tb_debug_fetch: buffer too small");
      memcpy(out, dims, sizeof(dims));
      return 0;
    default: return fail(c, "tb_debug_fetch: unknown item");
  }
  if (nbytes < need) return fail(c, "tb_debug_fetch: buffer too small (need " + std::to_string(need) + " bytes)");
  if (what == TB_DBG_L32 && d.L16) {
    // the factor of record is the fp16 copy (same 10-bit mantissa as the TF32 rounding; the wide panel solve does
    // not write the fp32 copy below the diagonal blocks): widen it, upper triangle zero
    const size_t nn = (size_t)d.ntp_all * d.ntp_all;
    std::vector<unsigned short> h(nn);
    TB_CUDA(c, cudaMemcpy(h.data(), d.L16 + (size_t)job * nn, nn * sizeof(unsigned short), cudaMemcpyDeviceToHost));
    float* o = static_cast<float*>(out);
    for (int r = 0; r < d.ntp_all; ++r)
      for (int q = 0; q < d.ntp_all; ++q) {
        float f = 0.f;
        if (q <= r) {
          const unsigned short b = h[(size_t)r * d.ntp_all + q];
          const int sign = b >> 15, ex = (b >> 10) & 31, man = b & 1023;
          f = ex == 0 ? std::ldexp((float)man, -24) : ex == 31 ? (man ? NAN : INFINITY) : std::ldexp((float)(man | 1024), ex - 25);
          if (sign) f = -f;
        }
        o[(size_t)r * d.ntp_all + q] = f;
      }
    return 0;
  }
  if (what == TB_DBG_C && c->last_c16) {
    // the wave stored int16 cross-products: widen to the int32 view the caller asked for
    std::vector<int16_t> h((size_t)d.rpad * d.rpad);
    const int16_t* src16 = reinterpret_cast<const int16_t*>(d.C) + (size_t)(job / d.n_slots) * d.rpad * d.rpad;
    TB_CUDA(c, cudaMemcpy(h.data(), src16, h.size() * sizeof(int16_t), cudaMemcpyDeviceToHost));
    int32_t* o = static_cast<int32_t*>(out);
    for (size_t i = 0; i < h.size(); ++i) o[i] = h[i];
    return 0;
  }
  TB_CUDA(c, cudaMemcpy(out, src, need, cudaMemcpyDeviceToHost));
  return 0;
}

int tb_set_option(tb_ctx* c, const char* name, long long value) {
  if (!c || !name) return -1;
  const std::string s(name);
  if (s == "profile") c->profile = value != 0;
  else if (s == "stop_after") c->stop_after = (int)value;
  else if (s == "workspace_mb") c->ws_limit = value > 0 ? (size_t)value << 20 : 0;
  else if (s == "max_wave") c->max_wave = (int)value;
  else if (s == "precision") c->precision = value != 0;
  else if (s == "fuse_scale") c->fuse_scale = value != 0;
  else if (s == "fuse_in_gram") c->fuse_in_gram = value != 0;
  else if (s == "solve_debug") tb_solve_mixed_set_debug((int)value);
  else if (s == "no_fallback") c->no_fallback = value != 0;     // diagnostics: keep the mixed-precision result of failed jobs
  else if (s == "blk0_scale32") c->blk0_scale32 = value != 0;   // A/B: block column 0 of the scaled matrix by its own scaling pass
  else if (s == "solve_pair") c->solve_pair = value < 0 ? 0 : value > 2 ? 2 : (int)value;
  else if (s == "gram_experiment") c->gram_experiment = (int)value;   // timing experiments only (results are wrong): 1 = no stores, 2 = no epilogue
  else if (s == "gram_pair") c->gram_pair = value < 0 ? 0 : value > 2 ? 2 : (int)value;
  else if (s == "wide_panel") c->wide_panel = value != 0;
  else if (s == "epi_warps") c->epi_warps = value == 8 ? 8 : 16;
  else if (s == "chain_inverse") c->chain_inverse = value != 0;  // A/B: 0 = trinv256_kernel after the fused chain
  else if (s == "chain_fused") c->chain_fused = (int)value;      // jobs per wave up to which the diagonal-block chain is one launch (-1: SM count, 0: never)
  else if (s == "t16") c->t16 = value != 0;                     // A/B: 0 = fp32 block columns all the way down (round-2 first version)
  else if (s == "panel_fused") c->panel_fused = value != 0;     // A/B: 0 = update, then the wide panel GEMM as its own launch
  else if (s == "narrow_c") c->narrow_c = value != 0;
  else if (s == "gram_fp4") c->gram_fp4 = value != 0;
  else if (s == "perm_rows") c->perm_rows = value != 0;
  else if (s == "storage") return fail(c, "tb_set_option: storage is fixed at tb_create_ex");
  else return fail(c, "tb_set_option: unknown option '" + s + "'");
  return 0;
}

int tb_get_info(const tb_ctx* c, const char* name, long long* value) {
  if (!c || !name || !value) return -1;
  const std::string s(name);
  if (s == "last_c16") *value = c->last_c16;
  else if (s == "last_fused_scale") *value = c->last_fused;
  else if (s == "last_mixed") *value = c->last_mixed;
  else if (s == "last_wave") *value = c->last_wave;
  else if (s == "storage") *value = c->storage;
  else if (s == "wide_panel") *value = c->wide_panel;
  else if (s == "t16") *value = c->t16;
  else if (s == "panel_fused") *value = c->panel_fused;
  else if (s == "epi_warps") *value = c->epi_warps;
  else if (s == "de_removed") *value = c->de.n_banned;
  else if (s == "last_fp4") *value = c->last_fp4;
  else if (s == "last_perm") *value = c->last_perm;
  else if (s == "last_split") *value = c->last_split;
  else if (s == "last_fallbacks") *value = c->last_fallbacks;
  else if (s == "last_issue_us") *value = c->last_issue_us;
  else if (s == "staged") *value = c->P;
  else return -1;
  return 0;
}

int tb_staged_offsets(const tb_ctx* c, int64_t* off_out, int n) {
  if (!c || !off_out) return -1;
  if (n < c->P + 1 || (int)c->h_off.size() < c->P + 1) return -1;
  for (int i = 0; i <= c->P; ++i) off_out[i] = c->h_off[i];
  return 0;
}

int tb_stage_times(tb_ctx* c, double* ms_out, uint64_t* launches_out) {
  if (!c) return -1;
  for (int i = 0; i < TB_ST_COUNT; ++i) {
    if (ms_out) ms_out[i] = c->stage_ms[i];
    if (launches_out) launches_out[i] = c->stage_launches[i];
  }
  return 0;
}

uint64_t tb_launch_count(const tb_ctx* c) { return c ? c->launches : 0; }

int tb_reset_counters(tb_ctx* c) {
  if (!c) return -1;
  for (int i = 0; i < TB_ST_COUNT; ++i) {
    c->stage_ms[i] = 0.0;
    c->stage_launches[i] = 0;
  }
  c->launches = 0;
  return 0;
}

int tb_last_wave(const tb_ctx* c) { return c ? c->last_wave : 0; }
int tb_last_precision(const tb_ctx* c) { return c ? (c->last_mixed ? 0 : 1) : -1; }

int tb_storage_info(const tb_ctx* c, int* storage, uint64_t* bytes) {
  if (!c) return -1;
  if (storage) *storage = c->storage;
  if (bytes) *bytes = (uint64_t)c->m * (uint64_t)(c->storage == TB_STORE_PACKED2 ? c->ldn / 4 : c->ldn);
  return 0;
}

int tb_marker_stats(tb_ctx* c, const int32_t* animals, int n_animals, const double* weights, double* sum_x,
                    double* sum_xx, double* sum_xw) {
  if (!c) return -1;
  if (!animals || !weights || !sum_x || !sum_xx || !sum_xw || n_animals <= 0) return fail(c, "tb_marker_stats: null or empty argument");
  TB_CUDA(c, cudaSetDevice(c->device));
  std::vector<int> pos(n_animals);
  for (int i = 0; i < n_animals; ++i) {
    if (animals[i] < 0 || animals[i] >= c->n) return fail(c, "tb_marker_stats: animal index out of range");
    pos[i] = c->pos_of[animals[i]];
  }
  int* d_pos = nullptr;
  double *d_w = nullptr, *d_out = nullptr;
  int rc = 0;
  auto ck = [&](cudaError_t e, const char* what) {
    if (e != cudaSuccess && rc == 0) rc = fail(c, std::string("tb_marker_stats ") + what + ": " + cudaGetErrorString(e), -2);
  };
  ck(cudaMalloc(&d_pos, (size_t)n_animals * sizeof(int)), "malloc");
  ck(cudaMalloc(&d_w, (size_t)n_animals * sizeof(double)), "malloc");
  ck(cudaMalloc(&d_out, (size_t)3 * c->m * sizeof(double)), "malloc");
  if (rc == 0) {
    cudaStream_t st = c->stream;
    ck(cudaMemcpyAsync(d_pos, pos.data(), (size_t)n_animals * sizeof(int), cudaMemcpyHostToDevice, st), "H2D");
    ck(cudaMemcpyAsync(d_w, weights, (size_t)n_animals * sizeof(double), cudaMemcpyHostToDevice, st), "H2D");
    ck(tb_launch_marker_stats(c->geno(), c->m, d_pos, d_w, n_animals, d_out, d_out + c->m, d_out + 2 * (size_t)c->m, st), "launch");
    c->launches += 1;
    ck(cudaMemcpyAsync(sum_x, d_out, (size_t)c->m * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H");
    ck(cudaMemcpyAsync(sum_xx, d_out + c->m, (size_t)c->m * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H");
    ck(cudaMemcpyAsync(sum_xw, d_out + 2 * (size_t)c->m, (size_t)c->m * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H");
    ck(cudaStreamSynchronize(st), "execution");
  }
  cudaFree(d_pos);
  cudaFree(d_w);
  cudaFree(d_out);
  return rc;
}

int tb_set_stream(tb_ctx* c, void* cuda_stream) {
  if (!c) return -1;
  TB_CUDA(c, cudaSetDevice(c->device));
  TB_CUDA(c, cudaStreamSynchronize(c->stream));
  c->stream = cuda_stream ? reinterpret_cast<cudaStream_t>(cuda_stream) : c->own_stream;
  return 0;
}

int tb_microbench(tb_ctx* c, int which, double* out) {
  if (!c || !out) return -1;
  TB_CUDA(c, cudaSetDevice(c->device));
  if (which == 0) {
    TB_CUDA(c, tb_microbench_dmma(c->n_sm, c->stream, out));
    c->launches += 4;
    return 0;
  }
  if (which >= 1 && which <= 6) {
    TB_CUDA(c, tb_microbench_umma(which, c->n_sm, c->stream, out));
    c->launches += which >= 3 ? 126 : 4;
    return 0;
  }
  return fail(c, "tb_microbench: unknown probe");
}

}  // extern "C"
