// Knockout local search on the device (SURVEY.md 8f row F4): tblup/local.py:50-76 walks the best individual's markers
// in order, evaluates the genome without marker i -- `evaluator.blup(genome[mask], ...)`, one sequential fitness
// evaluation per marker -- and keeps the marker out when the fitness improves.  Each decision depends on the drops
// accepted before it, so the sequence is greedy; here it runs as SPECULATIVE BATCHES through the ordinary pipeline:
//
//   base = genome[mask]  (device list)
//   candidates i .. i+B-1: base without its entry for marker i+c, built by one kernel straight into the staged batch
//   one batched evaluation (gather -> Gram -> Cholesky -> solve, like a generation)
//   scan in order: the first candidate that improves is accepted (exactly the reference's `fitness > best_fitness`,
//   NaN never wins); candidates after it were scored with that marker still present, so the next batch starts there.
//
// Each decision compares the fitness of the list the sequential loop would score at that step; a batch costs about what
// ONE single-genome evaluation costs (the pipeline is latency-bound below ~150 genomes), so the search is between 1x
// and Bx faster than the sequential loop depending on how often a drop is accepted.  The batch size adapts to the
// observed acceptance gaps.  A candidate's fitness is the same bits whatever batch it is scored in as long as the
// mixed-precision solve runs one CTA per matrix (option solve_pair 0; DESIGN section 4 states what the tests hold).
// tb_knockout_scan is the non-greedy companion: the fitness of every leave-one-out list of a fixed genome.
//
// Both calls score their candidates in an index buffer of their own and leave the staged batch (tb_stage_genomes)
// as they found it, on every way out, errors included: tb_eval_staged afterwards evaluates what the caller staged.
#include "tb_internal.h"
#include "../../include/tblup_b200.h"

namespace {

int ko_fail(TbCtx* c, const std::string& msg, int code = -1) {
  c->err = msg;
  return code;
}

// out[cand][t] = base[t] (t < q) or base[t + 1] (t >= q), q = q0 + cand: the list without its q-th entry
__global__ void knockout_lists_kernel(const int* __restrict__ base, int L, int q0, int* __restrict__ out) {
  const int cand = blockIdx.y, q = q0 + cand;
  int* dst = out + (size_t)cand * (L - 1);
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < L - 1; t += gridDim.x * blockDim.x)
    dst[t] = base[t < q ? t : t + 1];
}

// base <- base without its q-th entry (in place on a scratch copy; called once per accepted drop)
__global__ void knockout_drop_kernel(const int* __restrict__ src, int L, int q, int* __restrict__ dst) {
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < L - 1; t += gridDim.x * blockDim.x) dst[t] = src[t < q ? t : t + 1];
}

struct Scratch {
  int* base[2] = {nullptr, nullptr};
  double* fit = nullptr;
  int* idx = nullptr;             // the candidate lists of one batch
  size_t idx_cap = 0;
  ~Scratch() {
    cudaFree(base[0]);
    cudaFree(base[1]);
    cudaFree(fit);
    cudaFree(idx);
  }
};

// The caller's staged batch, set aside for the length of one call (the fp64 fallback of api.cu swaps its sub-batch in
// the same way).  Declared after the Scratch it points into, so that it is put back before that Scratch is freed.
struct StagedBatch {
  TbCtx* c;
  std::vector<long long> off;
  int* idx;
  size_t cap;
  int P;
  explicit StagedBatch(TbCtx* ctx) : c(ctx), idx(ctx->d_idx), cap(ctx->idx_cap), P(ctx->P) { off.swap(c->h_off); }
  ~StagedBatch() {
    c->h_off.swap(off);
    c->d_idx = idx;
    c->idx_cap = cap;
    c->P = P;
  }
};

// score candidates q0 .. q0 + B - 1 of the base list (length L) on row set `slot` -> h_fit[0 .. B); the candidate
// lists go to sc.idx (B (L - 1) entries, allocated by the caller) and are staged from there
int score_batch(TbCtx* c, Scratch& sc, const int* d_base, int L, int q0, int B, int slot, double h2, int mode_rule,
                double* d_fit, std::vector<double>& h_fit) {
  if ((size_t)B * (L - 1) > sc.idx_cap) return ko_fail(c, "internal: knockout batch exceeds its index buffer");
  dim3 grid((unsigned)std::min(32, (L - 1 + 255) / 256), (unsigned)B);
  knockout_lists_kernel<<<grid, 256, 0, c->stream>>>(d_base, L, q0, sc.idx);
  TB_CUDA(c, cudaGetLastError());
  c->launches += 1;
  c->d_idx = sc.idx;
  c->idx_cap = sc.idx_cap;
  c->h_off.resize(B + 1);
  for (int i = 0; i <= B; ++i) c->h_off[i] = (long long)i * (L - 1);
  c->P = B;
  const int32_t slots[1] = {slot};
  if (int rc = tb_internal_eval_device(c, slots, 1, h2, mode_rule, d_fit)) return rc;
  h_fit.resize(B);
  TB_CUDA(c, cudaMemcpyAsync(h_fit.data(), d_fit, (size_t)B * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  TB_CUDA(c, cudaStreamSynchronize(c->stream));
  tb_internal_collect_spans(c);
  return 0;
}

int check_args(TbCtx* c, const int32_t* genome, int k, int slot, double h2, int mode_rule, const char* who) {
  if (!genome || k < 2) return ko_fail(c, std::string(who) + ": need a genome of at least 2 markers");
  if (slot < 0 || slot >= TB_MAX_SLOTS || !c->slots[slot].valid) return ko_fail(c, std::string(who) + ": row set is not defined");
  if (!(h2 > 0.0) || !(h2 <= 1.0)) return ko_fail(c, std::string(who) + ": heritability must be in (0, 1]");
  if (mode_rule < 0 || mode_rule > 2) return ko_fail(c, std::string(who) + ": bad mode_rule");
  for (int i = 0; i < k; ++i)
    if (genome[i] < 0 || genome[i] >= c->m) return ko_fail(c, std::string(who) + ": marker index out of range");
  return 0;
}

}  // namespace

extern "C" {

int tb_knockout_scan(tb_ctx* c, const int32_t* genome, int k, int slot, double h2, int mode_rule, double* fitness_out) {
  if (!c) return -1;
  if (!fitness_out) return ko_fail(c, "tb_knockout_scan: null output");
  if (int rc = check_args(c, genome, k, slot, h2, mode_rule, "tb_knockout_scan")) return rc;
  TB_CUDA(c, cudaSetDevice(c->device));
  Scratch sc;
  StagedBatch staged(c);
  sc.idx_cap = (size_t)std::min(k, 1024) * (k - 1);
  TB_CUDA(c, cudaMalloc(&sc.idx, sc.idx_cap * sizeof(int)));
  TB_CUDA(c, cudaMalloc(&sc.base[0], (size_t)k * sizeof(int)));
  TB_CUDA(c, cudaMalloc(&sc.fit, (size_t)std::min(k, 1024) * sizeof(double)));
  TB_CUDA(c, cudaMemcpyAsync(sc.base[0], genome, (size_t)k * sizeof(int), cudaMemcpyHostToDevice, c->stream));
  std::vector<double> h;
  for (int q0 = 0; q0 < k; q0 += 1024) {
    const int B = std::min(1024, k - q0);
    if (int rc = score_batch(c, sc, sc.base[0], k, q0, B, slot, h2, mode_rule, sc.fit, h)) return rc;
    for (int i = 0; i < B; ++i) fitness_out[q0 + i] = h[i];
  }
  return 0;
}

int tb_knockout(tb_ctx* c, const int32_t* genome, int k, int slot, double h2, int mode_rule, double start_fitness,
                uint8_t* keep_out, double* best_fitness_out, int32_t* n_evals_out, int32_t* n_batches_out) {
  if (!c) return -1;
  if (!keep_out || !best_fitness_out) return ko_fail(c, "tb_knockout: null output");
  if (int rc = check_args(c, genome, k, slot, h2, mode_rule, "tb_knockout")) return rc;
  TB_CUDA(c, cudaSetDevice(c->device));
  Scratch sc;
  StagedBatch staged(c);
  sc.idx_cap = (size_t)std::min(k, 1024) * (k - 1);     // the largest batch: min(k, 1 024) lists of k - 1 markers
  TB_CUDA(c, cudaMalloc(&sc.idx, sc.idx_cap * sizeof(int)));
  TB_CUDA(c, cudaMalloc(&sc.base[0], (size_t)k * sizeof(int)));
  TB_CUDA(c, cudaMalloc(&sc.base[1], (size_t)k * sizeof(int)));
  TB_CUDA(c, cudaMalloc(&sc.fit, 1024 * sizeof(double)));
  TB_CUDA(c, cudaMemcpyAsync(sc.base[0], genome, (size_t)k * sizeof(int), cudaMemcpyHostToDevice, c->stream));
  for (int i = 0; i < k; ++i) keep_out[i] = 1;
  int cur = 0;          // which scratch buffer holds the current list
  int L = k;            // its length
  int kept_before = 0;  // markers kept among the original positions [0, i)
  double best = start_fitness;
  int evals = 0, batches = 0;
  int B_next = 32;
  std::vector<double> h;
  int i = 0;
  while (i < k && L >= 2) {
    const int B = std::min(std::min(B_next, 1024), k - i);
    if (int rc = score_batch(c, sc, sc.base[cur], L, kept_before, B, slot, h2, mode_rule, sc.fit, h)) return rc;
    ++batches;
    int used = B;
    bool accepted = false;
    for (int b = 0; b < B; ++b) {
      if (h[b] > best) {              // tblup/local.py:68 (NaN compares false: never accepted)
        best = h[b];
        keep_out[i + b] = 0;
        used = b + 1;
        accepted = true;
        break;
      }
    }
    evals += used;                    // evaluations whose result the greedy sequence actually consumed
    if (accepted) {
      const int q = kept_before + used - 1;      // position of the dropped marker in the current list
      knockout_drop_kernel<<<std::min(64, (L + 255) / 256), 256, 0, c->stream>>>(sc.base[cur], L, q, sc.base[cur ^ 1]);
      TB_CUDA(c, cudaGetLastError());
      c->launches += 1;
      cur ^= 1;
      L -= 1;
      kept_before += used - 1;
      // acceptance after `used` candidates: aim the next batch at about twice that gap
      B_next = std::max(16, std::min(1024, 2 * used + 8));
    } else {
      kept_before += used;
      B_next = std::min(1024, 2 * B);
    }
    i += used;
  }
  TB_CUDA(c, cudaStreamSynchronize(c->stream));
  *best_fitness_out = best;
  if (n_evals_out) *n_evals_out = evals;
  if (n_batches_out) *n_batches_out = batches;
  return 0;
}

}  // extern "C"
