// Internal declarations shared by the translation units of libtblup_b200.so (not part of the C-ABI).
#pragma once
#include <cuda_runtime.h>
#include <cuda.h>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>
#include <algorithm>

#define TB_MAX_SLOTS 64
#define TB_NB 64          // Cholesky block size (rows/cols per block column)
#define TB_GRAM_BM 128    // Gram tile rows
#define TB_GRAM_BN 256    // Gram tile cols
#define TB_GRAM_BK 128    // Gram K bytes per pipeline stage (one 128-byte swizzle span)
#define TB_GRAM_BN_FP4 224  // Gram tile cols of the fp4 (E2M1) variant: 2 x 224 accumulator columns + scale factors = TMEM
#define TB_GRAM_BK_FP4 256  // markers per k-block of the fp4 panel (128 bytes)

enum TbStage {
  TB_ST_H2D = 0,
  TB_ST_GATHER,
  TB_ST_CENTRE,
  TB_ST_GRAM,
  TB_ST_SCALE,
  TB_ST_CHOL_UPDATE,
  TB_ST_CHOL_PANEL,
  TB_ST_SOLVE,
  TB_ST_D2H,
  TB_ST_COUNT
};

struct TbRowSet {
  bool valid = false;
  int n_t = 0, n_v = 0;
  int ntp = 0;          // n_t rounded up to TB_NB
  int rows = 0;         // universe rows the Gram must cover (1 + max position used)
  int rpad = 0;         // rows rounded up to TB_GRAM_BM
  int* d_tpos = nullptr;        // [n_t] universe positions of the training animals
  int* d_vpos = nullptr;        // [n_v]
  int* d_colsum_train = nullptr;  // [m] dosage sums over the training animals
  double* d_yt_raw = nullptr;   // [ntp] (zero padded)
  double* d_yt_ctr = nullptr;   // [ntp] y_t minus its mean
  double* d_yv = nullptr;       // [n_v]
  double yt_mean = 0.0;         // mean phenotype of the training animals (intercept of the snp_blup model)
  std::vector<unsigned char> has_train;   // per 128-row universe block: contains a training animal
  bool contiguous = false;      // training animal b sits at universe position b
  // "contiguous with one hole": training animal i sits at i for i < hole0 and at i + gap beyond (hole0, gap multiples
  // of 8; gap = 0, hole0 = n_t when contiguous); valid_in_hole: the validation animals are exactly the hole, in order
  bool seg_ok = false;
  int hole0 = 0, gap = 0;
  bool valid_in_hole = false;
  // any OTHER row set can still be made a prefix by permuting the panel rows at gather time (training animals first,
  // then the validation animals; everyone else is dropped): d_rowmap[universe position] = panel row or -1,
  // d_ident = 0, 1, 2, ... (the position lists in panel order).  Needs disjoint, duplicate-free index lists.
  bool perm_ok = false;
  int* d_rowmap = nullptr;
  int* d_ident = nullptr;
  int rows_univ = 0;            // universe rows the gather has to visit (1 + max position used)
};

// resident genotypes as the kernels see them: exactly one of x (int8 dosages, [m][ldn]) and x2 (2-bit packed,
// [m][ld4], ld4 = ldn / 4, animal 4q + i of a marker in bits 2i..2i+1 of byte q) is non-null
struct TbGeno {
  const int8_t* x;
  int ldn;
  const uint8_t* x2;
  int ld4;
};

struct TbCtx {
  int device = 0;
  int n = 0, m = 0, ldn = 0;
  int8_t* d_x = nullptr;          // [m][ldn] SNP-major dosages, animals in universe order (storage 0)
  uint8_t* d_x2 = nullptr;        // [m][ldn / 4] the same matrix at 2 bits per dosage (storage 1; d_x is then freed)
  int storage = 0;
  TbGeno geno() const { return TbGeno{d_x, ldn, d_x2, ldn / 4}; }
  int* d_colsum_all = nullptr;    // [m]
  std::vector<double> y_univ;     // phenotypes in universe order (zeros when has_pheno is false)
  bool has_pheno = true;          // false: created without phenotypes (y = NULL), it only scores animals
  std::vector<int> pos_of;        // original animal index -> universe position
  TbRowSet slots[TB_MAX_SLOTS];
  cudaStream_t stream = nullptr;
  cudaStream_t own_stream = nullptr;

  // staged genomes
  int* d_idx = nullptr;           // flat marker lists
  size_t idx_cap = 0;
  std::vector<long long> h_off;   // [P+1]
  int P = 0;

  // wave workspace (grown on demand, reused)
  void* ws = nullptr;
  size_t ws_bytes = 0;
  size_t ws_limit = 0;            // user cap (0 = auto)
  int last_wave = 0;              // matrices per wave used by the last eval (diagnostics)

  // debug capture of the last wave's first individual
  int debug_keep = 0;

  std::vector<cudaEvent_t> ev_pool;     // events for profile mode
  size_t ev_used = 0;
  struct Span { int stage; size_t b, e; };
  std::vector<Span> spans;
  int profile = 0;                // 1: bracket every stage with events (serialises nothing: one stream)
  int stop_after = -1;            // debug: stop the pipeline after this stage
  int max_wave = 0;
  int precision = 0;              // 0: mixed (TF32 tensor-core Cholesky + fp64 refinement) when possible, 1: fp64
  int last_mixed = 0;
  int perm_rows = 1;              // 1: a single scattered row set becomes a prefix through a row permutation at gather time
  int last_perm = 0;
  int last_split = 0;             // the last multi-row-set evaluation ran one row set at a time (see eval_core)
  double* d_split = nullptr;      // [P] fitness of one row set while splitting
  size_t split_cap = 0;
  int gram_fp4 = 1;               // 1: E2M1 Gram (kind::mxf4) when the genotypes are resident in packed form
  int last_fp4 = 0;
  int narrow_c = 1;               // 1: int16 cross-products when every genome of the batch has 4 k <= 32 767
  int last_c16 = 0;
  double* d_fit_out = nullptr;    // device staging of the fitness vector for host-output calls
  size_t fit_cap = 0;
  int* d_fail = nullptr;          // [P * n_slots] per-job "mixed precision gave up" flags of the last evaluation
  size_t fail_cap = 0;
  long long last_issue_us = 0;    // host microseconds the last evaluation took to issue (diagnostics)
  int last_fallbacks = 0;         // jobs the last evaluation re-ran in fp64
  int last_fused = 0;
  int chain_inverse = 1;          // the fused chain kernel also forms the inverse of the 256-wide diagonal block
  int chain_fused = -1;           // fused diagonal-block chain (one launch per block column) for waves of at most this many jobs; -1: SM count
  int epi_warps = 16;             // epilogue warps of the Cholesky GEMM kernel (8: round-2 first version)
  int t16 = 1;                    // 1: block-column entries below the diagonal block live as halves in L16 between update and panel GEMM
  int panel_fused = 1;            // 1: with t16, those entries are updated and finished in one launch without leaving shared memory
  int wide_panel = 1;             // 1: 256-wide panel solve through the inverse of the diagonal block (chol_tc.cu)
  int fuse_scale = 1;             // 1: with one contiguous row set the scaled fp32 matrix is never written by a pass of
                                  //    its own (formed inside the Cholesky updates, or -- fuse_in_gram -- by the Gram epilogue)
  int fuse_in_gram = 0;           // 1: round-1 behaviour, the Gram epilogue writes the whole fp32 matrix
  int no_fallback = 0;
  int blk0_scale32 = 0;           // 1: block column 0 of the scaled matrix by scale32_kernel (round-2 first version)
  int gram_experiment = 0;
  int solve_pair = 1;             // solve with two CTAs per matrix: 0 never, 1 when the batch leaves half the CTA slots empty, 2 always
  int gram_pair = 2;              // Gram schedule: 0 one CTA per tile, 1 clusters of two CTAs sharing the B tile by TMA multicast,
                                  // 2 (default) tcgen05 CTA pairs: cta_group::2 MMAs, M = 256, each CTA holds half of the B tile
  int n_sm = 148;
  // layout of the last wave (for tb_debug_fetch)
  struct DbgLayout {
    int W = 0, n_slots = 0, rpad = 0, kstride = 0, centre_shared = 0;
    int32_t* C = nullptr; long long* s = nullptr; long long* SQ = nullptr;
    std::vector<double*> M, alpha, pred;
    float* L32 = nullptr; const unsigned short* L16 = nullptr; const float* Linv32 = nullptr; int* sweeps = nullptr;
    int ntp_all = 0;
    std::vector<int> ntp, n_v;
  } dbg;
  // on-device differential evolution (de.cu)
  struct DeState {
    int P = 0, k = 0;
    double *keys = nullptr, *child = nullptr, *fit = nullptr, *child_fit = nullptr, *raw_fit = nullptr;
    size_t raw_cap = 0;
    int *abc = nullptr, *fixed = nullptr, *take = nullptr;
    unsigned char* mask = nullptr;
    // SNP removal (tblup/evaluator.py:589-633): flags per marker, the same set as an ascending list, scratch rows
    unsigned char* banned = nullptr;
    int* banned_list = nullptr;
    int n_banned = 0;
    int* rows = nullptr;
    size_t rows_cap = 0;
    int* lens = nullptr;
    long long* d_off = nullptr;
  } de;
  double stage_ms[TB_ST_COUNT] = {};
  unsigned long long stage_launches[TB_ST_COUNT] = {};
  unsigned long long launches = 0;
  std::string err;
};

#define TB_CUDA(ctx, call)                                                                             \
  do {                                                                                                 \
    cudaError_t e__ = (call);                                                                          \
    if (e__ != cudaSuccess) {                                                                          \
      (ctx)->err = std::string(#call) + ": " + cudaGetErrorString(e__) + " @" + __FILE__ + ":" +       \
                   std::to_string(__LINE__);                                                           \
      return -2;                                                                                       \
    }                                                                                                  \
  } while (0)

__host__ __device__ static inline int tb_round_up(int x, int q) { return (x + q - 1) / q * q; }

// ---- launchers (each defined in its own .cu); all asynchronous on `st`, return cudaGetLastError() ----

// ingest.cu
cudaError_t tb_launch_transpose_rows(const int8_t* d_rows, int n_rows, int m, int8_t* d_x, int ldn, int pos0,
                                     cudaStream_t st);
cudaError_t tb_launch_colsum(const TbGeno& g, int m, const int* d_pos, int n_pos, int* d_colsum, cudaStream_t st);
cudaError_t tb_launch_marker_stats(const TbGeno& g, int m, const int* d_pos, const double* d_w, int n_pos, double* d_sx,
                                   double* d_sxx, double* d_sxw, cudaStream_t st);
cudaError_t tb_launch_pack2(const int8_t* d_x, int ldn, int m, uint8_t* d_x2, cudaStream_t st);
cudaError_t tb_launch_unpack2_perm(const uint8_t* d_rows2, int n_rows, int stride, const int* d_perm, int n,
                                   int8_t* d_x, int ldn, int j0, int* d_bad, cudaStream_t st);

// gather.cu
cudaError_t tb_launch_gather(const TbGeno& g, const int* d_idx, const long long* d_off, int w0, int W,
                             int rpad, int kstride, int8_t* d_panel, cudaStream_t st);
// fp4 panel: E2M1 nibbles, two markers per byte, kstride_b bytes per animal row (= padded k / 2), from packed genotypes
// d_rowmap (nullable): panel row of every universe position (-1 = not gathered), rows_univ = positions to visit
cudaError_t tb_launch_gather_fp4(const TbGeno& g, const int* d_idx, const long long* d_off, int w0, int W, int rpad,
                                 int kstride_b, int8_t* d_panel, cudaStream_t st, const int* d_rowmap = nullptr,
                                 int rows_univ = 0);
cudaError_t tb_gather_init();
cudaError_t tb_launch_centre_terms(const int8_t* d_panel, int rpad, int kstride, const int* d_idx,
                                   const long long* d_off, int w0, int W, int n_slots, const int* d_kblocks,
                                   const int* const* d_colsum_of, /* [W*n_slots] device ptrs */
                                   int* d_csg /* [W*n_slots][kstride] scratch */, long long* d_s, long long* d_SQ,
                                   cudaStream_t st,
                                   int fp4 = 0 /* 1: panel rows hold nibbles, kstride counts markers; 2: also split-byte sums + dp4a */);

// gram_tc.cu / gram_simt.cu
cudaError_t tb_gram_tc_init();
struct TbScaleJob;
// c16 != 0: d_C receives int16 entries (row stride still rpad elements); the caller guarantees 4 k <= 32 767.
// d_fuse_jobs != nullptr (one contiguous row set, mixed precision): the epilogue also writes the fp32 matrix
// A = G_tt + lambda I of every genome into d_L32 [W][ntp_all][ntp_all] (what tb_launch_scale32 would produce)
cudaError_t tb_launch_gram_tc(const int8_t* d_panel, int W, int rpad, int kstride, const int* d_kblocks,
                              const int* d_tiles, int n_tiles, int32_t* d_C, int n_sm, cudaStream_t st,
                              std::string* err, const TbScaleJob* d_fuse_jobs = nullptr, float* d_L32 = nullptr,
                              int ntp_all = 0, int c16 = 0, int fp4 = 0, int pair = 0);
cudaError_t tb_launch_gram_simt(const int8_t* d_panel, int W, int rpad, int kstride, const int* d_kblocks,
                                int32_t* d_C, cudaStream_t st);

// scale.cu
struct TbScaleJob {       // one (individual, rowset) matrix
  const int32_t* C;       // [rpad][rpad] lower triangle valid (int16 entries when the wave runs in C16 mode)
  const long long* s;     // [rpad]
  const long long* SQ;    // {S, Q}
  const int* tpos;
  const int* vpos;
  double* M;              // [ntp + n_v][ntp]: A on top (lower triangle + ridge), G_vt below
  long long N;            // animals behind the allele frequencies
  int n_t, n_v, ntp, rpad;
  double lambda;
  int hole0, gap, cw;     // "prefix with one aligned hole" (TbRowSet) and the genome's index in the wave (TbFromC)
};
cudaError_t tb_launch_scale(const TbScaleJob* d_jobs, int n_jobs, int max_rows, int max_ntp, cudaStream_t st);

// chol.cu
struct TbCholJob {
  double* M;        // [ntp + n_v][ntp]
  double* Linv;     // [ntp / TB_NB][TB_NB][TB_NB] inverses of the diagonal blocks
  int ntp;
  int* status;      // set to 1 if a pivot was not positive
};
cudaError_t tb_chol_init();
cudaError_t tb_launch_chol_update(const TbCholJob* d_jobs, int n_jobs, int max_ntp, int j, cudaStream_t st);
cudaError_t tb_launch_chol_diag(const TbCholJob* d_jobs, int n_jobs, int max_ntp, int j, cudaStream_t st);
cudaError_t tb_launch_chol_panel(const TbCholJob* d_jobs, int n_jobs, int max_ntp, int j, cudaStream_t st);

// solve.cu
struct TbSolveJob {
  const double* M;
  const double* Linv;
  const double* y_t;   // [ntp]
  const double* y_v;   // [n_v]
  const int* status;
  double* alpha;       // [ntp] scratch / debug
  double* pred;        // [n_v] scratch / debug
  double* fitness;     // one value
  int n_t, n_v, ntp;
};
cudaError_t tb_solve_init();
cudaError_t tb_launch_solve(const TbSolveJob* d_jobs, int n_jobs, int max_ntp, cudaStream_t st);

// solve_mixed.cu / chol_tc.cu (mixed-precision path)
struct TbSolveMixedJob {
  const float* L32;        // [ntp][ntp] TF32 Cholesky factor (lower)
  const void* L16;         // [ntp][ntp] the same factor in fp16 (same 10-bit mantissa): what the solve streams
  const float* Linv32;     // [ntp][64] inverses of its diagonal blocks
  const int32_t* C;        // [rpad][rpad] integer cross-products
  const long long* s;      // [rpad]
  const long long* SQ;     // {S, Q}
  const int* tpos;
  const int* vpos;
  const double* y_t;       // [ntp]
  const double* y_v;       // [n_v]
  const int* status;
  double* alpha;           // [ntp]
  double* pred;            // [n_v]
  double* fitness;
  int* sweeps;             // refinement sweeps used (diagnostics)
  int* fail;               // set to 1 when the mixed-precision solve did not reach the tolerance (or a pivot failed)
  long long N;
  int n_t, n_v, ntp, rpad;
  int hole0, gap, valid_in_hole;   // see TbRowSet (contiguous kernels only)
  double lambda;
  int cmax;                // bound on the cross-products of this genome: 4 k (every dosage <= 2)
};
cudaError_t tb_solve_mixed_init();
void tb_solve_mixed_set_debug(int v);
bool tb_solve_mixed_fits(int ntp);
cudaError_t tb_launch_solve_mixed(const TbSolveMixedJob* d_jobs, int n_jobs, int ntp, int contiguous, int c16, int hole,
                                  cudaStream_t st, int n_sm = 148, int pair_mode = 1);
// col_end > 0: only columns [0, col_end) (the first outer block column of the factorisation)
cudaError_t tb_launch_scale32(const TbScaleJob* d_jobs, int n_jobs, int ntp, float* L32, int c16, cudaStream_t st,
                              int col_end = 0);
// The fp32 matrix A = G_tt + lambda I is never materialised as a whole: block column J of the factorisation is formed
// inside the epilogue of ITS outer update, T = A[:, J] - L[:, 0:J] L[J, 0:J]^T, with A evaluated on the fly from the
// integer cross-products (2 or 4 bytes per entry instead of a 4-byte read of a matrix the Gram would have had to write).
// terms: per job [2][ntp] floats -- row terms -(2N/den) s_a, then column terms (2/den)(Q - N s_b) (zero beyond n_t);
// coef: per job {2 N^2 / den, lambda, n_t, hole0, gap, genome index}.  Row sets that are a prefix of the panel rows, or a
// prefix with one 8-aligned hole (k-fold training sets): training animal a sits at panel row a + (a >= hole0 ? gap : 0).
struct TbFuseCoef {
  float scale, lam;
  int n_t, hole0, gap, cw;
};
struct TbFromC {
  const void* C;        // [genomes][rpad][rpad] cross-products (int16 when c16)
  const float* terms;   // [n_jobs][2][ntp]
  const TbFuseCoef* coef;   // [n_jobs]
  int rpad, c16;
  int skip_blk0;        // block column 0 was already written by a scaling pass (A/B option)
};
cudaError_t tb_launch_fuse_terms(const TbScaleJob* d_jobs, int n_jobs, int ntp, float* terms, TbFuseCoef* coef,
                                 cudaStream_t st);
cudaError_t tb_chol_tc_init();
// Linv256 (nullable): [n_jobs][256][256] scratch for the inverses of the 256-wide diagonal blocks (wide panel path)
cudaError_t tb_chol_tc_factor(float* L32, float* Linv32, void* L16, float* Linv256, int* status, int n_jobs, int ntp,
                              int n_sm, cudaStream_t st, int* launches, std::string* err,
                              void (*mark)(void*, int, int), void* mark_ctx, const TbFromC* from_c = nullptr,
                              int t16 = 1, int epi_warps = 16, int chain_fused_jobs = 0, int panel_fused = 1);

// reml.cu: restricted log-likelihood of one (genome, h2) job after the fp64 factorisation of A = G_TT + lambda I
struct TbRemlJob {
  const double* M;       // [ntp][ntp] L (lower triangle) as chol.cu leaves it
  const double* Linv;    // [ntp / TB_NB][TB_NB][TB_NB] inverses of its diagonal blocks
  const double* y;       // [ntp] training phenotypes minus their mean (zero padded)
  const int* status;     // non-zero: a pivot was not positive
  double ymean;          // mean training phenotype (mu = ymean + b / a)
  int n_t, ntp;
  double* loglik;        // one value each
  double* sigma_g2;
  double* mu;
};
cudaError_t tb_reml_init();
cudaError_t tb_launch_reml(const TbRemlJob* d_jobs, int n_jobs, int max_ntp, cudaStream_t st);
// one chunk of a REML profile for eval_core: jobs (staged genome g, point s) for s < n, h2 of the job
// h2[g * ld + s0 + s] (ld = 0: one list shared by every genome), outputs at [g][n_out] entry s0 + s (device)
struct TbRemlReq {
  const double* h2;
  long long ld;
  int s0, n, n_out;
  double* d_loglik;
  double* d_sigma_g2;
  double* d_mu;
};

// microbench.cu
cudaError_t tb_microbench_dmma(int n_sm, cudaStream_t st, double* tflops);
cudaError_t tb_microbench_umma(int which, int n_sm, cudaStream_t st, double* tops);

// api.cu internals used by de.cu: evaluate the genomes already staged on the device (c->d_idx, c->h_off, c->P)
// into a device buffer [P * n_slots] (asynchronous on c->stream), and fold the profiling spans after a sync.
int tb_internal_eval_device(TbCtx* c, const int32_t* slots, int n_slots, double h2, int mode_rule, double* d_fit);
// the same on ONE row set, also writing every genome's solution: d_alpha [P][ntp of the row set], entry i of genome g
// belonging to the training animal at d_tpos[i] of the row set (entries beyond n_t are padding) -- used by tb_fit_effects
int tb_internal_eval_alpha(TbCtx* c, int slot, double h2, int mode_rule, double* d_fit, double* d_alpha);
// REML jobs (genome x h2 point) on ONE row set: gather, centring terms and Gram once per genome, then one fp64 A =
// G_TT + lambda_job I per job (no G_vt rows), the fp64 Cholesky whatever `precision` says, and reml_kernel
int tb_internal_eval_reml(TbCtx* c, int slot, int mode_rule, const TbRemlReq* req);
void tb_internal_collect_spans(TbCtx* c);
void tb_de_release(TbCtx* c);
