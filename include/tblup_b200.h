/* libtblup_b200 -- C ABI of the B200-native GBLUP fitness path.
 *
 * The reference (ianwhale/tblup, pure Python) has no FFI: its seam for this path is the evaluator
 * object that tblup/utils.py:48,59 builds through `get_evaluator(args)` and that
 * tblup/population.py:47,68 and main.py:35 call.  These entry points are what a ctypes binding placed
 * behind that seam needs (INTEGRATION.md shows the binding); each one names the reference code whose
 * work it takes over.  Conventions: plain pointers and sizes, caller keeps ownership of every host
 * buffer, return 0 on success / negative on error (message via tb_last_error), nothing throws across
 * the boundary, one host thread per context, every call returns with its results valid
 * (internally asynchronous on the context's own CUDA stream).
 */
#ifndef TBLUP_B200_H
#define TBLUP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct TbCtx tb_ctx;

#define TB_ABI_VERSION 1

/* branch rule of BlupParallelEvaluator.blup (tblup/evaluator.py:257-263) */
#define TB_MODE_AUTO 0    /* len(indices) > n  -> gblup, else snp_blup */
#define TB_MODE_GBLUP 1   /* allele frequencies over ALL animals, raw y      (evaluator.py:265-286) */
#define TB_MODE_SNPBLUP 2 /* frequencies over the training animals, centred y (evaluator.py:288-314) */

/* pipeline stages, index into tb_stage_times() and `stop_after` */
enum {
  TB_STAGE_H2D = 0, TB_STAGE_GATHER, TB_STAGE_CENTRE, TB_STAGE_GRAM, TB_STAGE_SCALE,
  TB_STAGE_CHOL_UPDATE, TB_STAGE_CHOL_PANEL, TB_STAGE_SOLVE, TB_STAGE_D2H, TB_STAGE_COUNT
};

/* what tb_debug_fetch() can copy back from the last wave (job = individual * n_slots + slot) */
enum {
  TB_DBG_C = 0,     /* int32  [rpad*rpad]      uncentred cross-products (lower triangle valid)      */
  TB_DBG_S = 1,     /* int64  [rpad]           s_a = sum_j x_aj colsum_j                             */
  TB_DBG_SQ = 2,    /* int64  [2]              S = sum colsum, Q = sum colsum^2                      */
  TB_DBG_M = 3,     /* double [(ntp+n_v)*ntp]  [A ; G_vt] (A holds L after the factorisation)        */
  TB_DBG_ALPHA = 4, /* double [ntp]                                                                  */
  TB_DBG_PRED = 5,  /* double [n_v]                                                                  */
  TB_DBG_DIMS = 6,  /* int32  [4]              rpad, ntp, n_v, kstride                               */
  TB_DBG_L32 = 7,   /* float  [ntp*ntp]        TF32 Cholesky factor (mixed precision mode only)      */
  TB_DBG_SWEEPS = 8, /* int32 [1]              refinement sweeps the solve needed (mixed mode)       */
  TB_DBG_LINV32 = 9  /* float [ntp/64][64][64]  inverses of the 64x64 diagonal blocks the solve applies (mixed mode) */
};

int tb_abi_version(void);

/* Message of the last failed call on ctx (ctx == NULL: last failed tb_create). */
const char* tb_last_error(const tb_ctx* ctx);

/* Upload a data set once.  Takes over `np.load(data_path)` / `np.load(labels_path)` of every worker
 * (tblup/evaluator.py:215-216).  geno: [n][m] dosages in {0,1,2}, animal-major (the .npy layout);
 * y: [n], or NULL for a context without phenotypes (it only scores animals with tb_predict_effects; row sets and
 * everything built on them are refused); perm: [n] or NULL, animal stored at "universe" position p is perm[p] (put the animals the
 * fitness reads first: training, validation, testing -- the Gram then only covers that prefix). */
int tb_create(const int8_t* geno, int n, int m, const double* y, const int32_t* perm, int device, tb_ctx** out);

/* Same, with the input layout and the resident storage chosen by the caller (the reference only knows the dense
 * float64 .npy of tblup/utils.py:95 / evaluator.py:188,215; at 20 000 x 500 000 that file would be 80 GB).
 * layout TB_LAYOUT_INT8_ANIMAL_MAJOR: geno = int8 [n][m] as above.
 * layout TB_LAYOUT_PACKED2_SNP_MAJOR: geno = uint8 [m][ceil(n/4)], marker-major, animal 4q+i of a marker in bits
 *   2i..2i+1 of byte q (the row layout and bit order of a PLINK .bed body), each 2-bit code being the dosage 0/1/2;
 *   code 3 is rejected (the reference has no missing-value handling).
 * storage TB_STORE_INT8: resident as int8 dosages (m x n bytes); TB_STORE_PACKED2: resident at 2 bits per dosage
 *   (m x n / 4 bytes), expanded inside the gather kernel.  Results are bit-identical between the two. */
#define TB_LAYOUT_INT8_ANIMAL_MAJOR 0
#define TB_LAYOUT_PACKED2_SNP_MAJOR 1
#define TB_STORE_INT8 0
#define TB_STORE_PACKED2 1
int tb_create_ex(const void* geno, int layout, int storage, int n, int m, const double* y, const int32_t* perm,
                 int device, tb_ctx** out);
int tb_destroy(tb_ctx* ctx);
/* A context on another GPU of the same box holding the same data set, filled by a device-to-device copy of the resident
 * matrix and column sums (NVLink peer copy) instead of a second host ingest -- the reference has every worker np.load()
 * the matrix again (tblup/evaluator.py:215-216).  Row sets are defined on the clone with tb_set_rowset as usual. */
int tb_clone(const tb_ctx* src, int device, tb_ctx** out);
/* resident genotype bytes and storage kind (TB_STORE_*) of a context */
int tb_storage_info(const tb_ctx* ctx, int* storage, uint64_t* bytes);

/* Define row set `slot`: the (train_indices, validation_indices) pair of tblup/evaluator.py:316-322,
 * :485-491, :555-561 (original animal indices).  Precomputes the training-row dosage sums
 * (np.mean(X_train, axis=0) of evaluator.py:304) and the centred phenotypes. */
int tb_set_rowset(tb_ctx* ctx, int slot, const int32_t* train, int n_train, const int32_t* valid, int n_valid);

/* Host helper (no device work, no context): pack P index lists -- the `genome` arrays of P individuals, each a
 * contiguous int32 (elem_bytes 4) or int64 (8) numpy buffer -- into one flat int32 list for tb_stage_genomes / tb_eval,
 * with numpy fancy-indexing semantics (tblup/evaluator.py:275, :298): an index in [-m, 0) wraps to index + m,
 * anything else outside [0, m) fails: returns -3 with *bad_index = the first offending value of the lowest-numbered
 * list that has one.  idx_off (P + 1 entries) receives the offsets.  Takes the place of the per-individual pickling of
 * evaluator.py:392-393 on the way to the workers; runs on up to 8 host threads for a generation-sized batch. */
int tb_pack_index_lists(const void* const* lists, const int64_t* lens, const int32_t* elem_bytes, int P, int64_t m,
                        int32_t* idx_flat, int64_t* idx_off, int64_t* bad_index);

/* Copy a batch of genomes (ragged marker-index lists, duplicates allowed; idx_off has P+1 entries) to
 * the device: the payload of P enqueue() calls (tblup/evaluator.py:227-241, :392-393). */
int tb_stage_genomes(tb_ctx* ctx, const int32_t* idx_flat, const int64_t* idx_off, int P);

/* Evaluate the staged batch on each listed row set: fitness_out[i * n_slots + s] =
 * BlupParallelEvaluator.blup(genome_i, train_s, valid_s, data, labels, h2) (tblup/evaluator.py:244-314),
 * the work of the worker loop at evaluator.py:205-225 and the gather at :396-398.
 * fitness_out is a host pointer, or a device pointer on ctx's device when out_is_device != 0. */
int tb_eval_staged(tb_ctx* ctx, const int32_t* slots, int n_slots, double h2, int mode_rule,
                   double* fitness_out, int out_is_device);

/* tb_stage_genomes + tb_eval_staged with host buffers: one call per _evaluate() (evaluator.py:380-405). */
int tb_eval(tb_ctx* ctx, const int32_t* slots, int n_slots, const int32_t* idx_flat, const int64_t* idx_off,
            int P, double h2, int mode_rule, double* fitness_out);

/* Raw uncentred cross-products of one genome over universe rows [0, rows): out[a*rows + b], b <= a
 * (upper triangle zero).  impl 0 = tcgen05 int8 kernel, 1 = plain dp4a verification kernel, 2 = tcgen05 fp4 (E2M1)
 * kernel (packed resident genotypes only); 3 / 4 = the int8 / fp4 kernel run as clusters of two CTAs that share the
 * B tile by TMA multicast (what evaluations use by default).
 * The integer part of make_grm (tblup/utils.py:17). */
int tb_gram_debug(tb_ctx* ctx, const int32_t* idx, int k, int rows, int impl, int32_t* out);

int tb_debug_fetch(tb_ctx* ctx, int what, int job, void* out, size_t nbytes);

/* options: "profile" (0/1: per-stage CUDA-event timing), "stop_after" (stage index, -1 = run all),
 * "workspace_mb" (cap for the wave workspace, 0 = auto), "max_wave" (cap individuals per wave, 0 = auto),
 * "precision" (0 = mixed: TF32 tensor-core Cholesky as preconditioner + fp64 refinement against the exact
 * integer operator [default]; 1 = fp64 Cholesky throughout),
 * "fuse_scale" (0/1, default 1: with one contiguous row set in mixed precision the Gram epilogue writes the scaled
 * fp32 matrix itself), "wide_panel" (0/1, default 1: 256-wide Cholesky panel through the inverse of the diagonal
 * block), "narrow_c" (0/1, default 1: int16 storage of the cross-products when 4 k <= 32 767 for the whole batch),
 * "gram_fp4" (0/1, default 1: with packed resident genotypes the Gram runs on E2M1 operands, tcgen05 kind::mxf4 --
 * dosages 0/1/2 are exact in E2M1 and the fp32 accumulators hold the same integers; 0 = int8 operands),
 * "gram_pair" (0/1, default 1: the Gram runs as clusters of two CTAs taking row blocks (I, I+1) of one column block together, the
 * shared B tile fetched half by each and TMA-multicast to both), "fuse_in_gram" (0/1, default 0: the Gram epilogue writes
 * the whole scaled fp32 matrix as in round 1; by default the Cholesky updates form it from the cross-products),
 * "perm_rows" (0/1, default 1: a single scattered row set -- Monte-Carlo split, unaligned fold, custom splitter -- is
 * turned into a prefix by permuting the panel rows at gather time, so it runs the contiguous kernels),
 * "solve_pair" (0 = one CTA per matrix, 2 = a cluster of two, 1 = by batch size [default]),
 * "t16" (0/1, default 1: the entries of a Cholesky block column below its diagonal block are kept as halves between
 * the update that forms them and the panel GEMM that finishes them in place; 0 = fp32 / TF32 as in the first version),
 * "panel_fused" (0/1, default 1: with t16, those entries are formed and finished in ONE launch after the diagonal
 * chain -- update, then product with the inverse of the diagonal block, the intermediate kept in shared memory; the
 * factor is bit-identical to 0 = the update of the whole block column, then the panel GEMM as its own launch),
 * "epi_warps" (8 or 16 [default]: epilogue warps of the Cholesky GEMM kernel), "chain_fused" (the 64 x 64
 * diagonal-block chain of a block column runs as ONE shared-memory kernel for waves of at most this many jobs;
 * -1 = the SM count [default], 0 = never), "chain_inverse" (0/1, default 1: that kernel also forms the inverse of the
 * 256-wide diagonal block).  The A/B options change speed, never results beyond the refinement tolerance. */
int tb_set_option(tb_ctx* ctx, const char* name, long long value);

/* Facts about the last evaluation / the context: "last_c16", "last_fused_scale", "last_mixed", "last_wave",
 * "storage", "wide_panel", "panel_fused", "de_removed" (size of the removed-marker set), "staged" (genomes staged), "last_fp4", "last_perm", "last_split",
 * "last_fallbacks" (jobs of the last evaluation whose mixed-precision solve gave up -- pivot breakdown or no
 * convergence, h2 close to 1 -- and that were evaluated again with the fp64 Cholesky). */
int tb_get_info(const tb_ctx* ctx, const char* name, long long* value);
/* Offsets (P + 1 entries, P = tb_get_info "staged") of the ragged batch currently staged on the device. */
int tb_staged_offsets(const tb_ctx* ctx, int64_t* off_out, int n);

/* Accumulated per-stage device milliseconds (valid with profile=1) and kernel launches since the last
 * tb_reset_counters(); either pointer may be NULL. */
int tb_stage_times(tb_ctx* ctx, double* ms_out, uint64_t* launches_out);
uint64_t tb_launch_count(const tb_ctx* ctx);
int tb_reset_counters(tb_ctx* ctx);
int tb_last_wave(const tb_ctx* ctx);
/* precision mode the last evaluation ran in: 0 = mixed, 1 = fp64 */
int tb_last_precision(const tb_ctx* ctx);

/* Run the context's work on a caller-owned CUDA stream (e.g. torch's current stream, so the caller's CUDA
 * events bracket it); NULL restores the context's own stream. */
int tb_set_stream(tb_ctx* ctx, void* cuda_stream);

/* Peak probes for roofline denominators (the Gram of tblup/utils.py:17 is reported against them): which = 0 -> fp64 DMMA
 * (mma.sync m8n8k4) TFLOP/s; 1 -> tcgen05 kind::i8 TOP/s and 2 -> tcgen05 kind::mxf4 (E2M1) TOP/s, M128 x N256 MMAs
 * issued back to back on shared-memory-resident operands, one CTA per SM (2 ops per multiply-accumulate): best of
 * three ~20 ms launches on random operand bits (burst); 3 / 4 -> the same two SUSTAINED (back to back for ~2.5 s, rate over
 * the last ~1.5 s, when the clock has settled under the board's power cap); 5 / 6 -> sustained with genotype-like operands
 * (dosages 0/1/2 at realistic frequencies: fewer toggling bits, a higher sustained clock). */
int tb_microbench(tb_ctx* ctx, int which, double* out);

/* ---- on-device differential evolution on random-key individuals (tblup/evolver.py:63-157 DE/rand/1 with binary
 * crossover, tblup/individual.py:132-167 random-key decode, tblup/selector.py:18-34 greedy selection) ----------
 * The P x m key matrix stays in HBM; a generation is evolve -> decode -> evaluate -> select without a host
 * round-trip of genomes.
 * tb_de_init: keys_host [P][m] (the reference's np.random.uniform(size=m) per individual) or NULL to draw them on
 * the device from `seed`.  tb_de_evaluate: fitness of the current population (generation 0,
 * tblup/population.py:47).  tb_de_step: one generation; abc [P][3] parent indices and fixed [P] forced crossover
 * positions, mask [P][m] (1 = take the mutant) may be given by the host (replaying the reference's own draws) or
 * be NULL (device draws from `seed`); F is the mutation intensity the caller chose for this generation
 * (evolver.py:147-151), take_out [P] (nullable) receives which children replaced their parent.
 * tb_de_get: what = 0 population fitness [P] f64, 1 last offspring fitness [P] f64, 2 population keys [P][m] f64,
 * 3 last offspring keys, 4 decoded genome of individual `which` [length] i32 (ascending index order),
 * 5 genomes of the last evaluated batch [P][length] i32. */
int tb_de_init(tb_ctx* ctx, int P, int length, const double* keys_host, uint64_t seed);
int tb_de_evaluate(tb_ctx* ctx, const int32_t* slots, int n_slots, double h2, int mode_rule);
int tb_de_step(tb_ctx* ctx, const int32_t* slots, int n_slots, double h2, int mode_rule, double F, double CR, int clip,
               const int32_t* abc, const int32_t* fixed, const uint8_t* mask, uint64_t seed, int32_t* take_out);
int tb_de_get(tb_ctx* ctx, int what, int which, void* out, size_t nbytes);
/* The same generation split in two, for a population whose keys are replicated on every GPU of a box and whose
 * EVALUATION is sharded (SURVEY.md 8e): tb_de_step_begin evolves the whole offspring population (same draws on every
 * rank, so no key ever crosses NVLink) and scores the offspring [first, first + count); the caller all-gathers the
 * offspring fitness in place (tb_de_device_ptr(ctx, 1) is the [P] device vector, e.g. ncclAllGather /
 * torch.distributed.all_gather_into_tensor); tb_de_step_end applies the greedy selection to all P individuals.
 * tb_de_evaluate_shard is the generation-0 counterpart (fills fit[first, first + count), tb_de_device_ptr(ctx, 0)). */
int tb_de_step_begin(tb_ctx* ctx, const int32_t* slots, int n_slots, double h2, int mode_rule, double F, double CR,
                     int clip, const int32_t* abc, const int32_t* fixed, const uint8_t* mask, uint64_t seed, int first,
                     int count);
int tb_de_step_end(tb_ctx* ctx, int32_t* take_out);
int tb_de_evaluate_shard(tb_ctx* ctx, const int32_t* slots, int n_slots, double h2, int mode_rule, int first, int count);
void* tb_de_device_ptr(tb_ctx* ctx, int what);
/* SNP removal on the device (tblup/evaluator.py:569-633, SNPRemovalHandler).  The removed set lives next to the keys:
 * once it is non-empty, tb_de_evaluate / tb_de_step score every individual on setdiff1d(genome, removed)
 * (evaluator.py:617; an individual left with no marker gets fitness 0.0, :618-620) and tb_de_evaluate_testing scores
 * union1d(genome, removed) on row set `slot` (evaluate_testing, evaluator.py:407-431; fitness_out: host, [P]).
 * tb_de_set_removed replaces the set with a host list; tb_de_ban_genome adds the decoded genome of individual
 * `which` of the current population (what genomes_to_evaluate does with the best individual, :603-606 -- the
 * reference always bans the whole genome, see SURVEY.md appendix A) without the list visiting the host.
 * tb_de_get: what = 6 removed markers (ascending) i32, 7 lengths of the last filtered batch [P] i32,
 * 8 the flat lists of the last evaluated batch. */
int tb_de_set_removed(tb_ctx* ctx, const int32_t* markers, int n);
int tb_de_ban_genome(tb_ctx* ctx, int which, int32_t* n_removed_out);
int tb_de_evaluate_testing(tb_ctx* ctx, int slot, double h2, int mode_rule, double* fitness_out);

/* ---- start-up scan of the top-SNPs seeder (tblup/seeder.py:144-160 get_sorted_indices, :202-210 p_value ->
 * sklearn.feature_selection.f_regression) ------------------------------------------------------------------------
 * Per-marker sums over a list of animals (original indices, duplicates allowed) with one weight each:
 * sum_x[j] = sum_i x_ij, sum_xx[j] = sum_i x_ij^2 (exact), sum_xw[j] = sum_i x_ij w_i -- everything f_regression needs
 * (with w = y - mean(y)) without the dense float64 matrix the reference slices (X[train]); all outputs host, [m] doubles. */
int tb_marker_stats(tb_ctx* ctx, const int32_t* animals, int n_animals, const double* weights, double* sum_x,
                    double* sum_xx, double* sum_xw);

/* ---- knockout local search (tblup/local.py:50-76, KnockoutLocalSearch.search) ------------------------------------
 * The reference walks the markers of the best genome in order and calls evaluator.blup(genome[mask], training_indices,
 * validation_indices, data, labels, h2) once per marker (local.py:65-66), keeping the marker out when the fitness
 * improves (`fitness > best_fitness`, local.py:68): len(genome) sequential single evaluations.
 * tb_knockout runs the same greedy sequence as speculative batches through the ordinary pipeline (candidate lists are
 * built on the device; a batch is rescored from the first accepted drop on, so every decision is the reference's):
 * genome [k] marker indices (duplicates allowed), row set `slot`, start_fitness = fitness of the whole genome;
 * keep_out [k] receives 1 for markers that stay and 0 for knocked-out ones (the reference's `mask`),
 * best_fitness_out the final fitness; n_evals_out (nullable) the evaluations the greedy sequence consumed (= what the
 * reference would have run), n_batches_out (nullable) the batched pipeline passes it took.
 * tb_knockout_scan: fitness_out[i] = blup(genome without its i-th entry) for every i (no greedy dependence). */
int tb_knockout(tb_ctx* ctx, const int32_t* genome, int k, int slot, double h2, int mode_rule, double start_fitness,
                uint8_t* keep_out, double* best_fitness_out, int32_t* n_evals_out, int32_t* n_batches_out);
int tb_knockout_scan(tb_ctx* ctx, const int32_t* genome, int k, int slot, double h2, int mode_rule, double* fitness_out);

/* ---- panel models: marker effects and breeding values (tblup/evaluator.py:284 forms the GBLUP predictions of every
 * animal and keeps the validation entries; :311-314 fits a Ridge model and discards it after one predict) ------------
 * tb_fit_effects solves every genome staged with tb_stage_genomes on row set `slot` exactly as tb_eval_staged does
 * (same branch rule, precision and fp64 fallback; fitness_out [P], nullable, receives the same values) and turns each
 * solution alpha into one effect per listed marker (flat, staged order, duplicates included):
 *   centre_q = colsum_q / N (2p over the N frequency animals of the branch),  d = (2 N S - Q) / (2 N^2),
 *   effect_q = (sum_{a in T} x_{a,q} alpha_a - centre_q sum_{a in T} alpha_a) / d,
 *   intercept = 0 (gblup) or the mean training phenotype (snp_blup) -- sklearn Ridge's coef_ / intercept_ there.
 * tb_predict_effects scores animals (original indices of ctx's data set) with P such models, given as the same flat
 * marker lists (idx_off: P + 1 offsets) and flat centre / effect arrays plus P intercepts:
 *   out[g * n_animals + b] = intercept_g + sum_q (x_{b,q} - centre_q) effect_q.
 * It reads only the resident genotypes, so a model fitted on one context scores the animals of any other context
 * holding the same markers (e.g. newly genotyped animals, created without phenotypes).  Both run in fp64 in a fixed
 * order: results are identical between the int8 and 2-bit storages and from run to run. */
int tb_fit_effects(tb_ctx* ctx, int slot, double h2, int mode_rule, double* effects_out, double* centre_out,
                   double* intercept_out, double* fitness_out);
int tb_predict_effects(tb_ctx* ctx, const int32_t* idx_flat, const int64_t* idx_off, int P, const double* centre,
                       const double* effects, const double* intercept, const int32_t* animals, int n_animals,
                       double* out);

/* ---- REML heritability: the restricted log-likelihood of a panel's genomic model as a profile in h2 ---------------
 * For a genome (marker list j_1..j_k, duplicates count twice) and row set `slot` with training animals T, n = n_t:
 *
 *     y_T = 1 mu + g + e,   g ~ N(0, sigma_g^2 G_TT),   e ~ N(0, sigma_e^2 I),   h2 = sigma_g^2 / (sigma_g^2 + sigma_e^2),   lambda = (1 - h2)/h2
 *
 * Here G_TT is exactly the matrix the fitness factors for that genome on that row set.  The same branch rule
 * (mode_rule, TB_MODE_AUTO: k > n -> gblup) picks the frequency animals: all n animals for gblup, the training animals
 * for snp_blup.  y_T is the raw training phenotype.  The intercept mu is a fixed effect of the model, so centring y
 * changes nothing.  With A = G_TT + lambda I = L L^T, u = L^-1 1 and v = L^-1 y_T:
 *
 *     a = u'u,  b = u'v,  c = v'v,  mu^ = b/a,  q = c - b^2/a,  sigma_g^2^ = q/(n - 1),  sigma_e^2^ = lambda sigma_g^2^
 *     l(h2) = -1/2 [ (n - 1)(log(2 pi sigma_g^2^) + 1) + log|A| + log a ],   log|A| = 2 sum_i log L_ii
 *
 * This is the restricted log-likelihood -1/2[log|V| + log|X'V^-1 X| + y'Py] - ((n-1)/2) log 2 pi with X = 1 and
 * V = sigma_g^2 A, maximised over sigma_g^2 in closed form.  So l is a one-dimensional profile in h2.  Padding rows of
 * the factor (identity) add 0 to log|A| and to every quadratic form.  For snp_blup, G_TT 1 = 0, so a = n/lambda.  The
 * formula needs no special case.
 *
 * tb_reml_profile evaluates l, sigma_g^2^ and mu^ for every genome staged with tb_stage_genomes at n_h2 points each:
 * h2 is one list of n_h2 values shared by every genome (per_genome = 0) or [P][n_h2] (per_genome != 0); the outputs
 * are host [P][n_h2], sigma_g2_out and mu_out may be NULL.  All points of a genome share its gather, centring terms
 * and Gram (64 points per pass); every point gets its own fp64 A and fp64 Cholesky, whatever the `precision` option
 * says (a determinant cannot be refined).  Results are identical between the storages and from run to run; a job
 * whose factorisation meets a non-positive pivot returns NaN in all three outputs.  Refused, with a tb_last_error
 * message: an h2 outside (0, 1), n_h2 < 1, an undefined row set, a context created without phenotypes, an empty
 * genome.  The context's options and its last-evaluation facts (tb_get_info "last_*") are unchanged afterwards; the
 * staged batch stays staged. */
int tb_reml_profile(tb_ctx* ctx, int slot, int mode_rule, const double* h2, int n_h2, int per_genome,
                    double* loglik_out, double* sigma_g2_out, double* mu_out);

#ifdef __cplusplus
}
#endif
#endif
