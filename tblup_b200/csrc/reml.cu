// REML heritability: the restricted log-likelihood of a marker panel's genomic model as a profile in h2.
//
// For a genome (marker list j_1..j_k, duplicates count twice) and row set `slot` with training animals T, n = n_t:
//
//     y_T = 1 mu + g + e,   g ~ N(0, sigma_g^2 G_TT),   e ~ N(0, sigma_e^2 I),   h2 = sigma_g^2 / (sigma_g^2 + sigma_e^2),   lambda = (1 - h2)/h2
//
// Here G_TT is exactly the matrix the fitness factors for that genome on that row set.  The same branch rule (mode_rule,
// MODE_AUTO: k > n -> gblup) picks the frequency animals: all n animals for gblup, the training animals for snp_blup.
// y_T is the raw training phenotype.  The intercept mu is a fixed effect of the model, so centring y changes nothing.
// With A = G_TT + lambda I = L L^T, u = L^-1 1 and v = L^-1 y_T:
//
//     a = u'u,  b = u'v,  c = v'v,  mu^ = b/a,  q = c - b^2/a,  sigma_g^2^ = q/(n - 1),  sigma_e^2^ = lambda sigma_g^2^
//     l(h2) = -1/2 [ (n - 1)(log(2 pi sigma_g^2^) + 1) + log|A| + log a ],   log|A| = 2 sum_i log L_ii
//
// This is the restricted log-likelihood -1/2[log|V| + log|X'V^-1 X| + y'Py] - ((n-1)/2) log 2 pi with X = 1 and
// V = sigma_g^2 A, maximised over sigma_g^2 in closed form.  So l is a one-dimensional profile in h2.  Padding rows of
// the factor (identity) add 0 to log|A| and to every quadratic form.  For snp_blup, G_TT 1 = 0, so a = n/lambda.  The
// formula needs no special case.
//
// reml_kernel runs one CTA per (genome, h2) job after the fp64 factorisation (chol.cu): log|A| as a fixed-order sum,
// then the blocked forward substitution of the two right-hand sides [y_T - ybar, 1] at once through L and the stored
// 64 x 64 diagonal-block inverses (the forward half of solve_kernel, with each 16-byte load of L serving both vectors;
// L streams once, there is no backward sweep), then a, b, c and the profile.  The right-hand side is the centred
// phenotype: v' = v - ybar u gives the same q (c' - b'^2/a = c - b^2/a) without the cancellation a large mean would
// cause, and mu^ = ybar + b'/a.  No atomics, fixed summation order: results are identical between the int8 and 2-bit
// storages and from run to run.  A job whose pivot failed returns NaN for l, sigma_g^2 and mu, never a wrong number.
#include "tb_internal.h"
#include "../../include/tblup_b200.h"

#include <cmath>

namespace {

constexpr int NB = TB_NB;
constexpr int RT = 512;   // threads
constexpr int REML_SMEM_MAX = 227 * 1024;

__device__ __forceinline__ double warp_sum(double v) {
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ double block_sum(double v, double* red) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
  for (int i = 0; i < RT / 32; ++i) t += red[i];
  return t;
}

__global__ void __launch_bounds__(RT) reml_kernel(const TbRemlJob* __restrict__ jobs) {
  extern __shared__ double rsm[];
  const TbRemlJob jb = jobs[blockIdx.x];
  const int ntp = jb.ntp, n_t = jb.n_t, nb = ntp / NB;
  double* zv = rsm;                // [ntp] v = L^-1 (y - ybar)
  double* zu = zv + ntp;           // [ntp] u = L^-1 1_T
  double* rv = zu + ntp;           // [NB]
  double* ru = rv + NB;            // [NB]
  double* red = ru + NB;           // [RT / 32]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const double* M = jb.M;

  // ---------------- forward: L [v u] = [y 1] ----------------
  for (int b = 0; b < nb; ++b) {
    const int kc = b * NB;
    for (int i = warp; i < NB; i += RT / 32) {
      const double2* row = reinterpret_cast<const double2*>(M + (size_t)(kc + i) * ntp);
      const double2* vv = reinterpret_cast<const double2*>(zv);
      const double2* uu = reinterpret_cast<const double2*>(zu);
      double sv0 = 0.0, sv1 = 0.0, su0 = 0.0, su1 = 0.0;
      int c = lane;
      for (; c + 32 < kc / 2; c += 64) {
        const double2 l0 = row[c], l1 = row[c + 32];
        const double2 v0 = vv[c], v1 = vv[c + 32], u0 = uu[c], u1 = uu[c + 32];
        sv0 += l0.x * v0.x + l0.y * v0.y;
        sv1 += l1.x * v1.x + l1.y * v1.y;
        su0 += l0.x * u0.x + l0.y * u0.y;
        su1 += l1.x * u1.x + l1.y * u1.y;
      }
      for (; c < kc / 2; c += 32) {
        const double2 l0 = row[c];
        const double2 v0 = vv[c], u0 = uu[c];
        sv0 += l0.x * v0.x + l0.y * v0.y;
        su0 += l0.x * u0.x + l0.y * u0.y;
      }
      const double sv = warp_sum(sv0 + sv1), su = warp_sum(su0 + su1);
      if (lane == 0) {
        rv[i] = jb.y[kc + i] - sv;
        ru[i] = (kc + i < n_t ? 1.0 : 0.0) - su;
      }
    }
    __syncthreads();
    {
      // [v u]_b = Linv_b [rv ru]   (8 threads per row, 8 columns each)
      const int i = tid >> 3, sub = tid & 7;
      const double* li = jb.Linv + (size_t)b * NB * NB + i * NB + sub * 8;
      double sv = 0.0, su = 0.0;
#pragma unroll
      for (int p = 0; p < 8; ++p) {
        const double l = li[p];
        sv += l * rv[sub * 8 + p];
        su += l * ru[sub * 8 + p];
      }
#pragma unroll
      for (int o = 1; o < 8; o <<= 1) {
        sv += __shfl_xor_sync(0xffffffffu, sv, o);
        su += __shfl_xor_sync(0xffffffffu, su, o);
      }
      if (sub == 0) {
        zv[kc + i] = sv;
        zu[kc + i] = su;
      }
    }
    __syncthreads();
  }

  // ---------------- log|A|, a = u'u, b = u'v, c = v'v (padding rows contribute exactly 0) ----------------
  double ld = 0.0, sa = 0.0, sb = 0.0, sc = 0.0;
  for (int i = tid; i < n_t; i += RT) {
    ld += log(M[(size_t)i * ntp + i]);
    const double u = zu[i], v = zv[i];
    sa += u * u;
    sb += u * v;
    sc += v * v;
  }
  ld = 2.0 * block_sum(ld, red);
  sa = block_sum(sa, red);
  sb = block_sum(sb, red);
  sc = block_sum(sc, red);
  if (tid == 0) {
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    double ll = nan, sg = nan, mu = nan;
    if (*jb.status == 0 && sa > 0.0) {
      // correctly rounded reciprocals instead of divisions: the division's slow path is a call, whose frame spills
      const double n1 = (double)(n_t - 1), ra = __drcp_rn(sa);
      const double q = sc - sb * sb * ra;
      if (q > 0.0) {
        sg = q * __drcp_rn(n1);
        ll = -0.5 * (n1 * (log(2.0 * M_PI * sg) + 1.0) + ld + log(sa));
        mu = jb.ymean + sb * ra;
      }
    }
    if (!isfinite(ll)) ll = sg = mu = nan;
    *jb.loglik = ll;
    *jb.sigma_g2 = sg;
    *jb.mu = mu;
  }
}

inline int reml_smem_bytes(int ntp) { return (2 * ntp + 2 * NB + RT / 32) * (int)sizeof(double); }

int rfail(TbCtx* c, const std::string& msg, int code = -1) {
  c->err = msg;
  return code;
}

}  // namespace

cudaError_t tb_reml_init() {
  return cudaFuncSetAttribute(reml_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, REML_SMEM_MAX);
}

cudaError_t tb_launch_reml(const TbRemlJob* d_jobs, int n_jobs, int max_ntp, cudaStream_t st) {
  const int smem = reml_smem_bytes(max_ntp);
  if (smem > REML_SMEM_MAX) return cudaErrorInvalidConfiguration;
  reml_kernel<<<n_jobs, RT, smem, st>>>(d_jobs);
  return cudaGetLastError();
}

extern "C" int tb_reml_profile(tb_ctx* c, int slot, int mode_rule, const double* h2, int n_h2, int per_genome,
                               double* loglik_out, double* sigma_g2_out, double* mu_out) {
  if (!c) return -1;
  if (!h2 || !loglik_out) return rfail(c, "tb_reml_profile: null argument");
  if (n_h2 < 1) return rfail(c, "tb_reml_profile: n_h2 must be at least 1");
  if (!c->has_pheno) return rfail(c, "tb_reml_profile: this context was created without phenotypes");
  if (c->P <= 0) return rfail(c, "tb_reml_profile: no genomes staged");
  if (slot < 0 || slot >= TB_MAX_SLOTS || !c->slots[slot].valid)
    return rfail(c, "tb_reml_profile: row set " + std::to_string(slot) + " is not defined");
  if (mode_rule < 0 || mode_rule > 2) return rfail(c, "tb_reml_profile: bad mode_rule");
  if (c->stop_after >= 0) return rfail(c, "tb_reml_profile: the stop_after debug option is set");
  const int P = c->P;
  for (int i = 0; i < P; ++i)
    if (c->h_off[i + 1] <= c->h_off[i]) return rfail(c, "tb_reml_profile: empty genome at position " + std::to_string(i));
  // h2 = 1 makes A = G_TT, singular for every snp_blup panel (G_TT 1 = 0) and whenever k < n_t
  const size_t n_vals = (size_t)n_h2 * (per_genome ? (size_t)P : 1);
  for (size_t i = 0; i < n_vals; ++i)
    if (!(h2[i] > 0.0 && h2[i] < 1.0))
      return rfail(c, "tb_reml_profile: heritability " + std::to_string(h2[i]) + " is outside (0, 1)");
  const TbRowSet& rs = c->slots[slot];
  if (reml_smem_bytes(rs.ntp) > REML_SMEM_MAX)
    return rfail(c, "tb_reml_profile: " + std::to_string(rs.n_t) + " training animals exceed the REML kernel's limit of " +
                        std::to_string((REML_SMEM_MAX / (int)sizeof(double) - 2 * NB - RT / 32) / 2 / NB * NB));
  TB_CUDA(c, cudaSetDevice(c->device));
  cudaStream_t st = c->stream;
  const size_t n_out = (size_t)P * n_h2;
  double* d_out = nullptr;
  TB_CUDA(c, cudaMalloc(&d_out, 3 * n_out * sizeof(double)));
  // the profile leaves the context as it found it: options are never touched, the facts of the last evaluation are
  // put back, and workspace grown for the fp64 matrices of the profile (up to 80 % of the free HBM) is released
  const int keep_mixed = c->last_mixed, keep_c16 = c->last_c16, keep_fused = c->last_fused, keep_fp4 = c->last_fp4;
  const int keep_wave = c->last_wave, keep_perm = c->last_perm, keep_split = c->last_split;
  const int keep_fallbacks = c->last_fallbacks;
  const long long keep_issue = c->last_issue_us;
  const size_t keep_ws = c->ws_bytes;
  TbRemlReq req{h2, per_genome ? (long long)n_h2 : 0LL, 0, 0, n_h2, d_out, d_out + n_out, d_out + 2 * n_out};
  int rc = 0;
  // TB_MAX_SLOTS points per pass: each pass gathers and forms the Gram of every genome once
  for (int s0 = 0; s0 < n_h2 && rc == 0; s0 += TB_MAX_SLOTS) {
    req.s0 = s0;
    req.n = std::min(TB_MAX_SLOTS, n_h2 - s0);
    rc = tb_internal_eval_reml(c, slot, mode_rule, &req);
  }
  cudaError_t ce = cudaSuccess;
  if (rc == 0) {
    ce = cudaMemcpyAsync(loglik_out, req.d_loglik, n_out * sizeof(double), cudaMemcpyDeviceToHost, st);
    if (ce == cudaSuccess && sigma_g2_out)
      ce = cudaMemcpyAsync(sigma_g2_out, req.d_sigma_g2, n_out * sizeof(double), cudaMemcpyDeviceToHost, st);
    if (ce == cudaSuccess && mu_out) ce = cudaMemcpyAsync(mu_out, req.d_mu, n_out * sizeof(double), cudaMemcpyDeviceToHost, st);
  }
  const cudaError_t se = cudaStreamSynchronize(st);
  tb_internal_collect_spans(c);
  cudaFree(d_out);
  if (c->ws_bytes > keep_ws) {
    cudaFree(c->ws);
    c->ws = nullptr;
    c->ws_bytes = 0;
    c->dbg = TbCtx::DbgLayout();                     // it pointed into the workspace
  }
  c->last_mixed = keep_mixed;
  c->last_c16 = keep_c16;
  c->last_fused = keep_fused;
  c->last_fp4 = keep_fp4;
  c->last_wave = keep_wave;
  c->last_perm = keep_perm;
  c->last_split = keep_split;
  c->last_fallbacks = keep_fallbacks;
  c->last_issue_us = keep_issue;
  if (rc) return rc;
  if (ce != cudaSuccess) return rfail(c, std::string("tb_reml_profile: D2H: ") + cudaGetErrorString(ce), -2);
  if (se != cudaSuccess) return rfail(c, std::string("tb_reml_profile: device execution failed: ") + cudaGetErrorString(se), -2);
  return 0;
}
