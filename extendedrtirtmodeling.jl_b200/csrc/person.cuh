// person.cuh -- the fused person-sweep kernel (K2 of SURVEY.md 2c), one launch per Gibbs sweep.
//
// Launch k (k = *sweep_ctr) performs, for every person row i of this GPU's shard, in the reference's
// scan order (SURVEY 7.1 pipeline "R"):
//   theta_k  | omega_k, a_k, b_k, beta_k, Sigma_k      drawSubjAbility / ...Null   Draw.pl.jl:49-80
//   zeta_k   | lambda_k, sigma2_k, theta_k, beta_k, Sigma_k, nu_k   drawSubjSpeed*  Draw.pl.jl:119-174
//   nu_{k+1} | zeta_k, theta_k, beta_k, Sigma_k        drawQrWeightsLatentQr       Draw.pl.jl:325-343
//   omega_{k+1} | a_k, b_k, theta_k                    drawRaPgRandomVariable      Draw.pl.jl:36-40
// and accumulates every sum over persons that the item / structural draws of sweep k+1 need
// (S0,S1,S2 = sum omega [1,theta,theta^2]; Ky = sum y theta; C = sum logT zeta; Gram of [1 X theta zeta nu])
// plus the Bernoulli and structural log-likelihood of state k (getLogLikelihood*, GibbsRtIrt.pl.jl:195-272).
// (k = 0 is the prologue: only the sweep-1 auxiliaries are drawn from the initial state.)
//
// Mapping: CTA = 128 threads = P persons x TPP threads; a tile of P rows of Y (u8), logT and omega is
// staged in shared memory with 1-D TMA bulk copies (the rows of a tile are contiguous in HBM), each
// thread walks 4-item groups of its own row with 128-bit shared loads, and the per-item statistics are
// reduced by re-reading the tile transposed (thread per item group).  omega is updated in place and
// written back with one TMA bulk store.  HBM traffic per cell: 1 B (Y) + 4 B (logT) + 4+4 B (omega) in f32.
#pragma once
#include <type_traits>
#include "layout.cuh"
#include "pg.cuh"
#include "pg_fast.cuh"

namespace erirt {

// ---------------- PTX helpers: mbarrier + 1-D TMA bulk copies ----------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile(
        "{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  } while (!ok);
}
__device__ __forceinline__ void tma_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tma_store_1d(void* gdst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(smem_src)),
               "r"(bytes)
               : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void l2_prefetch(const void* gsrc, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(gsrc), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---------------- 4-element group access ----------------
template <typename R>
struct Quad {
  R v[4];
};
__device__ __forceinline__ Quad<float> ld4(const float* p) {
  float4 t = *reinterpret_cast<const float4*>(p);
  Quad<float> q;
  q.v[0] = t.x; q.v[1] = t.y; q.v[2] = t.z; q.v[3] = t.w;
  return q;
}
__device__ __forceinline__ Quad<double> ld4(const double* p) {
  double2 t0 = *reinterpret_cast<const double2*>(p), t1 = *reinterpret_cast<const double2*>(p + 2);
  Quad<double> q;
  q.v[0] = t0.x; q.v[1] = t0.y; q.v[2] = t1.x; q.v[3] = t1.y;
  return q;
}
__device__ __forceinline__ void st4(float* p, const Quad<float>& q) {
  *reinterpret_cast<float4*>(p) = make_float4(q.v[0], q.v[1], q.v[2], q.v[3]);
}
__device__ __forceinline__ void st4(double* p, const Quad<double>& q) {
  *reinterpret_cast<double2*>(p) = make_double2(q.v[0], q.v[1]);
  *reinterpret_cast<double2*>(p + 2) = make_double2(q.v[2], q.v[3]);
}

// item-parameter arrays staged in shared memory (each Jp long, zero beyond J)
// PAR_IS2 holds 1/sigma2_j, or 1/(sigma2_j k2) for CrossQr; PAR_ISC = 1/sqrt(sigma2_j k2) (CrossQr)
enum ParIdx { PAR_A = 0, PAR_AB = 1, PAR_A2 = 2, PAR_A2B = 3, PAR_IS2 = 4, PAR_LAM = 5, PAR_RHO = 6, PAR_ISC = 7, PAR_COUNT = 8 };
// per-CTA scalars in the misc block (f64)
enum MiscD { MD_SUM_IS2 = 0, MD_SUM_RHO_IS2 = 1, MD_SUM_LOGS2K = 2, MD_COUNT = 4 };

// group index handled by thread q at step k: the TPP threads of one person and the persons of a quarter
// warp touch 8 distinct 16-byte bank groups (row pitch is an odd number of quads)
template <int TPP>
__device__ __forceinline__ int group_of(int q, int k) {
  constexpr int chunk = 8 / TPP;
  return (k / chunk) * 8 + q * chunk + (k % chunk);
}

// Box-Muller pair from two words (CrossQr cell weights: cosine branch for even items, sine branch for odd items)
__device__ __forceinline__ void normal_pair(uint32_t w0, uint32_t w1, float& zc, float& zs) {
  const float u = fminf(u01f(w0), 0.99999994f);
  const float t = -1.3862943611198906f * fast_lg2(u);
  const float rad = t * fast_rsqrt(t);
  float sn, cs;
  __sincosf(6.283185307179586f * u01f(w1), &sn, &cs);
  zc = rad * cs;
  zs = rad * sn;
}
__device__ __forceinline__ void normal_pair(uint32_t w0, uint32_t w1, double& zc, double& zs) {
  const double rad = sqrt(-2.0 * log(u01d(w0))), ang = 6.283185307179586476925286766559 * u01d(w1);
  zc = rad * cos(ang);
  zs = rad * sin(ang);
}

__device__ __noinline__ double pg_draw_cell_f64(PhiloxKey key, uint32_t gid, uint32_t sweep, int j, double z, uint32_t* na) {
  return pg_draw_exact<double>(key, gid, sweep, j, z, 0, na);
}

constexpr int STAT_FLUSH_TILES = 8;  // item statistics live in registers and are folded into f64 every 8 tiles

// resident CTAs per SM the register allocation is tuned for: the tile of TPP=2 leaves room for 3 CTAs, TPP=4 for 5, TPP=8 for 7.
// TPP = 4 is compiled for four (128 registers, no spills): measured against five (102 registers) CrossQr 1M x 100 runs 1.77 -> 1.70 ms
// per sweep and the fast kernel forced to TPP = 4 0.80 -> 0.75 ms (gpurun_out/ab_r02i.log, cqr_r02i.log); three (144 registers) is slower
template <int TPP>
constexpr int min_ctas_per_sm() {
  return TPP >= 8 ? 7 : (TPP == 4 ? 4 : 3);
}

// Float64: a tile row costs 17 bytes per cell, so shared memory holds three CTAs at most where TPP = 4 is chosen (J = 100: 54 KB);
// compiled for five the kernel had 96 registers and 684 bytes of spills in its cell loop
template <int TPP>
constexpr int min_ctas_f64() {
  return TPP >= 8 ? 4 : 3;
}

// ---------------- per-person conditionals, shared by person_sweep_kernel and person_sweep_fast_kernel ----------------
// The callers differ only in their inputs; every expression keeps the operand order and association of the sampler it states.

// quantile weights are kept in [1e-10, 1e10]
template <typename R>
__device__ __forceinline__ R clamp_nu(R x) {
  return x < R(1e-10) ? R(1e-10) : (x > R(1e10) ? R(1e10) : x);
}

// theta_k from the row sums sum a^2 omega, sum a^2 b omega, sum a kappa (drawSubjAbility / ...Null, Draw.pl.jl:49-80)
template <typename R>
__device__ __forceinline__ R theta_draw(int model, R xb1, R S11, R d_a2, R d_ab, R d_ak, R zn) {
  const R mu0 = (model == M_MLIRT || model == M_RTIRT) ? xb1 : R(0);
  const R var0 = (model == M_MLIRT) ? R(1) : S11;
  const R iv0 = rdiv(R(1), var0);
  const R parV = rdiv(R(1), iv0 + d_a2);
  const R parM = parV * (mu0 * iv0 + d_ak + d_ab);
  return parM + sqrt_of(parV) * zn;
}

// prior mean and variance of zeta_k given theta_k and nu_k (Draw.pl.jl:119-174); mu = 0, var = 1 for MlIrt, which has no zeta.
// has_rt, latent and qr are the kernel's flags of `model`: derived here again, they cost the Float64 kernel two selects.
template <typename R>
__device__ __forceinline__ void zeta_prior(int model, bool has_rt, bool latent, bool qr, R th, R nu, R xb1, R xb2, R beta_th, R S22, R k1,
                                           R k2, R& mu, R& var) {
  mu = R(0);
  var = R(1);
  if (has_rt) {
    if (model == M_RTIRT) { mu = xb2; var = S22; }
    else if (latent) {
      mu = fma(th, beta_th, xb1);
      var = S22;
      if (qr) { mu = fma(k1, nu, mu); var = S22 * (k2 * nu); }
    } else if (model == M_NULL) { mu = R(0); var = R(1); }  // Draw.pl.jl:120-121
    else { mu = R(0); var = S22; }
  }
}

// zeta_k from its prior and the likelihood's precision and numerator (the row sums of the model's response-time part)
template <typename R>
__device__ __forceinline__ R zeta_draw(R mu_z, R var_z, R prec, R num, R zn) {
  const R ivz = rdiv(R(1), var_z);
  const R parV = rdiv(R(1), ivz + prec);
  const R parM = parV * (mu_z * ivz + num);
  return parM + sqrt_of(parV) * zn;
}

// structural log-density of (theta_k, zeta_k) (getLogLikelihood*, GibbsRtIrt.pl.jl:195-272)
template <typename R>
__device__ __forceinline__ R struct_log_density(int model, R th, R ze, R xb1, R xb2, R mu_z, R var_z, R S11, R S12, R S22) {
  const R LOG2PI = R(1.8378770664093454835606594728112);
  if (model == M_MLIRT) {
    const R r = th - xb1;
    return R(-0.5) * LOG2PI - R(0.5) * r * r;
  } else if (model == M_LATENT || model == M_LATENTQR) {
    const R r = ze - mu_z;
    return R(-0.5) * (LOG2PI + rlog(var_z)) - R(0.5) * r * rdiv(r, var_z);
  } else {
    const R e1 = th - (model == M_RTIRT ? xb1 : R(0));
    const R e2 = ze - (model == M_RTIRT ? xb2 : R(0));
    const R det = S11 * S22 - S12 * S12;
    return -LOG2PI - R(0.5) * rlog(det) - R(0.5) * rdiv(S22 * e1 * e1 - R(2) * S12 * e1 * e2 + S11 * e2 * e2, det);
  }
}

// running moments (post burn-in) and the person trace of row pi at sweep k
template <typename R>
__device__ __forceinline__ void record_person(const PersonArgs<R>& A, int64_t pi, uint32_t k, bool moments, bool trace, bool has_rt, bool qr,
                                              R th, R ze, R nu) {
  if (moments) {
    double* m = A.mom + pi;  // fire-and-forget reductions (RED.ADD.F64): no round trip on the critical path
    atomicAdd(&m[0], (double)th);
    atomicAdd(&m[A.n_pad], (double)th * (double)th);
    if (has_rt) {
      atomicAdd(&m[2 * A.n_pad], (double)ze);
      atomicAdd(&m[3 * A.n_pad], (double)ze * (double)ze);
    }
    if (qr) {
      atomicAdd(&m[4 * A.n_pad], (double)nu);
      atomicAdd(&m[5 * A.n_pad], (double)nu * (double)nu);
    }
  }
  if (trace) {
    R* t = A.ptrace + ((int64_t)(k - 1) * 3) * A.n_pad + pi;
    t[0] = th;
    t[A.n_pad] = ze;
    t[2 * A.n_pad] = nu;
  }
}

// nu_{k+1} | zeta_k, theta_k, beta_k, Sigma_k (LatentQr, drawQrWeightsLatentQr, Draw.pl.jl:325-343)
template <typename R>
__device__ __forceinline__ R draw_nu_person(R th, R ze, R xb1, R beta_th, R S22, R k1, R k2, R zn, R un) {
  const R xb = fma(th, beta_th, xb1);
  const R isc = rdiv(R(1), sqrt_of(S22 * k2));
  const R parA = fabs(ze - xb) * isc;
  const R parB = sqrt_of(R(2) * k2 + k1 * k1) * isc;
  R mu = rdiv(parB, parA);
  if (!(mu >= R(1e-10))) mu = R(1e-10);
  const R ig = ig_msh<R>(mu, parB * parB, zn, un);
  return clamp_nu(rdiv(R(1), ig));
}

// the person's row u = [1 X theta zeta nu 1/nu] of the Gram (X is written in part 1); zero for a padding row
template <typename R>
__device__ __forceinline__ void write_u_row(R* u, bool pvalid, bool qr, int F, R th, R ze, R nu) {
  u[0] = pvalid ? R(1) : R(0);
  u[F + 1] = pvalid ? th : R(0);
  u[F + 2] = pvalid ? ze : R(0);
  u[F + 3] = (pvalid && qr) ? nu : R(0);
  u[F + 4] = (pvalid && qr) ? rdiv(R(1), nu) : R(0);  // weight of the nu-weighted Gram
}

// end of the kernel, called by every thread once its shared-memory atomics on s_scal are issued: add the CTA's accumulators (n_blocks
// per-item blocks, the Gram and, for LatentQr, its 1/nu-weighted twin, the scalars) to A.stats and let the last omega store drain.
// J and Jp are the kernel's copies: read from A.L in here, the item loop is no longer unrolled.
template <typename R>
__device__ __forceinline__ void flush_to_stats(const PersonArgs<R>& A, int J, int Jp, const double* s_acc_item, int n_blocks,
                                               const double* s_acc_gram, bool qr, const double* s_scal, int tid) {
  const Layout& L = A.L;
  __syncthreads();
  for (int t = tid; t < n_blocks * Jp; t += CTA_THREADS) {
    const int j = t % Jp;
    if (j < J) atomicAdd(&A.stats[L.s_S0 + t], s_acc_item[t]);
  }
  for (int t = tid; t < 2 * L.ntri; t += CTA_THREADS)
    if (t < L.ntri || qr) atomicAdd(&A.stats[L.s_gram + t], s_acc_gram[t]);
  if (tid < SC_COUNT) atomicAdd(&A.stats[L.s_scal + tid], s_scal[tid]);
  if (tid == 0) tma_store_wait_all();
}

// FAM = 0: the one-launch-per-sweep models (MlIrt, RtIrt, RtIrtNull, Latent, LatentQr) -- the hot configuration, with the
// Cross-family / evaluation code compiled out; FAM = 1: everything (Cross, CrossQr stages 1/2, stage 3 evaluation).
// BATCH: the replica-batch instantiation (layout.cuh BatchArgs), grid (gx, n_batch) with the replica in blockIdx.y
template <typename R, int TPP, int FAM, bool BATCH = false>
__global__ void __launch_bounds__(CTA_THREADS, (sizeof(R) == 8 ? min_ctas_f64<TPP>() : min_ctas_per_sm<TPP>())) person_sweep_kernel(KernelArgs<PersonArgs<R>, BATCH> A) {
  if constexpr (BATCH) to_replica(A, blockIdx.y);
  extern __shared__ __align__(128) unsigned char smem[];
  constexpr int P = CTA_THREADS / TPP;
  constexpr bool F32 = sizeof(R) == 4;
  const Layout& L = A.L;
  const int J = L.J, Jp = L.Jp, F = L.F, Dg = L.Dg, Dgp = A.S.Dgp, G = Jp / 4;
  const int model = A.model;
  const bool has_rt = model != M_MLIRT;
  const bool latent = model == M_LATENT || model == M_LATENTQR;
  const bool qr = model == M_LATENTQR;
  const bool reg_x = model == M_MLIRT || model == M_RTIRT || latent;  // models with a regression on [1 X]
  constexpr bool XF = FAM == 1;
  const bool cross = XF && (model == M_CROSS || model == M_CROSSQR);
  const bool cqr = XF && model == M_CROSSQR;
  const int stage = XF ? A.stage : 0;
  const bool eval = XF && stage == 3;  // log-likelihood of the current state only (DIC's D-hat): no draws, no stores
  const bool do_theta = stage != 2 && !eval, do_zeta = has_rt && stage != 1 && !eval, do_pg = stage != 1 && !eval;

  R* s_om = reinterpret_cast<R*>(smem + A.S.off_omega);
  R* s_lt = reinterpret_cast<R*>(smem + A.S.off_logt);
  R* s_nc = reinterpret_cast<R*>(smem + A.S.off_nuc);  // CrossQr nu tile
  uint8_t* s_y = smem + A.S.off_y;
  R* s_par = reinterpret_cast<R*>(smem + A.S.off_par);
  R* s_u = reinterpret_cast<R*>(smem + A.S.off_u);
  R* s_sum = reinterpret_cast<R*>(smem + A.S.off_sum);    // [P][4] row sums handed to the person phase
  R* s_beta = reinterpret_cast<R*>(smem + A.S.off_beta);  // beta (MAXD) then vec(Sigma) (4)
  double* s_acc_item = reinterpret_cast<double*>(smem + A.S.off_acc_item);
  double* s_acc_gram = reinterpret_cast<double*>(smem + A.S.off_acc_gram);
  uint32_t* s_queue = reinterpret_cast<uint32_t*>(smem + A.S.off_queue);
  double* s_miscd = reinterpret_cast<double*>(smem + A.S.off_misc);  // MD_COUNT + SC_COUNT doubles
  double* s_scal = s_miscd + MD_COUNT;
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_scal + SC_COUNT);
  uint32_t* s_qctl = reinterpret_cast<uint32_t*>(s_bar + 1);         // fast queue [0] count [1] head, exact queue [2] count [3] head

  const int tid = threadIdx.x, p = tid / TPP, q = tid % TPP;
  griddep_wait();    // parameters, sweep counter and cleared statistics come from the preceding global kernel (layout.cuh)
  if (*A.status <= -1000) return;  // a peer of the sharded chain timed out: the chain is dead
  const uint32_t k = *A.sweep_ctr;
  const bool do_draws = k >= 1 || (FAM == 1 && A.stage == 3);
  const double* par = A.params;

  // ---- stage item / structural parameters (state k) and clear accumulators ----
  for (int j = tid; j < Jp; j += CTA_THREADS) {
    double a = 0, b = 0, is2 = 0, lam = 0, rho = 0, isc = 0;
    if (j < J) {
      a = par[L.p_a + j];
      b = par[L.p_b + j];
      if (has_rt) {
        is2 = 1.0 / par[L.p_sigma2 + j];
        lam = par[L.p_lambda + j];
      }
      if (cross) rho = par[L.p_rho + j];
      if (cqr) {
        is2 = 1.0 / (par[L.p_sigma2 + j] * A.k2);
        isc = sqrt(is2);
      }
    }
    s_par[PAR_A * Jp + j] = (R)a;
    s_par[PAR_AB * Jp + j] = (R)(a * b);
    s_par[PAR_A2 * Jp + j] = (R)(a * a);
    s_par[PAR_A2B * Jp + j] = (R)(a * a * b);
    s_par[PAR_IS2 * Jp + j] = (R)is2;
    s_par[PAR_LAM * Jp + j] = (R)lam;
    if (cross) {  // these two arrays exist only in the Cross-family shared-memory plan
      s_par[PAR_RHO * Jp + j] = (R)rho;
      s_par[PAR_ISC * Jp + j] = (R)isc;
    }
  }
  if (tid < MAXD) s_beta[tid] = (R)par[L.p_beta + tid];
  if (tid < 4) s_beta[MAXD + tid] = has_rt ? (R)par[L.p_Sigma + tid] : (tid == 0 || tid == 3 ? R(1) : R(0));
  const int n_stat_blocks = cqr ? 7 : (cross ? 6 : 5);  // per-item statistic blocks of this model (shared-memory plan)
  for (int t = tid; t < n_stat_blocks * Jp; t += CTA_THREADS) s_acc_item[t] = 0.0;
  for (int t = tid; t < 2 * L.ntri; t += CTA_THREADS) s_acc_gram[t] = 0.0;
  if (tid < SC_COUNT) s_scal[tid] = 0.0;
  if (tid < 32) {  // sum_j 1/sigma2_j in f64
    double s1 = 0, s2 = 0, s3 = 0;
    if (has_rt)
      for (int j = tid; j < J; j += 32) {
        const double is2 = 1.0 / (cqr ? par[L.p_sigma2 + j] * A.k2 : par[L.p_sigma2 + j]);
        s1 += is2;
        if (cross) s2 += par[L.p_rho + j] * is2;
        if (cqr) s3 += log(par[L.p_sigma2 + j] * A.k2);
      }
    for (int o = 16; o; o >>= 1) {
      s1 += __shfl_xor_sync(0xffffffffu, s1, o);
      s2 += __shfl_xor_sync(0xffffffffu, s2, o);
      s3 += __shfl_xor_sync(0xffffffffu, s3, o);
    }
    if (tid == 0) {
      s_miscd[MD_SUM_IS2] = s1;
      s_miscd[MD_SUM_RHO_IS2] = s2;
      s_miscd[MD_SUM_LOGS2K] = s3;
      mbar_init(s_bar, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
  }
  __syncthreads();

  const R sum_is2 = (R)s_miscd[MD_SUM_IS2], sum_rho_is2 = (R)s_miscd[MD_SUM_RHO_IS2];
  const R S11 = s_beta[MAXD + 0], S12 = s_beta[MAXD + 2], S22 = s_beta[MAXD + 3];
  const R k1 = (R)A.k1, k2 = (R)A.k2;
  const int pb = F + 1;  // length of one regression block [1 X]
  const uint32_t iter_m = do_draws ? (k - 1) / (uint32_t)A.n_chain + 1 : 0;  // m of sweep k
  const bool post_burnin = do_draws && iter_m > (uint32_t)A.n_burnin;

  double acc_ll_bern = 0.0, acc_ll_struct = 0.0, acc_ll_rt = 0.0;
  uint32_t acc_defer = 0, acc_cells = 0;
  uint32_t parity = 0;
  const bool load_om = stage != 2 && !eval;  // K_b of the Cross family only writes omega
  const bool load_nc = cqr && do_draws;  // the prologue has no nu yet
  const uint32_t load_bytes = (uint32_t)(A.S.tile_real_bytes * ((has_rt ? 1 : 0) + (load_om ? 1 : 0) + (load_nc ? 1 : 0)) + A.S.tile_y_bytes);
  const int nk = ((G + 7) / 8) * (8 / TPP);  // steps per thread over its 4-item groups

  // transposed-statistics role of this thread: item group eg, person class er (G <= CTA_THREADS is enforced by the host)
  const int Rc = CTA_THREADS / G;
  const bool e_active = tid < G * Rc;
  const int eg = tid % G, er = tid / G;
  R a0[4] = {0, 0, 0, 0}, a1[4] = {0, 0, 0, 0}, a2[4] = {0, 0, 0, 0}, ay[4] = {0, 0, 0, 0}, ac[4] = {0, 0, 0, 0}, ad[4] = {0, 0, 0, 0}, av[4] = {0, 0, 0, 0};
  auto flush_item_stats = [&]() {
    if (e_active) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int j = 4 * eg + e;
        atomicAdd(&s_acc_item[0 * Jp + j], (double)a0[e]);
        atomicAdd(&s_acc_item[1 * Jp + j], (double)a1[e]);
        atomicAdd(&s_acc_item[2 * Jp + j], (double)a2[e]);
        atomicAdd(&s_acc_item[3 * Jp + j], (double)ay[e]);
        atomicAdd(&s_acc_item[4 * Jp + j], (double)ac[e]);
        if (cross) atomicAdd(&s_acc_item[5 * Jp + j], (double)ad[e]);
        if (cqr) atomicAdd(&s_acc_item[6 * Jp + j], (double)av[e]);
        a0[e] = a1[e] = a2[e] = ay[e] = ac[e] = ad[e] = av[e] = R(0);
      }
    }
  };

  int tiles_done = 0;
  // tiles are dealt dynamically (see person_fast.cuh): tile blockIdx.x first, then from the device-wide counter
  volatile int* s_next = reinterpret_cast<volatile int*>(&s_miscd[MD_COUNT - 1]);  // spare slot of the misc block
  int tile = blockIdx.x;
  for (; tile < A.n_tiles; ++tiles_done) {
    const int64_t row0 = (int64_t)tile * P;
    if (tid == 0) {
      const uint32_t nxt = (uint32_t)gridDim.x + atomicAdd(A.tile_ctr, 1u);
      tma_store_wait_read();  // previous tile's omega store has finished reading shared memory
      mbar_expect_tx(s_bar, load_bytes);
      if (load_om) tma_load_1d(s_om, A.omega + row0 * Jp, (uint32_t)A.S.tile_real_bytes, s_bar);
      if (has_rt) tma_load_1d(s_lt, A.logT + row0 * Jp, (uint32_t)A.S.tile_real_bytes, s_bar);
      if (load_nc) tma_load_1d(s_nc, A.nu_cell + row0 * Jp, (uint32_t)A.S.tile_real_bytes, s_bar);
      tma_load_1d(s_y, A.Y + row0 * Jp, (uint32_t)A.S.tile_y_bytes, s_bar);
      *s_next = (int)nxt;
      s_qctl[0] = 0;
    }
    // ---- person phase, part 1 (one thread per person, coalesced): state k-1 and regression means ----
    const int64_t pi = row0 + tid;
    const bool pvalid = tid < P && pi < A.n_local;
    const uint32_t pgid = A.person_offset + (uint32_t)pi;
    R th = R(0), ze = R(0), nu = R(1), xb1 = R(0), xb2 = R(0);
    R zn_theta = R(0), zn_zeta = R(0), zn_nu = R(0), un_nu = R(0);  // variates drawn while the tile is in flight
    if (tid < P) {
      if (do_draws && !eval) {
        const uint4 w = philox(A.sched, pgid, k, make_site(DOM_PERSON, PK_NORMALS), 0);
        zn_theta = normal2r<R>(w.x, w.y);
        zn_zeta = normal2r<R>(w.z, w.w);
      }
      if (qr && !eval) {
        const uint4 w = philox(A.sched, pgid, k + 1, make_site(DOM_PERSON, PK_NU), 0);
        zn_nu = normal2r<R>(w.x, w.y);
        un_nu = u01<R>(w.z);
      }
      th = A.theta[pi];
      if (has_rt) ze = A.zeta[pi];
      if (qr) nu = A.nu[pi];
      if (reg_x) xb1 = s_beta[0];
      if (model == M_RTIRT) xb2 = s_beta[pb];
      for (int f = 0; f < F; ++f) {
        const R x = A.X[(int64_t)f * A.n_pad + pi];
        s_u[tid * Dgp + 1 + f] = pvalid ? x : R(0);
        if (reg_x) xb1 = fma(x, s_beta[1 + f], xb1);
        if (model == M_RTIRT) xb2 = fma(x, s_beta[pb + 1 + f], xb2);
      }
    }
    mbar_wait(s_bar, parity);
    parity ^= 1u;

    R* my_om = s_om + p * Jp;
    const R* my_lt = s_lt + p * Jp;
    const uint8_t* my_y = s_y + p * Jp;

    if (do_draws) {
      // ---- row sums over items (Draw.pl.jl:55-56, 137-138), TPP threads per person ----
      R sA2 = 0, sAB = 0, sAK = 0, sLT = 0;
      constexpr int CHUNK = 8 / TPP;  // consecutive groups owned by this thread inside each block of 8
      for (int g0 = q * CHUNK; g0 < G; g0 += 8) {
#pragma unroll
      for (int cc = 0; cc < CHUNK; ++cc) {
        const int g = g0 + cc;
        if (g >= G) continue;
        if (do_theta) {
          const Quad<R> om = ld4(my_om + 4 * g);
          const Quad<R> pA2 = ld4(s_par + PAR_A2 * Jp + 4 * g);
          const Quad<R> pA2B = ld4(s_par + PAR_A2B * Jp + 4 * g);
          const Quad<R> pA = ld4(s_par + PAR_A * Jp + 4 * g);
          const uint32_t yw = *reinterpret_cast<const uint32_t*>(my_y + 4 * g);
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            sA2 = fma(pA2.v[e], om.v[e], sA2);
            sAB = fma(pA2B.v[e], om.v[e], sAB);
            const R kap = ((yw >> (8 * e)) & 0xffu) ? R(0.5) : R(-0.5);
            sAK = fma(pA.v[e], kap, sAK);
          }
        }
        if (do_zeta) {
          const Quad<R> lt = ld4(my_lt + 4 * g);
          const Quad<R> pI = ld4(s_par + PAR_IS2 * Jp + 4 * g);
          const Quad<R> pL = ld4(s_par + PAR_LAM * Jp + 4 * g);
          if (!cqr) {
#pragma unroll
            for (int e = 0; e < 4; ++e) sLT = fma(pI.v[e], pL.v[e] - lt.v[e], sLT);  // sum_j (lambda_j - logT_ij)/sigma2_j
          } else {  // drawSubjSpeedCrossQr, Draw.pl.jl:192-206: weights 1/(sigma2_j k2 nu_ij)
            const Quad<R> nc = ld4(s_nc + p * Jp + 4 * g);
            const Quad<R> pR = ld4(s_par + PAR_RHO * Jp + 4 * g);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              if (4 * g + e < J) {
                const R t = rdiv(pI.v[e], nc.v[e]);
                sA2 += t;                                  // sum_j 1/(sigma2 k2 nu)
                sLT = fma(t, pL.v[e] - lt.v[e], sLT);      // sum_j (lambda - logT)/(sigma2 k2 nu)
                sAB = fma(t, pR.v[e], sAB);                // sum_j rho/(sigma2 k2 nu)
              }
            }
          }
        }
      }
      }
#pragma unroll
      for (int o = 1; o < TPP; o <<= 1) {
        sA2 += __shfl_xor_sync(0xffffffffu, sA2, o);
        sAB += __shfl_xor_sync(0xffffffffu, sAB, o);
        sAK += __shfl_xor_sync(0xffffffffu, sAK, o);
        sLT += __shfl_xor_sync(0xffffffffu, sLT, o);
      }
      if (q == 0) {
        R* d = s_sum + 4 * p;
        d[0] = sA2; d[1] = sAB; d[2] = sAK; d[3] = sLT;
      }
      __syncthreads();
      // ---- person phase, part 2: theta_k, zeta_k, structural log-density, moments ----
      if (tid < P) {
        const R* d = s_sum + 4 * tid;
        if (do_theta) th = theta_draw(model, xb1, S11, d[0], d[1], d[2], zn_theta);
        R mu_z, var_z;
        zeta_prior(model, has_rt, latent, qr, th, nu, xb1, xb2, s_beta[F + 1], S22, k1, k2, mu_z, var_z);
        if (do_zeta) {
          // Cross: sum_j (lambda - logT - theta rho_j)/sigma2;  CrossQr: the same weighted by 1/(k2 nu_ij), plus k1 sum_j 1/(sigma2 k2)
          const R prec = cqr ? d[0] : sum_is2;
          const R num = cqr ? d[3] - th * d[1] + k1 * sum_is2 : (cross ? d[3] - th * sum_rho_is2 : d[3]);
          ze = zeta_draw(mu_z, var_z, prec, num, zn_zeta);
        }
        if (pvalid && stage == 1) A.theta[pi] = th;  // K_a: theta_k only; everything else happens in K_b
        if (pvalid && stage != 1) {
          acc_ll_struct += (double)struct_log_density(model, th, ze, xb1, xb2, mu_z, var_z, S11, S12, S22);
          if (do_theta) A.theta[pi] = th;
          if (do_zeta) A.zeta[pi] = ze;
          record_person(A, pi, k, post_burnin && !eval, A.ptrace && !eval, has_rt, qr, th, ze, nu);
        }
      }
    }
    if (tid < P) {
      if (qr && !eval) {
        nu = draw_nu_person(th, ze, xb1, s_beta[F + 1], S22, k1, k2, zn_nu, un_nu);
        if (pvalid) A.nu[pi] = nu;
      }
      write_u_row(s_u + tid * Dgp, pvalid, qr, F, th, ze, nu);
      if (pvalid && do_pg) acc_cells += (uint32_t)J;
    }
    __syncthreads();
    const int next_tile = *s_next;  // written by thread 0 at the top of this tile; next written after at least one more barrier
    if (next_tile >= A.n_tiles - 2 * (int)gridDim.x) griddep_launch();  // last tile of this CTA: the global kernel may become resident once every CTA is here

    if (cqr && (do_pg || eval)) {
      // ---- CrossQr cell pass (thread per person row): response-time log-likelihood of state k with nu_k
      //      (getLogLikelihoodRtIrtCrossQr, GibbsRtIrtCross.pl.jl:240-258), then nu_{k+1} | state k
      //      (drawQrWeightsCrossQr, Draw.pl.jl:303-320), written in place.  Evaluation stage: the log-likelihood only ----
      const bool cvalid = (row0 + p) < A.n_local;
      const uint32_t cgid = A.person_offset + (uint32_t)(row0 + p);
      const R thc = s_u[p * Dgp + F + 1], zec = s_u[p * Dgp + F + 2];
      const R cB = sqrt_of(R(2) * k2 + k1 * k1);
      const bool nu_acc = A.nu_mom != nullptr && post_burnin && !eval;  // Post.mean.nu of GibbsRtIrtCross.pl.jl:310 as a running sum
      R llrt = R(0);
      // One 4-item group of this person's row.  FULL (a compile-time tag): the sampling pass of a complete group of a real person --
      // no per-cell validity tests and none of the run-time mode switches (evaluation stage, prologue, running moments) inside the
      // cell loop, the same arithmetic.  The cell-level draw was 40 % of the instructions of stage K_b, half of them control flow
      // (profiles/r02j_crossqr_kb_kernel_ncu_breakdown.txt).
      auto nu_group = [&](const int g, auto full_tag) {
        constexpr bool FULL = decltype(full_tag)::value;
        const bool g_draws = FULL ? true : do_draws, g_eval = FULL ? false : eval;
        Quad<R> nc;
        if (g_draws) nc = ld4(s_nc + p * Jp + 4 * g);
        const Quad<R> lt = ld4(my_lt + 4 * g);
        const Quad<R> pL = ld4(s_par + PAR_LAM * Jp + 4 * g);
        const Quad<R> pR = ld4(s_par + PAR_RHO * Jp + 4 * g);
        const Quad<R> pC = ld4(s_par + PAR_ISC * Jp + 4 * g);
        const Quad<R> pI = ld4(s_par + PAR_IS2 * Jp + 4 * g);
        R zn[4] = {R(0), R(0), R(0), R(0)}, un[4] = {R(0.5), R(0.5), R(0.5), R(0.5)};
        if (!g_eval) {
          const uint4 wA = philox(A.sched, cgid, k + 1, make_site(DOM_PERSON, PK_NU_CELL, (uint32_t)(2 * g)), 0);
          const uint4 wB = philox(A.sched, cgid, k + 1, make_site(DOM_PERSON, PK_NU_CELL, (uint32_t)(2 * g + 1)), 0);
          normal_pair(wA.x, wA.y, zn[0], zn[1]);
          normal_pair(wB.x, wB.y, zn[2], zn[3]);
          un[0] = u01<R>(wA.z); un[1] = u01<R>(wA.w); un[2] = u01<R>(wB.z); un[3] = u01<R>(wB.w);
        }
        if (!FULL && nu_acc && cvalid) {  // every cell is owned by exactly one thread of one CTA: plain read-modify-write
          double* m1 = A.nu_mom + (row0 + p) * (int64_t)Jp + 4 * g;
          double* m2 = m1 + A.n_pad * (int64_t)Jp;
#pragma unroll
          for (int e = 0; e < 4; ++e)
            if (4 * g + e < J) {
              const double v = (double)nc.v[e];
              m1[e] += v;
              m2[e] += v * v;
            }
        }
        Quad<R> out;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const R resid = lt.v[e] - pL.v[e] + zec + thc * pR.v[e];
          R nun = R(1);
          if (FULL || (cvalid && 4 * g + e < J)) {
            if (g_draws) {
              const R nu0 = nc.v[e];
              const R res = resid - k1 * nu0;
              llrt += R(-0.5) * (rlog(nu0) + res * res * rdiv(pI.v[e], nu0));
            }
            if (!g_eval) {
              const R parA = fabs(resid) * pC.v[e];
              const R parB = cB * pC.v[e];
              R mu = rdiv(parB, parA);
              if (!(mu >= R(1e-10))) mu = R(1e-10);
              const R ig = ig_msh<R>(mu, parB * parB, zn[e], un[e]);
              nun = clamp_nu(rdiv(R(1), ig));
            }
          }
          out.v[e] = nun;
        }
        if (!g_eval) st4(s_nc + p * Jp + 4 * g, out);
      };
      const bool full_row = cvalid && do_draws && !eval && !nu_acc;
      for (int kk = 0; kk < nk; ++kk) {
        const int g = group_of<TPP>(q, kk);
        if (g >= G) continue;
        if (full_row && 4 * g + 3 < J) nu_group(g, std::true_type{});
        else nu_group(g, std::false_type{});
      }
#pragma unroll
      for (int o = 1; o < TPP; o <<= 1) llrt += __shfl_xor_sync(0xffffffffu, llrt, o);
      if (q == 0 && cvalid && do_draws)
        acc_ll_rt += (double)llrt - 0.5 * ((double)J * 1.8378770664093454835606594728112 + s_miscd[MD_SUM_LOGS2K]);
    }
    if (do_pg) {
      // ---- omega_{k+1} ~ PG(1, a_k (theta_k - b_k)), Draw.pl.jl:36-40, and the Bernoulli log-likelihood of state k ----
      const bool valid = (row0 + p) < A.n_local;
      const uint32_t gid = A.person_offset + (uint32_t)(row0 + p);
      const R thp = s_u[p * Dgp + F + 1];
      float ll_tile = 0.f, ll_sabs = 0.f;
      u64 ll_prod = bc2(1.0f);
      int ll_npad = 0;
      double ll_lin = 0.0, ll_prodd = 1.0;  // f64: sum of y z - (z + |z|)/2 and product of 1 + e^{-|z|} over this thread's cells of the row
      uint32_t my_defer = 0;
      unsigned long long defer_mask = 0ull, rej_mask = 0ull;  // bit 4*kk+e: cell not certainly accepted / certainly rejected
      for (int kk = 0; kk < nk; ++kk) {
        const int g = group_of<TPP>(q, kk);
        if (g >= G) continue;
        Quad<R> out;
        if (!valid) {
          out.v[0] = out.v[1] = out.v[2] = out.v[3] = R(0);
          st4(my_om + 4 * g, out);
          continue;
        }
        const Quad<R> pA = ld4(s_par + PAR_A * Jp + 4 * g);
        const Quad<R> pAB = ld4(s_par + PAR_AB * Jp + 4 * g);
        const uint32_t yw = *reinterpret_cast<const uint32_t*>(my_y + 4 * g);
        if constexpr (F32) {
          const uint4 wA = philox(A.sched, gid, k + 1, make_site(DOM_PERSON, PK_PG, (uint32_t)(2 * g)), 0);
          const uint4 wB = philox(A.sched, gid, k + 1, make_site(DOM_PERSON, PK_PG, (uint32_t)(2 * g + 1)), 0);
          const int npad = 4 * g + 4 - J;  // > 0 only in groups holding padding cells
          float zs[4];
  #pragma unroll
          for (int e = 0; e < 4; ++e) {
            zs[e] = fmaf(pA.v[e], thp, -pAB.v[e]);
            ll_tile = fmaf(((yw >> (8 * e)) & 0xffu) ? 0.5f : -0.5f, zs[e], ll_tile);  // kappa z
          }
          uint32_t dm = 0, rm = 0;
          float o[4];
          pg_fast_pair<0>(pk2(zs[0], zs[1]), wA.x, wA.y, wA.z, wA.w, o[0], o[1], dm, rm, ll_prod, ll_sabs);
          pg_fast_pair<2>(pk2(zs[2], zs[3]), wB.x, wB.y, wB.z, wB.w, o[2], o[3], dm, rm, ll_prod, ll_sabs);
  #pragma unroll
          for (int e = 0; e < 4; ++e) {
            if (!(fabsf(zs[e]) <= PG_Z0MAX)) { o[e] = -2.0f; dm |= 1u << e; rm |= 1u << e; }  // no attempt 0 beyond |z| = 16
            if (npad > 0 && e >= 4 - npad) { o[e] = 0.f; dm &= ~(1u << e); ++ll_npad; }          // padding cells never count
            out.v[e] = o[e];
          }
          rm &= dm;
          defer_mask |= (unsigned long long)dm << (4 * kk);
          rej_mask |= (unsigned long long)rm << (4 * kk);
        } else {
          // Float64: attempt 0 of every cell without a branch (pg_attempt0_f64: both envelope pieces, first term of the series); the
          // cells it does not accept (4 %) go to the tile's work queue and are drawn by the exact loop, dealt over the whole CTA
          uint32_t dm = 0;
#pragma unroll 1
          for (int h = 0; h < 2; ++h) {  // one Philox block = the cell pair (4g + 2h, 4g + 2h + 1); rolled: one copy of the code
            const uint4 w = philox(A.sched, gid, k + 1, make_site(DOM_PERSON, PK_PG, (uint32_t)(2 * g + h)), 0);
            const R a0 = h ? pA.v[2] : pA.v[0], a1 = h ? pA.v[3] : pA.v[1];
            const R ab0 = h ? pAB.v[2] : pAB.v[0], ab1 = h ? pAB.v[3] : pAB.v[1];
            const uint32_t y2 = yw >> (16 * h);
            const R z0 = fma(a0, thp, -ab0), z1 = fma(a1, thp, -ab1);
            double om0 = pg_attempt0_f64((double)z0, w.x, w.y), om1 = pg_attempt0_f64((double)z1, w.z, w.w);
            const int j0 = 4 * g + 2 * h;
            // y z - ln(1 + e^z) = y z - (z + |z|)/2 - ln(1 + e^{-|z|}); the last term as a product per row: one log per thread and row
            // instead of a log1p per cell (14 % of the instructions of the f64 kernel, profiles/r02j_person_kernel_f64_ncu_breakdown.txt)
            if (j0 < J) {
              const R az = fabs(z0);
              ll_lin += (double)(((y2 & 0xffu) ? z0 : R(0)) - R(0.5) * (z0 + az));
              ll_prodd *= 1.0 + exp(-(double)az);
              if (om0 < 0.0) dm |= 1u << (2 * h);
            } else om0 = 0.0;
            if (j0 + 1 < J) {
              const R az = fabs(z1);
              ll_lin += (double)((((y2 >> 8) & 0xffu) ? z1 : R(0)) - R(0.5) * (z1 + az));
              ll_prodd *= 1.0 + exp(-(double)az);
              if (om1 < 0.0) dm |= 2u << (2 * h);
            } else om1 = 0.0;
            my_om[j0] = (R)om0;
            my_om[j0 + 1] = (R)om1;
          }
          defer_mask |= (unsigned long long)dm << (4 * kk);
        }
        if constexpr (!F32) continue;
        st4(my_om + 4 * g, out);
      }
      if constexpr (!F32) {
        if (valid) acc_ll_bern += ll_lin - log(ll_prodd);  // <= 64 factors in [1, 2]: no overflow
      }
      if constexpr (F32) {
        // kappa z - |z|/2 - ln(1 + e^{-|z|}); a padding cell has z = 0 and contributed -ln 2 through the product
        if (valid) acc_ll_bern += (double)(ll_tile - 0.5f * ll_sabs - PGF_LN2 * (fast_lg2(lo2(ll_prod)) + fast_lg2(hi2(ll_prod)) - (float)ll_npad));
      }
      {
        // ---- hand the cells that left the fast path to the tile's work queue: one shared-memory atomic per WARP reserves the
        //      slots of all its lanes (warp prefix sum), then every lane writes its own entries (bit 31: replay attempt 0) ----
        my_defer = (uint32_t)__popcll(defer_mask);
        uint32_t pre = my_defer;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const uint32_t t = __shfl_up_sync(0xffffffffu, pre, o);
          if ((tid & 31) >= o) pre += t;
        }
        const uint32_t wtotal = __shfl_sync(0xffffffffu, pre, 31);
        uint32_t wbase = 0;
        if ((tid & 31) == 31 && wtotal) wbase = atomicAdd(&s_qctl[0], wtotal);
        wbase = __shfl_sync(0xffffffffu, wbase, 31);
        uint32_t slot = wbase + pre - my_defer;
        while (defer_mask) {
          const int bit = __ffsll((long long)defer_mask) - 1;
          defer_mask &= defer_mask - 1ull;
          const bool replay0 = !((rej_mask >> bit) & 1ull);
          const int j = 4 * group_of<TPP>(q, bit >> 2) + (bit & 3);
          if (slot < (uint32_t)QCAP) s_queue[slot] = ((uint32_t)p << 16) | (uint32_t)j | (replay0 ? 0x80000000u : 0u);
          else {  // queue overflow: finish the cell here
            if constexpr (F32) {
              const float z = fmaf((float)s_par[PAR_A * Jp + j], (float)thp, -(float)s_par[PAR_AB * Jp + j]);
              my_om[j] = (R)pg_resolve_f32(A.key, gid, k + 1, j, z, replay0);
            } else {
              uint32_t na;
              my_om[j] = (R)pg_draw_cell_f64(A.key, gid, k + 1, j, (double)fma(s_par[PAR_A * Jp + j], thp, -s_par[PAR_AB * Jp + j]), &na);
            }
          }
          ++slot;
        }
      }
      acc_defer += my_defer;
      __syncthreads();

      {
        // ---- drain: a strided share of the queue per thread ----
        const uint32_t qn = min(s_qctl[0], (uint32_t)QCAP);
        for (uint32_t idx = tid; idx < qn; idx += CTA_THREADS) {
          const uint32_t e1 = s_queue[idx];
          const int j1 = (int)(e1 & 0xffffu), p1 = (int)((e1 >> 16) & 0x7fffu);
          if constexpr (F32) {
            const float z1 = fmaf((float)s_par[PAR_A * Jp + j1], (float)s_u[p1 * Dgp + F + 1], -(float)s_par[PAR_AB * Jp + j1]);
            s_om[p1 * Jp + j1] = (R)pg_resolve_f32(A.key, A.person_offset + (uint32_t)(row0 + p1), k + 1, j1, z1, (e1 >> 31) != 0u);
          } else {  // the exact loop from attempt 0 on; z is the expression of the main pass (same operands, same rounding)
            uint32_t na;
            const R z1 = fma(s_par[PAR_A * Jp + j1], s_u[p1 * Dgp + F + 1], -s_par[PAR_AB * Jp + j1]);
            s_om[p1 * Jp + j1] = (R)pg_draw_cell_f64(A.key, A.person_offset + (uint32_t)(row0 + p1), k + 1, j1, (double)z1, &na);
          }
        }
        __syncthreads();
      }
    }

    if (eval) {
      // ---- Bernoulli log-likelihood of the current state (no draws) ----
      const bool valid = (row0 + p) < A.n_local;
      const R thp = s_u[p * Dgp + F + 1];
      double llb = 0.0;
      if (valid)
        for (int kk = 0; kk < nk; ++kk) {
          const int g = group_of<TPP>(q, kk);
          if (g >= G) continue;
          const Quad<R> pA = ld4(s_par + PAR_A * Jp + 4 * g);
          const Quad<R> pAB = ld4(s_par + PAR_AB * Jp + 4 * g);
          const uint32_t yw = *reinterpret_cast<const uint32_t*>(my_y + 4 * g);
#pragma unroll 1
          for (int e = 0; e < 4; ++e) {
            if (4 * g + e >= J) continue;
            const double z = (double)fma(pA.v[e], thp, -pAB.v[e]);
            const double y = ((yw >> (8 * e)) & 0xffu) ? 1.0 : 0.0;
            const double az = fabs(z);
            llb += y * z - (0.5 * (z + az) + log1p(exp(-az)));
          }
        }
      acc_ll_bern += llb;
    }

    // ---- per-item statistics: thread per (item group, person class), tile read transposed, sums kept in registers ----
    if (e_active) {
      for (int pp = er; pp < P; pp += Rc) {
        const R tp = s_u[pp * Dgp + F + 1], zp = s_u[pp * Dgp + F + 2];
        if (do_pg) {
          const Quad<R> om = ld4(s_om + pp * Jp + 4 * eg);
          const uint32_t yw = *reinterpret_cast<const uint32_t*>(s_y + pp * Jp + 4 * eg);
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const R w = om.v[e];
            const R tw = tp * w;
            a0[e] += w;
            a1[e] += tw;
            a2[e] = fma(tp, tw, a2[e]);
            ay[e] += ((yw >> (8 * e)) & 0xffu) ? tp : R(0);
          }
        }
        if (has_rt && !cqr) {
          const Quad<R> lt = ld4(s_lt + pp * Jp + 4 * eg);
#pragma unroll
          for (int e = 0; e < 4; ++e) ac[e] = fma(lt.v[e], zp, ac[e]);
          if (cross) {
#pragma unroll
            for (int e = 0; e < 4; ++e) ad[e] = fma(lt.v[e], tp, ad[e]);
          }
        }
        if (cqr && s_u[pp * Dgp] != R(0)) {  // weighted statistics, w = 1/nu_ij, r = logT_ij + zeta_i (padding persons skipped)
          const Quad<R> lt = ld4(s_lt + pp * Jp + 4 * eg);
          const Quad<R> nc = ld4(s_nc + pp * Jp + 4 * eg);
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const R w = rdiv(R(1), nc.v[e]);
            const R r = lt.v[e] + zp;
            const R tw = tp * w;
            if (stage == 1) {  // K_a: A0..A5, V1 with (theta_k, zeta_{k-1}, nu_k)
              a0[e] += w;
              a1[e] += tw;
              a2[e] = fma(tw, r, a2[e]);
              ay[e] = fma(tw, tp, ay[e]);
              ac[e] = fma(r, w, ac[e]);
              ad[e] = fma(r * r, w, ad[e]);
              av[e] += nc.v[e];
            } else {           // K_b: A1', A2', A3' with (theta_k, zeta_k, nu_{k+1})
              ac[e] += tw;
              ad[e] = fma(tw, r, ad[e]);
              av[e] = fma(tw, tp, av[e]);
            }
          }
        }
      }
    }
    if ((tiles_done % STAT_FLUSH_TILES) == STAT_FLUSH_TILES - 1) flush_item_stats();
    // Gram of u = [1 X theta zeta nu] and its 1/nu-weighted twin: entry t is shared by the 4 lanes of a quad (persons
    // pp = lane mod 4 (mod 4)), so that all four warps of the CTA take part instead of one
    for (int t0 = 0; t0 < L.ntri; t0 += CTA_THREADS / 4) {
      const int t = t0 + (tid >> 2);
      double g0 = 0.0, g1 = 0.0;
      if (t < L.ntri) {
        int r = 0, rem = t;
        while (rem >= Dg - r) { rem -= Dg - r; ++r; }
        const int c = r + rem;
        for (int pp = tid & 3; pp < P; pp += 4) {
          const double ur = (double)s_u[pp * Dgp + r], uc = (double)s_u[pp * Dgp + c];
          g0 += ur * uc;
          if (qr) g1 += ur * uc * (double)s_u[pp * Dgp + F + 4];
        }
      }
      g0 += __shfl_xor_sync(0xffffffffu, g0, 1);
      g0 += __shfl_xor_sync(0xffffffffu, g0, 2);
      if (qr) {
        g1 += __shfl_xor_sync(0xffffffffu, g1, 1);
        g1 += __shfl_xor_sync(0xffffffffu, g1, 2);
      }
      if (t < L.ntri && (tid & 3) == 0) {
        s_acc_gram[t] += g0;
        if (qr) s_acc_gram[L.ntri + t] += g1;
      }
    }
    fence_proxy_async();
    __syncthreads();
    if (tid == 0 && do_pg) {
      tma_store_1d(A.omega + row0 * Jp, s_om, (uint32_t)A.S.tile_real_bytes);
      if (cqr) tma_store_1d(A.nu_cell + row0 * Jp, s_nc, (uint32_t)A.S.tile_real_bytes);
    }
    tile = next_tile;
  }
  flush_item_stats();

  // ---- flush CTA accumulators ----
  atomicAdd(&s_scal[SC_LL_BERN], acc_ll_bern);
  if (tid < P) atomicAdd(&s_scal[SC_LL_STRUCT], acc_ll_struct);
  if (cqr) atomicAdd(&s_scal[SC_LL_RT], acc_ll_rt);
  atomicAdd(&s_scal[SC_PG_DEFER], (double)acc_defer);
  if (tid < P) atomicAdd(&s_scal[SC_PG_CELLS], (double)acc_cells);
  flush_to_stats(A, J, Jp, s_acc_item, n_stat_blocks, s_acc_gram, qr, s_scal, tid);
}

// ---------------- parity / distribution-test kernels ----------------
template <typename R>
__global__ void k_pg_kernel(const double* z, int64_t rows, int cols, int64_t row0, PhiloxKey key, uint32_t sweep, double* out) {
  const int64_t n = rows * cols;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = t / cols;
    const int j = (int)(t % cols);
    const uint32_t gid = (uint32_t)(row0 + i);
    const R zz = (R)z[t];
    R om;
    om = pg_draw_exact<R>(key, gid, sweep, j, zz, 0);  // f64 only; the f32 test kernel is k_pg_fast_kernel (person_fast.cuh)
    out[t] = (double)om;
  }
}

template <typename R>
__global__ void k_nu_person_kernel(const double* mu, double lam, int64_t n, int64_t row0, PhiloxKey key, uint32_t sweep, double* out) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const uint4 w = philox(key, (uint32_t)(row0 + i), sweep, make_site(DOM_PERSON, PK_NU), 0);
    R x = ig_msh<R>((R)mu[i], (R)lam, normal2r<R>(w.x, w.y), u01<R>(w.z));
    R nu = R(1) / x;
    nu = nu < R(1e-10) ? R(1e-10) : (nu > R(1e10) ? R(1e10) : nu);
    out[i] = (double)nu;
  }
}

__global__ void k_philox_kernel(const uint32_t* ctr, const uint32_t* key, uint32_t* out) {
  PhiloxKey k{key[0], key[1]};
  uint4 w = philox(k, ctr[0], ctr[1], ctr[2], ctr[3]);
  out[0] = w.x; out[1] = w.y; out[2] = w.z; out[3] = w.w;
}

}  // namespace erirt
