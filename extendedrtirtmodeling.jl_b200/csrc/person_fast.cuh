// person_fast.cuh -- the f32 person-sweep kernel of the one-launch models (MlIrt, RtIrt, RtIrtNull, Latent, LatentQr):
// the hot configuration (BASELINE config 5 = LatentQr, 1M x 100, f32).  Same statement, data layout, Philox stream and
// statistics as person_sweep_kernel<float, TPP, 0> (person.cuh, which remains the f64 / Cross-family kernel), and the same
// per-person conditionals (the helpers in person.cuh); what differs is the instruction schedule of the per-cell loops:
//   * all per-cell arithmetic runs two cells per instruction on the packed FP32 pipe (FFMA2/FMUL2/FADD2, pg_fast.cuh);
//   * attempt 0 of the PG draw decides only "certainly accepted" / "certainly rejected" with constant bounds of a_1/a_0
//     (6 MUFU per cell instead of 10); undecided cells (0.5 %) are replayed with the a_1 term from a second work queue;
//   * of the Bernoulli log-likelihood  sum kappa z - |z|/2 - ln(1 + e^{-|z|})  the kernel accumulates only the last two terms
//     (the third as a product of (1 + e^{-|z|}): one lg2 per row instead of one per cell); the first is a function of statistics
//     the kernel reduces anyway,  sum_ij kappa_ij z_ij = sum_j a_j [(Ky_j - sum_i theta_i / 2) - b_j K0_j],  and is added by the
//     global kernel (GlobalArgs.kz_from_stats);
//   * the row sum  sum_j a_j kappa_ij  of drawSubjAbility (Draw.pl.jl:56) comes from a 16-entry table per 4-item group indexed by
//     the four responses (T_a[g][y] = sum_e kappa_e a_e), without touching the individual responses.
#pragma once
#include "person.cuh"
#include "pg_fast.cuh"

namespace erirt {

// slots of the f64 misc block as this kernel uses them (person.cuh's MiscD names the generic kernel's use of the same four doubles)
enum FastMiscD { FMD_SUM_IS2 = 0, FMD_SUM_LAM_IS2 = 1, FMD_AMAX = 2, FMD_ABMAX = 3 };
static_assert(FMD_ABMAX < MD_COUNT, "misc block too small");

constexpr int TAB_PITCH = 20;  // floats per item group in the response tables: groups g and g+4 fall on disjoint banks
constexpr int FAST_FLUSH_TILES = 16;  // item statistics live in f32 registers and are folded into the f64 accumulators every 16 tiles
// Phase timers of the diagnostic build (tools/make_tick_build.py, -DERIRT_TICKS): clock64() per warp at the phase boundaries.
#ifdef ERIRT_TICKS
#define PF_NTICK 16
__device__ unsigned long long g_ticks[PF_NTICK];
#define PF_TICK_DECL() unsigned long long _tk[PF_NTICK] = {0}; long long _t0 = clock64(), _t1
#define PF_TICK(n) do { _t1 = clock64(); if ((threadIdx.x & 31) == 0) _tk[n] += (unsigned long long)(_t1 - _t0); _t0 = _t1; } while (0)
#define PF_TICK_FLUSH() do { if ((threadIdx.x & 31) == 0) for (int n = 0; n < PF_NTICK; ++n) atomicAdd(&g_ticks[n], _tk[n]); } while (0)
#else
#define PF_TICK_DECL()
#define PF_TICK(n)
#define PF_TICK_FLUSH()
#endif

__device__ __forceinline__ uint32_t y_nibble(uint32_t yw) { return (yw * 0x01020408u) >> 24; }  // bytes 0/1 -> 4-bit index

// MODEL is a template parameter: each instantiation carries the code of one model only (less code to fetch, no model branches)
// BATCH: the replica-batch instantiation (layout.cuh BatchArgs), grid (gx, n_batch) with the replica in blockIdx.y
template <int TPP, int MODEL, bool BATCH = false>
__global__ void __launch_bounds__(CTA_THREADS, min_ctas_per_sm<TPP>()) person_sweep_fast_kernel(KernelArgs<PersonArgs<float>, BATCH> A) {
  if constexpr (BATCH) to_replica(A, blockIdx.y);
  extern __shared__ __align__(128) unsigned char smem[];
  constexpr int P = CTA_THREADS / TPP;
  typedef float R;
  const Layout& L = A.L;
  const int J = L.J, Jp = L.Jp, F = L.F, Dg = L.Dg, Dgp = A.S.Dgp, G = Jp / 4;
  constexpr int model = MODEL;
  constexpr bool has_rt = model != M_MLIRT;
  constexpr bool latent = model == M_LATENT || model == M_LATENTQR;
  constexpr bool qr = model == M_LATENTQR;
  constexpr bool reg_x = model == M_MLIRT || model == M_RTIRT || latent;  // models with a regression on [1 X]

  R* s_om = reinterpret_cast<R*>(smem + A.S.off_omega);
  R* s_lt = reinterpret_cast<R*>(smem + A.S.off_logt);
  uint8_t* s_y = smem + A.S.off_y;
  R* s_par = reinterpret_cast<R*>(smem + A.S.off_par);  // PAR_A: a, PAR_AB: -a b, PAR_A2: a^2, PAR_A2B: a^2 b, PAR_IS2: 1/sigma2
  R* s_u = reinterpret_cast<R*>(smem + A.S.off_u);
  R* s_beta = reinterpret_cast<R*>(smem + A.S.off_beta);  // beta (MAXD) then vec(Sigma) (4)
  R* s_ta = reinterpret_cast<R*>(smem + A.S.off_tab);     // [G][TAB_PITCH]  sum_e kappa_e a_e
  double* s_acc_item = reinterpret_cast<double*>(smem + A.S.off_acc_item);
  double* s_acc_gram = reinterpret_cast<double*>(smem + A.S.off_acc_gram);
  uint32_t* s_queue = reinterpret_cast<uint32_t*>(smem + A.S.off_queue);
  double* s_miscd = reinterpret_cast<double*>(smem + A.S.off_misc);  // MD_COUNT + SC_COUNT doubles
  double* s_scal = s_miscd + MD_COUNT;
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_scal + SC_COUNT);
  uint32_t* s_qctl = reinterpret_cast<uint32_t*>(s_bar + 1);  // [0]: packed counts of the CTA queue (low 16 bits standard, high 16 bits special)

  const int tid = threadIdx.x, p = tid / TPP, q = tid % TPP;
  const uint32_t qcap = (uint32_t)A.S.qcap, qstd = (uint32_t)A.S.qstd;  // work-queue capacity of this plan (erirt_b200.cu, make_smem_plan)
  TL_DECL(tl_entry);
  // ---- before the dependency wait (overlaps the tail of the preceding global kernel): clear the accumulators, arm the barrier ----
  for (int t = tid; t < 5 * Jp; t += CTA_THREADS) s_acc_item[t] = 0.0;
  for (int t = tid; t < 2 * L.ntri; t += CTA_THREADS) s_acc_gram[t] = 0.0;
  if (tid < SC_COUNT) s_scal[tid] = 0.0;
  if (tid == 0) {
    mbar_init(s_bar, 1);
    s_qctl[0] = 0;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  griddep_wait();    // parameters of state k, the sweep counter and the cleared statistics come from the preceding global kernel
  if (*A.status <= -1000) return;  // a peer of the sharded chain timed out: the chain is dead, do not spin through queued sweeps
  const uint32_t k = *A.sweep_ctr;
#ifdef ERIRT_TIMELINE
  if (tid == 0) {
    TL_MIN(k, 0, tl_entry); const unsigned long long t = tl_now(); TL_MIN(k, 1, t); TL_MAX(k, 2, t);
    if (k == TL_CTA_SWEEP && blockIdx.x < TL_CTAS) { g_tl_cta[blockIdx.x][0] = tl_smid(); g_tl_cta[blockIdx.x][1] = t; }
  }
#endif
  const bool do_draws = k >= 1;
  const double* par = A.params;

  // ---- stage item / structural parameters (state k) and the response tables ----
  for (int j = tid; j < Jp; j += CTA_THREADS) {
    double a = 0, b = 0, is2 = 0;
    if (j < J) {
      a = par[L.p_a + j];
      b = par[L.p_b + j];
      if (has_rt) is2 = 1.0 / par[L.p_sigma2 + j];
    }
    s_par[PAR_A * Jp + j] = (R)a;
    s_par[PAR_AB * Jp + j] = (R)(-a * b);
    s_par[PAR_A2 * Jp + j] = (R)(a * a);
    s_par[PAR_A2B * Jp + j] = (R)(a * a * b);
    s_par[PAR_IS2 * Jp + j] = (R)is2;
  }
  if (tid < MAXD) s_beta[tid] = (R)par[L.p_beta + tid];
  if (tid < 4) s_beta[MAXD + tid] = has_rt ? (R)par[L.p_Sigma + tid] : (tid == 0 || tid == 3 ? R(1) : R(0));
  if (tid < 32) {  // sum_j 1/sigma2_j, sum_j lambda_j/sigma2_j (f64), and the bound |z_ij| <= max|a| |theta_i| + max|a b|
    double s1 = 0, s2 = 0, amax = 0, abmax = 0;
    for (int j = tid; j < J; j += 32) {
      const double a = par[L.p_a + j], b = par[L.p_b + j];
      amax = fmax(amax, fabs(a));
      abmax = fmax(abmax, fabs(a * b));
      if (has_rt) {
        const double is2 = 1.0 / par[L.p_sigma2 + j];
        s1 += is2;
        s2 += par[L.p_lambda + j] * is2;
      }
    }
    for (int o = 16; o; o >>= 1) {
      s1 += __shfl_xor_sync(0xffffffffu, s1, o);
      s2 += __shfl_xor_sync(0xffffffffu, s2, o);
      amax = fmax(amax, __shfl_xor_sync(0xffffffffu, amax, o));
      abmax = fmax(abmax, __shfl_xor_sync(0xffffffffu, abmax, o));
    }
    if (tid == 0) {
      s_miscd[FMD_SUM_IS2] = s1;
      s_miscd[FMD_SUM_LAM_IS2] = s2;
      s_miscd[FMD_AMAX] = amax;
      s_miscd[FMD_ABMAX] = abmax;
    }
  }
  __syncthreads();
  // response table from the staged parameters (shared memory): T_a[g][y] = sum_e kappa_e a_e
  for (int t = tid; t < G * 16; t += CTA_THREADS) {
    const int g = t >> 4, yb = t & 15;
    const float4 a4 = *reinterpret_cast<const float4*>(s_par + PAR_A * Jp + 4 * g);
    const R k0 = (yb & 1) ? R(0.5) : R(-0.5), k1y = (yb & 2) ? R(0.5) : R(-0.5), k2y = (yb & 4) ? R(0.5) : R(-0.5), k3 = (yb & 8) ? R(0.5) : R(-0.5);
    s_ta[g * TAB_PITCH + yb] = fmaf(k0, a4.x, fmaf(k1y, a4.y, fmaf(k2y, a4.z, k3 * a4.w)));
  }
  __syncthreads();

  const R sum_is2 = (R)s_miscd[FMD_SUM_IS2], sum_lam_is2 = (R)s_miscd[FMD_SUM_LAM_IS2];
  const R z_amax = (R)s_miscd[FMD_AMAX], z_abmax = (R)s_miscd[FMD_ABMAX];
  const R S11 = s_beta[MAXD + 0], S12 = s_beta[MAXD + 2], S22 = s_beta[MAXD + 3];
  const R k1 = (R)A.k1, k2 = (R)A.k2;
  const int pb = F + 1;  // length of one regression block [1 X]
  const uint32_t iter_m = do_draws ? (k - 1) / (uint32_t)A.n_chain + 1 : 0;  // m of sweep k
  const bool post_burnin = do_draws && iter_m > (uint32_t)A.n_burnin;

  double acc_ll_bern = 0.0, acc_ll_struct = 0.0;
  uint32_t acc_defer = 0, acc_cells = 0;
  uint32_t parity = 0;
  const uint32_t load_bytes = (uint32_t)(A.S.tile_real_bytes * (has_rt ? 2 : 1) + A.S.tile_y_bytes);
  const int nk = ((G + 7) / 8) * (8 / TPP);  // steps per thread over its 4-item groups (nk <= 16 by the TPP choice)

  // cells of this thread that are real items (bit 4*kk+e), and the number of padding cells it walks over
  u64 valid_mask = 0ull;
  int n_pad_cells = 0;
  for (int kk = 0; kk < nk; ++kk) {
    const int g = group_of<TPP>(q, kk);
    if (g >= G) continue;
    for (int e = 0; e < 4; ++e) {
      if (4 * g + e < J) valid_mask |= 1ull << (4 * kk + e);
      else ++n_pad_cells;
    }
  }

  // transposed-statistics role of this thread: item group eg, person class er (G <= CTA_THREADS is enforced by the host)
  const int Rc = CTA_THREADS / G;
  ERIRT_CHECK(G >= 1 && G <= CTA_THREADS && Rc >= 1 && (size_t)A.S.off_misc + (MD_COUNT + SC_COUNT) * sizeof(double) + 24 <= (size_t)A.S.total);
  const bool e_active = tid < G * Rc;
  const int eg = tid % G, er = tid / G;
  u64 a0l = 0ull, a0h = 0ull, a1l = 0ull, a1h = 0ull, a2l = 0ull, a2h = 0ull, acl = 0ull, ach = 0ull;  // {items 0,1} / {items 2,3}
  R ay[4] = {0, 0, 0, 0};
  // Folding the f32 register sums into the CTA's f64 accumulators: the Rc person classes of an item group would collide on the
  // same 500 addresses (f64 shared atomics are CAS loops), so each class writes its 20 sums into its own slab of a staging area
  // -- the logT tile, dead between the statistics pass and the next tile's load -- and the slabs are added without atomics.
  // (MlIrt has no logT tile: inside the tile loop its folds go through the atomics below, the fold after the last tile uses the omega
  // tile once its store has drained -- with one tile per CTA, the launch-bound README problem, the atomics were 10 us of a 30 us sweep)
  const bool stage_fits = (size_t)Rc * 5 * Jp * sizeof(R) <= (size_t)A.S.tile_real_bytes;
  auto flush_item_stats = [&](const bool last) {  // called by all threads of the CTA at the same point
    const bool stage_flush = stage_fits && (has_rt || last);
    if (stage_flush) {
      R* stg = has_rt ? s_lt : s_om;
      if (!has_rt && tid == 0) tma_store_wait_read();  // the last tile's omega store no longer reads the buffer
      __syncthreads();  // every warp is done reading logT in the statistics pass
      if (e_active) {
        R* d = stg + (size_t)er * 5 * Jp + 4 * eg;
        *reinterpret_cast<float4*>(d + 0 * Jp) = make_float4(lo2(a0l), hi2(a0l), lo2(a0h), hi2(a0h));
        *reinterpret_cast<float4*>(d + 1 * Jp) = make_float4(lo2(a1l), hi2(a1l), lo2(a1h), hi2(a1h));
        *reinterpret_cast<float4*>(d + 2 * Jp) = make_float4(lo2(a2l), hi2(a2l), lo2(a2h), hi2(a2h));
        *reinterpret_cast<float4*>(d + 3 * Jp) = make_float4(ay[0], ay[1], ay[2], ay[3]);
        *reinterpret_cast<float4*>(d + 4 * Jp) = make_float4(lo2(acl), hi2(acl), lo2(ach), hi2(ach));
      }
      __syncthreads();
      for (int t = tid; t < 5 * Jp; t += CTA_THREADS) {
        double acc = 0.0;
        for (int r = 0; r < Rc; ++r) acc += (double)stg[(size_t)r * 5 * Jp + t];
        s_acc_item[t] += acc;
      }
      __syncthreads();  // the staging area is a tile buffer again after this point
    } else if (e_active) {
      const R v0[4] = {lo2(a0l), hi2(a0l), lo2(a0h), hi2(a0h)}, v1[4] = {lo2(a1l), hi2(a1l), lo2(a1h), hi2(a1h)};
      const R v2[4] = {lo2(a2l), hi2(a2l), lo2(a2h), hi2(a2h)}, vc[4] = {lo2(acl), hi2(acl), lo2(ach), hi2(ach)};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int j = 4 * eg + e;
        atomicAdd(&s_acc_item[0 * Jp + j], (double)v0[e]);
        atomicAdd(&s_acc_item[1 * Jp + j], (double)v1[e]);
        atomicAdd(&s_acc_item[2 * Jp + j], (double)v2[e]);
        atomicAdd(&s_acc_item[3 * Jp + j], (double)ay[e]);
        atomicAdd(&s_acc_item[4 * Jp + j], (double)vc[e]);
      }
    }
    ay[0] = ay[1] = ay[2] = ay[3] = R(0);
    a0l = a0h = a1l = a1h = a2l = a2h = acl = ach = 0ull;
  };

  int tiles_done = 0;
  PF_TICK_DECL();
  // Tiles are dealt dynamically: every CTA starts with tile blockIdx.x and then draws from a device-wide counter, so an SM that runs
  // slower (the finishing times of statically dealt CTAs were spread over five tile times, profiles/r02_sweep_timeline.txt) simply
  // takes fewer tiles.  Results do not depend on who processes a tile, except for the rounding of the per-CTA partial sums.
  int tile = blockIdx.x;
#ifdef ERIRT_TIMELINE
  if (tid == 0 && k == TL_CTA_SWEEP && blockIdx.x < TL_CTAS) g_tl_cta[blockIdx.x][2] = tl_now();
#endif
  for (; tile < A.n_tiles; ++tiles_done) {
    const int64_t row0 = (int64_t)tile * P;
    ERIRT_CHECK(tile >= 0 && tile < A.n_tiles && row0 + P <= A.n_pad);
    PF_TICK(13);  // tile-loop overhead / previous store issue
    if (tid == 0) {
      const uint32_t nxt = (uint32_t)gridDim.x + atomicAdd(A.tile_ctr, 1u);  // in flight while the store below drains
      mbar_expect_tx(s_bar, load_bytes);
      // the logT and Y buffers are free (every warp is past the statistics pass): their loads travel while the omega store drains
      if (has_rt) tma_load_1d(s_lt, A.logT + row0 * Jp, (uint32_t)A.S.tile_real_bytes, s_bar);
      tma_load_1d(s_y, A.Y + row0 * Jp, (uint32_t)A.S.tile_y_bytes, s_bar);
      tma_store_wait_read();  // previous tile's omega store has finished reading shared memory
      tma_load_1d(s_om, A.omega + row0 * Jp, (uint32_t)A.S.tile_real_bytes, s_bar);
      s_qctl[1] = nxt;
      if (nxt < (uint32_t)A.n_tiles) {  // pull the next tile of this CTA into L2 while this one is processed
        const int64_t rown = (int64_t)nxt * P;
        l2_prefetch(A.omega + rown * Jp, (uint32_t)A.S.tile_real_bytes);
        if (has_rt) l2_prefetch(A.logT + rown * Jp, (uint32_t)A.S.tile_real_bytes);
        l2_prefetch(A.Y + rown * Jp, (uint32_t)A.S.tile_y_bytes);
      }
    }
    // ---- person phase, part 1 (the first of the TPP lanes of a person): state k-1, regression means, the person's variates.
    //      Every warp serves its own persons, so nothing up to the work queues needs a CTA barrier ----
    const bool lead = q == 0;
    const int64_t pi = row0 + p;
    const bool pvalid = lead && pi < A.n_local;
    const uint32_t pgid = A.person_offset + (uint32_t)pi;
    R th = R(0), ze = R(0), nu = R(1), xb1 = R(0), xb2 = R(0);
    R zn_theta = R(0), zn_zeta = R(0), zn_nu = R(0), un_nu = R(0);
    if (lead) {
      // global loads first (independent, all in flight together), the variates while they travel
      th = A.theta[pi];
      if (has_rt) ze = A.zeta[pi];
      if (qr) nu = A.nu[pi];
      R xs[4] = {R(0), R(0), R(0), R(0)};
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (i < F) xs[i] = A.X[(int64_t)i * A.n_pad + pi];
      if (do_draws) {
        const uint4 w = philox(A.sched, pgid, k, make_site(DOM_PERSON, PK_NORMALS), 0);
        zn_theta = normal2f(w.x, w.y);
        zn_zeta = normal2f(w.z, w.w);
      }
      if (qr && TPP == 1) {
        const uint4 w = philox(A.sched, pgid, k + 1, make_site(DOM_PERSON, PK_NU), 0);
        zn_nu = normal2f(w.x, w.y);
        un_nu = u01f(w.z);
      }
      if (reg_x) xb1 = s_beta[0];
      if (model == M_RTIRT) xb2 = s_beta[pb];
      for (int f0 = 0; f0 < F; f0 += 4) {
        if (f0 > 0) {
#pragma unroll
          for (int i = 0; i < 4; ++i)
            if (f0 + i < F) xs[i] = A.X[(int64_t)(f0 + i) * A.n_pad + pi];
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int f = f0 + i;
          if (f < F) {
            const R x = xs[i];
            s_u[p * Dgp + 1 + f] = pvalid ? x : R(0);
            if (reg_x) xb1 = fmaf(x, s_beta[1 + f], xb1);
            if (model == M_RTIRT) xb2 = fmaf(x, s_beta[pb + 1 + f], xb2);
          }
        }
      }
    }
    if (qr && TPP >= 2) {  // the nu site's block is evaluated by the person's SECOND lane (idle otherwise) and handed to the first
      if (q == 1) {
        const uint4 w = philox(A.sched, pgid, k + 1, make_site(DOM_PERSON, PK_NU), 0);
        zn_nu = normal2f(w.x, w.y);
        un_nu = u01f(w.z);
      }
      const R zn_o = __shfl_down_sync(0xffffffffu, zn_nu, 1), un_o = __shfl_down_sync(0xffffffffu, un_nu, 1);
      if (lead) { zn_nu = zn_o; un_nu = un_o; }
    }
    PF_TICK(0);  // TMA issue, person part 1
    mbar_wait(s_bar, parity);
    parity ^= 1u;
    PF_TICK(1);  // TMA wait

    R* my_om = s_om + p * Jp;
    const R* my_lt = s_lt + p * Jp;
    const uint8_t* my_y = s_y + p * Jp;

    if (do_draws) {
      // ---- row sums over items (Draw.pl.jl:55-56, 137-138), TPP threads per person, two items per instruction ----
      u64 sA2 = 0ull, sAB = 0ull, sLT = 0ull, sA2b = 0ull, sABb = 0ull, sLTb = 0ull;  // two chains per sum
      R sAK = R(0);
      constexpr int CHUNK = 8 / TPP;  // consecutive groups owned by this thread inside each block of 8
      auto row_group = [&](const int g) {  // one 4-item group of this person's row
        const float4 om = *reinterpret_cast<const float4*>(my_om + 4 * g);
        const float4 pA2 = *reinterpret_cast<const float4*>(s_par + PAR_A2 * Jp + 4 * g);
        const float4 pA2B = *reinterpret_cast<const float4*>(s_par + PAR_A2B * Jp + 4 * g);
        const uint32_t yw = *reinterpret_cast<const uint32_t*>(my_y + 4 * g);
        const u64 o01 = pk2(om.x, om.y), o23 = pk2(om.z, om.w);
        sA2 = ffma2(pk2(pA2.x, pA2.y), o01, sA2);
        sA2b = ffma2(pk2(pA2.z, pA2.w), o23, sA2b);
        sAB = ffma2(pk2(pA2B.x, pA2B.y), o01, sAB);
        sABb = ffma2(pk2(pA2B.z, pA2B.w), o23, sABb);
        sAK += s_ta[g * TAB_PITCH + y_nibble(yw)];
        if (has_rt) {
          const float4 lt = *reinterpret_cast<const float4*>(my_lt + 4 * g);
          const float4 pI = *reinterpret_cast<const float4*>(s_par + PAR_IS2 * Jp + 4 * g);
          sLT = ffma2(pk2(pI.x, pI.y), pk2(lt.x, lt.y), sLT);
          sLTb = ffma2(pk2(pI.z, pI.w), pk2(lt.z, lt.w), sLTb);
        }
      };
      // whole chunks of CHUNK consecutive groups run without a branch inside (their shared-memory loads are issued together and the
      // six accumulator chains interleave); only the last, partial chunk of the row is guarded
      int g0 = q * CHUNK;
      for (; g0 + CHUNK <= G; g0 += 8) {
#pragma unroll
        for (int cc = 0; cc < CHUNK; ++cc) row_group(g0 + cc);
      }
      if (g0 < G) {
#pragma unroll
        for (int cc = 0; cc < CHUNK; ++cc)
          if (g0 + cc < G) row_group(g0 + cc);
      }
      sA2 = fadd2(sA2, sA2b);
      sAB = fadd2(sAB, sABb);
      sLT = fadd2(sLT, sLTb);
      R rA2 = lo2(sA2) + hi2(sA2), rAB = lo2(sAB) + hi2(sAB), rLT = lo2(sLT) + hi2(sLT);
#pragma unroll
      for (int o = 1; o < TPP; o <<= 1) {
        rA2 += __shfl_xor_sync(0xffffffffu, rA2, o);
        rAB += __shfl_xor_sync(0xffffffffu, rAB, o);
        sAK += __shfl_xor_sync(0xffffffffu, sAK, o);
        rLT += __shfl_xor_sync(0xffffffffu, rLT, o);
      }
      const float4 d = make_float4(rA2, rAB, sAK, sum_lam_is2 - rLT);  // all TPP lanes hold the person's sums
      PF_TICK(2);  // row sums
      // ---- person phase, part 2: theta_k, zeta_k, structural log-density, moments ----
      if (lead) {
        th = theta_draw(model, xb1, S11, d.x, d.y, d.z, zn_theta);
        R mu_z, var_z;
        zeta_prior(model, has_rt, latent, qr, th, nu, xb1, xb2, s_beta[F + 1], S22, k1, k2, mu_z, var_z);
        if (has_rt) ze = zeta_draw(mu_z, var_z, sum_is2, d.w, zn_zeta);
        if (pvalid) {
          acc_ll_struct += (double)struct_log_density(model, th, ze, xb1, xb2, mu_z, var_z, S11, S12, S22);
          A.theta[pi] = th;
          if (has_rt) A.zeta[pi] = ze;
          record_person(A, pi, k, post_burnin, A.ptrace != nullptr, has_rt, qr, th, ze, nu);
        }
      }
    }
    if (lead) {
      if (qr) {
        nu = draw_nu_person(th, ze, xb1, s_beta[F + 1], S22, k1, k2, zn_nu, un_nu);
        if (pvalid) A.nu[pi] = nu;
      }
      write_u_row(s_u + p * Dgp, pvalid, qr, F, th, ze, nu);
      if (pvalid) acc_cells += (uint32_t)J;
    }
    PF_TICK(4);  // person part 2, nu, u rows

    // ---- omega_{k+1} ~ PG(1, a_k (theta_k - b_k)), Draw.pl.jl:36-40, and the Bernoulli log-likelihood of state k ----
    const bool valid = (row0 + p) < A.n_local;
    const uint32_t gid = A.person_offset + (uint32_t)(row0 + p);
    const R thp = __shfl_sync(0xffffffffu, th, (tid & 31) & ~(TPP - 1));  // theta_k of this thread's person, from its first lane
    u64 dmask = 0ull, rmask = 0ull;  // bit 4*kk+e: cell not certainly accepted / certainly rejected
    if (valid) {
      const bool wide = !(fmaf(z_amax, fabsf(thp), z_abmax) <= PG_Z0MAX);  // some |z| of this row may exceed the attempt-0 range
      const u64 TH = bc2(thp);
      u64 prod = bc2(1.0f);
      R sabs = R(0);
      // one 4-item group: straight-line code (no branch inside), so that the groups of an iteration interleave when scheduled
      auto do_group = [&](const int g, uint32_t& dmu, uint32_t& rmu) {
        const float4 pA = *reinterpret_cast<const float4*>(s_par + PAR_A * Jp + 4 * g);
        const float4 pN = *reinterpret_cast<const float4*>(s_par + PAR_AB * Jp + 4 * g);
        const u64 z01 = ffma2(pk2(pA.x, pA.y), TH, pk2(pN.x, pN.y)), z23 = ffma2(pk2(pA.z, pA.w), TH, pk2(pN.z, pN.w));
        const uint4 wA = philox(A.sched, gid, k + 1, make_site(DOM_PERSON, PK_PG, (uint32_t)(2 * g)), 0);
        const uint4 wB = philox(A.sched, gid, k + 1, make_site(DOM_PERSON, PK_PG, (uint32_t)(2 * g + 1)), 0);
        float4 out;
        pg_fast_pair<0>(z01, wA.x, wA.y, wA.z, wA.w, out.x, out.y, dmu, rmu, prod, sabs);
        pg_fast_pair<2>(z23, wB.x, wB.y, wB.z, wB.w, out.z, out.w, dmu, rmu, prod, sabs);
        *reinterpret_cast<float4*>(my_om + 4 * g) = out;
      };
      if (!wide) {
        constexpr bool PAIRS = TPP <= 2;  // group_of(q, kk + 1) == group_of(q, kk) + 1 for even kk when 8/TPP is even
        for (int kk = 0; kk < nk; kk += PAIRS ? 2 : 1) {
          const int g0 = group_of<TPP>(q, kk);
          if (g0 >= G) continue;
          uint32_t dm0 = 0, rm0 = 0, dm1 = 0, rm1 = 0;
          if (PAIRS && g0 + 1 < G) {
            do_group(g0, dm0, rm0);
            do_group(g0 + 1, dm1, rm1);
          } else {
            do_group(g0, dm0, rm0);
          }
          dmask |= (u64)(dm0 | (dm1 << 4)) << (4 * kk);
          rmask |= (u64)(rm0 | (rm1 << 4)) << (4 * kk);
        }
      } else {
        // |theta| so large that some |z| may leave the range in which attempt 0 is defined (PG_Z0MAX): no fast evaluation for
        // this row -- every cell goes to the work queues, with the attempt-0 replay where attempt 0 exists.  Never taken with
        // sane parameters; kept exact for parity with the oracle.
        for (int kk = 0; kk < nk; ++kk) {
          const int g = group_of<TPP>(q, kk);
          if (g >= G) continue;
          uint32_t dm = 0, rm = 0;
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const R z = fmaf(s_par[PAR_A * Jp + 4 * g + e], thp, s_par[PAR_AB * Jp + 4 * g + e]);
            const R az = fabsf(z);
            if (e & 1) prod = ffma2(prod, pk2(0.f, fast_ex2(-PGF_LOG2E * az)), prod);
            else prod = ffma2(prod, pk2(fast_ex2(-PGF_LOG2E * az), 0.f), prod);
            sabs += az;
            my_om[4 * g + e] = -2.0f;
            dm |= 1u << e;
            if (!(az <= PG_Z0MAX)) rm |= 1u << e;
          }
          dmask |= (u64)dm << (4 * kk);
          rmask |= (u64)rm << (4 * kk);
        }
      }
      // - |z|/2 - ln(1 + e^{-|z|}) (sum kappa z is added by the global kernel); a padding cell has z = 0 and contributed -ln 2
      const R ll_row = R(-0.5) * sabs - PGF_LN2 * (fast_lg2(lo2(prod)) + fast_lg2(hi2(prod)) - (R)n_pad_cells);
      acc_ll_bern += (double)ll_row;
      dmask &= valid_mask;
      rmask &= dmask;
    }
    if (!valid || n_pad_cells) {  // padding persons / padding items hold omega = 0
      for (int kk = 0; kk < nk; ++kk) {
        const int g = group_of<TPP>(q, kk);
        if (g >= G) continue;
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (!valid || 4 * g + e >= J) my_om[4 * g + e] = R(0);
      }
    }
    PF_TICK(6);  // PG main pass
    {
      // ---- hand the cells that left the fast path to the tile's work queues: one shared-memory atomic per WARP reserves the
      //      slots of all its lanes in both queues (packed counts, warp prefix sum), then every lane writes its entries ----
      const u64 smask = dmask & rmask, umask = dmask & ~rmask;  // standard (certainly rejected) / special (undecided)
      const uint32_t n_std = (uint32_t)__popcll(smask), n_spc = (uint32_t)__popcll(umask);
      acc_defer += n_std + n_spc;
      uint32_t pre = n_std | (n_spc << 16);
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, pre, o);
        if ((tid & 31) >= o) pre += t;
      }
      const uint32_t wtotal = __shfl_sync(0xffffffffu, pre, 31);
      uint32_t wbase = 0;
      if ((tid & 31) == 31 && wtotal) wbase = atomicAdd(&s_qctl[0], wtotal);
      wbase = __shfl_sync(0xffffffffu, wbase, 31);
      uint32_t slot_s = (wbase & 0xffffu) + (pre & 0xffffu) - n_std;
      uint32_t slot_u = (wbase >> 16) + (pre >> 16) - n_spc;
      // bit 4*kk+e of a mask -> item index: the thread owns 32/TPP consecutive items in every block of 32
      constexpr int BPB = 32 / TPP;
      auto push = [&](uint32_t m, int bit0, uint32_t& slot, const uint32_t cap, const uint32_t qbase, const uint32_t flag) {
        while (m) {
          const int bit = bit0 + __ffs((int)m) - 1;
          m &= m - 1u;
          const int j = ((bit / BPB) << 5) + q * BPB + (bit % BPB);
          ERIRT_CHECK(j >= 0 && j < J && qbase + cap <= qcap);
          if (slot < cap) s_queue[qbase + slot] = ((uint32_t)p << 16) | (uint32_t)j | flag;
          else {  // queue overflow: finish the cell here
            const float z = fmaf(s_par[PAR_A * Jp + j], thp, s_par[PAR_AB * Jp + j]);
            my_om[j] = pg_resolve_f32(A.key, gid, k + 1, j, z, flag != 0u);
          }
          ++slot;
        }
      };
      if (wtotal) {
        push((uint32_t)smask, 0, slot_s, qstd, 0u, 0u);
        push((uint32_t)(smask >> 32), 32, slot_s, qstd, 0u, 0u);
        push((uint32_t)umask, 0, slot_u, qcap - qstd, qstd, 0x80000000u);
        push((uint32_t)(umask >> 32), 32, slot_u, qcap - qstd, qstd, 0x80000000u);
      }
    }
    PF_TICK(7);  // queue push
    __syncthreads();
    PF_TICK(8);  // barrier
    const int next_tile = (int)s_qctl[1];  // written by thread 0 at the top of this tile; next written after two more barriers
    // the deal has reached its last round: once every CTA is here the global kernel of the sweep may become resident beside the
    // person CTAs (about two and a half tile times before the end: its rehearsal pass takes one) and rehearse; released earlier it would only slow its SM down
    if (next_tile >= A.n_tiles - 2 * (int)gridDim.x) griddep_launch();
    if (next_tile < A.n_tiles && tid >= 32 && tid < 32 + 3 + F) {      // person vectors of the next tile (theta, zeta, nu, X columns) towards L2
      const int a = tid - 32;
      const R* src = a == 0 ? A.theta : (a == 1 ? A.zeta : (a == 2 ? A.nu : A.X + (int64_t)(a - 3) * A.n_pad));
      l2_prefetch(src + (int64_t)next_tile * P, (uint32_t)(P * sizeof(R)));
    }

    {
      // ---- drain, one phase over the CTA's queue (the load of the four warps is balanced: a warp-local queue was measured 7 %
      //      slower, r02 profiles): standard entries (Method-A retry rounds, two cells in flight per thread) are dealt from
      //      thread 0 upwards, special entries (undecided attempt 0: replay it with the a_1 term) from the last thread downwards ----
      const uint32_t qc = s_qctl[0];
      const uint32_t qn = min(qc & 0xffffu, qstd), qu = min(qc >> 16, qcap - qstd);
      for (uint32_t idx = tid; idx < qn; idx += 2 * CTA_THREADS) {
        const bool has2 = idx + CTA_THREADS < qn;
        const uint32_t e1 = s_queue[idx], e2 = s_queue[has2 ? idx + CTA_THREADS : idx];
        const int j1 = (int)(e1 & 0xffffu), p1 = (int)(e1 >> 16), j2 = (int)(e2 & 0xffffu), p2 = (int)(e2 >> 16);
        ERIRT_CHECK(j1 < J && p1 < P && j2 < J && p2 < P);
        const float z1 = fmaf(s_par[PAR_A * Jp + j1], s_u[p1 * Dgp + F + 1], s_par[PAR_AB * Jp + j1]);
        const float z2 = fmaf(s_par[PAR_A * Jp + j2], s_u[p2 * Dgp + F + 1], s_par[PAR_AB * Jp + j2]);
        const uint32_t g1 = A.person_offset + (uint32_t)(row0 + p1), g2 = A.person_offset + (uint32_t)(row0 + p2);
        // retry block r carries two Method-A attempts (c <= 1/t) or one Method-B attempt (c > 1/t: with a wide ability distribution a
        // third of the queued cells); a poisoned (NaN) state is passed through instead of spinning
        const bool b1 = 0.5f * fabsf(z1) > (float)PG_CSWITCH, b2 = 0.5f * fabsf(z2) > (float)PG_CSWITCH;
        float om1 = (z1 == z1) ? -2.0f : z1, om2 = (has2 && z2 == z2) ? -2.0f : (has2 ? z2 : 0.0f);
#pragma unroll 1
        for (uint32_t r = 1; r < PG_MAX_ATTEMPTS && (om1 < 0.f || om2 < 0.f); ++r) {
          const uint4 w1 = philox(A.sched, g1, k + 1, make_site(DOM_PERSON, PK_PG_RETRY, (uint32_t)j1), r);
          const uint4 w2 = philox(A.sched, g2, k + 1, make_site(DOM_PERSON, PK_PG_RETRY, (uint32_t)j2), r);
          const float o1 = b1 ? pg_fast_attemptB(z1, w1) : pg_exact_pair(z1, w1.x, w1.y, w1.z, w1.w);
          const float o2 = b2 ? pg_fast_attemptB(z2, w2) : pg_exact_pair(z2, w2.x, w2.y, w2.z, w2.w);
          if (om1 < 0.f) om1 = o1;
          if (om2 < 0.f) om2 = o2;
        }
        if (om1 < 0.f) om1 = 0.25f * (float)PG_T;
        if (om2 < 0.f) om2 = 0.25f * (float)PG_T;
        s_om[p1 * Jp + j1] = om1;
        if (has2) s_om[p2 * Jp + j2] = om2;
      }
      for (uint32_t idx = (uint32_t)(CTA_THREADS - 1 - tid); idx < qu; idx += CTA_THREADS) {
        const uint32_t e1 = s_queue[qstd + idx];
        const int j1 = (int)(e1 & 0xffffu), p1 = (int)((e1 >> 16) & 0x7fffu);
        ERIRT_CHECK(qstd + idx < qcap && j1 < J && p1 < P && (e1 >> 31));
        const float z1 = fmaf(s_par[PAR_A * Jp + j1], s_u[p1 * Dgp + F + 1], s_par[PAR_AB * Jp + j1]);
        s_om[p1 * Jp + j1] = pg_resolve_f32(A.key, A.person_offset + (uint32_t)(row0 + p1), k + 1, j1, z1, true);
      }
    }
    PF_TICK(9);  // drain
    __syncthreads();  // the whole tile (omega_{k+1}, u rows) is final: the transposed passes below read across warps
    if (tid == 0) s_qctl[0] = 0;  // next written by the push of the next tile, two barriers from here
    PF_TICK(10);  // barrier

    // ---- per-item statistics: thread per (item group, person class), tile read transposed, sums kept in registers ----
    if (e_active) {
      const R* r_om = s_om + er * Jp + 4 * eg;
      const uint8_t* r_y = s_y + er * Jp + 4 * eg;
      const R* r_u = s_u + er * Dgp + F + 1;
      const int step = Rc * Jp, ustep = Rc * Dgp;
      const R* r_lt = s_lt + er * Jp + 4 * eg;
      for (int pp = er; pp < P; pp += Rc, r_om += step, r_lt += step, r_y += step, r_u += ustep) {
        const R tp = r_u[0];
        const float4 om = *reinterpret_cast<const float4*>(r_om);
        const uint32_t yw = *reinterpret_cast<const uint32_t*>(r_y);
        const u64 o01 = pk2(om.x, om.y), o23 = pk2(om.z, om.w), T1 = bc2(tp), T2 = bc2(tp * tp);
        a0l = fadd2(a0l, o01);
        a0h = fadd2(a0h, o23);
        a1l = ffma2(T1, o01, a1l);
        a1h = ffma2(T1, o23, a1h);
        a2l = ffma2(T2, o01, a2l);
        a2h = ffma2(T2, o23, a2h);
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (yw & (1u << (8 * e))) ay[e] += tp;
        if (has_rt) {
          const u64 Z = bc2(r_u[1]);
          const float4 lt = *reinterpret_cast<const float4*>(r_lt);
          acl = ffma2(pk2(lt.x, lt.y), Z, acl);
          ach = ffma2(pk2(lt.z, lt.w), Z, ach);
        }
      }
    }
    PF_TICK(11);  // statistics pass
    if ((tiles_done % FAST_FLUSH_TILES) == FAST_FLUSH_TILES - 1) flush_item_stats(false);
    // Gram of u = [1 X theta zeta nu] and its 1/nu-weighted twin: entry t is shared by the 4 lanes of a quad (persons
    // pp = lane mod 4 (mod 4)), so that all four warps of the CTA take part instead of one
    for (int t0 = 0; t0 < L.ntri; t0 += CTA_THREADS / 4) {
      const int t = t0 + (tid >> 2);
      float g0 = 0.f, g1 = 0.f;  // f32 over the <= 32 persons of a lane, f64 across tiles
      if (t < L.ntri) {
        int r = 0, rem = t;
        while (rem >= Dg - r) { rem -= Dg - r; ++r; }
        const int c = r + rem;
        const R* u = s_u + (tid & 3) * Dgp;
        for (int pp = tid & 3; pp < P; pp += 4, u += 4 * Dgp) {
          const float pr = u[r] * u[c];
          g0 += pr;
          if (qr) g1 = fmaf(pr, u[F + 4], g1);
        }
      }
      g0 += __shfl_xor_sync(0xffffffffu, g0, 1);
      g0 += __shfl_xor_sync(0xffffffffu, g0, 2);
      if (qr) {
        g1 += __shfl_xor_sync(0xffffffffu, g1, 1);
        g1 += __shfl_xor_sync(0xffffffffu, g1, 2);
      }
      if (t < L.ntri && (tid & 3) == 0) {
        s_acc_gram[t] += (double)g0;
        if (qr) s_acc_gram[L.ntri + t] += (double)g1;
      }
    }
    PF_TICK(12);  // flush + Gram
    fence_proxy_async();
    __syncthreads();
    if (tid == 0) tma_store_1d(A.omega + row0 * Jp, s_om, (uint32_t)A.S.tile_real_bytes);
    tile = next_tile;
  }
  PF_TICK_FLUSH();
#ifdef ERIRT_TIMELINE
  if (tid == 0 && k == TL_CTA_SWEEP && blockIdx.x < TL_CTAS) { g_tl_cta[blockIdx.x][4] = tl_now(); g_tl_cta[blockIdx.x][5] = (unsigned long long)tiles_done; }
#endif
  flush_item_stats(true);

  // ---- flush CTA accumulators ----
  {  // warp totals by shuffle, then one shared-memory atomic per warp and quantity (f64 shared atomics are CAS loops)
    double v0 = acc_ll_bern, v1 = acc_ll_struct;
    uint32_t c0 = acc_defer, c1 = acc_cells;
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      v0 += __shfl_xor_sync(0xffffffffu, v0, o);
      v1 += __shfl_xor_sync(0xffffffffu, v1, o);
      c0 += __shfl_xor_sync(0xffffffffu, c0, o);
      c1 += __shfl_xor_sync(0xffffffffu, c1, o);
    }
    if ((tid & 31) == 0) {
      atomicAdd(&s_scal[SC_LL_BERN], v0);
      atomicAdd(&s_scal[SC_LL_STRUCT], v1);
      atomicAdd(&s_scal[SC_PG_DEFER], (double)c0);
      atomicAdd(&s_scal[SC_PG_CELLS], (double)c1);
    }
  }
  flush_to_stats(A, J, Jp, s_acc_item, 5, s_acc_gram, qr, s_scal, tid);
#ifdef ERIRT_TIMELINE
  __syncthreads();
  if (tid == 0) {
    const unsigned long long t = tl_now();
    TL_MAX(k, 3, t);
    if (k == TL_CTA_SWEEP && blockIdx.x < TL_CTAS) g_tl_cta[blockIdx.x][3] = t;
  }
#endif
}

// ---------------- parity / distribution-test kernel of the f32 PG path: the same functions as the sampler ----------------
__global__ void k_pg_fast_kernel(const double* z, int64_t rows, int cols, int64_t row0, PhiloxKey key, uint32_t sweep, double* out) {
  const int pairs = (cols + 1) / 2;
  const int64_t n = rows * pairs;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = t / pairs;
    const int j0 = 2 * (int)(t % pairs);
    const bool has1 = j0 + 1 < cols;
    const uint32_t gid = (uint32_t)(row0 + i);
    const float za = (float)z[i * cols + j0], zb = has1 ? (float)z[i * cols + j0 + 1] : 0.f;
    const uint4 w = philox(key, gid, sweep, make_site(DOM_PERSON, PK_PG, (uint32_t)(j0 >> 1)), 0);
    float oa, ob, sabs = 0.f;
    uint32_t dm = 0, rm = 0;
    u64 prod = bc2(1.0f);
    pg_fast_pair<0>(pk2(za, zb), w.x, w.y, w.z, w.w, oa, ob, dm, rm, prod, sabs);
    if (!(fabsf(za) <= PG_Z0MAX)) { dm |= 1u; rm |= 1u; }
    if (!(fabsf(zb) <= PG_Z0MAX)) { dm |= 2u; rm |= 2u; }
    if (dm & 1u) oa = pg_resolve_f32(key, gid, sweep, j0, za, !(rm & 1u));
    if (dm & 2u) ob = pg_resolve_f32(key, gid, sweep, j0 + 1, zb, !(rm & 2u));
    out[i * cols + j0] = (double)oa;
    if (has1) out[i * cols + j0 + 1] = (double)ob;
  }
}

}  // namespace erirt
