// layout.cuh -- device data layout shared by the kernels and the host orchestration (DESIGN.md "Data layout in HBM").
#pragma once
#include <cstdint>
#include <type_traits>
#include "rng.cuh"

namespace erirt {

constexpr int CTA_THREADS = 128;  // person-sweep CTA; tile = CTA_THREADS / TPP persons
constexpr int MAXD = 32;          // largest dense system solved in the global kernel (2*(nFeat+1) <= 32)
constexpr int QCAP = 1024;        // PG fast-retry queue capacity per tile (overflow is handled inline)

constexpr int N_ITEM_STATS = 7;   // S0, S1, S2, Ky, C, D, (V);  CrossQr K_a: A0..A5, V1;  CrossQr K_b: S0, S1, S2, Ky, A1', A2', A3'
enum ModelId { M_MLIRT = 0, M_RTIRT = 1, M_NULL = 2, M_CROSS = 3, M_CROSSQR = 4, M_LATENT = 5, M_LATENTQR = 6 };

// statistics scalars (f64), accumulated by the person kernel and consumed by the global kernel
enum StatScalar {
  SC_LL_BERN = 0,    // sum_ij y z - log(1+e^z) at state k
  SC_LL_STRUCT = 1,  // sum_i structural log-density at state k
  SC_PG_DEFER = 2,   // PG cells that left the fast path (diagnostic)
  SC_PG_CELLS = 3,
  SC_LL_RT = 4,      // response-time log-likelihood summed per cell (CrossQr only; the other models use sufficient statistics)
  SC_COUNT = 8
};

// Offsets (in f64 elements) into the parameter vector written by the global kernel and the statistics
// vector written by the person kernel.  Jp = padded item count (row pitch of the tiles, multiple of 4, odd
// number of 16-byte quads so that row-strided 128-bit shared-memory accesses are conflict free).
struct Layout {
  int J, Jp, F, Dg, ntri;
  int p_a, p_b, p_lambda, p_sigma2, p_rho, p_beta, p_Sigma, p_count;
  int s_S0, s_S1, s_S2, s_Ky, s_C, s_D, s_V, s_gram, s_gramw, s_scal, s_count;
};

// Programmatic dependent launch (sm_90+): the kernels of a chain are launched with cudaLaunchAttributeProgrammaticStreamSerialization,
// so a kernel's CTAs may become resident while its predecessor still runs.  Everything that reads what the predecessor wrote comes
// after griddep_wait() (returns once the predecessor grid has completed and its writes are visible); griddep_launch() lets the
// successor's CTAs be scheduled.  Both are no-ops for a kernel launched without the attribute.
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void griddep_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// Index checks of the diagnostic build (-DERIRT_CHECKS, tools/make_tick_build.py): a failing check traps the kernel (device assert)
#ifdef ERIRT_CHECKS
#include <cassert>
#define ERIRT_CHECK(c) assert(c)
#else
#define ERIRT_CHECK(c)
#endif

// Sweep timeline of the diagnostic build (-DERIRT_TIMELINE, tools/make_tick_build.py): %globaltimer stamps (ns) per sweep slot
#ifdef ERIRT_TIMELINE
#define TL_SLOTS 256
#define TL_N 16
__device__ unsigned long long g_timeline[TL_SLOTS][TL_N];
#define TL_CTAS 1024
#define TL_CTA_SWEEP 60
__device__ unsigned long long g_tl_cta[TL_CTAS][6];  // person launch of sweep TL_CTA_SWEEP: per CTA smid, past-wait, tile loop start, end, tile loop end, tiles
__device__ __forceinline__ unsigned tl_smid() { unsigned v; asm volatile("mov.u32 %0, %%smid;" : "=r"(v)); return v; }
__device__ __forceinline__ unsigned long long tl_now() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#define TL_DECL(v) unsigned long long v = tl_now()
#define TL_MIN(k, i, v) atomicMin(&g_timeline[(k) % TL_SLOTS][i], (v))
#define TL_MAX(k, i, v) atomicMax(&g_timeline[(k) % TL_SLOTS][i], (v))
#else
#define TL_DECL(v)
#define TL_MIN(k, i, v)
#define TL_MAX(k, i, v)
#endif

__host__ __device__ inline int tri_index(int r, int c, int Dg) {  // r <= c, row-major upper triangle
  return r * Dg - (r * (r - 1)) / 2 + (c - r);
}

inline Layout make_layout(int J, int F) {
  Layout L;
  L.J = J;
  L.F = F;
  int q = (J + 3) / 4;
  if ((q & 1) == 0) ++q;
  L.Jp = 4 * q;
  L.Dg = F + 4;  // u_i = [1, X_i(1..F), theta_i, zeta_i, nu_i]
  L.ntri = L.Dg * (L.Dg + 1) / 2;
  int o = 0;
  L.p_a = o; o += L.Jp;
  L.p_b = o; o += L.Jp;
  L.p_lambda = o; o += L.Jp;
  L.p_sigma2 = o; o += L.Jp;
  L.p_rho = o; o += L.Jp;
  L.p_beta = o; o += MAXD;
  L.p_Sigma = o; o += 4;
  L.p_count = o;
  o = 0;
  L.s_S0 = o; o += L.Jp;
  L.s_S1 = o; o += L.Jp;
  L.s_S2 = o; o += L.Jp;
  L.s_Ky = o; o += L.Jp;
  L.s_C = o; o += L.Jp;
  L.s_D = o; o += L.Jp;  // sum_i theta_i logT_ij (Cross family)
  L.s_V = o; o += L.Jp;  // seventh per-item block (CrossQr)
  L.s_gram = o; o += L.ntri;
  L.s_gramw = o; o += L.ntri;
  L.s_scal = o; o += SC_COUNT;
  L.s_count = o;
  return L;
}

// dynamic shared-memory plan of the person kernel (byte offsets)
struct SmemPlan {
  int P;  // persons per tile
  int tile_real_bytes, tile_y_bytes;
  int off_omega, off_logt, off_nuc, off_y, off_par, off_u, off_sum, off_beta, off_acc_item, off_acc_gram, off_queue, off_tab, off_misc, total;
  int Dgp;  // pitch of the U tile (elements)
  int qcap, qstd;  // f32 fast kernel: entries of the tile's work queue, and how many of them belong to the standard end
};

template <typename R>
struct PersonArgs {
  // tiles, person-major, row pitch Jp, n_pad rows (n_pad multiple of 128; padding rows are zero)
  const uint8_t* Y;
  const R* logT;
  R* omega;
  R* nu_cell;  // CrossQr: cell-level quantile weights, same tiling as omega
  // person vectors (n_pad) and covariates, column-major [F][n_pad]
  R* theta;
  R* zeta;
  R* nu;
  const R* X;
  double* mom;    // [6][n_pad] running sum / sum of squares of theta, zeta, nu (post burn-in)
  R* ptrace;      // optional [cap][3][n_pad] person trace (theta, zeta, nu) or nullptr
  double* nu_mom; // optional (CrossQr, cfg.nu_cell_moments) [2][n_pad][Jp] post-burn-in sum / sum of squares of the cell weights, or nullptr
  const double* params;
  double* stats;
  const uint32_t* sweep_ctr;  // k: this launch draws theta_k, zeta_k (k >= 1) and omega_{k+1}, nu_{k+1}
  uint32_t* tile_ctr;         // work counter of the launch: tile blockIdx.x first, then gridDim.x + atomicAdd(tile_ctr, 1); the global kernel zeroes it
  const int* status;          // sticky error flag of the chain; <= -1000: a peer of the sharded chain timed out, every launch returns at once
  int64_t n_local, n_pad;
  uint32_t person_offset;
  int n_tiles;
  Layout L;
  SmemPlan S;
  int model, n_chain, n_burnin;
  int stage;  // 0: whole sweep in one launch; Cross family: 1 = K_a (theta + its statistics), 2 = K_b (zeta, omega, statistics)
  double k1, k2;
  PhiloxKey key;
  PhiloxSched sched;  // key schedule of `key` (constant-bank operands of the hot Philox rounds)
};

struct GlobalArgs {
  double* params;
  double* stats;
  double* stats_prev;  // reduced statistics of the previous sweep (input of the instruction-cache rehearsal, global.cuh), or nullptr
  int rehearse;        // 1: run the rehearsal pass before the dependency wait
  uint32_t* tile_ctr;  // work counter of the person launches, zeroed at the end of every global kernel
  uint32_t* sweep_ctr;
  // constants from ingest (already all-reduced over shards)
  const double* T1;   // sum_i logT_ij
  const double* T2;   // sum_i logT_ij^2
  const double* K0;   // sum_i kappa_ij
  const double* XtX;  // [1 X]'[1 X], (F+1)^2 column-major
  const double* consts;  // [0]=mean(logT) [1]=std(logT)
  // traces, row per sweep
  double* tr_items_ra;  // [cap][2J]  a, b
  double* tr_items_rt;  // [cap][2J]  lambda, sigma2
  double* tr_qr;        // [cap][qw]
  double* tr_ll;        // [cap]
  int* status;          // sticky numeric error flag
  double* ll_out;       // stage 3: log-likelihood of the current state
  int64_t n_total;
  int cap, qw;
  Layout L;
  int model, intercept, onepl, cov2one, compat;
  int stage;  // 0/2: full draw + trace + counter; 1 (Cross family): lambda, sigma2 only
  int kz_from_stats;  // 1: SC_LL_BERN lacks sum_ij kappa_ij z_ij (f32 fast person kernel); add it from Ky, sum theta, K0 and a_k, b_k
  double k1, k2;
  PhiloxKey key;
  // one-shot peer exchange of the statistics (person-sharded chains, NVLink peer memory); peer_bufs == nullptr: not used
  double* const* peer_bufs;  // [world] base of every GPU's exchange buffer: [2 parities][world][xstride] 16-byte packets (global.cuh)
  uint32_t* xseq;            // exchanges completed so far (identical on every GPU)
  int world, rank, xstride;
};

// consts vector of a handle (f64): T1[Jp] T2[Jp] K0[Jp] XtX[MAXD*MAXD/4 >= (F+1)^2] sums[2]
inline int consts_count(const Layout& L) { return 3 * L.Jp + MAXD * MAXD / 4 + 2; }

// ---- replica batches (DESIGN.md 6.6) ----
// A batched handle holds n_batch independent problems of one configuration.  Each of its device buffers is n_batch copies of the
// standalone buffer, back to back; these are the lengths of one copy (elements of the buffer's type; Y: bytes).  The sweep,
// tile and status counters are one element per replica.
struct ReplicaSizes {
  int64_t cells;     // Y, logT, omega: n_pad * Jp
  int64_t vec;       // theta, zeta, nu: n_pad
  int64_t x;         // X [max(F,1)][n_pad]
  int64_t mom;       // running moments [6][n_pad]
  int64_t params;    // p_count
  int64_t stats;     // s_count + 2 (statistics and the last sweep's PG diagnostics); stats_prev alike
  int64_t consts;    // consts_count
  int64_t derived;   // mean and sd of logT (4)
  int64_t tr_items;  // [cap][2J], trace of a, b and of lambda, sigma2
  int64_t tr_qr;     // [cap][qw]
  int64_t tr_ll;     // [cap]
};
inline ReplicaSizes replica_sizes(int64_t n_pad, const Layout& L, int cap, int qw) {
  ReplicaSizes z;
  z.cells = n_pad * L.Jp;
  z.vec = n_pad;
  z.x = n_pad * (L.F > 0 ? L.F : 1);
  z.mom = 6 * n_pad;
  z.params = L.p_count;
  z.stats = L.s_count + 2;
  z.consts = consts_count(L);
  z.derived = 4;
  z.tr_items = (int64_t)cap * 2 * L.J;
  z.tr_qr = (int64_t)cap * qw;
  z.tr_ll = cap;
  return z;
}

// Kernel parameters of a replica-batch launch: the arguments of replica 0's standalone launch (its key excepted), the replica sizes,
// and seed and chain, from which replica r derives its key make_key(seed + r, chain).  The person launch is a (gx, n_batch) grid and
// the global launch n_batch CTAs.
template <typename Args>
struct BatchArgs : Args {
  ReplicaSizes z;
  uint64_t seed;
  uint32_t chain;
};
// The parameter of a sweep kernel: the standalone arguments, or those of a batch (the BATCH instantiation)
template <typename Args, bool BATCH>
using KernelArgs = typename std::conditional<BATCH, BatchArgs<Args>, const Args>::type;

// Replica r's standalone arguments, in place, once at kernel entry: every pointer moves by r copies, and every index inside the kernels
// stays as it is.  The Cross-family buffers (nu_cell, nu_mom) and the person trace are not part of a batch and stay null.  The key
// schedule of replica r is built here, in registers: the constant bank cannot be indexed by the replica without serialising the hot
// Philox rounds.
template <typename R>
__device__ __forceinline__ void to_replica(BatchArgs<PersonArgs<R>>& A, uint32_t r) {
  const ReplicaSizes& z = A.z;
  A.Y += r * z.cells;
  A.logT += r * z.cells;
  A.omega += r * z.cells;
  A.theta += r * z.vec;
  A.zeta += r * z.vec;
  A.nu += r * z.vec;
  A.X += r * z.x;
  A.mom += r * z.mom;
  A.params += r * z.params;
  A.stats += r * z.stats;
  A.sweep_ctr += r;
  A.tile_ctr += r;
  A.status += r;
  A.key = make_key(A.seed + r, A.chain);
  A.sched = make_sched(A.key);
}
__device__ __forceinline__ void to_replica(BatchArgs<GlobalArgs>& A, uint32_t r) {
  const ReplicaSizes& z = A.z;
  A.params += r * z.params;
  A.stats += r * z.stats;
  if (A.stats_prev) A.stats_prev += r * z.stats;
  A.tile_ctr += r;
  A.sweep_ctr += r;
  A.T1 += r * z.consts;
  A.T2 += r * z.consts;
  A.K0 += r * z.consts;
  A.XtX += r * z.consts;
  A.consts += r * z.derived;
  A.tr_items_ra += r * z.tr_items;
  A.tr_items_rt += r * z.tr_items;
  A.tr_qr += r * z.tr_qr;
  A.tr_ll += r * z.tr_ll;
  A.status += r;
  A.ll_out += r;
  A.key = make_key(A.seed + r, A.chain);
}

}  // namespace erirt
