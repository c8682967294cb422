// erirt_b200.cu -- host orchestration and the C ABI of include/erirt_b200.h.
//
// Replaces the body of the seven sample! methods of the reference (SURVEY.md 3.2 / 8b):
//   for m in 1:nIter, l in 1:nChain ... end       /root/reference/src/GibbsRtIrt.pl.jl:289-324
// by   P(0) G(1) [P(k) (allreduce) G(k+1)]_{k=1..}   on one CUDA stream, optionally replayed from a CUDA graph.
// No CPU fallback exists: every entry point fails with ERIRT_E_CUDA when no sm_100 device is usable.
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <string>
#include <mutex>
#include <vector>

#include "../../include/erirt_b200.h"
#include "global.cuh"
#include "diagnostics.cuh"
#include "layout.cuh"
#include "person.cuh"
#include "person_fast.cuh"

using namespace erirt;

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local std::string g_err;
// ERIRT_TIMING=1: host-side wall-clock marks of the set-up calls on stderr (diagnostic)
struct HostTimer {
  bool on = getenv("ERIRT_TIMING") != nullptr;
  std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
  void mark(const char* what) {
    if (!on) return;
    const auto t1 = std::chrono::steady_clock::now();
    fprintf(stderr, "[erirt timing] %-28s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(t1 - t0).count());
    t0 = t1;
  }
};
static int fail(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}
#define CU(expr)                                                                                         \
  do {                                                                                                   \
    cudaError_t _e = (expr);                                                                             \
    if (_e != cudaSuccess) return fail(ERIRT_E_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)
// CU for a function that holds stream-ordered staging buffers: its lambda `cleanup` frees them before the error is returned
#define CUX(expr)                                                                                        \
  do {                                                                                                   \
    cudaError_t _e = (expr);                                                                             \
    if (_e != cudaSuccess) {                                                                             \
      cleanup();                                                                                         \
      return fail(ERIRT_E_CUDA, "%s failed: %s", #expr, cudaGetErrorString(_e));                        \
    }                                                                                                    \
  } while (0)

static int pick_device(int device) {
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) return fail(ERIRT_E_CUDA, "no CUDA device available (%s); this engine has no CPU fallback", cudaGetErrorString(e));
  if (device < 0 || device >= ndev) return fail(ERIRT_E_ARG, "device %d out of range [0,%d)", device, ndev);
  CU(cudaSetDevice(device));
  return 0;
}

// ------------------------------------------------------------------------------------------------
// NCCL through dlopen (no link-time dependency; single-GPU use never touches it)
// ------------------------------------------------------------------------------------------------
namespace nccl {
typedef struct ncclComm* comm_t;
typedef struct { char internal[128]; } unique_id;
typedef int (*fn_get_unique_id)(unique_id*);
typedef int (*fn_comm_init_rank)(comm_t*, int, unique_id, int);
typedef int (*fn_all_reduce)(const void*, void*, size_t, int, int, comm_t, cudaStream_t);
typedef int (*fn_comm_destroy)(comm_t);
typedef const char* (*fn_get_error_string)(int);
static void* lib = nullptr;
static fn_get_unique_id get_unique_id;
static fn_comm_init_rank comm_init_rank;
static fn_all_reduce all_reduce;
static fn_comm_destroy comm_destroy;
static fn_get_error_string get_error_string;
constexpr int kFloat64 = 8, kSum = 0;  // ncclDouble, ncclSum
static int load() {
  if (lib) return 0;
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  for (const char* n : names) {
    lib = dlopen(n, RTLD_NOW | RTLD_NOLOAD);
    if (lib) break;
  }
  if (!lib)
    for (const char* n : names) {
      lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
      if (lib) break;
    }
  if (!lib) return fail(ERIRT_E_NCCL, "cannot dlopen libnccl.so.2: %s", dlerror());
  get_unique_id = (fn_get_unique_id)dlsym(lib, "ncclGetUniqueId");
  comm_init_rank = (fn_comm_init_rank)dlsym(lib, "ncclCommInitRank");
  all_reduce = (fn_all_reduce)dlsym(lib, "ncclAllReduce");
  comm_destroy = (fn_comm_destroy)dlsym(lib, "ncclCommDestroy");
  get_error_string = (fn_get_error_string)dlsym(lib, "ncclGetErrorString");
  if (!get_unique_id || !comm_init_rank || !all_reduce || !comm_destroy || !get_error_string) {
    lib = nullptr;
    return fail(ERIRT_E_NCCL, "libnccl is missing required symbols");
  }
  return 0;
}
}  // namespace nccl
#define NC(expr)                                                                                     \
  do {                                                                                               \
    int _e = (expr);                                                                                 \
    if (_e != 0) return fail(ERIRT_E_NCCL, "%s failed: %s", #expr, nccl::get_error_string(_e));      \
  } while (0)

// ------------------------------------------------------------------------------------------------
// ingest kernels (K8): Julia column-major float64 -> person-major tiles
// ------------------------------------------------------------------------------------------------
template <typename SrcT, typename OutT, bool AS_U8>
__global__ void pack_transpose_kernel(const SrcT* __restrict__ src, int64_t ld, int64_t n, int J, OutT* __restrict__ dst, int Jp) {
  __shared__ double tile[32][33];
  const int64_t i0 = (int64_t)blockIdx.x * 32;
  const int j0 = blockIdx.y * 32;
  for (int jj = threadIdx.y; jj < 32; jj += blockDim.y) {
    const int64_t i = i0 + threadIdx.x;
    const int j = j0 + jj;
    tile[jj][threadIdx.x] = (i < n && j < J) ? (double)src[i + ld * j] : 0.0;
  }
  __syncthreads();
  for (int ii = threadIdx.y; ii < 32; ii += blockDim.y) {
    const int64_t i = i0 + ii;
    const int j = j0 + threadIdx.x;
    if (i < n && j < J) {
      const double v = tile[threadIdx.x][ii];
      if (AS_U8) dst[i * Jp + j] = (OutT)(v > 0.5 ? 1 : 0);
      else dst[i * Jp + j] = (OutT)v;
    }
  }
}
// row-major padded [n][Jp] <-> column-major [n][J] float64 (data and state get/set; a person vector or one column of X is J = Jp = 1)
template <typename R>
__global__ void tile_to_colmajor_kernel(const R* __restrict__ src, int64_t n, int J, int Jp, double* __restrict__ dst) {
  const int64_t total = n * J;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = t % n;
    const int j = (int)(t / n);
    dst[t] = (double)src[i * Jp + j];
  }
}
template <typename R>
__global__ void colmajor_to_tile_kernel(const double* __restrict__ src, int64_t n, int J, int Jp, R* __restrict__ dst) {
  const int64_t total = n * J;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = t % n;
    const int j = (int)(t / n);
    dst[i * Jp + j] = (R)src[t];
  }
}
// column sums over persons in two deterministic stages (the grouping depends only on n, not on how the columns were chunked):
// part[(j)*COLSUM_PARTS + p] = sum over the p-th contiguous slice of rows of f(src[i + ld*j]);  mode 0: v, 1: v^2, 2: (v > 0.5) - 0.5
#define COLSUM_PARTS 32
template <typename SrcT>
__global__ void colsum_part_kernel(const SrcT* __restrict__ src, int64_t ld, int64_t n, int mode, double* __restrict__ part) {
  __shared__ double red[256];
  const int j = blockIdx.x, p = blockIdx.y;
  const int64_t per = (n + COLSUM_PARTS - 1) / COLSUM_PARTS;
  const int64_t lo = p * per, hi = lo + per < n ? lo + per : n;
  double acc = 0.0;
  for (int64_t i = lo + threadIdx.x; i < hi; i += blockDim.x) {
    const double v = (double)src[i + ld * j];
    acc += mode == 0 ? v : (mode == 1 ? v * v : ((v > 0.5 ? 1.0 : 0.0) - 0.5));
  }
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int o = blockDim.x / 2; o; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) part[(int64_t)j * COLSUM_PARTS + p] = red[0];
}
__global__ void colsum_finish_kernel(const double* __restrict__ part, int J, double* __restrict__ out, int parts = COLSUM_PARTS) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= J) return;
  double acc = 0.0;
  for (int p = 0; p < parts; ++p) acc += part[(int64_t)j * parts + p];
  out[j] = acc;
}
// post-burn-in mean and SD from the running sums: tiled [n_pad][Jp] (the N x J cell weights of CrossQr), results column-major [n][J];
// a person vector is J = Jp = 1.  No FMA contraction: same bits as the host formula
__global__ void tile_moments_kernel(const double* __restrict__ s1, const double* __restrict__ s2, int64_t n, int J, int Jp, double cnt,
                                    double* __restrict__ mean, double* __restrict__ sd) {
  const int64_t total = n * J;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = t % n;
    const int j = (int)(t / n);
    if (cnt <= 0.0) { mean[t] = sd[t] = __longlong_as_double(0x7ff8000000000000LL); continue; }
    const double a = s1[i * Jp + j], b = s2[i * Jp + j], m = a / cnt;
    mean[t] = m;
    sd[t] = cnt > 1.0 ? sqrt(fmax(0.0, __dsub_rn(b, __dmul_rn(__dmul_rn(cnt, m), m)) / (cnt - 1.0))) : 0.0;
  }
}
// column sums of the packed tiles (erirt_generate_data: the data never existed in column-major form), same two-stage scheme with
// TILE_COLSUM_PARTS row slices (one block each, thread per column: a warp reads a contiguous piece of a row)
#define TILE_COLSUM_PARTS 1024
template <typename R>
__global__ void tile_colsum_part_kernel(const uint8_t* __restrict__ Y, const R* __restrict__ T, int64_t n, int Jp, double* __restrict__ part) {
  const int j = threadIdx.x, p = blockIdx.x;
  if (j >= Jp) return;
  const int64_t per = (n + TILE_COLSUM_PARTS - 1) / TILE_COLSUM_PARTS;
  const int64_t lo = p * per, hi = lo + per < n ? lo + per : n;
  double t1 = 0.0, t2 = 0.0, k0 = 0.0;
#pragma unroll 4
  for (int64_t i = lo; i < hi; ++i) {
    k0 += Y[i * Jp + j] ? 0.5 : -0.5;
    if (T) { const double v = (double)T[i * Jp + j]; t1 += v; t2 += v * v; }
  }
  part[((int64_t)(0 * Jp + j)) * TILE_COLSUM_PARTS + p] = t1;
  part[((int64_t)(1 * Jp + j)) * TILE_COLSUM_PARTS + p] = t2;
  part[((int64_t)(2 * Jp + j)) * TILE_COLSUM_PARTS + p] = k0;
}

// ---- device-side data generator: the N x J part of setData* (src/SimTools.jl:117-368) straight into the packed tiles ----
//   Y_ij ~ Bernoulli(logistic(a_j (theta_i - b_j)))                                   (:131, :165, :241, :329, :363)
//   logT_ij = lambda_j - zeta_i - theta_i rho_j + e_ij,  e_ij by `err`:
//     0: N(0, sigma2_j) with logT truncated to (0, inf)  (Null / RtIrt, :136-139, :170-173)
//     1: N(0, 1)                                         (Latent*, :336)
//     2: N(0, 0.3)  3: t(5)  4: Gamma(0.5, 1) - 1        (Cross "norm" / "tail" / "skew", :236-247)
struct GenArgs {
  uint8_t* Y;
  void* logT;
  const double *theta, *zeta, *a, *b, *lam, *sd, *rho;  // person vectors [n], item vectors [Jp]
  int64_t n;
  int J, Jp, err, has_rt;
  uint32_t person_offset;
  PhiloxKey key;
};
__device__ __forceinline__ void bm_pair(uint32_t w0, uint32_t w1, double& c, double& s) {
  const double r = sqrt(-2.0 * log(u01d(w0)));
  double sn, cs;
  sincospi(2.0 * u01d(w1), &sn, &cs);
  c = r * cs;
  s = r * sn;
}
template <typename R>
__global__ void generate_data_kernel(const GenArgs A) {
  const int G = A.Jp / 4;
  const int64_t total = A.n * G;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = t / G;
    const int g = (int)(t % G);
    const uint32_t gid = A.person_offset + (uint32_t)i;
    const double th = A.theta[i], ze = A.zeta ? A.zeta[i] : 0.0;
    const uint4 wy = philox(A.key, gid, 0u, make_site(DOM_DATA, DK_Y, (uint32_t)g), 0u);
    const uint32_t wys[4] = {wy.x, wy.y, wy.z, wy.w};
    uint32_t ypack = 0u;
    R lt[4] = {R(0), R(0), R(0), R(0)};
#pragma unroll 1
    for (int e = 0; e < 4; ++e) {
      const int j = 4 * g + e;
      if (j >= A.J) break;
      const double eta = A.a[j] * (th - A.b[j]);
      if (u01d(wys[e]) < 1.0 / (1.0 + exp(-eta))) ypack |= 1u << (8 * e);
      if (!A.has_rt) continue;
      const double mu = A.lam[j] - ze - th * A.rho[j];
      const uint32_t site = make_site(DOM_DATA, DK_LOGT, (uint32_t)j);
      double x;
      if (A.err == 0) {
        x = site_tnorm_pos(A.key, gid, 0u, site, mu, A.sd[j]);
      } else {
        const uint4 wa = philox(A.key, gid, 0u, site, 0u);
        const double z = normal2(wa.x, wa.y);
        if (A.err == 1) x = mu + z;
        else if (A.err == 2) x = mu + 0.3 * z;
        else if (A.err == 4) x = mu + (0.5 * z * z - 1.0);
        else {  // t(5) = Z / sqrt(chi2_5 / 5)
          const uint4 wb = philox(A.key, gid, 0u, make_site(DOM_DATA, DK_AUX, (uint32_t)j), 0u);
          double n1, n2, n3, n4;
          bm_pair(wb.x, wb.y, n1, n2);
          bm_pair(wb.z, wb.w, n3, n4);
          const double n5 = normal2(wa.z, wa.w);
          x = mu + z / sqrt((n1 * n1 + n2 * n2 + n3 * n3 + n4 * n4 + n5 * n5) / 5.0);
        }
      }
      lt[e] = (R)x;
    }
    *reinterpret_cast<uint32_t*>(A.Y + i * A.Jp + 4 * g) = ypack;
    if (A.has_rt) {
      R* d = (R*)A.logT + i * A.Jp + 4 * g;
#pragma unroll
      for (int e = 0; e < 4; ++e) d[e] = lt[e];
    }
  }
}
// XtX[r + pb*c] = sum_i x_ir x_ic, x = [1 X]
__global__ void xtx_kernel(const double* __restrict__ X, int64_t ld, int64_t n, int pb, double* __restrict__ out) {
  __shared__ double red[256];
  const int r = blockIdx.x % pb, c = blockIdx.x / pb;
  double acc = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
    const double xr = r == 0 ? 1.0 : X[i + ld * (r - 1)];
    const double xc = c == 0 ? 1.0 : X[i + ld * (c - 1)];
    acc += xr * xc;
  }
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int o = blockDim.x / 2; o; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[r + pb * c] = red[0];
}

// ------------------------------------------------------------------------------------------------
// handle
// ------------------------------------------------------------------------------------------------
struct erirt_handle {
  erirt_config cfg{};
  Layout L{};
  SmemPlan S{};      // plan of the sampling kernel of this engine
  SmemPlan S_gen{};  // plan of the generic kernel (== S unless the engine samples with the f32 fast kernel; used by the evaluation stage)
  int tpp = 1, tpp_gen = 1;
  int grid_gen = 0;
  int sm_count = 0;
  int grid = 0;
  size_t rsz = 4;
  double k1 = 0.0, k2 = 0.0;  // (1 - 2q) / (q (1 - q)) and 2 / (q (1 - q)) of q = cfg.q_rt
  PhiloxKey key{};            // make_key(cfg.seed, cfg.chain)
  int64_t n_pad = 0;
  int cap = 0, qw = 0;
  int nb = 1;        // replicas of a batched handle (erirt_create_batch): every per-replica buffer below holds nb copies
  ReplicaSizes z{};  // lengths of one copy
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  // device buffers
  char* arena = nullptr;  // the one device allocation every pointer below is a slice of
  std::vector<size_t> guard_offs;  // ERIRT_GUARDS=1: offsets of the 256-byte guard zones that follow every slice (erirt_debug_check_guards)
  uint8_t* dY = nullptr;
  void *dNuCell = nullptr, *dLogT = nullptr, *dOmega = nullptr, *dTheta = nullptr, *dZeta = nullptr, *dNu = nullptr, *dX = nullptr, *dPtrace = nullptr;
  double* dStatsPrev = nullptr;  // reduced statistics of the previous sweep: input of the global kernel's rehearsal pass
  uint32_t* dTileCtr = nullptr;  // work counter of the person launches (dynamic tile dealing)
  double *dMom = nullptr, *dParams = nullptr, *dStats = nullptr, *dConstsLocal = nullptr, *dConsts = nullptr, *dDerived = nullptr;
  double* dLlOut = nullptr;
  double* dNuMom = nullptr;    // CrossQr with cfg.nu_cell_moments: [2][n_pad][Jp] running sum / sum of squares of the cell weights
  double* dColPart = nullptr;  // [3][Jp][COLSUM_PARTS] partial column sums of the ingest
  double *dTrRa = nullptr, *dTrRt = nullptr, *dTrQr = nullptr, *dTrLl = nullptr;
  uint32_t* dSweep = nullptr;
  int* dStatus = nullptr;
  // consts vector layout (f64): T1[Jp] T2[Jp] K0[Jp] XtX[MAXD*MAXD/4 >= pb*pb] sums[2]
  int c_T1 = 0, c_T2 = 0, c_K0 = 0, c_XtX = 0, c_sums = 0, c_count = 0;
  bool data_set = false, consts_final = false, prologue_done = false;
  int64_t sweeps_done = 0;
  double last_ms = 0.0, person_ms = 0.0;
  std::vector<cudaEvent_t> kev;  // event pairs around person launches (time_kernels)
  size_t kev_used = 0;
  // NCCL
  nccl::comm_t comm = nullptr;
  int rank = 0, world = 1;
  // one-shot peer exchange (NVLink peer memory, CUDA IPC between the per-GPU processes)
  double* xbuf = nullptr;             // this GPU's exchange buffer
  double** dPeerBufs = nullptr;       // device array [world] of every GPU's exchange buffer
  uint32_t* dXseq = nullptr;
  int xstride = 0;
  bool peer_ready = false;
  int peer_cache_slot = -1;           // the g_peer_cache entry that owns xbuf / dPeerBufs / dXseq and the peer mappings (-1: none yet)
  // graph
  cudaGraphExec_t graph_exec = nullptr;
  cudaGraphExec_t graph_multi = nullptr;  // GRAPH_SWEEPS sweeps in one graph
};

static int launch_person(erirt_handle* h, int stage);
static int launch_global(erirt_handle* h, int stage);
static int finalize_constants(erirt_handle* h);
// fn(float{}) or fn(double{}): the real type R of the handle's device state, for launches of a kernel template over R
template <typename Fn>
static auto with_real(const erirt_handle* h, Fn&& fn) { return h->cfg.dtype == ERIRT_F32 ? fn(float{}) : fn(double{}); }
static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// `fast`: plan of person_sweep_fast_kernel (f32, one-launch models): the generic plan plus the response tables
static SmemPlan make_smem_plan(const Layout& L, int tpp, size_t rsz, bool has_rt, bool cqr, bool cross, bool fast) {
  SmemPlan S{};
  S.P = CTA_THREADS / tpp;
  S.tile_real_bytes = (int)(S.P * L.Jp * rsz);
  S.tile_y_bytes = S.P * L.Jp;
  S.Dgp = L.Dg + 2;  // + 1/nu column, padded to an odd count to spread banks
  if ((S.Dgp & 1) == 0) ++S.Dgp;
  size_t o = 0;
  S.off_omega = (int)o; o = align_up(o + S.tile_real_bytes, 128);
  S.off_logt = (int)o; if (has_rt) o = align_up(o + S.tile_real_bytes, 128);
  S.off_nuc = (int)o; if (cqr) o = align_up(o + S.tile_real_bytes, 128);
  S.off_y = (int)o; o = align_up(o + S.tile_y_bytes, 128);
  S.off_par = (int)o; o = align_up(o + (cross ? PAR_COUNT : PAR_RHO) * L.Jp * rsz, 128);
  S.off_u = (int)o; o = align_up(o + (size_t)S.P * S.Dgp * rsz, 128);
  S.off_sum = (int)o; o = align_up(o + (size_t)S.P * 4 * rsz, 128);
  S.off_beta = (int)o; o = align_up(o + (size_t)(MAXD + 4) * rsz, 128);
  S.off_acc_item = (int)o; o = align_up(o + (cqr ? 7 : (cross ? 6 : 5)) * L.Jp * sizeof(double), 128);
  S.off_acc_gram = (int)o; o = align_up(o + 2 * L.ntri * sizeof(double), 128);
  // Work queue of the cells that leave the PG fast path.  4 % of the cells do at the benchmark configuration, but attempt 0 is always a
  // Method-A attempt and its acceptance falls with |z|: data with a wide ability distribution (the regression models with |beta| ~ 1:
  // BASELINE configs 1 and 2) defer 15-30 % of their cells.  Small tiles therefore get a queue of up to 45 % of their cells as long
  // as the plan stays below 64 KB (three CTAs per SM either way); an overflowing queue is still handled inline, cell by cell.
  S.qcap = QCAP;
  if (fast) {
    size_t rest = 0;  // what follows the queue in the plan
    rest += align_up((size_t)(L.Jp / 4) * TAB_PITCH * rsz, 128) + align_up((MD_COUNT + SC_COUNT) * sizeof(double) + 8 + 16, 128);
    const size_t budget = 64 * 1024;
    const int want = (int)align_up((size_t)(0.45 * S.P * L.Jp), 256);
    while (S.qcap < want && S.qcap < 16384 && o + (size_t)(S.qcap + 256) * sizeof(uint32_t) + rest <= budget) S.qcap += 256;
  }
  S.qstd = (S.qcap * 3) / 4;
  S.off_queue = (int)o; o = align_up(o + (size_t)S.qcap * sizeof(uint32_t), 128);
  S.off_tab = (int)o; if (fast) o = align_up(o + (size_t)(L.Jp / 4) * TAB_PITCH * rsz, 128);  // response table of the f32 fast kernel
  S.off_misc = (int)o; o = align_up(o + (MD_COUNT + SC_COUNT) * sizeof(double) + 8 + 16, 128);
  S.total = (int)o;
  return S;
}

// batch: the replica-batch instantiation of the kernel (BATCH = true)
template <typename R, int TPP, int FAM>
static const void* person_kernel_ptr_t(bool batch) {
  return batch ? (const void*)person_sweep_kernel<R, TPP, FAM, true> : (const void*)person_sweep_kernel<R, TPP, FAM>;
}
template <typename R, int FAM>
static const void* person_kernel_ptr(int tpp, bool batch) {
  switch (tpp) {
    case 1: return person_kernel_ptr_t<R, 1, FAM>(batch);
    case 2: return person_kernel_ptr_t<R, 2, FAM>(batch);
    case 4: return person_kernel_ptr_t<R, 4, FAM>(batch);
    default: return person_kernel_ptr_t<R, 8, FAM>(batch);
  }
}
template <int TPP, int MODEL>
static const void* person_fast_kernel_ptr_t(bool batch) {
  return batch ? (const void*)person_sweep_fast_kernel<TPP, MODEL, true> : (const void*)person_sweep_fast_kernel<TPP, MODEL>;
}
template <int MODEL>
static const void* person_fast_kernel_ptr_m(int tpp, bool batch) {
  switch (tpp) {
    case 1: return person_fast_kernel_ptr_t<1, MODEL>(batch);
    case 2: return person_fast_kernel_ptr_t<2, MODEL>(batch);
    case 4: return person_fast_kernel_ptr_t<4, MODEL>(batch);
    default: return person_fast_kernel_ptr_t<8, MODEL>(batch);
  }
}
static const void* person_fast_kernel_ptr(int tpp, int model, bool batch) {
  switch (model) {
    case M_MLIRT: return person_fast_kernel_ptr_m<M_MLIRT>(tpp, batch);
    case M_RTIRT: return person_fast_kernel_ptr_m<M_RTIRT>(tpp, batch);
    case M_NULL: return person_fast_kernel_ptr_m<M_NULL>(tpp, batch);
    case M_LATENT: return person_fast_kernel_ptr_m<M_LATENT>(tpp, batch);
    default: return person_fast_kernel_ptr_m<M_LATENTQR>(tpp, batch);
  }
}
// Stage 0 is the sweep of the one-launch models, stages 1 and 2 the two halves of a Cross-family sweep, stage 3 the evaluation.
// Stage 0 in f32 runs person_sweep_fast_kernel (plan h->S); every other stage runs the generic kernel (plan h->S_gen).
static bool runs_fast_kernel(const erirt_handle* h, int stage) { return stage == 0 && h->cfg.dtype == ERIRT_F32; }
static const void* person_kernel_for(const erirt_handle* h, int stage) {
  const bool batch = h->nb > 1;
  if (runs_fast_kernel(h, stage)) return person_fast_kernel_ptr(h->tpp, h->cfg.model, batch);
  if (stage == 0) return person_kernel_ptr<double, 0>(h->tpp, batch);  // Cross-family and evaluation code compiled out
  return h->cfg.dtype == ERIRT_F32 ? person_kernel_ptr<float, 1>(h->tpp_gen, batch) : person_kernel_ptr<double, 1>(h->tpp_gen, batch);
}
static const void* global_kernel_for(const erirt_handle* h) {
  return h->nb > 1 ? (const void*)global_draw_kernel<true> : (const void*)global_draw_kernel<>;
}

static int qr_small_width(int model, int J, int F) {
  switch (model) {
    case M_MLIRT: return F + 1;
    case M_RTIRT: case M_NULL: return 2 * (F + 1) + 4;
    case M_CROSS: case M_CROSSQR: return J + 4;
    default: return F + 2 + 4;
  }
}
static int beta_len(int model, int F) {
  switch (model) {
    case M_MLIRT: return F + 1;
    case M_RTIRT: case M_NULL: return 2 * (F + 1);
    case M_LATENT: case M_LATENTQR: return F + 2;
    default: return 0;
  }
}

// ------------------------------------------------------------------------------------------------
// create / destroy
// ------------------------------------------------------------------------------------------------
extern "C" int erirt_version(void) { return ERIRT_ABI_VERSION; }
extern "C" const char* erirt_last_error(void) { return g_err.c_str(); }

// Exchange buffers and their CUDA IPC mappings are kept for the next handle of the process (same device, rank, world and slot size):
// opening the seven peer mappings of an 8-GPU chain costs ~40 ms per erirt_create + attach, more than 100 sweeps of the benchmark.
// The stamps are sequence numbers that simply keep counting (xseq is cached with the buffer), so a reused buffer needs no reset;
// every rank of a sharded program makes the same calls, hence the same reuse decisions.  erirt_trim_pool releases the entries
// that are not in use.
struct PeerCacheEntry {
  int device = -1, world = 0, rank = -1, xstride = 0;
  double* xbuf = nullptr;
  double** dPeerBufs = nullptr;
  uint32_t* dXseq = nullptr;
  std::vector<void*> opened;
  std::vector<char> handles;  // world x 64 bytes the mappings were opened from
  bool in_use = false;
};
static std::mutex g_peer_mu;
static std::vector<PeerCacheEntry> g_peer_cache;
static void peer_cache_release_entry(PeerCacheEntry& c) {
  for (void* p : c.opened) cudaIpcCloseMemHandle(p);
  c.opened.clear();
  c.handles.clear();
  if (c.xbuf) cudaFree(c.xbuf);
  if (c.dPeerBufs) cudaFree(c.dPeerBufs);
  if (c.dXseq) cudaFree(c.dXseq);
  c.xbuf = nullptr; c.dPeerBufs = nullptr; c.dXseq = nullptr; c.device = -1;
}

static int free_handle(erirt_handle* h) {
  if (!h) return 0;
  cudaSetDevice(h->cfg.device);
  if (h->graph_exec) cudaGraphExecDestroy(h->graph_exec);
  if (h->graph_multi) cudaGraphExecDestroy(h->graph_multi);
  if (h->comm && nccl::comm_destroy) nccl::comm_destroy(h->comm);
  if (h->peer_cache_slot >= 0) {  // buffers and mappings stay with the cache
    if (h->stream) cudaStreamSynchronize(h->stream);
    std::lock_guard<std::mutex> lk(g_peer_mu);
    g_peer_cache[h->peer_cache_slot].in_use = false;
  }
  if (h->arena && h->stream) {  // all device buffers of the handle: back to the pool
    cudaFreeAsync(h->arena, h->stream);
    cudaStreamSynchronize(h->stream);
  } else if (h->arena) cudaFree(h->arena);
  for (cudaEvent_t e : h->kev) cudaEventDestroy(e);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
  return 0;
}

extern "C" int erirt_create(const erirt_config* cfg, erirt_handle** out) { return erirt_create_batch(cfg, 1, out); }

extern "C" int erirt_create_batch(const erirt_config* cfg, int32_t n_batch, erirt_handle** out) {
  if (!cfg || !out) return fail(ERIRT_E_ARG, "null argument");
  *out = nullptr;
  if (n_batch < 1 || n_batch > 65535) return fail(ERIRT_E_ARG, "n_batch %d outside [1, 65535]", n_batch);
  if (n_batch > 1 && (cfg->model == ERIRT_RTIRT_CROSS || cfg->model == ERIRT_RTIRT_CROSSQR))
    return fail(ERIRT_E_UNSUPPORTED, "replica batches of the Cross family are not supported (two-stage sweep)");
  if (n_batch > 1 && cfg->person_trace) return fail(ERIRT_E_UNSUPPORTED, "replica batches keep no person trace (person_trace = 1)");
  if (cfg->abi_version != ERIRT_ABI_VERSION) return fail(ERIRT_E_ARG, "abi_version %d != %d", cfg->abi_version, ERIRT_ABI_VERSION);
  if (cfg->model < 0 || cfg->model > 6) return fail(ERIRT_E_ARG, "unknown model %d", cfg->model);
  if (cfg->n_subj < 1 || cfg->n_item < 1 || cfg->n_feat < 0) return fail(ERIRT_E_ARG, "bad dimensions");
  if (cfg->n_subj_total < cfg->n_subj || cfg->subj_offset < 0 || cfg->subj_offset + cfg->n_subj > cfg->n_subj_total)
    return fail(ERIRT_E_ARG, "inconsistent shard: n_subj=%lld offset=%lld total=%lld", (long long)cfg->n_subj,
                (long long)cfg->subj_offset, (long long)cfg->n_subj_total);
  if (cfg->n_subj_total > 0xffffffffLL) return fail(ERIRT_E_ARG, "n_subj_total exceeds the 32-bit person counter");
  if (2 * (cfg->n_feat + 1) > MAXD) return fail(ERIRT_E_ARG, "n_feat %d too large (2*(n_feat+1) <= %d)", cfg->n_feat, MAXD);
  if (cfg->n_item > 500) return fail(ERIRT_E_ARG, "n_item %d too large (<= 500)", cfg->n_item);
  if (cfg->n_iter < 1 || cfg->n_chain < 1) return fail(ERIRT_E_ARG, "n_iter and n_chain must be >= 1");
  if (cfg->dtype != ERIRT_F32 && cfg->dtype != ERIRT_F64) return fail(ERIRT_E_ARG, "dtype must be ERIRT_F32 or ERIRT_F64");
  if (!(cfg->q_rt > 0.0 && cfg->q_rt < 1.0)) return fail(ERIRT_E_ARG, "qRt must be between 0 and 1");  // Draw.pl.jl:476

  HostTimer tm;
  if (int rc = pick_device(cfg->device)) return rc;
  // three attributes, not cudaGetDeviceProperties: that call was measured at 3-260 ms per erirt_create on this box
  struct { int major, minor, multiProcessorCount; } prop;
  CU(cudaDeviceGetAttribute(&prop.major, cudaDevAttrComputeCapabilityMajor, cfg->device));
  CU(cudaDeviceGetAttribute(&prop.minor, cudaDevAttrComputeCapabilityMinor, cfg->device));
  CU(cudaDeviceGetAttribute(&prop.multiProcessorCount, cudaDevAttrMultiProcessorCount, cfg->device));
  tm.mark("create: device properties");
  if (prop.major < 10) return fail(ERIRT_E_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", cfg->device, prop.major, prop.minor);

  {  // staging buffers and the full-size buffers of a handle are stream-ordered allocations: keep up to ERIRT_POOL_KEEP_MB (default
     // 4096) of freed memory in the device's default pool instead of returning it to the driver at every synchronisation, so that the
     // next sample! of the process does not pay for mapping its gigabyte again.  erirt_trim_pool() gives it back.
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, cfg->device) == cudaSuccess) {
      const char* env = getenv("ERIRT_POOL_KEEP_MB");
      uint64_t thr = (uint64_t)(env ? atoll(env) : 4096) << 20;
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    }
  }
  erirt_handle* h = new erirt_handle();
  h->cfg = *cfg;
  h->nb = n_batch;
  h->sm_count = prop.multiProcessorCount;
  h->rsz = cfg->dtype == ERIRT_F32 ? 4 : 8;
  h->k1 = (1.0 - 2.0 * cfg->q_rt) / (cfg->q_rt * (1.0 - cfg->q_rt));
  h->k2 = 2.0 / (cfg->q_rt * (1.0 - cfg->q_rt));
  h->key = make_key(cfg->seed, cfg->chain);
  h->L = make_layout(cfg->n_item, cfg->n_feat);
  const bool has_rt = cfg->model != ERIRT_MLIRT;
  // threads per person: smallest TPP whose shared-memory plan leaves room for >= 3 CTAs per SM (75 KB + 1 KB reserved each)
  const bool is_cross = cfg->model == ERIRT_RTIRT_CROSS || cfg->model == ERIRT_RTIRT_CROSSQR;
  const bool is_cqr = cfg->model == ERIRT_RTIRT_CROSSQR;
  const bool fast_engine = cfg->dtype == ERIRT_F32 && !is_cross;
  const int n_groups = h->L.Jp / 4;
  auto choose = [&](bool fast, int& tpp, SmemPlan& S) -> const char* {
    for (tpp = 1; tpp < 8; tpp *= 2) {
      SmemPlan s = make_smem_plan(h->L, tpp, h->rsz, has_rt, is_cqr, is_cross, fast);
      if (s.total <= 75 * 1024 && n_groups <= 16 * tpp) break;
    }
    // Float64 (the generic kernel): a cell costs thousands of instructions, so a problem with fewer tiles than two per SM is
    // spread over more, smaller tiles (measured at BASELINE configs 1-3: 2x the sweeps/s from TPP 1 -> 8; the f32 kernels, whose
    // sweep is bound by the per-tile latency chain, gain nothing: profiles/r02_summary.md)
    // (for a large problem TPP = 8 was 7 % faster while the cell loop was one divergent exact draw per cell; with the branch-free
    // attempt 0 the 168-register TPP = 4 instantiation wins, 4.0 against 5.3 ms per sweep at 1M x 100)
    // (a replica batch counts the tiles of all its replicas)
    if (!fast && cfg->dtype == ERIRT_F64)
      while (tpp < 8 && (int64_t)align_up((size_t)cfg->n_subj, 128) * n_batch / (CTA_THREADS / tpp) < 2 * (int64_t)h->sm_count) tpp *= 2;
    if (n_groups > 16 * tpp) return "too many items for this TPP (at most 64*TPP - 4)";
    S = make_smem_plan(h->L, tpp, h->rsz, has_rt, is_cqr, is_cross, fast);
    if (S.total > 227 * 1024) return "n_item needs more shared memory per CTA than an SM has";
    return nullptr;
  };
  if (const char* msg = choose(fast_engine, h->tpp, h->S)) { delete h; return fail(ERIRT_E_UNSUPPORTED, "%s (n_item %d)", msg, cfg->n_item); }
  if (fast_engine) {
    if (const char* msg = choose(false, h->tpp_gen, h->S_gen)) { delete h; return fail(ERIRT_E_UNSUPPORTED, "%s (n_item %d)", msg, cfg->n_item); }
  } else {
    h->tpp_gen = h->tpp;
    h->S_gen = h->S;
  }
  h->n_pad = (int64_t)align_up((size_t)cfg->n_subj, 128);
  h->cap = cfg->n_iter * cfg->n_chain;
  h->qw = qr_small_width(cfg->model, cfg->n_item, cfg->n_feat);
  h->z = replica_sizes(h->n_pad, h->L, h->cap, h->qw);

  {
    tm.mark("create: pool attr, plans");
    cudaError_t ce = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
    if (ce != cudaSuccess) { free_handle(h); return fail(ERIRT_E_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(ce)); }
    cudaEventCreate(&h->ev0);
    cudaEventCreate(&h->ev1);
  }
  // Every device buffer of the handle is a slice of ONE zero-initialised block from the device's stream-ordered pool: one allocation
  // and one memset at create, one free at destroy (dozens of cudaMalloc / cudaFree calls, each a driver round trip and, for cudaFree,
  // a device-wide synchronisation, made create and destroy take 10-250 ms), and the next handle of the process finds the memory in
  // the pool again.
  const size_t cells = (size_t)h->n_pad * h->L.Jp;
  h->c_T1 = 0; h->c_T2 = h->L.Jp; h->c_K0 = 2 * h->L.Jp; h->c_XtX = 3 * h->L.Jp; h->c_sums = h->c_XtX + MAXD * MAXD / 4;
  h->c_count = consts_count(h->L);
  {
    struct Req { void** p; size_t bytes; };
    std::vector<Req> reqs;
    // every buffer but the ingest scratch dColPart holds one copy per replica (ReplicaSizes)
    auto want = [&](void** p, size_t bytes) {
      if (p != (void**)&h->dColPart) bytes *= (size_t)n_batch;
      reqs.push_back({p, align_up(bytes > 0 ? bytes : 16, 256)});
    };
    const size_t vec = (size_t)h->n_pad * h->rsz, D = sizeof(double);
    want((void**)&h->dY, cells);
    want(&h->dOmega, cells * h->rsz);
    if (has_rt) want(&h->dLogT, cells * h->rsz);
    if (cfg->model == ERIRT_RTIRT_CROSSQR) want(&h->dNuCell, cells * h->rsz);
    if (cfg->model == ERIRT_RTIRT_CROSSQR && cfg->nu_cell_moments) want((void**)&h->dNuMom, 2 * cells * D);
    want(&h->dTheta, vec);
    want(&h->dZeta, vec);
    want(&h->dNu, vec);
    want(&h->dX, vec * (cfg->n_feat > 0 ? cfg->n_feat : 1));
    want((void**)&h->dMom, (size_t)6 * h->n_pad * D);
    if (cfg->person_trace) want(&h->dPtrace, (size_t)h->cap * 3 * vec);
    want((void**)&h->dParams, (size_t)h->L.p_count * D);
    want((void**)&h->dStats, (size_t)(h->L.s_count + 2) * D);
    want((void**)&h->dStatsPrev, (size_t)(h->L.s_count + 2) * D);
    want((void**)&h->dTileCtr, sizeof(uint32_t));
    want((void**)&h->dConstsLocal, (size_t)h->c_count * D);
    want((void**)&h->dConsts, (size_t)h->c_count * D);
    want((void**)&h->dDerived, 4 * D);
    want((void**)&h->dColPart, (size_t)3 * h->L.Jp * COLSUM_PARTS * D);
    want((void**)&h->dTrRa, (size_t)h->cap * 2 * cfg->n_item * D);
    want((void**)&h->dTrRt, (size_t)h->cap * 2 * cfg->n_item * D);
    want((void**)&h->dTrQr, (size_t)h->cap * h->qw * D);
    want((void**)&h->dTrLl, (size_t)h->cap * D);
    want((void**)&h->dSweep, sizeof(uint32_t));
    want((void**)&h->dStatus, sizeof(int));
    want((void**)&h->dLlOut, D);
    // ERIRT_GUARDS=1 (debugging; compute-sanitizer is not available on every pool): every slice is followed by a 256-byte guard zone
    // filled with 0xA5, and erirt_debug_check_guards() counts the guard bytes a kernel, a bulk copy or an ingest pass has overwritten
    const char* env_guard = getenv("ERIRT_GUARDS");
    const size_t guard = (env_guard && atoi(env_guard) > 0) ? 256 : 0;
    size_t total = 0;
    for (const Req& r : reqs) total += r.bytes + guard;
    tm.mark("create: stream, events");
    cudaError_t ae = cudaMallocAsync((void**)&h->arena, total, h->stream);
    tm.mark("create: cudaMallocAsync");
    if (ae == cudaSuccess) ae = cudaMemsetAsync(h->arena, 0, total, h->stream);
    if (ae != cudaSuccess) { free_handle(h); return fail(ERIRT_E_CUDA, "allocating %zu bytes of device memory: %s", total, cudaGetErrorString(ae)); }
    size_t off = 0;
    for (const Req& r : reqs) {
      *r.p = h->arena + off;
      off += r.bytes;
      if (guard) {
        cudaMemsetAsync(h->arena + off, 0xA5, guard, h->stream);
        h->guard_offs.push_back(off);
        off += guard;
      }
    }
  }
  // default parameters == setInitialValues (a = 1, sigma2 = 1, Sigma = I; src/GibbsRtIrt.pl.jl:122-133)
  {
    std::vector<double> p(h->L.p_count, 0.0);
    for (int j = 0; j < cfg->n_item; ++j) { p[h->L.p_a + j] = 1.0; p[h->L.p_sigma2 + j] = 1.0; }
    p[h->L.p_Sigma + 0] = 1.0; p[h->L.p_Sigma + 3] = 1.0;
    const std::vector<double> one = p;
    for (int r = 1; r < n_batch; ++r) p.insert(p.end(), one.begin(), one.end());
    cudaMemcpyAsync(h->dParams, p.data(), p.size() * sizeof(double), cudaMemcpyHostToDevice, h->stream);
    cudaStreamSynchronize(h->stream);  // p is a local; also orders the zero-fill before any default-stream access below
  }
  // kernel attributes / occupancy-sized persistent grid
  tm.mark("create: memset, params, sync");
  const void* kfn = person_kernel_for(h, is_cross ? 1 : 0);
  cudaError_t ce = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, h->S.total);
  if (ce == cudaSuccess) ce = cudaFuncSetAttribute(person_kernel_for(h, 1), cudaFuncAttributeMaxDynamicSharedMemorySize, h->S_gen.total);
  if (ce != cudaSuccess) { free_handle(h); return fail(ERIRT_E_CUDA, "cudaFuncSetAttribute(%d bytes): %s", h->S.total, cudaGetErrorString(ce)); }
  int occ = 0;
  ce = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kfn, CTA_THREADS, h->S.total);
  if (ce != cudaSuccess || occ < 1) { free_handle(h); return fail(ERIRT_E_CUDA, "person kernel does not fit on an SM: %s", cudaGetErrorString(ce)); }
  const int n_tiles = (int)(h->n_pad / h->S.P);
  // A replica batch launches grid x n_batch CTAs: the grid of a replica is sized so that the whole launch stays within the resident
  // slots where it can (one CTA per replica at least)
  h->grid = std::max(1, std::min(n_tiles, h->sm_count * occ / n_batch));
  // A full grid leaves ONE slot free: with dynamic tile dealing no person CTA exits before the last round, so the global kernel of the
  // sweep (256 threads, 80 registers, ~55 KB) could otherwise not become resident early enough to finish its rehearsal pass
  // (global.cuh) before the person kernel ends; the slot costs 1/444 of the person kernel's throughput
  if (h->grid * n_batch == h->sm_count * occ && h->grid > 1) h->grid -= 1;
  // test hook: ERIRT_MAX_GRID caps the persistent grid, so that a small problem gives every CTA many tiles (the cross-tile register
  // accumulators and their 16-tile fold are otherwise reached only at benchmark size); results do not depend on the grid
  const char* env_grid = getenv("ERIRT_MAX_GRID");
  const int max_grid = env_grid && atoi(env_grid) > 0 ? atoi(env_grid) : (1 << 30);
  h->grid = std::min(h->grid, max_grid);
  {  // the global kernel stages the statistics in dynamic shared memory on top of its ~42 KB of static scratch
    const size_t gsm = (size_t)(h->L.s_count + 2 + (h->L.F + 1) * (h->L.F + 1) + 5 * h->L.Jp) * sizeof(double);
    ce = cudaFuncSetAttribute(global_kernel_for(h), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gsm);
    if (ce != cudaSuccess) { free_handle(h); return fail(ERIRT_E_CUDA, "cudaFuncSetAttribute(global_draw_kernel, %zu bytes): %s", gsm, cudaGetErrorString(ce)); }
  }
  {
    int occ_gen = 0;
    ce = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_gen, person_kernel_for(h, 1), CTA_THREADS, h->S_gen.total);
    if (ce != cudaSuccess || occ_gen < 1) { free_handle(h); return fail(ERIRT_E_CUDA, "generic person kernel does not fit on an SM: %s", cudaGetErrorString(ce)); }
    h->grid_gen = std::min(std::min((int)(h->n_pad / h->S_gen.P), std::max(1, h->sm_count * occ_gen / n_batch)), max_grid);
  }
  tm.mark("create: func attrs, occupancy");
  *out = h;
  return 0;
}

extern "C" int erirt_destroy(erirt_handle* h) { return free_handle(h); }
extern "C" int erirt_trim_pool(int32_t device) {
  CU(cudaSetDevice(device));
  cudaMemPool_t pool;
  CU(cudaDeviceGetDefaultMemPool(&pool, device));
  CU(cudaDeviceSynchronize());
  CU(cudaMemPoolTrimTo(pool, 0));
  {
    std::lock_guard<std::mutex> lk(g_peer_mu);
    for (PeerCacheEntry& c : g_peer_cache)
      if (!c.in_use && c.device == device) peer_cache_release_entry(c);
  }
  return 0;
}

// ------------------------------------------------------------------------------------------------
// data
// ------------------------------------------------------------------------------------------------
// Pack columns [c0, c0+nc) of replica r's Y / logT (column-major, on the device) into its person-major tiles and add their partial
// column sums.
template <typename R, typename YT>
static void pack_columns(erirt_handle* h, int r, const YT* dYc, int64_t ldY, const double* dTc, int64_t ldT, int c0, int nc) {
  const int64_t n = h->cfg.n_subj;
  const int Jp = h->L.Jp;
  dim3 blk(32, 8), grd((unsigned)((n + 31) / 32), (unsigned)((nc + 31) / 32));
  dim3 cg((unsigned)nc, COLSUM_PARTS);
  pack_transpose_kernel<YT, uint8_t, true><<<grd, blk, 0, h->stream>>>(dYc, ldY, n, nc, h->dY + r * h->z.cells + c0, Jp);
  colsum_part_kernel<YT><<<cg, 256, 0, h->stream>>>(dYc, ldY, n, 2, h->dColPart + (size_t)(2 * Jp + c0) * COLSUM_PARTS);
  if (dTc) {
    pack_transpose_kernel<double, R, false><<<grd, blk, 0, h->stream>>>(dTc, ldT, n, nc, (R*)h->dLogT + r * h->z.cells + c0, Jp);
    colsum_part_kernel<double><<<cg, 256, 0, h->stream>>>(dTc, ldT, n, 0, h->dColPart + (size_t)(0 * Jp + c0) * COLSUM_PARTS);
    colsum_part_kernel<double><<<cg, 256, 0, h->stream>>>(dTc, ldT, n, 1, h->dColPart + (size_t)(1 * Jp + c0) * COLSUM_PARTS);
  }
}

// The start of every ingest: zero the packed Y / logT of every replica (the padding cells stay zero) and the constants the ingest adds up
static int clear_data(erirt_handle* h) {
  const size_t cells = (size_t)h->z.cells * h->nb;
  CU(cudaMemsetAsync(h->dY, 0, cells, h->stream));
  if (h->cfg.model != ERIRT_MLIRT) CU(cudaMemsetAsync(h->dLogT, 0, cells * h->rsz, h->stream));
  CU(cudaMemsetAsync(h->dConstsLocal, 0, (size_t)h->z.consts * h->nb * sizeof(double), h->stream));
  return 0;
}

// The end of every ingest of replica r, after its Y / logT are packed: X (column-major float64 [n][F], leading dimension ldX; a host
// buffer unless x_on_device) into dX, the constants in f64 (T1, T2, K0 are consecutive Jp-blocks of the consts vector, finished from
// `part`: [3 Jp][parts] partial column sums; X'X), then a synchronisation, after which the replica's data is in place.
static int finish_ingest(erirt_handle* h, int r, const double* X, int64_t ldX, bool x_on_device, const double* part, int parts) {
  const int64_t n = h->cfg.n_subj;
  const int Jp = h->L.Jp, F = h->cfg.n_feat, pb = F + 1;
  double* staged = nullptr;
  auto cleanup = [&]() { if (staged) cudaFreeAsync(staged, h->stream); };
  if (F > 0 && !x_on_device) {
    CUX(cudaMallocAsync((void**)&staged, (size_t)n * F * sizeof(double), h->stream));
    CUX(cudaMemcpy2DAsync(staged, n * sizeof(double), X, ldX * sizeof(double), n * sizeof(double), F, cudaMemcpyHostToDevice, h->stream));
    X = staged;
    ldX = n;
  }
  for (int f = 0; f < F; ++f)
    with_real(h, [&](auto rr) {
      using R = decltype(rr);
      colmajor_to_tile_kernel<R><<<1024, 256, 0, h->stream>>>(X + ldX * f, n, 1, 1, (R*)h->dX + r * h->z.x + (int64_t)f * h->n_pad);
    });
  double* consts = h->dConstsLocal + r * h->z.consts;
  colsum_finish_kernel<<<(3 * Jp + 127) / 128, 128, 0, h->stream>>>(part, 3 * Jp, consts + h->c_T1, parts);
  xtx_kernel<<<pb * pb, 256, 0, h->stream>>>(X, ldX, n, pb, consts + h->c_XtX);
  CUX(cudaGetLastError());
  cleanup();
  staged = nullptr;
  CUX(cudaStreamSynchronize(h->stream));
  h->data_set = true;
  h->consts_final = false;
  return 0;
}

// Ingest (K8) of replica r: rows [r n_subj, (r+1) n_subj) of the caller's matrices.  on_device: the three matrices are device buffers
// and are packed in place.  Otherwise they are host buffers and are streamed through one bounded staging buffer in chunks of whole
// columns (H2D copy, pack, next chunk: the staging memory stays at <= 64 MB instead of a second copy of the data set, and the packed
// tiles are the only full-size device copy).
template <typename YT>
static int ingest_replica(erirt_handle* h, int r, const YT* Y, int64_t ldY, const double* T, int64_t ldT, const double* X, int64_t ldX,
                          bool on_device) {
  const bool has_rt = h->cfg.model != ERIRT_MLIRT;
  const int64_t n = h->cfg.n_subj;
  const int J = h->cfg.n_item, Jp = h->L.Jp;
  Y += r * n;
  if (T) T += r * n;
  if (X) X += r * n;
  CU(cudaMemsetAsync(h->dColPart, 0, (size_t)3 * Jp * COLSUM_PARTS * sizeof(double), h->stream));
  if (on_device) {
    with_real(h, [&](auto rr) { pack_columns<decltype(rr), YT>(h, r, Y, ldY, T, ldT, 0, J); });
    return finish_ingest(h, r, X, ldX, true, h->dColPart, COLSUM_PARTS);
  }
  // stream-ordered allocations: cudaFree of large blocks is a device-wide synchronisation (measured up to 0.9 s for GB-sized blocks)
  char* stage = nullptr;
  auto cleanup = [&]() { if (stage) cudaFreeAsync(stage, h->stream); };
  const size_t col_bytes = (size_t)n * (sizeof(YT) + (has_rt ? sizeof(double) : 0));
  int cc = (int)std::max<size_t>(1, std::min<size_t>((size_t)J, ((size_t)64 << 20) / col_bytes));
  const size_t y_bytes = align_up((size_t)n * cc * sizeof(YT), 256);
  CUX(cudaMallocAsync((void**)&stage, y_bytes + (has_rt ? (size_t)n * cc * sizeof(double) : 0), h->stream));
  YT* sY = (YT*)stage;
  double* sT = has_rt ? (double*)(stage + y_bytes) : nullptr;
  for (int c0 = 0; c0 < J; c0 += cc) {
    const int nc = std::min(cc, J - c0);
    CUX(cudaMemcpy2DAsync(sY, n * sizeof(YT), Y + ldY * c0, ldY * sizeof(YT), n * sizeof(YT), nc, cudaMemcpyHostToDevice, h->stream));
    if (has_rt) CUX(cudaMemcpy2DAsync(sT, n * sizeof(double), T + ldT * c0, ldT * sizeof(double), n * sizeof(double), nc, cudaMemcpyHostToDevice, h->stream));
    with_real(h, [&](auto rr) { pack_columns<decltype(rr), YT>(h, r, sY, n, sT, n, c0, nc); });
  }
  cleanup();
  return finish_ingest(h, r, X, ldX, false, h->dColPart, COLSUM_PARTS);
}

// Ingest of every replica: the matrices have n_batch * n_subj rows, replica r's in rows [r n_subj, (r+1) n_subj).  The constants of a
// replica come from its rows alone, by the code of a standalone ingest, so they carry the same bits.
template <typename YT>
static int ingest(erirt_handle* h, const YT* Y, int64_t ldY, const double* T, int64_t ldT, const double* X, int64_t ldX, bool on_device) {
  if (!h || !Y) return fail(ERIRT_E_ARG, "null argument");
  const bool has_rt = h->cfg.model != ERIRT_MLIRT;
  if (has_rt && !T) return fail(ERIRT_E_ARG, "logT is required for this model");
  if (h->cfg.n_feat > 0 && !X) return fail(ERIRT_E_ARG, "X is required when n_feat > 0");
  CU(cudaSetDevice(h->cfg.device));
  const int64_t n = h->cfg.n_subj * h->nb;
  if (ldY < n || (has_rt && ldT < n) || (h->cfg.n_feat > 0 && ldX < n))
    return fail(ERIRT_E_ARG, h->nb > 1 ? "leading dimension smaller than n_batch * n_subj" : "leading dimension smaller than n_subj");
  if (!has_rt) T = nullptr;
  if (int rc = clear_data(h)) return rc;
  for (int r = 0; r < h->nb; ++r)
    if (int rc = ingest_replica(h, r, Y, ldY, T, ldT, X, ldX, on_device)) return rc;
  return 0;
}

// ---- data generated on the device (SURVEY 8f-1) ----
// Replica r: the person vectors and X start at its first row, the item vectors at its first item; data seed `seed`
static int generate_replica(erirt_handle* h, int r, const double* theta, const double* zeta, const double* a, const double* b,
                            const double* lambda, const double* sigma2, const double* rho, const double* X, int64_t ldX,
                            int32_t error_type, uint64_t seed) {
  const bool has_rt = h->cfg.model != ERIRT_MLIRT;
  const int64_t n = h->cfg.n_subj;
  const int J = h->cfg.n_item, Jp = h->L.Jp;
  HostTimer tm;
  // device copy of the small inputs: [theta n][zeta n][a Jp][b Jp][lambda Jp][sd Jp][rho Jp]; the person vectors go straight from
  // the caller's buffers, the item vectors through a small host block
  std::vector<double> hit((size_t)5 * Jp, 0.0);
  double* it = hit.data();
  for (int j = 0; j < J; ++j) {
    it[j] = a[j];
    it[Jp + j] = b[j];
    it[2 * Jp + j] = has_rt ? lambda[j] : 0.0;
    it[3 * Jp + j] = sigma2 ? std::sqrt(sigma2[j]) : 1.0;
    it[4 * Jp + j] = rho ? rho[j] : 0.0;
  }
  double *dbuf = nullptr, *dpart = nullptr;  // dpart: [3][Jp][TILE_COLSUM_PARTS]
  auto cleanup = [&]() { if (dbuf) cudaFreeAsync(dbuf, h->stream); if (dpart) cudaFreeAsync(dpart, h->stream); };
  CUX(cudaMallocAsync((void**)&dbuf, ((size_t)2 * n + 5 * Jp) * sizeof(double), h->stream));
  CUX(cudaMemcpyAsync(dbuf, theta, n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  if (has_rt) CUX(cudaMemcpyAsync(dbuf + n, zeta, n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  CUX(cudaMemcpyAsync(dbuf + 2 * n, hit.data(), hit.size() * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  tm.mark("generate: host staging, H2D");
  GenArgs A{};
  A.Y = h->dY + r * h->z.cells;
  A.logT = has_rt ? (char*)h->dLogT + r * h->z.cells * h->rsz : nullptr;
  A.theta = dbuf; A.zeta = has_rt ? dbuf + n : nullptr;
  A.a = dbuf + 2 * n; A.b = A.a + Jp; A.lam = A.a + 2 * Jp; A.sd = A.a + 3 * Jp; A.rho = A.a + 4 * Jp;
  A.n = n; A.J = J; A.Jp = Jp; A.err = error_type; A.has_rt = has_rt ? 1 : 0;
  A.person_offset = (uint32_t)h->cfg.subj_offset;
  A.key = make_key(seed, 0xDA7Au);
  with_real(h, [&](auto r) { generate_data_kernel<decltype(r)><<<h->sm_count * 8, 256, 0, h->stream>>>(A); });
  CUX(cudaMallocAsync((void**)&dpart, (size_t)3 * Jp * TILE_COLSUM_PARTS * sizeof(double), h->stream));
  with_real(h, [&](auto r) {
    using R = decltype(r);
    tile_colsum_part_kernel<R><<<TILE_COLSUM_PARTS, Jp, 0, h->stream>>>(A.Y, (const R*)A.logT, n, Jp, dpart);
  });
  const int rc = finish_ingest(h, r, X, ldX, false, dpart, TILE_COLSUM_PARTS);
  cleanup();
  tm.mark("generate: launches, device work");
  return rc;
}

// A batch generates replica r from rows [r n_subj, (r+1) n_subj) of theta, zeta and X, items [r n_item, (r+1) n_item) of the item
// vectors, and data seed seed + r: the data set a standalone handle generates from the same inputs with that seed.
extern "C" int erirt_generate_data(erirt_handle* h, const double* theta, const double* zeta, const double* a, const double* b,
                                   const double* lambda, const double* sigma2, const double* rho, const double* X, int64_t ldX,
                                   int32_t error_type, uint64_t seed) {
  if (!h || !theta || !a || !b) return fail(ERIRT_E_ARG, "null argument");
  const bool has_rt = h->cfg.model != ERIRT_MLIRT;
  if (has_rt && (!zeta || !lambda)) return fail(ERIRT_E_ARG, "zeta and lambda are required for a response-time model");
  if (error_type < 0 || error_type > 4) return fail(ERIRT_E_ARG, "error_type must be 0 (truncated normal), 1 (unit normal), 2 (norm), 3 (tail) or 4 (skew)");
  if (has_rt && error_type == 0 && !sigma2) return fail(ERIRT_E_ARG, "sigma2 is required for error_type 0");
  const int64_t n = h->cfg.n_subj;
  const int J = h->cfg.n_item;
  if (h->cfg.n_feat > 0 && (!X || ldX < n * h->nb))
    return fail(ERIRT_E_ARG, h->nb > 1 ? "X (leading dimension >= n_batch * n_subj) is required when n_feat > 0"
                                       : "X (leading dimension >= n_subj) is required when n_feat > 0");
  CU(cudaSetDevice(h->cfg.device));
  if (int rc = clear_data(h)) return rc;
  auto at = [](const double* p, int64_t off) { return p ? p + off : nullptr; };
  for (int r = 0; r < h->nb; ++r)
    if (int rc = generate_replica(h, r, theta + r * n, at(zeta, r * n), a + (int64_t)r * J, b + (int64_t)r * J, at(lambda, (int64_t)r * J),
                                  at(sigma2, (int64_t)r * J), at(rho, (int64_t)r * J), at(X, r * n), ldX, error_type, seed + (uint64_t)r))
      return rc;
  return 0;
}

// The data set held by the handle (ingested or generated), back in Julia's column-major Float64 (logT as stored: f32-rounded in f32 mode)
extern "C" int erirt_get_data(erirt_handle* h, double* Y, int64_t ldY, double* logT, int64_t ldT) {
  if (!h || (!Y && !logT)) return fail(ERIRT_E_ARG, "null argument");
  if (!h->data_set) return fail(ERIRT_E_STATE, "no data set: call erirt_set_data or erirt_generate_data first");
  const int64_t n = h->cfg.n_subj;
  const int J = h->cfg.n_item, Jp = h->L.Jp;
  if ((Y && ldY < n * h->nb) || (logT && ldT < n * h->nb))
    return fail(ERIRT_E_ARG, h->nb > 1 ? "leading dimension smaller than n_batch * n_subj" : "leading dimension smaller than n_subj");
  if (logT && h->cfg.model == ERIRT_MLIRT) return fail(ERIRT_E_ARG, "GibbsMlIrt has no response times");
  CU(cudaSetDevice(h->cfg.device));
  double* tmp = nullptr;
  CU(cudaMallocAsync((void**)&tmp, (size_t)n * J * sizeof(double), h->stream));
  cudaError_t e = cudaSuccess;
  for (int r = 0; r < h->nb && e == cudaSuccess; ++r) {  // replica r: rows [r n, (r+1) n)
    if (Y) {
      tile_to_colmajor_kernel<uint8_t><<<1024, 256, 0, h->stream>>>(h->dY + r * h->z.cells, n, J, Jp, tmp);
      e = cudaMemcpy2DAsync(Y + r * n, ldY * sizeof(double), tmp, n * sizeof(double), n * sizeof(double), J, cudaMemcpyDeviceToHost, h->stream);
      if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    }
    if (logT && e == cudaSuccess) {
      with_real(h, [&](auto rr) {
        using R = decltype(rr);
        tile_to_colmajor_kernel<R><<<1024, 256, 0, h->stream>>>((const R*)h->dLogT + r * h->z.cells, n, J, Jp, tmp);
      });
      e = cudaMemcpy2DAsync(logT + r * n, ldT * sizeof(double), tmp, n * sizeof(double), n * sizeof(double), J, cudaMemcpyDeviceToHost, h->stream);
      if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);  // tmp is reused by the next replica
    }
  }
  cudaFreeAsync(tmp, h->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  if (e != cudaSuccess) return fail(ERIRT_E_CUDA, "get_data: %s", cudaGetErrorString(e));
  return 0;
}

extern "C" int erirt_set_data_device(erirt_handle* h, const double* dYc, int64_t ldY, const double* dTc, int64_t ldT,
                                     const double* dXc, int64_t ldX) {
  return ingest<double>(h, dYc, ldY, dTc, ldT, dXc, ldX, true);
}
extern "C" int erirt_set_data(erirt_handle* h, const double* Y, int64_t ldY, const double* logT, int64_t ldT, const double* X, int64_t ldX) {
  return ingest<double>(h, Y, ldY, logT, ldT, X, ldX, false);
}
extern "C" int erirt_set_data_y8(erirt_handle* h, const uint8_t* Y, int64_t ldY, const double* logT, int64_t ldT, const double* X, int64_t ldX) {
  return ingest<uint8_t>(h, Y, ldY, logT, ldT, X, ldX, false);
}

// all-reduce the ingest constants over shards once, derive mean/std of logT
static int finalize_constants(erirt_handle* h) {
  if (h->consts_final) return 0;
  CU(cudaMemcpyAsync(h->dConsts, h->dConstsLocal, (size_t)h->z.consts * h->nb * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
  if (h->world > 1) {
    if (h->peer_ready) {
      peer_allreduce_kernel<<<1, 512, 0, h->stream>>>(h->dPeerBufs, h->dXseq, h->world, h->rank, h->xstride, h->dConsts, h->c_count, h->dStatus);
      CU(cudaGetLastError());
    } else if (h->comm) {
      NC(nccl::all_reduce(h->dConsts, h->dConsts, (size_t)h->c_count, nccl::kFloat64, nccl::kSum, h->comm, h->stream));
    } else {
      return fail(ERIRT_E_STATE, "sharded chain without a communicator: call erirt_peer_attach (or erirt_comm_init with an NCCL id) first");
    }
  }
  std::vector<double> c((size_t)h->z.consts * h->nb);
  CU(cudaMemcpyAsync(c.data(), h->dConsts, c.size() * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  std::vector<double> derived;  // 4 per replica
  for (int r = 0; r < h->nb; ++r) {
    const double* cr = c.data() + r * h->z.consts;
    double s1 = 0, s2 = 0;
    for (int j = 0; j < h->cfg.n_item; ++j) { s1 += cr[h->c_T1 + j]; s2 += cr[h->c_T2 + j]; }
    const double n = (double)h->cfg.n_subj_total * h->cfg.n_item;
    double d[4] = {0, 1, 0, 0};
    if (h->cfg.model != ERIRT_MLIRT) {
      d[0] = s1 / n;                                   // mean(Data.logT)   Draw.pl.jl:215
      d[1] = std::sqrt((s2 - s1 * s1 / n) / (n - 1.0));  // std(Data.logT)
    }
    derived.insert(derived.end(), d, d + 4);
  }
  CU(cudaMemcpyAsync(h->dDerived, derived.data(), derived.size() * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  h->consts_final = true;
  return 0;
}

// ------------------------------------------------------------------------------------------------
// state
// ------------------------------------------------------------------------------------------------
// Device storage [n_subj][Jp] of R of a person field, seen by the caller as column-major [n_subj][J] float64: the person vectors
// theta / zeta / nu are J = Jp = 1; omega and the N x J nu of CrossQr are the tiles.  CrossQr's nu is drawn before it is read (no
// initial value is needed); setting it serves erirt_loglik_current (D-hat at Post.mean, GibbsRtIrtCross.pl.jl:344-352)
struct PersonField { void* p; int J, Jp; };
static bool person_field(const erirt_handle* h, int field, PersonField* f) {
  const int J = h->cfg.n_item, Jp = h->L.Jp;
  switch (field) {
    case ERIRT_THETA: *f = {h->dTheta, 1, 1}; return true;
    case ERIRT_ZETA: *f = {h->dZeta, 1, 1}; return true;
    case ERIRT_NU: *f = h->cfg.model == ERIRT_RTIRT_CROSSQR ? PersonField{h->dNuCell, J, Jp} : PersonField{h->dNu, 1, 1}; return true;
    case ERIRT_OMEGA: *f = {h->dOmega, J, Jp}; return true;
  }
  return false;
}
static int param_slot(erirt_handle* h, int field, int* off, int* len) {
  const Layout& L = h->L;
  const int J = h->cfg.n_item;
  switch (field) {
    case ERIRT_A: *off = L.p_a; *len = J; return 0;
    case ERIRT_B: *off = L.p_b; *len = J; return 0;
    case ERIRT_LAMBDA: *off = L.p_lambda; *len = J; return 0;
    case ERIRT_SIGMA2: *off = L.p_sigma2; *len = J; return 0;
    case ERIRT_RHO: *off = L.p_rho; *len = J; return 0;
    case ERIRT_BETA: *off = L.p_beta; *len = beta_len(h->cfg.model, h->cfg.n_feat); return 0;
    case ERIRT_SIGMA_P: *off = L.p_Sigma; *len = 4; return 0;
  }
  return -1;
}

// A batch stacks replicas: a person field has n_batch * n_subj rows (column-major, replica r in rows [r n_subj, (r+1) n_subj)), a
// parameter n_batch consecutive blocks of its standalone length.
extern "C" int erirt_set_state(erirt_handle* h, int32_t field, const double* v, int64_t n) {
  if (!h || !v) return fail(ERIRT_E_ARG, "null argument");
  CU(cudaSetDevice(h->cfg.device));
  PersonField pf;
  int off, len;
  const int64_t ns = h->cfg.n_subj;
  if (person_field(h, field, &pf)) {
    const int64_t want = ns * pf.J * h->nb;
    if (n != want) return fail(ERIRT_E_ARG, "field %d expects %lld values, got %lld", field, (long long)want, (long long)n);
    const int64_t stride = pf.J == 1 ? h->z.vec : h->z.cells;  // one replica's copy of the device field
    double* tmp;
    CU(cudaMallocAsync((void**)&tmp, ns * pf.J * sizeof(double), h->stream));
    for (int r = 0; r < h->nb; ++r) {
      cudaMemcpy2DAsync(tmp, ns * sizeof(double), v + r * ns, ns * h->nb * sizeof(double), ns * sizeof(double), pf.J, cudaMemcpyHostToDevice,
                        h->stream);
      with_real(h, [&](auto rr) {
        using R = decltype(rr);
        colmajor_to_tile_kernel<R><<<1024, 256, 0, h->stream>>>(tmp, ns, pf.J, pf.Jp, (R*)pf.p + r * stride);
      });
    }
    cudaFreeAsync(tmp, h->stream);
    cudaError_t e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) return fail(ERIRT_E_CUDA, "set_state: %s", cudaGetErrorString(e));
    return 0;
  }
  if (param_slot(h, field, &off, &len) == 0) {
    if (n != (int64_t)len * h->nb) return fail(ERIRT_E_ARG, "field %d expects %lld values, got %lld", field, (long long)len * h->nb, (long long)n);
    for (int r = 0; r < h->nb && len > 0; ++r)
      CU(cudaMemcpy(h->dParams + r * h->z.params + off, v + (int64_t)r * len, len * sizeof(double), cudaMemcpyHostToDevice));
    return 0;
  }
  return fail(ERIRT_E_ARG, "unknown field %d", field);
}

extern "C" int erirt_get_state(erirt_handle* h, int32_t field, double* out, int64_t n) {
  if (!h || !out) return fail(ERIRT_E_ARG, "null argument");
  CU(cudaSetDevice(h->cfg.device));
  PersonField pf;
  int off, len;
  const int64_t ns = h->cfg.n_subj;
  if (person_field(h, field, &pf)) {
    const int64_t want = ns * pf.J * h->nb;
    if (n != want) return fail(ERIRT_E_ARG, "field %d expects %lld values, got %lld", field, (long long)want, (long long)n);
    const int64_t stride = pf.J == 1 ? h->z.vec : h->z.cells;
    double* tmp;
    CU(cudaMallocAsync((void**)&tmp, ns * pf.J * sizeof(double), h->stream));
    for (int r = 0; r < h->nb; ++r) {
      with_real(h, [&](auto rr) {
        using R = decltype(rr);
        tile_to_colmajor_kernel<R><<<1024, 256, 0, h->stream>>>((const R*)pf.p + r * stride, ns, pf.J, pf.Jp, tmp);
      });
      cudaMemcpy2DAsync(out + r * ns, ns * h->nb * sizeof(double), tmp, ns * sizeof(double), ns * sizeof(double), pf.J, cudaMemcpyDeviceToHost,
                        h->stream);
    }
    cudaFreeAsync(tmp, h->stream);
    cudaError_t e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) return fail(ERIRT_E_CUDA, "get_state: %s", cudaGetErrorString(e));
    return 0;
  }
  if (param_slot(h, field, &off, &len) == 0) {
    if (n != (int64_t)len * h->nb) return fail(ERIRT_E_ARG, "field %d expects %lld values, got %lld", field, (long long)len * h->nb, (long long)n);
    CU(cudaStreamSynchronize(h->stream));
    for (int r = 0; r < h->nb && len > 0; ++r)
      CU(cudaMemcpy(out + (int64_t)r * len, h->dParams + r * h->z.params + off, len * sizeof(double), cudaMemcpyDeviceToHost));
    return 0;
  }
  return fail(ERIRT_E_ARG, "unknown field %d", field);
}

// ------------------------------------------------------------------------------------------------
// sampling
// ------------------------------------------------------------------------------------------------
template <typename R>
static PersonArgs<R> make_person_args(erirt_handle* h, int stage) {
  PersonArgs<R> A{};
  A.stage = stage;
  A.Y = h->dY;
  A.logT = (const R*)h->dLogT;
  A.omega = (R*)h->dOmega;
  A.nu_cell = (R*)h->dNuCell;
  A.theta = (R*)h->dTheta;
  A.zeta = (R*)h->dZeta;
  A.nu = (R*)h->dNu;
  A.X = (const R*)h->dX;
  A.mom = h->dMom;
  A.ptrace = (R*)h->dPtrace;
  A.nu_mom = h->dNuMom;
  A.params = h->dParams;
  A.stats = h->dStats;
  A.sweep_ctr = h->dSweep;
  A.tile_ctr = h->dTileCtr;
  A.status = h->dStatus;
  A.n_local = h->cfg.n_subj;
  A.n_pad = h->n_pad;
  A.person_offset = (uint32_t)h->cfg.subj_offset;
  A.S = runs_fast_kernel(h, stage) ? h->S : h->S_gen;
  A.n_tiles = (int)(h->n_pad / A.S.P);
  A.L = h->L;
  A.model = h->cfg.model;
  A.n_chain = h->cfg.n_chain;
  A.n_burnin = h->cfg.n_burnin;
  A.k1 = h->k1;
  A.k2 = h->k2;
  A.key = h->key;
  A.sched = make_sched(h->key);
  return A;
}

static GlobalArgs make_global_args(erirt_handle* h, int stage) {
  GlobalArgs A{};
  A.stage = stage;
  A.params = h->dParams;
  A.stats = h->dStats;
  A.stats_prev = h->dStatsPrev;
  {
    // The rehearsal pays when the person launch in front of this kernel is long enough to hide it (about 20 us) and big enough to
    // have flushed the instruction caches: more than one tile per CTA.  Behind a one-round launch (the small problems) it would only
    // delay the real pass.
    const bool fast = runs_fast_kernel(h, stage);
    // A replica batch does not rehearse (its CTAs would fetch the same code in parallel).
    const int64_t tiles = h->n_pad / (fast ? h->S.P : h->S_gen.P);
    A.rehearse = h->nb == 1 && tiles > (fast ? h->grid : h->grid_gen) ? 1 : 0;
  }
  A.tile_ctr = h->dTileCtr;
  A.sweep_ctr = h->dSweep;
  A.T1 = h->dConsts + h->c_T1;
  A.T2 = h->dConsts + h->c_T2;
  A.K0 = h->dConsts + h->c_K0;
  A.XtX = h->dConsts + h->c_XtX;
  A.consts = h->dDerived;
  A.tr_items_ra = h->dTrRa;
  A.tr_items_rt = h->dTrRt;
  A.tr_qr = h->dTrQr;
  A.tr_ll = h->dTrLl;
  A.status = h->dStatus;
  A.ll_out = h->dLlOut;
  A.n_total = h->cfg.n_subj_total;
  A.cap = h->cap;
  A.qw = h->qw;
  A.L = h->L;
  A.model = h->cfg.model;
  A.intercept = h->cfg.intercept;
  A.onepl = h->cfg.itemtype_1pl;
  A.cov2one = h->cfg.cov2one;
  A.compat = h->cfg.compat;
  A.kz_from_stats = runs_fast_kernel(h, stage) ? 1 : 0;
  A.k1 = h->k1;
  A.k2 = h->k2;
  A.key = h->key;
  A.peer_bufs = h->peer_ready ? h->dPeerBufs : nullptr;
  A.xseq = h->dXseq;
  A.world = h->world;
  A.rank = h->rank;
  A.xstride = h->xstride;
  return A;
}

// Every kernel of the sweep chain is launched with programmatic stream serialization (griddep_wait / griddep_launch in the
// kernels, layout.cuh): a kernel's CTAs may become resident, and run what does not depend on its predecessor, while the predecessor
// is still running.
static cudaError_t launch_chain_kernel(const void* kfn, dim3 grid, dim3 block, void** args, size_t smem, cudaStream_t stream) {
  cudaLaunchConfig_t lc{};
  lc.gridDim = grid;
  lc.blockDim = block;
  lc.dynamicSmemBytes = smem;
  lc.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  lc.attrs = at;
  lc.numAttrs = 1;
  return cudaLaunchKernelExC(&lc, kfn, args);
}

// A replica batch launches the BATCH instantiations of the kernels (layout.cuh BatchArgs): the person grid gains a replica dimension,
// the global kernel one CTA per replica.
static int launch_person(erirt_handle* h, int stage) {
  const void* kfn = person_kernel_for(h, stage);
  return with_real(h, [&](auto r) -> int {
    PersonArgs<decltype(r)> A = make_person_args<decltype(r)>(h, stage);
    BatchArgs<PersonArgs<decltype(r)>> B{A, h->z, h->cfg.seed, h->cfg.chain};  // A: replica 0
    void* args[] = {h->nb > 1 ? (void*)&B : (void*)&A};
    CU(launch_chain_kernel(kfn, dim3(stage == 0 ? h->grid : h->grid_gen, h->nb), dim3(CTA_THREADS), args, A.S.total, h->stream));
    return 0;
  });
}
static int launch_global(erirt_handle* h, int stage) {
  if (h->world > 1 && !h->peer_ready && !h->comm)
    return fail(ERIRT_E_STATE, "sharded chain (world %d) without an exchange: the peer buffers were detached and there is no NCCL communicator", h->world);
  if (h->comm && !h->peer_ready)  // fallback: the exchange is otherwise fused into the kernel below
    NC(nccl::all_reduce(h->dStats, h->dStats, (size_t)h->L.s_count, nccl::kFloat64, nccl::kSum, h->comm, h->stream));
  GlobalArgs G = make_global_args(h, stage);
  BatchArgs<GlobalArgs> B{G, h->z, h->cfg.seed, h->cfg.chain};
  const size_t gsm = (size_t)(h->L.s_count + 2 + (h->L.F + 1) * (h->L.F + 1) + 5 * h->L.Jp) * sizeof(double);  // staged statistics, X'X, raw variates
  void* args[] = {h->nb > 1 ? (void*)&B : (void*)&G};
  CU(launch_chain_kernel(global_kernel_for(h), dim3(h->nb), dim3(G_THREADS), args, gsm, h->stream));
  return 0;
}

// one sweep on h->stream:  P(k) [allreduce] G(k+1);  Cross family: K_a(k) [ar] G_a(k) K_b(k) [ar] G_b(k+1)
static int enqueue_step(erirt_handle* h, bool prologue) {
  const bool cross = h->cfg.model == ERIRT_RTIRT_CROSS || h->cfg.model == ERIRT_RTIRT_CROSSQR;
  const bool timed = h->cfg.time_kernels && h->kev_used + 2 <= h->kev.size();
  int rc;
  if (cross && !prologue) {
    if ((rc = launch_person(h, 1))) return rc;
    if ((rc = launch_global(h, 1))) return rc;
  }
  if (timed) CU(cudaEventRecord(h->kev[h->kev_used], h->stream));
  if ((rc = launch_person(h, cross ? 2 : 0))) return rc;
  if (timed) {
    CU(cudaEventRecord(h->kev[h->kev_used + 1], h->stream));
    h->kev_used += 2;
  }
  return launch_global(h, cross ? 2 : 0);
}

constexpr int GRAPH_SWEEPS = 16;  // sweeps of the long CUDA graph of erirt_sample

extern "C" int erirt_sample(erirt_handle* h, int64_t n_sweeps) {
  if (!h) return fail(ERIRT_E_ARG, "null handle");
  if (!h->data_set) return fail(ERIRT_E_STATE, "erirt_set_data has not been called");
  if (n_sweeps < 0) return fail(ERIRT_E_ARG, "n_sweeps < 0");
  if (h->sweeps_done + n_sweeps > h->cap) return fail(ERIRT_E_ARG, "trace capacity exceeded: %lld + %lld > n_iter*n_chain = %d",
                                                      (long long)h->sweeps_done, (long long)n_sweeps, h->cap);
  CU(cudaSetDevice(h->cfg.device));
  int rc = finalize_constants(h);
  if (rc) return rc;
  if (!h->prologue_done) {
    CU(cudaMemsetAsync(h->dSweep, 0, h->nb * sizeof(uint32_t), h->stream));
    CU(cudaMemsetAsync(h->dStats, 0, h->z.stats * h->nb * sizeof(double), h->stream));
    rc = enqueue_step(h, true);  // P(0), G(1)
    if (rc) return rc;
    h->prologue_done = true;
  }
  h->kev_used = 0;
  if (h->cfg.time_kernels) {
    const size_t want = (size_t)std::min<int64_t>(n_sweeps, 4096) * 2;
    while (h->kev.size() < want) {
      cudaEvent_t e;
      CU(cudaEventCreate(&e));
      h->kev.push_back(e);
    }
  }
  const bool graphs = h->cfg.use_graph && !h->cfg.time_kernels && n_sweeps > 0;
  // The sweeps are replayed from two CUDA graphs: one of GRAPH_SWEEPS sweeps and one of a single sweep for the remainder.  Inside a
  // graph the kernels overlap their neighbours through the programmatic-dependent-launch edges; a graph boundary serialises, so the
  // long graph also keeps the launch-bound small problems busy.  Both are captured on the first call, before the timed region of this
  // call starts.
  if (graphs) {
    auto capture = [&](int sweeps, cudaGraphExec_t* exec) -> int {
      cudaGraph_t graph;
      CU(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
      int r = 0;
      for (int t = 0; t < sweeps && !r; ++t) r = enqueue_step(h, false);
      cudaError_t e = cudaStreamEndCapture(h->stream, &graph);
      if (r) return r;
      if (e != cudaSuccess) return fail(ERIRT_E_CUDA, "graph capture failed: %s", cudaGetErrorString(e));
      e = cudaGraphInstantiate(exec, graph, 0);
      cudaGraphDestroy(graph);
      if (e != cudaSuccess) return fail(ERIRT_E_CUDA, "graph instantiate failed: %s", cudaGetErrorString(e));
      return 0;
    };
    if (!h->graph_exec && (rc = capture(1, &h->graph_exec))) return rc;
    if (!h->graph_multi && (rc = capture(GRAPH_SWEEPS, &h->graph_multi))) return rc;
  }
  CU(cudaEventRecord(h->ev0, h->stream));
  if (graphs) {
    int64_t left = n_sweeps;
    for (; left >= GRAPH_SWEEPS; left -= GRAPH_SWEEPS) CU(cudaGraphLaunch(h->graph_multi, h->stream));
    for (; left > 0; --left) CU(cudaGraphLaunch(h->graph_exec, h->stream));
  } else {
    for (int64_t t = 0; t < n_sweeps; ++t) {
      rc = enqueue_step(h, false);
      if (rc) return rc;
    }
  }
  CU(cudaEventRecord(h->ev1, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  float ms = 0.f;
  CU(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
  h->last_ms = ms;
  h->person_ms = 0.0;
  if (h->kev_used) {
    double tot = 0.0;
    for (size_t t = 0; t + 1 < h->kev_used; t += 2) {
      float kms = 0.f;
      CU(cudaEventElapsedTime(&kms, h->kev[t], h->kev[t + 1]));
      tot += kms;
    }
    h->person_ms = tot / (double)(h->kev_used / 2);
  }
  h->sweeps_done += n_sweeps;
  std::vector<int> status(h->nb);  // sticky, one per replica
  CU(cudaMemcpy(status.data(), h->dStatus, h->nb * sizeof(int), cudaMemcpyDeviceToHost));
  if (status[0] <= -1000) return fail(ERIRT_E_NCCL, "peer exchange timed out waiting for rank %d (a GPU of the sharded chain is gone); the chain is unusable", -1000 - status[0]);
  for (int r = 0; r < h->nb; ++r) {
    if (status[r] == 0) continue;
    if (h->nb == 1) return fail(ERIRT_E_NUMERIC, "a posterior covariance was not positive definite at sweep %d (PosDefException in the reference)", status[r]);
    return fail(ERIRT_E_NUMERIC, "replica %d: a posterior covariance was not positive definite at sweep %d (PosDefException in the reference)", r, status[r]);
  }
  return 0;
}

// ------------------------------------------------------------------------------------------------
// results
// ------------------------------------------------------------------------------------------------
static int64_t full_width(const erirt_handle* h, int which) {
  const int64_t N = h->cfg.n_subj, J = h->cfg.n_item;
  switch (which) {
    case ERIRT_TRACE_RA: return N + 2 * J;
    case ERIRT_TRACE_RT: return h->cfg.model == ERIRT_MLIRT ? 0 : N + 2 * J;
    case ERIRT_TRACE_QR: return h->qw + (h->cfg.model == ERIRT_RTIRT_LATENTQR ? N : 0);
    case ERIRT_TRACE_LOGLIKE: return 1;
  }
  return -1;
}
extern "C" int64_t erirt_trace_width(erirt_handle* h, int32_t which) { return h ? full_width(h, which) : -1; }

// Post.<which>[:, first_col + c0 .. first_col + c0 + nc, l] in Julia's layout (iteration fastest), assembled on the device:
// dst[m + n_iter * c];  sweep s = m * n_chain + l;  NaN for sweeps not yet run.  Small (item / structural) columns come from the
// sweep-major trace [s][small_w], person columns from the person trace [s][3][n_pad].
template <typename R>
__global__ void trace_gather_kernel(double* __restrict__ dst, int64_t n_iter, int64_t nc, int64_t col0, int64_t l, int64_t n_chain, int64_t done,
                                    const double* __restrict__ small, int64_t small0, int64_t small_w,
                                    const R* __restrict__ ptrace, int pfield, int64_t pcol0, int64_t n_subj, int64_t n_pad) {
  const int64_t total = n_iter * nc;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t m = t % n_iter, col = col0 + t / n_iter, s = m * n_chain + l;
    double v = __longlong_as_double(0x7ff8000000000000LL);
    if (s < done) {
      if (col >= small0 && col < small0 + small_w) v = small[s * small_w + (col - small0)];
      else if (ptrace && col >= pcol0 && col < pcol0 + n_subj) v = (double)ptrace[(s * 3 + pfield) * n_pad + (col - pcol0)];
    }
    dst[t] = v;
  }
}

// Where the columns of trace `which` come from: columns [small0, small0 + small_w) from the sweep-major trace small [s][small_w],
// columns [pcol0, pcol0 + pn) from field pfield of the person trace (pn = 0: the trace has no person columns).
struct TraceSource {
  const double* small;
  int64_t small0, small_w;
  int64_t small_stride;  // replica batch: length of one replica's copy of `small`
  int pfield;
  int64_t pcol0, pn;
  bool person_cols;  // [first_col, first_col + n_cols) includes person columns
};
// Checks [first_col, first_col + n_cols) against the trace's width and resolves `which`.  Whether person columns may be read without
// a person trace is each caller's rule: erirt_get_trace refuses them only once a sweep has run (before that every value it returns
// is NaN), erirt_trace_ess_rhat refuses them always.
static int trace_source(const erirt_handle* h, int which, int64_t first_col, int64_t n_cols, TraceSource* src) {
  const int64_t W = full_width(h, which);
  if (W <= 0) return fail(ERIRT_E_ARG, "trace %d does not exist for this model", which);
  if (first_col < 0 || n_cols < 0 || first_col + n_cols > W) return fail(ERIRT_E_ARG, "columns [%lld,%lld) outside [0,%lld)", (long long)first_col, (long long)(first_col + n_cols), (long long)W);
  const int64_t N = h->cfg.n_subj, J = h->cfg.n_item;
  // column ranges: person block [0,N) for ra/rt, trailing nu block for LatentQr qr
  TraceSource s{nullptr, 0, 0, 0, 0, -1, 0, false};
  if (which == ERIRT_TRACE_RA) { s.small = h->dTrRa; s.small0 = N; s.small_w = 2 * J; s.small_stride = h->z.tr_items; s.pfield = 0; s.pcol0 = 0; s.pn = N; }
  else if (which == ERIRT_TRACE_RT) { s.small = h->dTrRt; s.small0 = N; s.small_w = 2 * J; s.small_stride = h->z.tr_items; s.pfield = 1; s.pcol0 = 0; s.pn = N; }
  else if (which == ERIRT_TRACE_QR) {
    s.small = h->dTrQr; s.small_w = h->qw; s.small_stride = h->z.tr_qr;
    if (h->cfg.model == ERIRT_RTIRT_LATENTQR) { s.pfield = 2; s.pcol0 = h->qw; s.pn = N; }
  } else { s.small = h->dTrLl; s.small_w = 1; s.small_stride = h->z.tr_ll; }
  s.person_cols = first_col < s.pcol0 + s.pn && first_col + n_cols > s.pcol0;
  *src = s;
  return 0;
}

// Columns [col0, col0 + nc) of chain l of replica rep into dst [nc][n_iter] (trace_gather_kernel)
static void gather_trace(erirt_handle* h, const TraceSource& s, int rep, double* dst, int64_t col0, int64_t nc, int64_t l) {
  const int64_t nIter = h->cfg.n_iter;
  const int grid = (int)std::min<int64_t>((nIter * nc + 255) / 256, (int64_t)h->sm_count * 16);
  const double* small = s.small + rep * s.small_stride;
  with_real(h, [&](auto r) {
    using R = decltype(r);
    trace_gather_kernel<R><<<grid, 256, 0, h->stream>>>(dst, nIter, nc, col0, l, h->cfg.n_chain, h->sweeps_done, small, s.small0, s.small_w,
                                                         (const R*)h->dPtrace, s.pfield, s.pcol0, s.pn, h->n_pad);
  });
}

extern "C" int erirt_get_trace(erirt_handle* h, int32_t which, int64_t first_col, int64_t n_cols, double* out) {
  if (!h || !out) return fail(ERIRT_E_ARG, "null argument");
  TraceSource src;
  if (int rc = trace_source(h, which, first_col, n_cols, &src)) return rc;
  CU(cudaSetDevice(h->cfg.device));
  const int64_t nIter = h->cfg.n_iter, nChain = h->cfg.n_chain;
  if (src.person_cols && h->sweeps_done > 0 && !h->dPtrace)
    return fail(ERIRT_E_STATE, "person columns requested but person_trace = 0 (use erirt_get_moments)");
  if (n_cols == 0) return 0;
  // assembled on the device in column chunks of <= 64 MB per chain (Julia's layout makes such a chunk contiguous in `out`), one D2H copy each
  const int64_t chunk_cols = std::max<int64_t>(1, std::min<int64_t>(n_cols, ((int64_t)64 << 20) / (nIter * (int64_t)sizeof(double))));
  double* tmp = nullptr;
  CU(cudaMallocAsync((void**)&tmp, (size_t)nIter * chunk_cols * sizeof(double), h->stream));
  cudaError_t e = cudaSuccess;
  // a batch appends the replica as the last axis: out[m + n_iter * (c + n_cols * (l + n_chain * r))]
  for (int r = 0; r < h->nb && e == cudaSuccess; ++r)
    for (int64_t l = 0; l < nChain && e == cudaSuccess; ++l)
      for (int64_t c0 = 0; c0 < n_cols && e == cudaSuccess; c0 += chunk_cols) {
        const int64_t nc = std::min(chunk_cols, n_cols - c0);
        gather_trace(h, src, r, tmp, first_col + c0, nc, l);
        e = cudaMemcpyAsync(out + nIter * (c0 + n_cols * (l + nChain * r)), tmp, (size_t)nIter * nc * sizeof(double), cudaMemcpyDeviceToHost,
                            h->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);  // tmp is reused by the next chunk
      }
  cudaFreeAsync(tmp, h->stream);
  if (e != cudaSuccess) return fail(ERIRT_E_CUDA, "get_trace: %s", cudaGetErrorString(e));
  return 0;
}

// ---- convergence diagnostics on the device (diagnostics.cuh) ----
// dx: device block [n_chain][n_cols][n_iter]; results copied to the host arrays ess / rhat (n_cols each)
static int run_ess_rhat(const double* dx, int64_t n_iter, int64_t n_cols, int64_t n_chain, int64_t skip, int64_t n_used, cudaStream_t st,
                        double* ess, double* rhat) {
  if (n_cols == 0) return 0;
  const int64_t n = n_used / 2, N = 2 * n_chain * n;
  int64_t npad = 2;
  while (npad < N) npad <<= 1;
  DiagArgs A{};
  A.x = dx; A.n_iter = n_iter; A.n_cols = n_cols; A.skip = skip; A.n_used = n_used; A.n_chain = (int)n_chain; A.npad = npad;
  const size_t smem = (size_t)npad * (sizeof(double) + sizeof(uint32_t));
  A.use_smem = smem <= (size_t)200 * 1024 ? 1 : 0;
  double* scratch = nullptr;
  const size_t zb = align_up((size_t)n_cols * (size_t)std::max<int64_t>(N, 1) * sizeof(double), 256);
  const size_t kb = A.use_smem ? 0 : align_up((size_t)n_cols * npad * sizeof(double), 256);
  const size_t ib = A.use_smem ? 0 : align_up((size_t)n_cols * npad * sizeof(uint32_t), 256);
  const size_t ob = align_up((size_t)2 * n_cols * sizeof(double), 256);
  CU(cudaMallocAsync((void**)&scratch, zb + kb + ib + ob, st));
  unsigned char* base = reinterpret_cast<unsigned char*>(scratch);
  A.z = scratch;
  A.keys = reinterpret_cast<double*>(base + zb);
  A.idx = reinterpret_cast<uint32_t*>(base + zb + kb);
  A.ess = reinterpret_cast<double*>(base + zb + kb + ib);
  A.rhat = A.ess + n_cols;
  cudaError_t e = cudaSuccess;
  if (A.use_smem) e = cudaFuncSetAttribute((const void*)ess_rhat_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e == cudaSuccess) {
    ess_rhat_kernel<<<(unsigned)n_cols, DIAG_THREADS, A.use_smem ? smem : 0, st>>>(A);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaMemcpyAsync(ess, A.ess, (size_t)n_cols * sizeof(double), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(rhat, A.rhat, (size_t)n_cols * sizeof(double), cudaMemcpyDeviceToHost, st);
  cudaFreeAsync(scratch, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return fail(ERIRT_E_CUDA, "ess_rhat: %s", cudaGetErrorString(e));
  return 0;
}

extern "C" int erirt_ess_rhat(const double* x, int64_t n_iter, int64_t n_cols, int64_t n_chain, int64_t skip, int32_t device,
                              double* ess, double* rhat) {
  if (!x || !ess || !rhat) return fail(ERIRT_E_ARG, "null argument");
  if (n_iter < 1 || n_cols < 0 || n_chain < 1 || n_chain > 32 || skip < 0 || skip > n_iter) return fail(ERIRT_E_ARG, "ess_rhat: bad dimensions (1 <= n_chain <= 32, 0 <= skip <= n_iter)");
  if (n_cols > 2147483647LL) return fail(ERIRT_E_ARG, "ess_rhat: too many columns");
  if (int prc = pick_device(device)) return prc;
  double* dx = nullptr;
  const size_t bytes = (size_t)n_iter * n_cols * n_chain * sizeof(double);
  if (bytes == 0) return 0;
  CU(cudaMallocAsync((void**)&dx, bytes, 0));
  cudaError_t e = cudaMemcpyAsync(dx, x, bytes, cudaMemcpyHostToDevice, 0);
  int rc = 0;
  if (e == cudaSuccess) rc = run_ess_rhat(dx, n_iter, n_cols, n_chain, skip, n_iter - skip, 0, ess, rhat);
  cudaFreeAsync(dx, 0);
  cudaStreamSynchronize(0);
  if (e != cudaSuccess) return fail(ERIRT_E_CUDA, "ess_rhat: %s", cudaGetErrorString(e));
  return rc;
}

extern "C" int erirt_trace_ess_rhat(erirt_handle* h, int32_t which, int64_t first_col, int64_t n_cols, int64_t skip, double* ess, double* rhat) {
  if (!h || !ess || !rhat) return fail(ERIRT_E_ARG, "null argument");
  TraceSource src;
  if (int rc = trace_source(h, which, first_col, n_cols, &src)) return rc;
  CU(cudaSetDevice(h->cfg.device));
  const int64_t nIter = h->cfg.n_iter, nChain = h->cfg.n_chain;
  const int64_t done_iter = h->sweeps_done / nChain;  // complete iterations (every chain has drawn)
  if (nChain > 32) return fail(ERIRT_E_ARG, "ess_rhat: at most 32 chains");
  if (skip < 0 || skip > done_iter) return fail(ERIRT_E_ARG, "skip %lld outside [0, %lld] completed iterations", (long long)skip, (long long)done_iter);
  if (src.person_cols && !h->dPtrace) return fail(ERIRT_E_STATE, "person columns requested but person_trace = 0");
  if (n_cols == 0) return 0;
  // the columns are gathered into [chain][column][iteration] in chunks of <= 256 MB and never leave the device
  const int64_t chunk_cols = std::max<int64_t>(1, std::min<int64_t>(n_cols, ((int64_t)256 << 20) / (nIter * nChain * (int64_t)sizeof(double))));
  double* tmp = nullptr;
  CU(cudaMallocAsync((void**)&tmp, (size_t)nIter * chunk_cols * nChain * sizeof(double), h->stream));
  int rc = 0;
  // a batch returns n_batch * n_cols results, replica-major
  for (int r = 0; r < h->nb && rc == 0; ++r)
    for (int64_t c0 = 0; c0 < n_cols && rc == 0; c0 += chunk_cols) {
      const int64_t nc = std::min(chunk_cols, n_cols - c0);
      for (int64_t l = 0; l < nChain; ++l) gather_trace(h, src, r, tmp + nIter * nc * l, first_col + c0, nc, l);
      rc = run_ess_rhat(tmp, nIter, nc, nChain, skip, done_iter - skip, h->stream, ess + r * n_cols + c0, rhat + r * n_cols + c0);
    }
  cudaFreeAsync(tmp, h->stream);
  cudaStreamSynchronize(h->stream);
  return rc;
}

extern "C" int erirt_get_moments(erirt_handle* h, int32_t field, double* mean, double* sd, int64_t n) {
  if (!h || !mean) return fail(ERIRT_E_ARG, "null argument");
  int slot = field == ERIRT_THETA ? 0 : (field == ERIRT_ZETA ? 1 : (field == ERIRT_NU ? 2 : -1));
  if (slot < 0) return fail(ERIRT_E_ARG, "moments exist for THETA, ZETA and NU only");
  const bool nu_cell = field == ERIRT_NU && h->cfg.model == ERIRT_RTIRT_CROSSQR;
  if (nu_cell && !h->dNuMom) return fail(ERIRT_E_STATE, "the running moments of the N x J weights of CrossQr need erirt_config.nu_cell_moments = 1");
  PersonField pf;
  person_field(h, field, &pf);
  if (n != h->cfg.n_subj * pf.J * h->nb)
    return fail(ERIRT_E_ARG, nu_cell ? "expects n_subj * n_item values" : (h->nb > 1 ? "expects n_batch * n_subj values" : "expects n_subj values"));
  CU(cudaSetDevice(h->cfg.device));
  CU(cudaStreamSynchronize(h->stream));
  const int64_t nChain = h->cfg.n_chain;
  const int64_t first = (int64_t)h->cfg.n_burnin * nChain;  // sweeps with m > n_burnin
  const int64_t cnt = h->sweeps_done > first ? h->sweeps_done - first : 0;
  // mean and SD are finished on the device and copied straight into the caller's buffers (pinned buffers make this a plain DMA)
  double* tmp = nullptr;
  CU(cudaMallocAsync((void**)&tmp, (size_t)2 * n * sizeof(double), h->stream));
  const int64_t nr = n / h->nb;  // values of one replica
  for (int r = 0; r < h->nb; ++r) {
    // running sum and sum of squares of the field, laid out like it: [2][n_pad][Jp]
    const double* s1 = nu_cell ? h->dNuMom : h->dMom + r * h->z.mom + (size_t)(2 * slot) * h->n_pad;
    tile_moments_kernel<<<1024, 256, 0, h->stream>>>(s1, s1 + (size_t)h->n_pad * pf.Jp, h->cfg.n_subj, pf.J, pf.Jp, (double)cnt, tmp + r * nr, tmp + n + r * nr);
  }
  cudaError_t e = cudaMemcpyAsync(mean, tmp, n * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess && sd) e = cudaMemcpyAsync(sd, tmp + n, n * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
  cudaFreeAsync(tmp, h->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  if (e != cudaSuccess) return fail(ERIRT_E_CUDA, "get_moments: %s", cudaGetErrorString(e));
  return 0;
}

extern "C" int erirt_loglik_current(erirt_handle* h, double* out) {
  if (!h || !out) return fail(ERIRT_E_ARG, "null argument");
  if (!h->data_set) return fail(ERIRT_E_STATE, "erirt_set_data has not been called");
  CU(cudaSetDevice(h->cfg.device));
  int rc = finalize_constants(h);
  if (rc) return rc;
  if (!h->prologue_done) CU(cudaMemsetAsync(h->dStats, 0, h->z.stats * h->nb * sizeof(double), h->stream));
  if ((rc = launch_person(h, 3))) return rc;
  if ((rc = launch_global(h, 3))) return rc;
  CU(cudaMemcpyAsync(out, h->dLlOut, h->nb * sizeof(double), cudaMemcpyDeviceToHost, h->stream));  // one per replica
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

extern "C" int64_t erirt_debug_check_guards(erirt_handle* h) {
  if (!h) return fail(ERIRT_E_ARG, "null handle");
  if (h->guard_offs.empty()) return -1;  // the handle was created without ERIRT_GUARDS=1
  cudaSetDevice(h->cfg.device);
  if (cudaStreamSynchronize(h->stream) != cudaSuccess) return fail(ERIRT_E_CUDA, "stream synchronize failed");
  int64_t bad = 0;
  std::vector<unsigned char> buf(256);
  for (size_t off : h->guard_offs) {
    if (cudaMemcpy(buf.data(), h->arena + off, 256, cudaMemcpyDeviceToHost) != cudaSuccess) return fail(ERIRT_E_CUDA, "guard read-back failed");
    for (unsigned char c : buf) bad += c != 0xA5;
  }
  return bad;
}

extern "C" int erirt_get_stats(erirt_handle* h, erirt_stats* out) {
  if (!h || !out) return fail(ERIRT_E_ARG, "null argument");
  CU(cudaSetDevice(h->cfg.device));
  memset(out, 0, sizeof(*out));
  out->sweeps_done = h->sweeps_done;
  out->last_sample_ms = h->last_ms;
  out->person_kernel_ms = h->person_ms;
  out->launches_per_sweep = (h->cfg.model == ERIRT_RTIRT_CROSS || h->cfg.model == ERIRT_RTIRT_CROSSQR) ? 4 : 2;
  out->sm_count = h->sm_count;
  const int64_t N = h->cfg.n_subj, J = h->cfg.n_item, F = h->cfg.n_feat;
  const int64_t r = (int64_t)h->rsz;
  const bool has_rt = h->cfg.model != ERIRT_MLIRT;
  int64_t per_cell = 1 + 2 * r + (has_rt ? r : 0);
  if (h->cfg.model == ERIRT_RTIRT_CROSS) per_cell = 2 * (1 + 2 * r);  // K_a reads Y, logT, omega; K_b reads Y, logT, writes omega
  if (h->cfg.model == ERIRT_RTIRT_CROSSQR) per_cell = (1 + 3 * r) + (1 + 4 * r);  // K_a: Y, logT, omega, nu; K_b: Y, logT, nu r/w, omega w
  int nv = has_rt ? 2 : 1;
  if (h->cfg.model == ERIRT_RTIRT_LATENTQR) nv = 3;
  out->bytes_per_sweep = (N * J * per_cell + N * r * (2 * nv + F)) * h->nb;  // a batch reports totals over its replicas
  double d[2] = {0, 0};
  CU(cudaStreamSynchronize(h->stream));
  for (int b = 0; b < h->nb; ++b) {
    double db[2];
    CU(cudaMemcpy(db, h->dStats + b * h->z.stats + h->L.s_count, sizeof(db), cudaMemcpyDeviceToHost));
    d[0] += db[0];
    d[1] += db[1];
  }
  out->pg_deferred_frac = d[1] > 0 ? d[0] / d[1] : 0.0;
  return 0;
}

// ------------------------------------------------------------------------------------------------
// checkpoint / resume: every mutable device buffer of the chain (state, auxiliaries, Philox sweep counter, running moments,
// traces) behind a header that pins the configuration it belongs to.  The data (Y, logT, X) is not part of it.
// ------------------------------------------------------------------------------------------------
struct CkHeader {
  char magic[8];
  int32_t abi, model, dtype, n_item, n_feat, n_iter, n_chain, n_burnin, person_trace, prologue_done;
  int64_t n_subj, n_subj_total, subj_offset, sweeps_done, payload_bytes;
  uint64_t seed;
  uint32_t chain, pad;
  // sampler flags: a checkpoint continues the SAME chain only under the same keyword arguments
  int32_t intercept, itemtype_1pl, cov2one, compat, nu_cell_moments, pad2;
  double q_rt;
};
struct CkSeg { void* p; size_t bytes; };
static std::vector<CkSeg> ck_segments(erirt_handle* h) {
  const size_t cells = (size_t)h->n_pad * h->L.Jp, vec = (size_t)h->n_pad * h->rsz, J = (size_t)h->cfg.n_item, cap = (size_t)h->cap;
  std::vector<CkSeg> v;
  v.push_back({h->dOmega, cells * h->rsz});
  if (h->dNuCell) v.push_back({h->dNuCell, cells * h->rsz});
  v.push_back({h->dTheta, vec});
  v.push_back({h->dZeta, vec});
  v.push_back({h->dNu, vec});
  v.push_back({h->dMom, (size_t)6 * h->n_pad * sizeof(double)});
  v.push_back({h->dParams, (size_t)h->L.p_count * sizeof(double)});
  v.push_back({h->dStats, (size_t)(h->L.s_count + 2) * sizeof(double)});
  v.push_back({h->dSweep, sizeof(uint32_t)});
  v.push_back({h->dStatus, sizeof(int)});
  v.push_back({h->dTrRa, cap * 2 * J * sizeof(double)});
  v.push_back({h->dTrRt, cap * 2 * J * sizeof(double)});
  v.push_back({h->dTrQr, cap * (size_t)h->qw * sizeof(double)});
  v.push_back({h->dTrLl, cap * sizeof(double)});
  if (h->dPtrace) v.push_back({h->dPtrace, cap * 3 * vec});
  if (h->dNuMom) v.push_back({h->dNuMom, 2 * cells * sizeof(double)});
  return v;
}
static CkHeader ck_header(erirt_handle* h) {
  CkHeader H{};
  memcpy(H.magic, "ERIRTCK2", 8);
  const erirt_config& c = h->cfg;
  H.abi = ERIRT_ABI_VERSION; H.model = c.model; H.dtype = c.dtype; H.n_item = c.n_item; H.n_feat = c.n_feat; H.n_iter = c.n_iter;
  H.n_chain = c.n_chain; H.n_burnin = c.n_burnin; H.person_trace = c.person_trace ? 1 : 0; H.prologue_done = h->prologue_done ? 1 : 0;
  H.n_subj = c.n_subj; H.n_subj_total = c.n_subj_total; H.subj_offset = c.subj_offset; H.sweeps_done = h->sweeps_done;
  H.seed = c.seed; H.chain = c.chain;
  H.intercept = c.intercept; H.itemtype_1pl = c.itemtype_1pl; H.cov2one = c.cov2one; H.compat = c.compat;
  H.nu_cell_moments = c.nu_cell_moments ? 1 : 0; H.q_rt = c.q_rt;
  for (const CkSeg& sg : ck_segments(h)) H.payload_bytes += (int64_t)sg.bytes;
  return H;
}
// checkpoints, sharding and the peer exchange are per chain: a replica batch refuses them
static int refuse_batch(const erirt_handle* h, const char* what) {
  return fail(ERIRT_E_UNSUPPORTED, "%s is not supported on a replica batch (n_batch = %d)", what, h->nb);
}
extern "C" int64_t erirt_checkpoint_size(erirt_handle* h) {
  if (!h) { fail(ERIRT_E_ARG, "null handle"); return -1; }
  if (h->nb > 1) return refuse_batch(h, "erirt_checkpoint_size");
  return (int64_t)sizeof(CkHeader) + ck_header(h).payload_bytes;
}
extern "C" int erirt_checkpoint_save(erirt_handle* h, void* buf, int64_t size) {
  if (!h || !buf) return fail(ERIRT_E_ARG, "null argument");
  if (h->nb > 1) return refuse_batch(h, "erirt_checkpoint_save");
  const CkHeader H = ck_header(h);
  const int64_t need = (int64_t)sizeof(CkHeader) + H.payload_bytes;
  if (size < need) return fail(ERIRT_E_ARG, "checkpoint buffer of %lld bytes, %lld needed", (long long)size, (long long)need);
  CU(cudaSetDevice(h->cfg.device));
  CU(cudaStreamSynchronize(h->stream));
  memcpy(buf, &H, sizeof(H));
  char* dst = (char*)buf + sizeof(H);
  for (const CkSeg& sg : ck_segments(h)) {
    CU(cudaMemcpyAsync(dst, sg.p, sg.bytes, cudaMemcpyDeviceToHost, h->stream));
    dst += sg.bytes;
  }
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}
extern "C" int erirt_checkpoint_load(erirt_handle* h, const void* buf, int64_t size) {
  if (!h || !buf) return fail(ERIRT_E_ARG, "null argument");
  if (h->nb > 1) return refuse_batch(h, "erirt_checkpoint_load");
  if (size < (int64_t)sizeof(CkHeader)) return fail(ERIRT_E_ARG, "checkpoint shorter than its header");
  CkHeader H;
  memcpy(&H, buf, sizeof(H));
  if (memcmp(H.magic, "ERIRTCK2", 8) != 0) return fail(ERIRT_E_ARG, "not an erirt checkpoint (bad magic)");
  CkHeader W = ck_header(h);
  // everything but the progress fields must match the handle: a checkpoint continues THE SAME chain on the same shard
  W.sweeps_done = H.sweeps_done; W.prologue_done = H.prologue_done;
  if (memcmp(&H, &W, sizeof(H)) != 0)
    return fail(ERIRT_E_ARG, "checkpoint belongs to another configuration (model %d dtype %d %lld x %d, F=%d, nIter=%d nChain=%d, shard %lld+%lld, seed %llu chain %u, "
                "intercept %d 1pl %d cov2one %d compat %d qRt %g)",
                H.model, H.dtype, (long long)H.n_subj, H.n_item, H.n_feat, H.n_iter, H.n_chain, (long long)H.subj_offset, (long long)H.n_subj,
                (unsigned long long)H.seed, H.chain, H.intercept, H.itemtype_1pl, H.cov2one, H.compat, H.q_rt);
  if (size < (int64_t)sizeof(CkHeader) + H.payload_bytes) return fail(ERIRT_E_ARG, "checkpoint truncated: %lld of %lld bytes", (long long)size, (long long)(sizeof(CkHeader) + H.payload_bytes));
  if (H.sweeps_done < 0 || H.sweeps_done > h->cap) return fail(ERIRT_E_ARG, "checkpoint holds %lld sweeps, capacity is %d", (long long)H.sweeps_done, h->cap);
  CU(cudaSetDevice(h->cfg.device));
  CU(cudaStreamSynchronize(h->stream));
  const char* src = (const char*)buf + sizeof(H);
  for (const CkSeg& sg : ck_segments(h)) {
    CU(cudaMemcpyAsync(sg.p, src, sg.bytes, cudaMemcpyHostToDevice, h->stream));
    src += sg.bytes;
  }
  CU(cudaStreamSynchronize(h->stream));
  h->sweeps_done = H.sweeps_done;
  h->prologue_done = H.prologue_done != 0;
  return 0;
}

// ------------------------------------------------------------------------------------------------
// NCCL plumbing
// ------------------------------------------------------------------------------------------------
extern "C" int erirt_nccl_unique_id(void* id128) {
  if (!id128) return fail(ERIRT_E_ARG, "null argument");
  int rc = nccl::load();
  if (rc) return rc;
  nccl::unique_id id;
  NC(nccl::get_unique_id(&id));
  memcpy(id128, &id, 128);
  return 0;
}
extern "C" int erirt_comm_init(erirt_handle* h, int32_t rank, int32_t world, const void* id128) {
  if (!h) return fail(ERIRT_E_ARG, "null argument");
  if (h->nb > 1) return refuse_batch(h, "erirt_comm_init");
  if (world < 1 || rank < 0 || rank >= world) return fail(ERIRT_E_ARG, "bad rank/world");
  if (h->prologue_done) return fail(ERIRT_E_STATE, "erirt_comm_init must precede erirt_sample");
  CU(cudaSetDevice(h->cfg.device));
  if (id128) {  // NCCL communicator (fallback exchange); id128 == NULL: rank/world only, the peer exchange is attached next
    int rc = nccl::load();
    if (rc) return rc;
    nccl::unique_id id;
    memcpy(&id, id128, 128);
    NC(nccl::comm_init_rank(&h->comm, world, id, rank));
  }
  h->rank = rank;
  h->world = world;
  h->consts_final = false;
  return 0;
}

extern "C" int erirt_peer_export(erirt_handle* h, void* ipc_handle64) {
  if (!h || !ipc_handle64) return fail(ERIRT_E_ARG, "null argument");
  if (h->nb > 1) return refuse_batch(h, "erirt_peer_export");
  if (h->world < 2) return fail(ERIRT_E_STATE, "erirt_peer_export needs erirt_comm_init with world >= 2 first");
  if (h->prologue_done) return fail(ERIRT_E_STATE, "erirt_peer_export must precede erirt_sample");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handle size");
  CU(cudaSetDevice(h->cfg.device));
  if (!h->xbuf) {
    h->xstride = (int)align_up((size_t)std::max(h->L.s_count, h->c_count), 16);  // the statistics per sweep, the ingest constants once
    std::lock_guard<std::mutex> lk(g_peer_mu);
    for (size_t t = 0; t < g_peer_cache.size(); ++t) {
      PeerCacheEntry& c = g_peer_cache[t];
      if (!c.in_use && c.device == h->cfg.device && c.world == h->world && c.rank == h->rank && c.xstride == h->xstride && c.xbuf) {
        c.in_use = true;
        h->peer_cache_slot = (int)t;
        h->xbuf = c.xbuf; h->dPeerBufs = c.dPeerBufs; h->dXseq = c.dXseq;
        break;
      }
    }
  }
  if (!h->xbuf) {
    const size_t bytes = (size_t)2 * h->world * h->xstride * 16 + 256;  // [2 parities][world][xstride] 16-byte packets (global.cuh)
    auto alloc = [&]() -> int {
      CU(cudaMalloc((void**)&h->xbuf, bytes));
      CU(cudaMemset(h->xbuf, 0, bytes));
      CU(cudaMalloc((void**)&h->dPeerBufs, h->world * sizeof(double*)));
      CU(cudaMalloc((void**)&h->dXseq, sizeof(uint32_t)));
      CU(cudaMemset(h->dXseq, 0, sizeof(uint32_t)));
      CU(cudaDeviceSynchronize());
      return 0;
    };
    if (int rc = alloc()) {  // the buffers belong to no cache entry yet: free what was allocated
      if (h->xbuf) cudaFree(h->xbuf);
      if (h->dPeerBufs) cudaFree(h->dPeerBufs);
      if (h->dXseq) cudaFree(h->dXseq);
      h->xbuf = nullptr; h->dPeerBufs = nullptr; h->dXseq = nullptr;
      return rc;
    }
    std::lock_guard<std::mutex> lk(g_peer_mu);
    PeerCacheEntry c;
    c.device = h->cfg.device; c.world = h->world; c.rank = h->rank; c.xstride = h->xstride;
    c.xbuf = h->xbuf; c.dPeerBufs = h->dPeerBufs; c.dXseq = h->dXseq; c.in_use = true;
    g_peer_cache.push_back(c);
    h->peer_cache_slot = (int)g_peer_cache.size() - 1;
  }
  cudaIpcMemHandle_t hd;
  CU(cudaIpcGetMemHandle(&hd, h->xbuf));
  memcpy(ipc_handle64, &hd, 64);
  return 0;
}
extern "C" int erirt_peer_attach(erirt_handle* h, const void* ipc_handles) {
  if (!h || !ipc_handles) return fail(ERIRT_E_ARG, "null argument");
  if (h->nb > 1) return refuse_batch(h, "erirt_peer_attach");
  if (!h->xbuf) return fail(ERIRT_E_STATE, "erirt_peer_export has not been called");
  if (h->prologue_done) return fail(ERIRT_E_STATE, "erirt_peer_attach must precede erirt_sample");
  CU(cudaSetDevice(h->cfg.device));
  {
    std::lock_guard<std::mutex> lk(g_peer_mu);
    PeerCacheEntry& c = g_peer_cache[h->peer_cache_slot];
    if (c.handles.size() == (size_t)64 * h->world && memcmp(c.handles.data(), ipc_handles, c.handles.size()) == 0) {
      h->peer_ready = true;  // same peers, same buffers: the mappings (and the device table of their addresses) are still in place
      return 0;
    }
    for (void* p : c.opened) cudaIpcCloseMemHandle(p);  // the peers changed (a rank restarted): map afresh
    c.opened.clear();
    c.handles.clear();
  }
  std::vector<double*> ptrs(h->world, nullptr);
  std::vector<void*> opened;
  for (int r = 0; r < h->world; ++r) {
    if (r == h->rank) { ptrs[r] = h->xbuf; continue; }
    cudaIpcMemHandle_t hd;
    memcpy(&hd, (const char*)ipc_handles + (size_t)64 * r, 64);
    void* p = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&p, hd, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      for (void* q : opened) cudaIpcCloseMemHandle(q);
      return fail(ERIRT_E_CUDA, "cudaIpcOpenMemHandle(rank %d): %s (the GPUs must be peers on one node, one process each)", r, cudaGetErrorString(e));
    }
    opened.push_back(p);
    ptrs[r] = (double*)p;
  }
  {
    std::lock_guard<std::mutex> lk(g_peer_mu);
    PeerCacheEntry& c = g_peer_cache[h->peer_cache_slot];
    c.opened = opened;
    c.handles.assign((const char*)ipc_handles, (const char*)ipc_handles + (size_t)64 * h->world);
  }
  CU(cudaMemcpy(h->dPeerBufs, ptrs.data(), h->world * sizeof(double*), cudaMemcpyHostToDevice));
  h->peer_ready = true;
  return 0;
}

extern "C" int erirt_peer_detach(erirt_handle* h) {
  if (!h) return fail(ERIRT_E_ARG, "null handle");
  if (h->nb > 1) return refuse_batch(h, "erirt_peer_detach");
  CU(cudaSetDevice(h->cfg.device));
  CU(cudaStreamSynchronize(h->stream));  // (the peer mappings stay open with the cached exchange buffer, for the next handle)
  // Later sweeps go through ncclAllReduce when the chain has an NCCL communicator; a chain created with
  // erirt_comm_init(..., NULL) has no exchange left and launch_global refuses to run (ERIRT_E_STATE) instead of drawing
  // the item / structural parameters from the local shard's statistics only.
  h->peer_ready = false;
  // both captured graphs carry GlobalArgs.peer_bufs, the exchange just detached
  if (h->graph_exec) { cudaGraphExecDestroy(h->graph_exec); h->graph_exec = nullptr; }
  if (h->graph_multi) { cudaGraphExecDestroy(h->graph_multi); h->graph_multi = nullptr; }
  return 0;
}

// ------------------------------------------------------------------------------------------------
// parity entry points
// ------------------------------------------------------------------------------------------------
// n float64 inputs to the device, `launch(grid, din, dout)` enqueues the kernel on the default stream, n float64 results back
template <typename Launch>
static int run_parity_kernel(const char* name, int32_t device, const double* in, int64_t n, double* out, Launch launch) {
  if (int rc = pick_device(device)) return rc;
  if (n == 0) return 0;
  double *din = nullptr, *dout = nullptr;
  CU(cudaMalloc((void**)&din, n * sizeof(double)));
  CU(cudaMalloc((void**)&dout, n * sizeof(double)));
  CU(cudaMemcpy(din, in, n * sizeof(double), cudaMemcpyHostToDevice));
  launch((int)std::min<int64_t>((n + 255) / 256, 148 * 8), din, dout);
  cudaError_t e = cudaDeviceSynchronize();
  if (e == cudaSuccess) e = cudaMemcpy(out, dout, n * sizeof(double), cudaMemcpyDeviceToHost);
  cudaFree(din);
  cudaFree(dout);
  if (e != cudaSuccess) return fail(ERIRT_E_CUDA, "%s: %s", name, cudaGetErrorString(e));
  return 0;
}

extern "C" int erirt_k_pg(const double* z, int64_t rows, int32_t cols, int64_t row0, uint64_t seed, uint32_t chain,
                          uint32_t sweep, int32_t dtype, int32_t device, double* out) {
  if (!z || !out || rows < 0 || cols < 1) return fail(ERIRT_E_ARG, "bad argument");
  const PhiloxKey key = make_key(seed, chain);
  return run_parity_kernel("erirt_k_pg", device, z, rows * cols, out, [&](int grid, const double* dz, double* dout) {
    if (dtype == ERIRT_F32) k_pg_fast_kernel<<<grid, 256>>>(dz, rows, cols, row0, key, sweep, dout);
    else k_pg_kernel<double><<<grid, 256>>>(dz, rows, cols, row0, key, sweep, dout);
  });
}

extern "C" int erirt_k_nu_person(const double* mu, double lam, int64_t n, int64_t row0, uint64_t seed, uint32_t chain,
                                 uint32_t sweep, int32_t dtype, int32_t device, double* out) {
  if (!mu || !out || n < 0) return fail(ERIRT_E_ARG, "bad argument");
  const PhiloxKey key = make_key(seed, chain);
  return run_parity_kernel("erirt_k_nu_person", device, mu, n, out, [&](int grid, const double* dm, double* dout) {
    if (dtype == ERIRT_F32) k_nu_person_kernel<float><<<grid, 256>>>(dm, lam, n, row0, key, sweep, dout);
    else k_nu_person_kernel<double><<<grid, 256>>>(dm, lam, n, row0, key, sweep, dout);
  });
}

extern "C" int erirt_k_philox(const uint32_t ctr[4], const uint32_t key[2], int32_t device, uint32_t out[4]) {
  if (!ctr || !key || !out) return fail(ERIRT_E_ARG, "bad argument");
  int rc = pick_device(device);
  if (rc) return rc;
  uint32_t* d = nullptr;
  CU(cudaMalloc((void**)&d, 10 * sizeof(uint32_t)));
  CU(cudaMemcpy(d, ctr, 4 * sizeof(uint32_t), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(d + 4, key, 2 * sizeof(uint32_t), cudaMemcpyHostToDevice));
  k_philox_kernel<<<1, 1>>>(d, d + 4, d + 6);
  cudaError_t e = cudaMemcpy(out, d + 6, 4 * sizeof(uint32_t), cudaMemcpyDeviceToHost);
  cudaFree(d);
  if (e != cudaSuccess) return fail(ERIRT_E_CUDA, "erirt_k_philox: %s", cudaGetErrorString(e));
  return 0;
}
