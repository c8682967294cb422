// global.cuh -- item and structural draws from the reduced sufficient statistics (K3/K4/K6/K7 of SURVEY.md 2c).
//
// One CTA, launched after the person kernel P(k).  When persons are sharded over GPUs the all-reduce of the statistics is
// fused into this kernel (one-shot exchange over NVLink peer memory, see the top of global_draw_kernel; an ncclAllReduce
// in front of the launch is the fallback when no peer buffers are attached); every GPU then runs the draws redundantly
// with the same Philox key, so the new parameters need no broadcast.
//   1. log-likelihood of state k: Bernoulli + structural parts arrive in the statistics, the response-time
//      part is evaluated from sufficient statistics (getLogLikelihood*, GibbsRtIrt.pl.jl:262-272)
//   2. parameters of sweep k+1 in the reference's order (SURVEY 3.2), every sum over persons expanded into
//      S0,S1,S2,Ky,C, the Gram matrix and the ingest constants T1,T2,K0,X'X (SURVEY 7.1):
//        beta   drawSubjCoefficients :380-393 | ...Latent :399-416 | getSubjCoefficientsMlIrt :351-357 | ...LatentQr :446-458
//        Sigma  drawSubjCovariance :499-515 | ...Null :522-535 | ...Latent :563-579 | ...LatentQr :585-606
//        b      drawItemDifficulty :98-105,   a  drawItemDiscrimination :88-93   (MlIrt: a before b)
//        lambda drawItemIntensity :215-220,   sigma2  drawItemTimeResidual :257-262
//   3. trace row k+1 (Post.ra/rt/qr item + structural columns, GibbsRtIrt.pl.jl:319-321), statistics reset.
// All arithmetic is f64.
#pragma once
#include "layout.cuh"

namespace erirt {

// warp 0: structural block (cooperatively); warps 1..7: item draws; all warps: raw variates, reductions.  256 threads at <= 80
// registers fit beside two resident person CTAs of the hot configuration (168 registers each), i.e. as soon as ONE person CTA of some SM has finished
// its tiles, so the parameter-independent part of this kernel (everything before griddep_wait) runs beside the person kernel's tail.
constexpr int G_THREADS = 256;

// ---- small dense SPD helpers, warp-cooperative: all 32 lanes of ONE warp call them at the same point with the same arguments;
//      matrices are column-major in shared memory, n <= 32 = MAXD, lane i owns row i (or column i).  The structural block is a
//      dependent chain that sits on the critical path of every sweep (the person kernels wait for it): on one lane a 12 x 12
//      solve took 29 us (profiles/r02_sweep_timeline.txt), spread over the lanes its depth is O(n^2) shared-memory round trips.
//      Products are subtracted in the order of the textbook serial loops in the factor and the forward substitution, in another
//      order in the back substitution and the inverse, and divisions by the diagonal are multiplications by its reciprocal: the
//      results are within a few ulp of the oracle's serial code (the parity tests hold 1e-9 over whole chains). ----
// idiag (n doubles) receives 1 / L_jj: the substitutions below multiply by it instead of dividing (an f64 division is ~100 cycles of
// a dependent chain that every sweep waits for).  (Rows kept in registers with the columns travelling by shuffle were measured no
// faster: the structural block is bound by its many short dependent f64 chains, not by this factorisation; profiles/r02_summary.md.)
__device__ inline bool chol_lower(int n, const double* A, double* Lm, double* idiag, int lane) {
  // right-looking: Lm starts as the lower triangle of A, column j is scaled and its outer product leaves the trailing rows
  for (int t = lane; t < n * n; t += 32) {
    const int r = t % n, c = t / n;
    Lm[t] = r >= c ? A[t] : 0.0;
  }
  bool ok = true;
  #pragma unroll 1
  for (int j = 0; j < n; ++j) {
    __syncwarp();
    const double djj = Lm[j + n * j];
    if (!(djj > 0.0)) { ok = false; break; }  // uniform: every lane reads the same element
    const double d = sqrt(djj), id = 1.0 / d;
    double lij = 0.0;
    if (lane > j && lane < n) lij = Lm[lane + n * j] * id;
    __syncwarp();
    if (lane == j) { Lm[j + n * j] = d; idiag[j] = id; }
    if (lane > j && lane < n) Lm[lane + n * j] = lij;
    __syncwarp();  // column j is final
    if (lane > j && lane < n) {
      #pragma unroll 1
      for (int c = j + 1; c <= lane; ++c) Lm[lane + n * c] -= lij * Lm[c + n * j];
    }
  }
  __syncwarp();
  return ok;
}
// sol = A^{-1} rhs through the Cholesky factor (Lm: n*n scratch, idiag: n).  sol may alias rhs.
__device__ inline bool spd_solve(int n, const double* A, const double* rhs, double* sol, double* Lm, double* idiag, int lane) {
  if (!chol_lower(n, A, Lm, idiag, lane)) return false;
  double sv = lane < n ? rhs[lane] : 0.0;
  #pragma unroll 1
  for (int k = 0; k < n; ++k) {  // forward: y_k = s_k / L_kk, rows below lose L_ik y_k
    const double yk = __shfl_sync(0xffffffffu, sv, k) * idiag[k];
    if (lane == k) sv = yk;
    else if (lane > k && lane < n) sv -= Lm[lane + n * k] * yk;
  }
  #pragma unroll 1
  for (int k = n - 1; k >= 0; --k) {  // backward: x_k = s_k / L_kk, rows above lose L_ki x_k
    const double xk = __shfl_sync(0xffffffffu, sv, k) * idiag[k];
    if (lane == k) sv = xk;
    else if (lane < k) sv -= Lm[k + n * lane] * xk;
  }
  __syncwarp();
  if (lane < n) sol[lane] = sv;
  __syncwarp();
  return true;
}
// Ainv = A^{-1}: lane j solves A x = e_j (column j) by the two substitutions; Lm and Y are n*n scratch, none of the four may alias
__device__ inline bool spd_inverse(int n, const double* A, double* Ainv, double* Lm, double* Y, double* idiag, int lane) {
  if (!chol_lower(n, A, Lm, idiag, lane)) return false;
  if (lane < n) {
    double* y = Y + n * lane;     // column `lane` of L^{-1}: zero above its diagonal, so the rows start there
    double* x = Ainv + n * lane;  // column `lane` of A^{-1}
    #pragma unroll 1
    for (int i = 0; i < lane; ++i) y[i] = 0.0;
    #pragma unroll 1
    for (int i = lane; i < n; ++i) {
      double sacc = i == lane ? 1.0 : 0.0;
      #pragma unroll 1
      for (int k = lane; k < i; ++k) sacc -= Lm[i + n * k] * y[k];
      y[i] = sacc * idiag[i];
    }
    #pragma unroll 1
    for (int i = n - 1; i >= 0; --i) {
      double sacc = y[i];
      #pragma unroll 1
      for (int k = i + 1; k < n; ++k) sacc -= Lm[k + n * i] * x[k];
      x[i] = sacc * idiag[i];
    }
  }
  __syncwarp();
  return true;
}
// sum over the lanes of a warp (butterfly: every lane gets the total)
__device__ inline double warp_sum(double v) {
  #pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// quadratic form b' M b and bilinear a' b (every lane returns the result)
__device__ inline double quad_form(int n, const double* M, const double* b, int lane) {
  double t = 0.0;
  if (lane < n) {
    double x = 0.0;
    #pragma unroll 1
    for (int q = 0; q < n; ++q) x += M[lane + n * q] * b[q];
    t = b[lane] * x;
  }
  return warp_sum(t);
}
__device__ inline double dotn(int n, const double* a, const double* b, int lane) {
  return warp_sum(lane < n ? a[lane] * b[lane] : 0.0);
}

__device__ inline void cov2one_2x2(double* S) {  // Draw.pl.jl:507-511
  const double r12 = S[2] / sqrt(S[0]) / sqrt(S[3]), r21 = S[1] / sqrt(S[0]) / sqrt(S[3]);
  S[0] = 1.0; S[3] = 1.0; S[2] = r12; S[1] = r21;
}

// rand(InverseWishart(df, Psi)) = inv(rand(Wishart(df, inv(Psi)))), Wishart by Bartlett's decomposition
__device__ inline void inv_wishart2(PhiloxKey key, uint32_t sweep, double df, const double Psi[4], double out[4], const double* graw) {
  const double det = Psi[0] * Psi[3] - Psi[1] * Psi[2];
  const double S[4] = {Psi[3] / det, -Psi[1] / det, -Psi[2] / det, Psi[0] / det};
  const double l11 = sqrt(S[0]), l21 = S[1] / l11, l22 = sqrt(S[3] - l21 * l21);
  const uint32_t site = make_site(DOM_GLOBAL, GK_SIGMAP);
  const double a11 = sqrt(2.0 * gamma_from_raw(key, 0, sweep, site, 0.5 * df, graw[0], graw[1]));
  const double a22 = sqrt(2.0 * gamma_from_raw(key, 1, sweep, site, 0.5 * (df - 1.0), graw[2], graw[3]));
  const double a21 = graw[4];
  const double x11 = l11 * a11, x21 = l21 * a11 + l22 * a21, x22 = l22 * a22;
  const double w11 = x11 * x11, w21 = x21 * x11, w22 = x21 * x21 + x22 * x22;
  const double dw = w11 * w22 - w21 * w21;
  out[0] = w22 / dw; out[1] = -w21 / dw; out[2] = -w21 / dw; out[3] = w11 / dw;
}

#ifdef ERIRT_TICKS
__device__ long long g_gticks[16];
__device__ long long g_g0;
#define G_TICK(n, who) do { if (tid == (who)) g_gticks[n] = clock64() - _g0; } while (0)
#define S_TICK(n) (g_gticks[n] = clock64() - g_g0)
#else
#define G_TICK(n, who)
#define S_TICK(n)
#endif

struct GramView {  // accessors into the upper-triangular Gram of u = [1, X(1..F), theta, zeta, nu]
  const double* g;
  int Dg, F;
  __device__ double at(int r, int c) const { return r <= c ? g[tri_index(r, c, Dg)] : g[tri_index(c, r, Dg)]; }
  __device__ int th() const { return F + 1; }
  __device__ int ze() const { return F + 2; }
  __device__ int nu() const { return F + 3; }
};

// ---- fused one-shot all-reduce over NVLink peer memory (one CTA; all its threads call it at the same point) ----
// Every GPU owns an exchange buffer of 16-byte packets [2 parities][world slots][S]; a double travels as two self-validating 8-byte
// words {low 32 bits, seq} {high 32 bits, seq} (the LL protocol of NCCL: an aligned 8-byte store is delivered whole, so a word whose
// flag equals the sequence number of this exchange carries this exchange's data).  A thread stores its elements into slot
// [parity][rank] of EVERY GPU's buffer (fire and forget over NVLink), then polls the world slots of its OWN buffer and sums them in
// rank order (bitwise the same result on every GPU).  No fence, no separate flag, no CTA barrier between sending and receiving: the
// latency of the exchange is one NVLink store.  Two parities suffice: a GPU writes a slot again two exchanges later, and it cannot
// finish the exchange in between before the slot's owner has sent its data for it, i.e. has finished reading the earlier one.
__device__ inline void peer_allreduce_sum(double* const* peer_bufs, uint32_t* xseq, int world, int rank, int S, const double* src,
                                          int count, double* dst, int* status, int tid, int nthreads) {
  const uint32_t seq = *xseq + 1u;
  const int par = (int)(seq & 1u);
  ERIRT_CHECK(count <= S && rank >= 0 && rank < world);
  for (int t = tid; t < count; t += nthreads) {
    const unsigned long long bits = (unsigned long long)__double_as_longlong(src[t]);
    const unsigned long long w0 = (bits & 0xffffffffull) | ((unsigned long long)seq << 32), w1 = (bits >> 32) | ((unsigned long long)seq << 32);
    for (int r = 0; r < world; ++r) {
      ulonglong2* slot = reinterpret_cast<ulonglong2*>(peer_bufs[r]) + ((size_t)par * world + rank) * S + t;
      asm volatile("st.relaxed.sys.global.v2.u64 [%0], {%1, %2};" ::"l"(slot), "l"(w0), "l"(w1) : "memory");
    }
  }
  const ulonglong2* mine = reinterpret_cast<const ulonglong2*>(peer_bufs[rank]) + (size_t)par * world * S;
  const long long t_start = clock64();
  bool dead = false;
  for (int t = tid; t < count; t += nthreads) {
    double acc = 0.0;
    for (int r0 = 0; r0 < world; r0 += 8) {
      // the packets of eight ranks are requested together (one L2 round trip instead of eight in a row: polled one by one the
      // receive loop was ~8 us of the sweep at 8 GPUs), then each is validated and re-polled until it carries this exchange
      unsigned long long w0[8], w1[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        w0[i] = w1[i] = 0ull;
        if (r0 + i < world) {
          const ulonglong2* pk = mine + (size_t)(r0 + i) * S + t;
          asm volatile("ld.relaxed.sys.global.v2.u64 {%0, %1}, [%2];" : "=l"(w0[i]), "=l"(w1[i]) : "l"(pk) : "memory");
        }
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if (r0 + i < world) {
          const ulonglong2* pk = mine + (size_t)(r0 + i) * S + t;
          while ((uint32_t)(w0[i] >> 32) != seq || (uint32_t)(w1[i] >> 32) != seq) {
            if (dead || clock64() - t_start > 20000000000LL) {  // ~10 s: a peer is gone; flag it instead of hanging the GPU
              if (!dead) atomicExch(status, -1000 - (r0 + i));
              dead = true;
              break;
            }
            asm volatile("ld.relaxed.sys.global.v2.u64 {%0, %1}, [%2];" : "=l"(w0[i]), "=l"(w1[i]) : "l"(pk) : "memory");
          }
          acc += __longlong_as_double((long long)((w0[i] & 0xffffffffull) | (w1[i] << 32)));
        }
      }
    }
    dst[t] = acc;
  }
  __syncthreads();  // every thread has read *xseq; dst is complete
  if (tid == 0) *xseq = seq;
}
// the same exchange on its own, for the one-time ingest constants
__global__ void __launch_bounds__(512) peer_allreduce_kernel(double* const* peer_bufs, uint32_t* xseq, int world, int rank, int S,
                                                             double* buf, int count, int* status) {
  if (*status <= -1000) return;
  peer_allreduce_sum(peer_bufs, xseq, world, rank, S, buf, count, buf, status, (int)threadIdx.x, (int)blockDim.x);
}

struct GScratch {
  double M[MAXD * MAXD], V[MAXD * MAXD], Lc[MAXD * MAXD], T[MAXD * MAXD], XX[MAXD * MAXD];
  double rhs[MAXD], mean[MAXD], z[MAXD], beta[MAXD], Sigma[4];
  double idiag[MAXD];  // reciprocal diagonal of the current Cholesky factor
  double zn[MAXD];  // N(0,1) of the global beta site, unit t (precomputed on separate lanes)
  double graw[6];   // attempt-0 raw material of the Sigma site: (normal, uniform) of units 0, 1, 2
};

// mean + chol(V).L * z with z_t ~ N(0,1) at the global beta site; returns false if V is not SPD (warp-cooperative)
__device__ inline bool mvn_draw(int d, GScratch& w, int lane) {
  if (!chol_lower(d, w.V, w.Lc, w.idiag, lane)) return false;
  if (lane < d) {
    double acc = w.mean[lane];
    #pragma unroll 1
    for (int q = 0; q <= lane; ++q) acc += w.Lc[lane + d * q] * w.zn[q];
    w.beta[lane] = acc;
  }
  __syncwarp();
  return true;
}

// w.XX = x'x and w.rhs = x'y of the Latent family (x = [1 X θ]), one element per lane
__device__ inline void latent_prebuild(const GlobalArgs& A, const double* XtX, const GramView& Gm, GScratch& w, int tid, int nthreads) {
  const int F = A.L.F, pb = F + 1, d = F + 2;
  const bool qrm = A.model == M_LATENTQR;
  for (int t = tid; t < d * d + d; t += nthreads) {
    if (t < d * d) {
      const int r = t % d, q = t / d;
      w.XX[r + d * q] = (r < pb && q < pb) ? XtX[r + pb * q] : Gm.at(r, q);
    } else {
      const int r = t - d * d;
      w.rhs[r] = Gm.at(r, Gm.ze()) - (qrm ? A.k1 * Gm.at(r, Gm.nu()) : 0.0);
    }
  }
}

// Structural draws of sweep s, executed by the 32 lanes of warp 0 together: vector work is dealt over the lanes, scalar work is
// computed redundantly by every lane (same values), results are left in w.beta / w.Sigma.
__device__ inline bool structural_draws(const GlobalArgs& A, const double* XtX, uint32_t s, const GramView& Gm, const GramView& Gw, GScratch& w,
                                        int lane) {
  const Layout& L = A.L;
  const int F = L.F, pb = F + 1, model = A.model;
  const double N = (double)A.n_total;
  const int TH = Gm.th(), ZE = Gm.ze(), NU = Gm.nu();
  const double Sth2 = Gm.at(TH, TH), Sze2 = Gm.at(ZE, ZE), Sthze = Gm.at(TH, ZE);
  const double add = (A.compat & 1) ? 0.0 : 1.0;  // `1/σβ₀^2 .+ M` adds to EVERY element (Draw.pl.jl:386,410; quirk Q1)
  bool ok = true;
  double Sig[4] = {w.Sigma[0], w.Sigma[1], w.Sigma[2], w.Sigma[3]};
  __syncwarp();
  if (model == M_MLIRT) {
    if (lane < pb) w.rhs[lane] = Gm.at(lane, TH);
    __syncwarp();
    ok = spd_solve(pb, XtX, w.rhs, w.beta, w.Lc, w.idiag, lane);  // getSubjCoefficientsMlIrt
    if (!A.intercept && lane == 0) w.beta[0] = 0.0;
  } else if (model == M_RTIRT) {
    const int d = 2 * pb;
    const double S11 = Sig[0], S12 = Sig[2], S22 = Sig[3], det = S11 * S22 - S12 * S12;
    const double iO[4] = {S22 / det, -S12 / det, -S12 / det, S11 / det};
    for (int t = lane; t < d * d; t += 32) {
      const int rr = t % d, cc = t / d, br = rr / pb, r = rr % pb, bc = cc / pb, q = cc % pb;
      w.M[t] = iO[br + 2 * bc] * XtX[r + pb * q] + add + ((add == 0.0 && rr == cc) ? 1.0 : 0.0);
    }
    __syncwarp();
    ok = spd_inverse(d, w.M, w.V, w.Lc, w.T, w.idiag, lane);
    if (lane < d) {  // vec(x'η invΩ')
      const int c = lane / pb, r = lane % pb;
      w.rhs[lane] = Gm.at(r, TH) * iO[c + 0] + Gm.at(r, ZE) * iO[c + 2];
    }
    __syncwarp();
    if (lane < d) {
      double acc = 0.0;
      #pragma unroll 1
      for (int q = 0; q < d; ++q) acc += w.V[lane + d * q] * w.rhs[q];
      w.mean[lane] = acc;
    }
    __syncwarp();
    ok = ok && mvn_draw(d, w, lane);
    if (!A.intercept && lane == 0) { w.beta[0] = 0.0; w.beta[pb] = 0.0; }
    __syncwarp();
    // e'e, e = [θ ζ] - xβ   (drawSubjCovariance)
    const double* b1 = w.beta;
    const double* b2 = w.beta + pb;
    double q11 = 0, q12 = 0, q22 = 0, l1t = 0, l1z = 0, l2t = 0, l2z = 0;
    if (lane < pb) {
      const int r = lane;
      double x1 = 0, x2 = 0;
      #pragma unroll 1
      for (int q = 0; q < pb; ++q) { x1 += XtX[r + pb * q] * b1[q]; x2 += XtX[r + pb * q] * b2[q]; }
      q11 = b1[r] * x1; q12 = b1[r] * x2; q22 = b2[r] * x2;
      l1t = b1[r] * Gm.at(r, TH); l1z = b1[r] * Gm.at(r, ZE);
      l2t = b2[r] * Gm.at(r, TH); l2z = b2[r] * Gm.at(r, ZE);
    }
    q11 = warp_sum(q11); q12 = warp_sum(q12); q22 = warp_sum(q22);
    l1t = warp_sum(l1t); l1z = warp_sum(l1z); l2t = warp_sum(l2t); l2z = warp_sum(l2z);
    const double E11 = Sth2 - 2.0 * l1t + q11, E12 = Sthze - l1z - l2t + q12, E22 = Sze2 - 2.0 * l2z + q22;
    const double Psi[4] = {E11 + 1.0, E12, E12, E22 + 1.0};
    inv_wishart2(A.key, s, N + 3.0, Psi, Sig, w.graw);
    if (A.cov2one) cov2one_2x2(Sig);
  } else if (model == M_NULL) {
    for (int t = lane; t < 2 * pb; t += 32) w.beta[t] = 0.0;
    const double Psi[4] = {Sth2 + 1.0, Sthze, Sthze, Sze2 + 1.0};
    inv_wishart2(A.key, s, N + 3.0, Psi, Sig, w.graw);  // drawSubjCovarianceNull
    if (A.cov2one) cov2one_2x2(Sig);
  } else if (model == M_CROSS || model == M_CROSSQR) {
    // drawSubjCovarianceCross, Draw.pl.jl:542-557
    const double parA = 1e-3 + N / 2.0, parB = 1e-3 + Sze2 / 2.0;
    const double sv = parB / gamma_from_raw(A.key, 0, s, make_site(DOM_GLOBAL, GK_SIGMAP), parA, w.graw[0], w.graw[1]);
    Sig[0] = 1.0; Sig[1] = 0.0; Sig[2] = 0.0; Sig[3] = sv;
    if (A.cov2one) cov2one_2x2(Sig);
  } else if (model == M_LATENT || model == M_LATENTQR) {
    const int d = F + 2;
    const bool qrm = model == M_LATENTQR;
    // x = [1 X θ]: x'x (ingest constant bordered by the θ column of the Gram) and x'y, y = ζ (Latent) or ζ - k1 ν (LatentQr),
    // were built by all lanes in latent_prebuild
    double yy = Sze2;
    if (qrm) yy += -2.0 * A.k1 * Gm.at(ZE, NU) + A.k1 * A.k1 * Gm.at(NU, NU);
    if (!qrm) {  // drawSubjCoefficientsLatent
      const double iO = 1.0 / Sig[3];
      for (int t = lane; t < d * d; t += 32) w.M[t] = iO * w.XX[t] + add + ((add == 0.0 && t % d == t / d) ? 1.0 : 0.0);
      __syncwarp();
      ok = spd_inverse(d, w.M, w.V, w.Lc, w.T, w.idiag, lane);
      if (lane < d) {
        double acc = 0.0;
        #pragma unroll 1
        for (int q = 0; q < d; ++q) acc += w.V[lane + d * q] * (w.rhs[q] * iO);
        w.mean[lane] = acc;
      }
      __syncwarp();
      ok = ok && mvn_draw(d, w, lane);
    } else {  // getSubjCoefficientsLatentQr: the tall Kronecker system collapses to OLS (SURVEY a21)
      ok = spd_solve(d, w.XX, w.rhs, w.beta, w.Lc, w.idiag, lane);
    }
    if (!A.intercept && lane == 0) w.beta[0] = 0.0;
    __syncwarp();
    // residual sum of squares r = y - xβ
    const double ss = yy - 2.0 * dotn(d, w.beta, w.rhs, lane) + quad_form(d, w.XX, w.beta, lane);
    double parA, parB;
    if (!qrm) {
      parA = 1e-3 + N / 2.0;
      parB = 1e-3 + ss / 2.0;
    } else {
      const double Snu = Gm.at(0, NU), Snu2 = Gm.at(NU, NU);
      parA = 1e-3 + N * 3.0 / 2.0;
      double scale;
      if (A.compat & 2) {
        // Σ r_i²/(2 k2 ν_i) from the 1/ν-weighted Gram: y/ν terms
        for (int t = lane; t < d * d; t += 32) w.T[t] = Gw.at(t % d, t / d);
        if (lane < d) w.mean[lane] = Gw.at(lane, ZE) - A.k1 * Gm.at(0, lane);  // Σ x (ζ - k1 ν)/ν
        __syncwarp();
        const double yyw = Gw.at(ZE, ZE) - 2.0 * A.k1 * Gm.at(0, ZE) + A.k1 * A.k1 * Snu;
        const double ssw = yyw - 2.0 * dotn(d, w.beta, w.mean, lane) + quad_form(d, w.T, w.beta, lane);
        scale = ssw / (2.0 * A.k2);
      } else {
        // as written: sum(r.^2 / (2 k2e)) with vector / vector (quirk Q2, Draw.pl.jl:594)
        scale = ss * (2.0 * A.k2 * Snu) / (4.0 * A.k2 * A.k2 * Snu2);
      }
      parB = 1e-3 + scale + Snu;
    }
    const double sv = parB / gamma_from_raw(A.key, 0, s, make_site(DOM_GLOBAL, GK_SIGMAP), parA, w.graw[0], w.graw[1]);
    Sig[0] = 1.0; Sig[1] = 0.0; Sig[2] = 0.0; Sig[3] = sv;
    if (A.cov2one) cov2one_2x2(Sig);
  }
  __syncwarp();
  if (lane == 0) { w.Sigma[0] = Sig[0]; w.Sigma[1] = Sig[1]; w.Sigma[2] = Sig[2]; w.Sigma[3] = Sig[3]; }
  return ok;
}

__device__ inline void global_raw_variates(const GlobalArgs& A, uint32_t s, double* sRaw, GScratch& w, int tid) {
  // attempt-0 raw material of every site of sweep s, one task per lane: it does not depend on the parameters, and an f64 Box-Muller
  // (log, sqrt, cospi) is a long dependent chain
  const int J = A.L.J, Jp = A.L.Jp;
  for (int t = tid; t < 4 * J + MAXD + 3; t += G_THREADS) {
    if (t < 4 * J) {
      const int j = t >> 2, kind = t & 3;
      const uint32_t ik = kind == 0 ? IK_B : (kind == 1 ? IK_A : (kind == 2 ? IK_LAMBDA : IK_SIGMA2));
      const uint4 wd = philox(A.key, (uint32_t)j, s, make_site(DOM_ITEM, ik), 0);
      if (kind < 3) sRaw[kind * Jp + j] = normal2(wd.x, wd.y);
      else { sRaw[3 * Jp + j] = normal2(wd.x, wd.y); sRaw[4 * Jp + j] = u01d(wd.z); }
    } else if (t < 4 * J + MAXD) {
      const int u = t - 4 * J;
      const uint4 wd = philox(A.key, (uint32_t)u, s, make_site(DOM_GLOBAL, GK_BETA), 0);
      w.zn[u] = normal2(wd.x, wd.y);
    } else {
      const int u = t - 4 * J - MAXD;
      const uint4 wd = philox(A.key, (uint32_t)u, s, make_site(DOM_GLOBAL, GK_SIGMAP), 0);
      w.graw[2 * u] = normal2(wd.x, wd.y);
      w.graw[2 * u + 1] = u01d(wd.z);
    }
  }
}

// BATCH: the replica-batch instantiation (layout.cuh BatchArgs), one CTA per replica
template <bool BATCH = false>
__global__ void __maxnreg__(80) global_draw_kernel(KernelArgs<GlobalArgs, BATCH> A) {
  if constexpr (BATCH) to_replica(A, blockIdx.x);
#ifdef ERIRT_TICKS
  const long long _g0 = clock64();
  if (threadIdx.x == 0) g_g0 = _g0;
#endif
  __shared__ GScratch w;
  __shared__ double sRed[G_THREADS];
  const Layout& L = A.L;
  const int J = L.J, F = L.F, Dg = L.Dg, tid = threadIdx.x;
  const int model = A.model;
  const bool has_rt = model != M_MLIRT;
  const double N = (double)A.n_total;
  double* par = A.params;
  // Stage the reduced statistics and X'X in shared memory first: the structural block reads them element by element in
  // dependent loops, and every such read would otherwise be an L2 round trip (the person kernel's atomics left them in L2).
  extern __shared__ double g_dyn[];
  double* st = g_dyn;                     // [s_count + 2] local copy of the statistics (read-only below)
  double* sXtX = g_dyn + L.s_count + 2;   // [(F+1)^2]
  double* sRaw = sXtX + (F + 1) * (F + 1);  // [5][Jp] attempt-0 raw material of the item sites: z_b, z_a, z_lambda, x_sigma2, u_sigma2
  const int Jp = L.Jp;
  // ---- 0. before the dependency wait: what does not depend on the person launch P(k) that may still be running.  The sweep
  //      counter and the parameters were written by the previous global kernel, which completed before any CTA of P(k) let this
  //      kernel be scheduled (P's griddep_launch follows its own griddep_wait). ----
  TL_DECL(tl_entry);
  const uint32_t k = *A.sweep_ctr;  // person launch P(k)
  const uint32_t s = k + 1;         // sweep whose parameters are drawn now
  ERIRT_CHECK(2 * (F + 1) <= MAXD && F + 2 <= MAXD && L.J <= L.Jp);
  for (int t = tid; t < (F + 1) * (F + 1); t += G_THREADS) sXtX[t] = A.XtX[t];
  if (A.stage == 0 || A.stage == 2) global_raw_variates(A, s, sRaw, w, tid);
  // Two passes over the body below.  Pass 0 is a REHEARSAL that runs before the dependency wait, on the reduced statistics of the
  // previous sweep (A.stats_prev) and with every global store suppressed: this kernel runs once per sweep on an SM whose instruction
  // caches the person kernel has flushed, and its ~4000 executed instructions are fetched cold (measured: 16 us after the wait, of
  // which the arithmetic is a fraction).  The rehearsal pulls exactly the code (and the constants T1, T2, K0) the real pass needs
  // into the caches while the person kernel is still finishing its last tiles; pass 1 is the real one.
  const int first_pass = (A.rehearse && (A.stage == 0 || A.stage == 2) && k >= 1) ? 0 : 1;
#pragma unroll 1
  for (int pass = first_pass; pass < 2; ++pass) {
  const bool real = pass == 1;
  __syncthreads();  // the previous pass has finished with the shared scratch
  if (tid < MAXD) w.beta[tid] = par[L.p_beta + tid];  // one lane each: a single lane copying global -> shared pays a round trip per element
  if (tid >= 64 && tid < 68) w.Sigma[tid - 64] = par[L.p_Sigma + tid - 64];
  if (real) {
#ifdef ERIRT_TIMELINE
    __syncthreads();
    if (tid == 0) { g_timeline[k % TL_SLOTS][4] = tl_entry; g_timeline[k % TL_SLOTS][5] = tl_now(); }
#endif
    griddep_wait();  // P(k) has completed: its statistics (and, sharded, nothing else) are visible
#ifdef ERIRT_TIMELINE
    if (tid == 0) g_timeline[k % TL_SLOTS][6] = tl_now();
#endif
    if (*A.status <= -1000) return;   // a peer timed out in an earlier exchange: no draws from partial sums, no further 10 s waits
    if (A.peer_bufs) {
      peer_allreduce_sum(A.peer_bufs, A.xseq, A.world, A.rank, A.xstride, A.stats, L.s_count, st, A.status, tid, G_THREADS);
      if (*reinterpret_cast<volatile int*>(A.status) <= -1000) return;  // timed out in this exchange (uniform: written before the CTA barrier)
    } else {
      for (int t = tid; t < L.s_count; t += G_THREADS) st[t] = A.stats[t];
    }
  } else {
    for (int t = tid; t < L.s_count; t += G_THREADS) st[t] = A.stats_prev[t];
  }
  __syncthreads();
  G_TICK(0, 0);  // staging done
#ifdef ERIRT_TIMELINE
  if (real && tid == 0) g_timeline[k % TL_SLOTS][7] = tl_now();
#endif
  const GramView Gm{st + L.s_gram, Dg, F};
  const GramView Gw{st + L.s_gramw, Dg, F};
  const double Sth = Gm.at(0, Gm.th()), Sth2 = Gm.at(Gm.th(), Gm.th()), Sthze = Gm.at(Gm.th(), Gm.ze());
  const double Sze = Gm.at(0, Gm.ze()), Sze2 = Gm.at(Gm.ze(), Gm.ze());
  const double LOG2PI = 1.8378770664093454835606594728112;
  const bool cross = model == M_CROSS || model == M_CROSSQR;
  const double mu_lam = has_rt ? A.consts[0] : 0.0, sd_lam = has_rt ? A.consts[1] : 1.0;

  if (A.stage == 1) {
    // ---- G_a of the Cross family: lambda_k, sigma2_k from (theta_k, zeta_{k-1}, rho_k)   Draw.pl.jl:225-231, 267-273 ----
    for (int j = tid; j < J; j += G_THREADS) {
      const double s2 = par[L.p_sigma2 + j], rho = par[L.p_rho + j];
      const double T1 = A.T1[j], T2 = A.T2[j];
      const double pv = 1.0 / (sd_lam * sd_lam);
      double lam, s2n;
      if (model == M_CROSS) {
        const double C = st[L.s_C + j], D = st[L.s_D + j];
        const double parV = 1.0 / (pv + N / s2);
        const double parM = parV * (mu_lam * pv + (T1 + Sze + rho * Sth) / s2);
        lam = site_tnorm_pos(A.key, (uint32_t)j, k, make_site(DOM_ITEM, IK_LAMBDA), parM, sqrt(parV));
        const double Q = T2 - 2.0 * lam * T1 + N * lam * lam + 2.0 * (C - lam * Sze) + Sze2 + rho * rho * Sth2 +
                         2.0 * rho * (D - lam * Sth + Sthze);
        s2n = (1e-3 + Q / 2.0) / site_gamma(A.key, (uint32_t)j, k, make_site(DOM_ITEM, IK_SIGMA2), 1e-3 + N / 2.0);
      } else {
        // CrossQr (Draw.pl.jl:239-251, 278-288): weights w = 1/nu, r = logT + zeta; A0=Σw A1=Σθw A2=Σθrw A3=Σθ²w A4=Σrw A5=Σr²w V1=Σν
        const double A0 = st[L.s_S0 + j], A1 = st[L.s_S1 + j], A2 = st[L.s_S2 + j], A3 = st[L.s_Ky + j], A4 = st[L.s_C + j],
                     A5 = st[L.s_D + j], V1 = st[L.s_V + j];
        const double R1 = T1 + Sze, k1 = A.k1, k2 = A.k2;
        const double parV = 1.0 / (pv + A0 / (s2 * k2));
        const double parM = parV * (mu_lam * pv + (A4 + rho * A1 - k1 * N) / (s2 * k2));
        lam = site_tnorm_pos(A.key, (uint32_t)j, k, make_site(DOM_ITEM, IK_LAMBDA), parM, sqrt(parV));
        const double SS = A5 + lam * lam * A0 + rho * rho * A3 + k1 * k1 * V1 - 2.0 * lam * A4 + 2.0 * rho * A2 - 2.0 * k1 * R1 -
                          2.0 * lam * rho * A1 + 2.0 * lam * k1 * N - 2.0 * rho * k1 * Sth;
        s2n = (1e-3 + SS / (2.0 * k2) + V1) / site_gamma(A.key, (uint32_t)j, k, make_site(DOM_ITEM, IK_SIGMA2), 1e-3 + N * 3.0 / 2.0);
      }
      par[L.p_lambda + j] = lam;
      par[L.p_sigma2 + j] = s2n;
      if (k >= 1 && (int)(k - 1) < A.cap) {
        A.tr_items_rt[(size_t)(k - 1) * 2 * J + j] = lam;
        A.tr_items_rt[(size_t)(k - 1) * 2 * J + J + j] = s2n;
      }
    }
    __syncthreads();
    for (int t = tid; t < L.s_count; t += G_THREADS) A.stats[t] = 0.0;
    if (tid == 0) *A.tile_ctr = 0u;
    return;
  }

  // ---- 1. log-likelihood of state k ----
  if (k >= 1 || A.stage == 3) {
    double part = 0.0;
    if (model == M_CROSSQR) {
      if (tid == 0) part = st[L.s_scal + SC_LL_RT];
    } else if (has_rt || A.kz_from_stats)
      for (int j = tid; j < J; j += G_THREADS) {
        if (has_rt) {
          const double lam = par[L.p_lambda + j], s2 = par[L.p_sigma2 + j];
          double Q = A.T2[j] - 2.0 * lam * A.T1[j] + N * lam * lam + 2.0 * (st[L.s_C + j] - lam * Sze) + Sze2;
          if (cross) {  // residual logT - lambda + zeta + theta rho_j  (getLogLikelihoodRtIrtCross, GibbsRtIrtCross.pl.jl:158-169)
            const double rho = par[L.p_rho + j];
            Q += rho * rho * Sth2 + 2.0 * rho * (st[L.s_D + j] - lam * Sth + Sthze);
          }
          part += -0.5 * N * (LOG2PI + log(s2)) - 0.5 * Q / s2;
        }
        // sum_i kappa_ij z_ij = a_j [(Ky_j - sum_i theta_i / 2) - b_j K0_j] at state k: the part of the Bernoulli term the f32
        // person kernel leaves to its statistics (Ky = sum_i y_ij theta_i, K0 = sum_i kappa_ij)
        if (A.kz_from_stats) part += par[L.p_a + j] * ((st[L.s_Ky + j] - 0.5 * Sth) - par[L.p_b + j] * A.K0[j]);
      }
    for (int o = 16; o; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    if ((tid & 31) == 0) sRed[tid >> 5] = part;
    __syncthreads();
    if (tid == 0) {
      double tot = 0.0;
      for (int t = 0; t < G_THREADS / 32; ++t) tot += sRed[t];
      sRed[0] = tot;
    }
    __syncthreads();
    if (A.stage == 3) {  // evaluation only: report and leave every parameter untouched
      if (tid == 0) *A.ll_out = st[L.s_scal + SC_LL_BERN] + sRed[0] + st[L.s_scal + SC_LL_STRUCT];
      __syncthreads();
      for (int t = tid; t < L.s_count; t += G_THREADS) A.stats[t] = 0.0;
      if (tid == 0) *A.tile_ctr = 0u;
      return;
    }
    if (real && tid == 0 && (int)(k - 1) < A.cap) A.tr_ll[k - 1] = st[L.s_scal + SC_LL_BERN] + sRed[0] + st[L.s_scal + SC_LL_STRUCT];
  }

  G_TICK(1, 0);  // log-likelihood done
#ifdef ERIRT_TIMELINE
  if (real && tid == 0) g_timeline[k % TL_SLOTS][8] = tl_now();
#endif
  if (model == M_LATENT || model == M_LATENTQR) latent_prebuild(A, sXtX, Gm, w, tid, G_THREADS);
  __syncthreads();
#ifdef ERIRT_TIMELINE
  if (real && tid == 0) g_timeline[k % TL_SLOTS][13] = tl_now();
#endif
  G_TICK(6, 0);  // raw variates done
  // ---- 2a. structural draws (warp 0, cooperatively), 2b. item draws (warps 1..) ----
  if (tid < 32) {
    if (!structural_draws(A, sXtX, s, Gm, Gw, w, tid) && tid == 0 && real) atomicExch(A.status, (int)s);
    G_TICK(2, 0);  // structural block done
#ifdef ERIRT_TIMELINE
    if (real && tid == 0) g_timeline[k % TL_SLOTS][11] = tl_now();
#endif
  }
  // item draws on warps 1..: the structural block of warp 0 runs concurrently.  Two tasks per item, dealt so that a warp holds one
  // kind: (b, a) [MlIrt: (a, b)] and the response-time pair (lambda, sigma2) [Cross family: rho], which do not depend on each other
  for (int t = tid - 32; t >= 0 && t < 2 * J; t += G_THREADS - 32) {
    const int part = t / J, j = t - part * J;
    if (part == 0) {
      const double S0 = st[L.s_S0 + j], S1 = st[L.s_S1 + j], S2 = st[L.s_S2 + j];
      const double K0 = A.K0[j], K1 = st[L.s_Ky + j] - 0.5 * Sth;  // Σκ, Σκθ
      double a = par[L.p_a + j], b = par[L.p_b + j];
      auto draw_b = [&]() {  // drawItemDifficulty
        const double parV = 1.0 / (1.0 + a * a * S0);
        const double parM = parV * (0.0 - (a * K0 - a * a * S1));
        double v = parM + sqrt(parV) * sRaw[0 * Jp + j];
        b = v < -4.0 ? -4.0 : (v > 4.0 ? 4.0 : v);
      };
      auto draw_a = [&]() {  // drawItemDiscrimination
        const double parV = 1.0 / (1.0 + (S2 - 2.0 * b * S1 + b * b * S0));
        const double parM = parV * (1.0 + (K1 - b * K0));
        a = tnorm_pos_from_raw(A.key, (uint32_t)j, s, make_site(DOM_ITEM, IK_A), parM, sqrt(parV), sRaw[1 * Jp + j]);
        if (A.onepl) a = 1.0;
      };
      if (model == M_MLIRT) { draw_a(); draw_b(); }  // GibbsRtIrt.pl.jl:233-237 (quirk Q8)
      else { draw_b(); draw_a(); }
      if (real) {
        par[L.p_a + j] = a;
        par[L.p_b + j] = b;
      }
    } else if (cross) {  // drawSubjCorrCross, Draw.pl.jl:463-469 (state k: theta_k, zeta_k, lambda_k, sigma2_k)
      const double s2 = par[L.p_sigma2 + j], lam = par[L.p_lambda + j];
      double parV, parM;
      if (model == M_CROSS) {
        parV = 1.0 / (1.0 + Sth2 / s2);
        parM = parV * (0.0 + (lam * Sth - Sthze - st[L.s_D + j]) / s2);
      } else {  // drawSubjCorrCrossQr, Draw.pl.jl:474-489 with A1'=Σθ/ν, A2'=Σθ(logT+ζ)/ν, A3'=Σθ²/ν at nu_{k+1}
        const double A1 = st[L.s_C + j], A2 = st[L.s_D + j], A3 = st[L.s_V + j];
        parV = 1.0 / (1.0 + A3 / (s2 * A.k2));
        parM = parV * (0.0 + (lam * A1 - A2 + A.k1 * Sth) / (s2 * A.k2));
      }
      const double rho_new = parM + sqrt(parV) * site_normal(A.key, (uint32_t)j, s, make_site(DOM_ITEM, IK_RHO));
      if (real) par[L.p_rho + j] = rho_new;
    } else if (has_rt) {
      const double s2 = par[L.p_sigma2 + j];
      const double T1 = A.T1[j], T2 = A.T2[j], C = st[L.s_C + j];
      // drawItemIntensity
      const double pv = 1.0 / (sd_lam * sd_lam);
      const double parV = 1.0 / (pv + N / s2);
      const double parM = parV * (mu_lam * pv + (T1 + Sze) / s2);
      const double lam = tnorm_pos_from_raw(A.key, (uint32_t)j, s, make_site(DOM_ITEM, IK_LAMBDA), parM, sqrt(parV), sRaw[2 * Jp + j]);
      // drawItemTimeResidual: Σ_i (logT - λ + ζ)²
      const double Q = T2 - 2.0 * lam * T1 + N * lam * lam + 2.0 * (C - lam * Sze) + Sze2;
      const double parA = 1e-3 + N / 2.0, parB = 1e-3 + Q / 2.0;
      const double s2n = parB / gamma_from_raw(A.key, (uint32_t)j, s, make_site(DOM_ITEM, IK_SIGMA2), parA, sRaw[3 * Jp + j], sRaw[4 * Jp + j]);
      if (real) {
        par[L.p_lambda + j] = lam;
        par[L.p_sigma2 + j] = s2n;
      }
    }
  }
  G_TICK(3, 32);  // item draws of lane 32 done
#ifdef ERIRT_TIMELINE
  if (real && tid == 32) g_timeline[k % TL_SLOTS][12] = tl_now();
  if (real && tid == G_THREADS - 1) g_timeline[k % TL_SLOTS][14] = tl_now();
#endif
  __syncthreads();
  G_TICK(4, 0);
  if (real) griddep_launch();  // the CTAs of the next person launch become resident and arm their barriers while the trace row is written
#ifdef ERIRT_TIMELINE
  if (real && tid == 0) g_timeline[k % TL_SLOTS][9] = tl_now();
#endif
  if (real) {
    if (tid < MAXD) par[L.p_beta + tid] = w.beta[tid];
    if (tid >= 64 && tid < 68) par[L.p_Sigma + tid - 64] = w.Sigma[tid - 64];
  }
  __syncthreads();

  // ---- 3. trace row of sweep s, statistics reset ----
  if ((int)k < A.cap) {
    for (int j = tid; j < J; j += G_THREADS) {
      const double va = par[L.p_a + j], vb = par[L.p_b + j];
      if (real) {
        A.tr_items_ra[(size_t)k * 2 * J + j] = va;
        A.tr_items_ra[(size_t)k * 2 * J + J + j] = vb;
      }
      if (has_rt && !cross) {
        const double vl = par[L.p_lambda + j], vs = par[L.p_sigma2 + j];
        if (real) {
          A.tr_items_rt[(size_t)k * 2 * J + j] = vl;
          A.tr_items_rt[(size_t)k * 2 * J + J + j] = vs;
        }
      }
    }
    const int nb = cross ? J : ((model == M_MLIRT) ? F + 1 : ((model == M_RTIRT || model == M_NULL) ? 2 * (F + 1) : F + 2));
    for (int t = tid; t < A.qw; t += G_THREADS) {
      double v = t < nb ? (cross ? par[L.p_rho + t] : par[L.p_beta + t]) : par[L.p_Sigma + (t - nb)];
      if (real) A.tr_qr[(size_t)k * A.qw + t] = v;
    }
  }
  }  // pass
  if (tid == 0) {
    A.stats[L.s_count] = st[L.s_scal + SC_PG_DEFER];      // keep the diagnostics of the last sweep
    A.stats[L.s_count + 1] = st[L.s_scal + SC_PG_CELLS];
  }
  __syncthreads();
  for (int t = tid; t < L.s_count; t += G_THREADS) {
    A.stats[t] = 0.0;
    if (A.stats_prev) A.stats_prev[t] = st[t];  // the next launch rehearses on these
  }
  G_TICK(5, 0);  // trace + reset done
  if (tid == 0) { *A.sweep_ctr = k + 1; *A.tile_ctr = 0u; }
#ifdef ERIRT_TIMELINE
  if (tid == 0) {
    g_timeline[k % TL_SLOTS][10] = tl_now();
    // slots of the person launch of sweep k+1 start from their identity values
    g_timeline[(k + 1) % TL_SLOTS][0] = ~0ull; g_timeline[(k + 1) % TL_SLOTS][1] = ~0ull;
    g_timeline[(k + 1) % TL_SLOTS][2] = 0ull; g_timeline[(k + 1) % TL_SLOTS][3] = 0ull;
  }
#endif
}

}  // namespace erirt
