// Device-side building blocks shared by the kernels in abd_b200.cu.
//
// Everything here restates, per individual and in closed form, what the reference graph
// computes with dense (G,G,N) tensors:
//   constrain()        abd.py:640-667 (+ :560-601, :732-771, :774-862)    integer prologue
//   traj_*()           abd.py:242-274, :296-306, :329-341, :367-391       titer trajectories
//   row_eval()         abd.py:445-469, :556-557                           OD-row likelihood
//   finalize_*()       PyMC priors / transforms / Bernoulli terms invoked at abd.py:329-340,
//                      :367-388, :424-427, :464-467
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace abd {

// Gap masks are uint32_t (G <= 31), uint64_t (G <= 63) or u128 (G <= 127): the top bit of a mask word carries the
// waner bit (PackedState.rw, IndState.vacw).
using u128 = unsigned __int128;
// Length of the per-gap tables a kernel instantiated for mask type M keeps in shared memory (powers of rho, visiting
// order): one entry per mask bit, but at least 64, the size the 32- and 64-bit kernels were tuned with (the grid
// planner derives tiles and chains per CTA from their occupancy).
template <typename M>
constexpr int kGapTab = sizeof(M) * 8 > 64 ? (int)sizeof(M) * 8 : 64;
constexpr int kNSums = 16;
constexpr double kHalfLog2Pi = 0.918938533204672741780329736406;  // log(sqrt(2 pi))

// ---- indexes into theta13 -------------------------------------------------------------
enum Theta {
  N_PERM = 0, N_TEMP, N_RHO, N_INIT, S_PERM, S_RHO, S_INIT,
  N_B, N_D, N_SIGMA, S_B, S_D, S_SIGMA
};
// ---- indexes into the per-chain raw sums ------------------------------------------------
enum Sums {
  SN_0 = 0, SN_1, SN_2, SN_QINIT, SN_QPERM, SN_QTEMP, SN_QRHO,
  SS_0, SS_1, SS_2, SS_QINIT, SS_QPERM, SS_QRHO,
  S_KI, S_KW, S_PAD
};

// position of each theta13 entry inside q17
__constant__ const int kQOfTheta[13] = {1, 2, 3, 4, 5, 6, 10, 11, 12, 13, 14, 15, 16};
// transform of each q17 entry: 0 none, 1 log, 2 logodds
__constant__ const int kQTransform[17] = {2, 1, 1, 2, 0, 1, 2, 2, 1, 1, 0, 0, 0, 1, 0, 0, 1};
constexpr int kQ_P = 0, kQ_PW = 7;

struct Chunks {
  int n;               // number of time chunks (1 => OneTimeChunk rule)
  uint64_t mask[3];    // bit t set <=> gap t belongs to the chunk
  uint64_t mask_hi[3]; // the same for gaps 64..127 (128-bit layout only)
};

struct Totals {        // sizes over ALL shards (Bernoulli terms and likelihood constants)
  double rows_n, rows_s, bits_i, bits_w;
};

// prior of one continuous RV, in the form the finaliser needs
struct PriorSpec {
  int kind;      // 0 Normal(mu,sigma)  1 Gamma(alpha,beta)  2 Beta(a,b)  3 Exponential(lam)
  double a, b;   // (mu, sigma) | (alpha, beta) | (a, b) | (lam, -)
  double c;      // additive normalising constant
};
struct Priors {
  PriorSpec v[17];
};

// ---- bit helpers -------------------------------------------------------------------------
__device__ __forceinline__ int ctz(uint32_t v) { return __ffs((int)v) - 1; }
__device__ __forceinline__ int ctz(uint64_t v) { return __ffsll((long long)v) - 1; }
__device__ __forceinline__ int popc(uint32_t v) { return __popc(v); }
__device__ __forceinline__ int popc(uint64_t v) { return __popcll(v); }
__device__ __forceinline__ int ctz(u128 v) {
  const int lo = __ffsll((long long)(uint64_t)v), hi = __ffsll((long long)(uint64_t)(v >> 64));
  return lo ? lo - 1 : (hi ? 63 + hi : -1);
}
__device__ __forceinline__ int popc(u128 v) { return __popcll((uint64_t)v) + __popcll((uint64_t)(v >> 64)); }
// warp shuffle of a mask (two 64-bit shuffles for the 128-bit layout)
template <typename M>
__device__ __forceinline__ M shfl_mask(M v, int src) {
  if constexpr (sizeof(M) > 8) {
    const uint64_t lo = __shfl_sync(0xffffffffu, (uint64_t)v, src), hi = __shfl_sync(0xffffffffu, (uint64_t)(v >> 64), src);
    return ((M)hi << 64) | lo;
  } else {
    return __shfl_sync(0xffffffffu, v, src);
  }
}
template <typename M>
__device__ __forceinline__ M chunk_mask(const Chunks& ch, int k) {
  if constexpr (sizeof(M) > 8) return ((M)ch.mask_hi[k] << 64) | ch.mask[k];
  else return (M)ch.mask[k];
}
template <typename M>
__device__ __forceinline__ M low_mask(int t) {  // bits 0..t inclusive
  return (M)(~(M)0) >> (sizeof(M) * 8 - 1 - t);
}

// i_raw column (as a bit mask over gaps) -> constrained infection mask.
//   one chunk : i = mask3(i_raw | pcrpos)                                   abd.py:640-649
//   k chunks  : per chunk, PCR+ bits replace the column if any, else keep only the first
//               raw infection of the chunk (abd.py:658-667, :691-697, :722-729, :792-818);
//   then no infection within 3 gaps after an accepted one, scanning from t = 0 on the OUTPUT
//   (abd.py:560-601).
template <typename M>
__device__ __forceinline__ M constrain(M raw, M pcr, const Chunks& ch) {
  M m;
  if (ch.n == 1) {
    m = raw | pcr;
  } else {
    m = 0;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      if (k < ch.n) {
        const M cm = chunk_mask<M>(ch, k);
        const M p = pcr & cm, r = raw & cm;
        m |= p ? p : (r & (~r + 1));
      }
    }
  }
  M out = 0;
  while (m) {
    const M b = m & (~m + 1);
    out |= b;
    m &= ~(b | (b << 1) | (b << 2) | (b << 3));
  }
  return out;
}

__device__ __forceinline__ double ipow(double r, int k) {
  double acc = 1.0, b = r;
  while (k) {
    if (k & 1) acc *= b;
    b *= b;
    k >>= 1;
  }
  return acc;
}

// N antigen at gap t: P = 1[any infection <= t], T = sum_{s in inf, s<=t} rho^(t-s),
// dT = dT/drho.  pwd[k] = {rho^k, k rho^(k-1)} (one 16-byte shared-memory load per event).
template <typename M>
__device__ __forceinline__ void traj_n(M inf, int t, const double2* pwd, double& P, double& T, double& dT) {
  M e = inf & low_mask<M>(t);
  P = e ? 1.0 : 0.0;
  T = 0.0;
  dT = 0.0;
  while (e) {
    const double2 v = pwd[t - ctz(e)];
    e &= e - 1;
    T += v.x;
    dT += v.y;
  }
}

// S antigen: exposure = i + v (a month with both counts twice, abd.py:378-386).
// w == 0 => rho_ind = 1 (abd.py:374): U = number of exposures so far, dU/drho_s = 0.
// One loop over the months with any exposure (its trip count in a warp is the largest number of
// exposed months, not the largest number of infections plus the largest number of vaccinations).
template <typename M>
__device__ __forceinline__ void traj_s(M inf, M vac, int w, int t, const double2* pwd, double& P, double& U, double& dU) {
  const M lm = low_mask<M>(t);
  const M e = inf & lm, v = vac & lm;
  M u = e | v;
  const M both = e & v;
  P = u ? 1.0 : 0.0;
  U = 0.0;
  dU = 0.0;
  if (w) {
    while (u) {
      const int s = ctz(u);
      const double2 p = pwd[t - s];
      const double cnt = ((both >> s) & 1) ? 2.0 : 1.0;
      u &= u - 1;
      U = fma(cnt, p.x, U);
      dU = fma(cnt, p.y, dU);
    }
  } else {
    U = (double)(popc(e) + popc(v));
  }
}

// value-only versions for the Gibbs kernel
template <typename M>
__device__ __forceinline__ double mu_n_at(M inf, int t, const double* pw, double init, double perm,
                                          double temp) {
  M e = inf & low_mask<M>(t);
  double T = 0.0;
  const double P = e ? perm : 0.0;
  while (e) {
    T += pw[t - ctz(e)];
    e &= e - 1;
  }
  return init + P + temp * T;
}
template <typename M>
__device__ __forceinline__ double mu_s_at(M inf, M vac, int w, int t, const double* pw, double init,
                                          double perm) {
  const M lm = low_mask<M>(t);
  M e = inf & lm, v = vac & lm;
  const double P = (e | v) ? perm : 0.0;
  double U = 0.0;
  if (w) {
    while (e) {
      U += pw[t - ctz(e)];
      e &= e - 1;
    }
    while (v) {
      U += pw[t - ctz(v)];
      v &= v - 1;
    }
  } else {
    U = (double)(popc(e) + popc(v));
  }
  return init + P + U;
}

// ---- fast fp64 exp / reciprocal for the OD-row hot loop -------------------------------------
// exp(z) = 2^(k/64) * exp(r),  k = rint(z * 64/ln2),  r = z - k ln2/64  (|r| <= ln2/128):
// 64-entry table of 2^(j/64) (shared memory) x degree-5 polynomial; < 1.5 ulp for -745 <= z
// <= 709 (checked against libm in tests/test_gpu_parity.py::test_fast_math).  Results below
// 2^-1021 are flushed to 0 (the caller only needs 1/(1+E)).  NaN in -> NaN out.
constexpr int kExpTab = 64;
// 2^(j/64), j = 0..63, correctly rounded (generated with 60-digit decimal arithmetic)
__device__ const double kExp2Tab[kExpTab] = {
    0x1.0000000000000p+0, 0x1.02c9a3e778061p+0, 0x1.059b0d3158574p+0, 0x1.0874518759bc8p+0,
    0x1.0b5586cf9890fp+0, 0x1.0e3ec32d3d1a2p+0, 0x1.11301d0125b51p+0, 0x1.1429aaea92de0p+0,
    0x1.172b83c7d517bp+0, 0x1.1a35beb6fcb75p+0, 0x1.1d4873168b9aap+0, 0x1.2063b88628cd6p+0,
    0x1.2387a6e756238p+0, 0x1.26b4565e27cddp+0, 0x1.29e9df51fdee1p+0, 0x1.2d285a6e4030bp+0,
    0x1.306fe0a31b715p+0, 0x1.33c08b26416ffp+0, 0x1.371a7373aa9cbp+0, 0x1.3a7db34e59ff7p+0,
    0x1.3dea64c123422p+0, 0x1.4160a21f72e2ap+0, 0x1.44e086061892dp+0, 0x1.486a2b5c13cd0p+0,
    0x1.4bfdad5362a27p+0, 0x1.4f9b2769d2ca7p+0, 0x1.5342b569d4f82p+0, 0x1.56f4736b527dap+0,
    0x1.5ab07dd485429p+0, 0x1.5e76f15ad2148p+0, 0x1.6247eb03a5585p+0, 0x1.6623882552225p+0,
    0x1.6a09e667f3bcdp+0, 0x1.6dfb23c651a2fp+0, 0x1.71f75e8ec5f74p+0, 0x1.75feb564267c9p+0,
    0x1.7a11473eb0187p+0, 0x1.7e2f336cf4e62p+0, 0x1.82589994cce13p+0, 0x1.868d99b4492edp+0,
    0x1.8ace5422aa0dbp+0, 0x1.8f1ae99157736p+0, 0x1.93737b0cdc5e5p+0, 0x1.97d829fde4e50p+0,
    0x1.9c49182a3f090p+0, 0x1.a0c667b5de565p+0, 0x1.a5503b23e255dp+0, 0x1.a9e6b5579fdbfp+0,
    0x1.ae89f995ad3adp+0, 0x1.b33a2b84f15fbp+0, 0x1.b7f76f2fb5e47p+0, 0x1.bcc1e904bc1d2p+0,
    0x1.c199bdd85529cp+0, 0x1.c67f12e57d14bp+0, 0x1.cb720dcef9069p+0, 0x1.d072d4a07897cp+0,
    0x1.d5818dcfba487p+0, 0x1.da9e603db3285p+0, 0x1.dfc97337b9b5fp+0, 0x1.e502ee78b3ff6p+0,
    0x1.ea4afa2a490dap+0, 0x1.efa1bee615a27p+0, 0x1.f50765b6e4540p+0, 0x1.fa7c1819e90d8p+0};
__device__ __forceinline__ void fill_exp_table(double* tab, int tid, int nthreads) {
  for (int j = tid; j < kExpTab; j += nthreads) tab[j] = kExp2Tab[j];
}
__device__ __forceinline__ double fast_exp(double z, const double* __restrict__ tab) {
  constexpr double kInv = 92.33248261689366;            // 64 / ln 2
  constexpr double kMagic = 6755399441055744.0;         // 1.5 * 2^52
  constexpr double kLn2Hi = 0.01083042469326756;        // ln2/64, low 21 mantissa bits zero
  constexpr double kLn2Lo = 2.9815858269852933e-12;     // ln2/64 - kLn2Hi
  const double zc = (z < -750.0) ? -750.0 : z;
  const double t = fma(zc, kInv, kMagic);
  const int k = __double2loint(t);
  const double kd = t - kMagic;
  double r = fma(kd, -kLn2Hi, zc);
  r = fma(kd, -kLn2Lo, r);
  double p = fma(r, 8.3333333333333332e-03, 4.1666666666666664e-02);
  p = fma(p, r, 1.6666666666666666e-01);
  p = fma(p, r, 0.5);
  p = fma(p * r, r, r);
  const double T = tab[k & (kExpTab - 1)];
  double res = fma(T, p, T);
  const int e = k >> 6;
  res = __hiloint2double(__double2hiint(res) + (e << 20), __double2loint(res));
  res = (e < -1021) ? 0.0 : res;
  return (z != z) ? z : res;
}
// 1/x for normal x >= 1: MUFU seed + two Newton steps (full fp64 accuracy to ~1 ulp)
__device__ __forceinline__ double fast_rcp(double x) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  double e = fma(-x, r, 1.0);
  r = fma(r, e, r);
  e = fma(-x, r, 1.0);
  r = fma(r, e, r);
  return r;
}

// 1/x for normal x >= 1 with one cubic step: e = 1 - x r (|e| <= 2^-19.9 after the MUFU seed, which
// reads only the high word of x), r' = r (1 + e + e^2): remaining error e^3 < 2^-59, < 1 ulp overall.
__device__ __forceinline__ double fast_rcp3(double x) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  const double e = fma(-x, r, 1.0);
  const double t = fma(e, e, e);
  return fma(r, t, r);
}

// One OD row: s = 1/(1+E), E = exp(-b (x - m));  r = od - d s;  q = r s (1 - s).
// 1 - s is formed as E s (no cancellation); E is capped so that E s stays finite.
__device__ __forceinline__ void row_eval(double x, double od, double m, double b, double d,
                                         const double* __restrict__ tab, double& s, double& r,
                                         double& q, double& xm) {
  xm = x - m;
  double z = -b * xm;
  z = (z > 700.0) ? 700.0 : z;  // NaN stays NaN
  const double E = fast_exp(z, tab);
  s = fast_rcp(1.0 + E);
  r = fma(-d, s, od);
  q = r * s * (E * s);
}
// The same with E handed in (factored mode: E = exp(-b x) * exp(b m), one exp per (individual,
// gap) cell and a per-chain table over the cohort's few distinct dilutions instead of one exp per
// row).  The caller guarantees E <= e^700 (or NaN).
__device__ __forceinline__ void row_eval_E(double E, double od, double d, double& s, double& r, double& q) {
  s = fast_rcp3(1.0 + E);
  r = fma(-d, s, od);
  q = r * s * (E * s);
}
__device__ __forceinline__ double row_resid2(double x, double od, double m, double b, double d,
                                             const double* __restrict__ tab) {
  double z = -b * (x - m);
  z = (z > 700.0) ? 700.0 : z;
  const double s = fast_rcp(1.0 + fast_exp(z, tab));
  const double r = fma(-d, s, od);
  return r * r;
}

// ---- warp reduction of 16 doubles with 16 (not 80) 64-bit shuffles ----------------------------
// Butterfly that halves the number of values a lane carries at every step.  Afterwards lane l
// holds the warp total of value  k(l) = 8 b4 + 4 b3 + 2 b2 + b1  (b_i = bit i of l); both lanes
// of a pair (l, l^1) hold the same total.  Summation order is fixed => deterministic.
__device__ __forceinline__ double warp_reduce16(const double (&v)[16], int lane) {
  double a8[8], a4[4], a2[2], a1;
  const bool h16 = lane & 16, h8 = lane & 8, h4 = lane & 4, h2 = lane & 2;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const double send = h16 ? v[k] : v[k + 8], keep = h16 ? v[k + 8] : v[k];
    a8[k] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const double send = h8 ? a8[k] : a8[k + 4], keep = h8 ? a8[k + 4] : a8[k];
    a4[k] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
  }
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const double send = h4 ? a4[k] : a4[k + 2], keep = h4 ? a4[k + 2] : a4[k];
    a2[k] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
  }
  {
    const double send = h2 ? a2[0] : a2[1], keep = h2 ? a2[1] : a2[0];
    a1 = keep + __shfl_xor_sync(0xffffffffu, send, 2);
  }
  return a1 + __shfl_xor_sync(0xffffffffu, a1, 1);
}
__device__ __forceinline__ int warp_reduce16_index(int lane) {
  return ((lane >> 4) & 1) * 8 + ((lane >> 3) & 1) * 4 + ((lane >> 2) & 1) * 2 + ((lane >> 1) & 1);
}

// ---- programmatic dependent launch (PDL) ------------------------------------------------------
// launch_dependents: the next kernel in the stream may start being scheduled (it still blocks in
// its own griddep_wait until this grid has completed and flushed).  wait: block until every
// kernel this launch depends on has completed.  Both are no-ops without the launch attribute.
__device__ __forceinline__ void griddep_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ---- mbarrier + 1-D bulk async copy (TMA) -------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@!p bra WAIT_%=;\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// global -> shared, size and both addresses multiples of 16 bytes; completes on `bar`
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

__device__ __forceinline__ double softplus(double y) {  // log(1 + e^y)
  return log1p(exp(-fabs(y))) + fmax(y, 0.0);
}

// q17 entry -> constrained value
__device__ __forceinline__ double backward(double y, int transform) {
  if (transform == 1) return exp(y);
  if (transform == 2) return 1.0 / (1.0 + exp(-y));
  return y;
}

// ---- finalisation: raw sums -> loglik / joint logp and gradients ---------------------------------
// Split in a "pre" part that depends only on the parameters (logs, exps, priors, transforms --
// computed while the rows are still being processed) and a cheap "post" part that needs the sums.
struct LikPre {
  double lsn, lss;   // log sigma
  double ivn, ivs;   // 1 / sigma^2
  double isn, iss;   // 1 / sigma
};
__device__ __forceinline__ LikPre lik_pre(double sn, double ss) {
  LikPre p;
  p.lsn = log(sn);
  p.lss = log(ss);
  p.isn = 1.0 / sn;
  p.iss = 1.0 / ss;
  p.ivn = p.isn * p.isn;
  p.ivs = p.iss * p.iss;
  return p;
}

// Data log-likelihood and gradient w.r.t. theta13 from the raw sums.  The finaliser is inlined in
// several kernels (k_sums, k_finalize) that must agree BITWISE, so every product / sum is spelled
// with non-contractible intrinsics: the compiler may not pick different FMA contractions per copy.
__device__ __forceinline__ double mul_(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double add_(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ void finalize_loglik_post(const double* th, const LikPre& lp, const double* S,
                                                     const Totals& tot, double* loglik, double* g) {
  const double ln = add_(mul_(mul_(-0.5, S[SN_0]), lp.ivn), -mul_(tot.rows_n, add_(kHalfLog2Pi, lp.lsn)));
  const double ls = add_(mul_(mul_(-0.5, S[SS_0]), lp.ivs), -mul_(tot.rows_s, add_(kHalfLog2Pi, lp.lss)));
  *loglik = add_(ln, ls);
  if (!g) return;
  g[N_D] = mul_(S[SN_1], lp.ivn);
  g[N_B] = mul_(mul_(th[N_D], S[SN_2]), lp.ivn);
  g[N_SIGMA] = mul_(add_(mul_(S[SN_0], lp.ivn), -tot.rows_n), lp.isn);
  const double cn = mul_(mul_(-th[N_D], th[N_B]), lp.ivn);
  g[N_INIT] = mul_(cn, S[SN_QINIT]);
  g[N_PERM] = mul_(cn, S[SN_QPERM]);
  g[N_TEMP] = mul_(cn, S[SN_QTEMP]);
  g[N_RHO] = mul_(mul_(cn, th[N_TEMP]), S[SN_QRHO]);
  g[S_D] = mul_(S[SS_1], lp.ivs);
  g[S_B] = mul_(mul_(th[S_D], S[SS_2]), lp.ivs);
  g[S_SIGMA] = mul_(add_(mul_(S[SS_0], lp.ivs), -tot.rows_s), lp.iss);
  const double cs = mul_(mul_(-th[S_D], th[S_B]), lp.ivs);
  g[S_INIT] = mul_(cs, S[SS_QINIT]);
  g[S_PERM] = mul_(cs, S[SS_QPERM]);
  g[S_RHO] = mul_(cs, S[SS_QRHO]);
}
__device__ inline void finalize_loglik(const double* th, const double* S, const Totals& tot,
                                       double* loglik, double* g) {
  finalize_loglik_post(th, lik_pre(th[N_SIGMA], th[S_SIGMA]), S, tot, loglik, g);
}

// Prior + transform of value variable k at unconstrained value y, minus what needs the sums:
//   logp_k = lpA (+ K lx + (n - K) l1mx   for the two Bernoulli probabilities)
//   dlogp_k = dA (+ K omx - (n - K) x) + f * d loglik / d x_k
struct PriorPre {
  double lpA, dA, f, lx, l1mx, x, omx;
};
// (not inlined: one copy of this cold code per kernel, and the same arithmetic in every kernel)
__device__ __noinline__ PriorPre prior_pre(int k, double y, const PriorSpec& ps) {
  PriorPre o;
  o.lx = o.l1mx = o.x = o.omx = 0.0;
  const int tr = kQTransform[k];
  if (tr == 0) {  // Normal, no transform
    const double z = (y - ps.a) / ps.b;
    o.lpA = -0.5 * z * z + ps.c;
    o.dA = -z / ps.b;
    o.f = 1.0;
  } else if (tr == 1) {  // log transform: x = e^y, log|J| = y
    const double x = exp(y);
    if (ps.kind == 1) {  // Gamma(alpha, beta)
      o.lpA = ps.c - ps.b * x + (ps.a - 1.0) * y + y;
      o.dA = -ps.b * x + (ps.a - 1.0) + 1.0;
    } else {  // Exponential(lam)
      o.lpA = ps.c - ps.a * x + y;
      o.dA = -ps.a * x + 1.0;
    }
    o.f = x;
  } else {  // logodds transform: x = sigmoid(y), log|J| = log x + log(1 - x); Beta(a, b) prior
    o.lx = -softplus(-y);
    o.l1mx = -softplus(y);
    o.x = exp(o.lx);
    o.omx = exp(o.l1mx);
    const double ca = ps.a - 1.0, cb = ps.b - 1.0;
    o.lpA = ps.c + (ca == 0.0 ? 0.0 : ca * o.lx) + (cb == 0.0 ? 0.0 : cb * o.l1mx) + o.lx + o.l1mx;
    o.dA = (ca + 1.0) * o.omx - (cb + 1.0) * o.x;
    o.f = o.x * o.omx;
  }
  return o;
}

// Joint logp over (q17, i_raw, waner) in PyMC's unconstrained space and d logp / d q17, by one
// full warp: lane k < 17 owns value variable k; the 17 terms are summed by a fixed-order shuffle
// tree (deterministic).  pre[k] = prior_pre(k, q[k], ...), th = the 13 constrained parameters.
__device__ inline void finalize_logp_post(int lane, const PriorPre* pre, const double* th, const LikPre& lk,
                                          const double* S, const Totals& tot, double* logp, double* dlogp) {
  double g13[13], ll;
  finalize_loglik_post(th, lk, S, tot, &ll, g13);
  double lp = 0.0;
  if (lane < 17) {
    const int k = lane;
    double gl = 0.0;  // d loglik / d (constrained value of slot k)
#pragma unroll
    for (int j = 0; j < 13; ++j) gl = (kQOfTheta[j] == k) ? g13[j] : gl;
    const PriorPre p = pre[k];
    lp = p.lpA;
    double d = p.dA;
    if (k == kQ_P || k == kQ_PW) {  // Bernoulli(i_raw | p) abd.py:427, Bernoulli(waner | p_waner) abd.py:373
      const double K = (k == kQ_P) ? S[S_KI] : S[S_KW];
      const double nK = ((k == kQ_P) ? tot.bits_i : tot.bits_w) - K;
      lp = add_(lp, add_(K == 0.0 ? 0.0 : mul_(K, p.lx), nK == 0.0 ? 0.0 : mul_(nK, p.l1mx)));
      d = add_(d, add_(mul_(K, p.omx), -mul_(nK, p.x)));
    }
    d = fma(gl, p.f, d);
    if (dlogp) dlogp[k] = d;
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) lp = add_(lp, __shfl_down_sync(0xffffffffu, lp, off));
  if (lane == 0) *logp = add_(ll, lp);
}

// Philox4x32-10 (Salmon et al. 2011), counter-based: one call yields 4 x 32 random bits.
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
  constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
    const uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += W0;
    key.y += W1;
  }
  return ctr;
}
// (0, 1] uniform from 32 bits
__device__ __forceinline__ double u01(uint32_t r) { return ((double)r + 1.0) * 2.3283064365386963e-10; }

}  // namespace abd
