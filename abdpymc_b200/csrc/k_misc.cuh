// Small kernels: the two ends of an HMC transition, the Deterministics, the SM copy kernel for
// pinned host memory, and the fast-math test hook.
#pragma once
#include "abd_kernels_common.cuh"

namespace {
using namespace abd;

// ------------------------------------------------------------------------------------------
// k_hmc_begin / k_hmc_end -- the two ends of an HMC transition, one warp per chain
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
k_hmc_begin(const int C, const double* __restrict__ q, const double* __restrict__ grad, const double* __restrict__ logp,
            const double* __restrict__ linv_t, const uint64_t seed, const uint64_t iter, double* __restrict__ qw,
            double* __restrict__ pw, double* __restrict__ gw, double* __restrict__ h0, const unsigned chain_offset) {
  const int c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (c >= C) return;
  double z = 0.0;
  if (lane < 17) {  // Box-Muller on two of the four Philox words
    const uint4 r = philox4x32_10(make_uint4((uint32_t)lane, (uint32_t)c + chain_offset, (uint32_t)iter, 0x484d4331u),
                                  make_uint2((uint32_t)seed, (uint32_t)(seed >> 32) ^ (uint32_t)(iter >> 32)));
    z = sqrt(-2.0 * log(u01(r.x))) * cospi(2.0 * u01(r.y));
  }
  double p = 0.0, kin = z * z;
  for (int j = 0; j < 17; ++j) {
    const double zj = __shfl_sync(0xffffffffu, z, j);
    if (lane < 17) p = fma(linv_t[lane * 17 + j], zj, p);
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) kin += __shfl_xor_sync(0xffffffffu, kin, off);
  if (lane < 17) {
    qw[(size_t)c * 17 + lane] = q[(size_t)c * 17 + lane];
    gw[(size_t)c * 17 + lane] = grad[(size_t)c * 17 + lane];
    pw[(size_t)c * 17 + lane] = p;
  }
  if (lane == 0) h0[c] = -logp[c] + 0.5 * kin;
}

__global__ void __launch_bounds__(128)
k_hmc_end(const int C, double* __restrict__ q, double* __restrict__ grad, double* __restrict__ logp,
          const double* __restrict__ qw, const double* __restrict__ pw, const double* __restrict__ gw,
          const double* __restrict__ lpw, const double* __restrict__ inv_mass, const double* __restrict__ h0,
          const uint64_t seed, const uint64_t iter, double* __restrict__ accept_out, double* __restrict__ da,
          double* __restrict__ eps, const int adapt, const double target, const unsigned chain_offset) {
  const int c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (c >= C) return;
  const double p = lane < 17 ? pw[(size_t)c * 17 + lane] : 0.0;
  double v = 0.0;
  for (int j = 0; j < 17; ++j) {
    const double pj = __shfl_sync(0xffffffffu, p, j);
    if (lane < 17) v = fma(inv_mass[lane * 17 + j], pj, v);
  }
  double kin = p * v;
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) kin += __shfl_xor_sync(0xffffffffu, kin, off);
  const double h1 = -lpw[c] + 0.5 * kin;
  double dh = h0[c] - h1;
  if (!isfinite(dh)) dh = -INFINITY;
  const double acc = exp(fmin(dh, 0.0));
  const uint4 r = philox4x32_10(make_uint4(0u, (uint32_t)c + chain_offset, (uint32_t)iter, 0x41434331u),
                                make_uint2((uint32_t)seed, (uint32_t)(seed >> 32) ^ (uint32_t)(iter >> 32)));
  const bool take = (u01(r.x) - 2.3283064365386963e-10) < acc;  // u in [0, 1)
  if (take && lane < 17) {
    q[(size_t)c * 17 + lane] = qw[(size_t)c * 17 + lane];
    grad[(size_t)c * 17 + lane] = gw[(size_t)c * 17 + lane];
  }
  if (lane == 0) {
    if (take) logp[c] = lpw[c];
    accept_out[c] = acc;
    if (adapt) {  // Nesterov dual averaging of log(step size): gamma 0.05, t0 10, kappa 0.75
      double* s = da + (size_t)c * 4;
      const double t = s[3] + 1.0, eta = 1.0 / (t + 10.0);
      const double hbar = (1.0 - eta) * s[1] + eta * (target - acc);
      const double log_eps = s[0] - sqrt(t) / 0.05 * hbar;
      const double w = pow(t, -0.75);
      s[1] = hbar;
      s[2] = w * log_eps + (1.0 - w) * s[2];
      s[3] = t;
      eps[c] = exp(log_eps);
    }
  }
}

// ------------------------------------------------------------------------------------------
// k_determ
// ------------------------------------------------------------------------------------------
// STREAM: streaming (evict-first) stores.  Outputs larger than the L2 go straight to HBM (72 -> 84 %
// of the copy peak at 32 chains x 10k individuals); small outputs stay ordinary stores so that the
// consumer (the sampler's running means) finds them in L2 (8.4 us instead of 10.4 at 4 chains).
template <typename M, bool STREAM>
__global__ void __launch_bounds__(128)
k_determ(const DevCohort dc, const double* __restrict__ theta13, const int8_t* __restrict__ i_raw,
         const int8_t* __restrict__ waner, int8_t* __restrict__ out_i, double* __restrict__ out_mu_n,
         double* __restrict__ out_mu_s) {
  const int c = blockIdx.y, n = blockIdx.x * blockDim.x + threadIdx.x;
  const int G = dc.G, N = dc.N;
  __shared__ double s_th[16];
  if (threadIdx.x < 13) s_th[threadIdx.x] = theta13[(size_t)c * 13 + threadIdx.x];
  __syncthreads();
  if (n >= N) return;
  const M raw = load_column<M>(i_raw + (size_t)c * G * N + n, G, N);
  const int w = waner[(size_t)c * N + n] != 0;
  const M inf = constrain<M>(raw, reinterpret_cast<const M*>(dc.pcr)[n], dc.ch);
  const M vac = reinterpret_cast<const M*>(dc.vac)[n];
  const double rho_n = s_th[N_RHO], rho_s = w ? s_th[S_RHO] : 1.0;
  double T = 0.0, U = 0.0, Pn = 0.0, Ps = 0.0;
  for (int t = 0; t < G; ++t) {  // the recurrence of abd.py:277-293
    const int it = (int)((inf >> t) & 1), vt = (int)((vac >> t) & 1);
    T = T * rho_n + it;
    U = U * rho_s + (it + vt);
    if (it) Pn = 1.0;
    if (it | vt) Ps = 1.0;
    const size_t o = ((size_t)c * G + t) * N + n;
    const double mn = s_th[N_PERM] * Pn + s_th[N_TEMP] * T + s_th[N_INIT];
    const double ms = s_th[S_PERM] * Ps + U + s_th[S_INIT];
    if constexpr (STREAM) {
      if (out_i) __stcs(reinterpret_cast<signed char*>(out_i) + o, (signed char)it);
      if (out_mu_n) __stcs(out_mu_n + o, mn);
      if (out_mu_s) __stcs(out_mu_s + o, ms);
    } else {
      if (out_i) out_i[o] = (int8_t)it;
      if (out_mu_n) out_mu_n[o] = mn;
      if (out_mu_s) out_mu_s[o] = ms;
    }
  }
}

// Streaming posterior summaries (SURVEY 8f-2): the same recurrence, but instead of writing every
// chain's (G, N) arrays the kernel ADDS the sum over the C chains to running totals sum_i, sum_mu_n,
// sum_mu_s (G, N) -- what the consumers of the InferenceData need are posterior means
// (survival.py:68-69, timelines.py:274).  One thread per individual, chains in order (the result
// does not depend on the launch geometry); 3 x 8 G N bytes added to per 8 chains instead of 17 G N
// written per chain and then reduced by a dozen framework kernels.
template <typename M>
__global__ void __launch_bounds__(128)
k_determ_accum(const DevCohort dc, const int C, const double* __restrict__ theta, const int theta_is_q,
               const int8_t* __restrict__ i_raw, const int8_t* __restrict__ waner, double* __restrict__ sum_i,
               double* __restrict__ sum_mu_n, double* __restrict__ sum_mu_s) {
  constexpr int KC = 8;  // chains advanced together: their sum is formed in registers, in chain order
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  const int G = dc.G, N = dc.N;
  __shared__ double s_th[KC][13];
  M pcr = 0, vac = 0;
  if (n < N) {
    pcr = reinterpret_cast<const M*>(dc.pcr)[n];
    vac = reinterpret_cast<const M*>(dc.vac)[n];
  }
  for (int c0 = 0; c0 < C; c0 += KC) {
    const int nc = min(KC, C - c0);
    __syncthreads();
    if ((int)threadIdx.x < nc * 13) s_th[threadIdx.x / 13][threadIdx.x % 13] = load_param(theta, theta_is_q, c0 + threadIdx.x / 13, threadIdx.x % 13);
    __syncthreads();
    if (n >= N) continue;
    M inf[KC];
    double T[KC], U[KC], rho_s[KC];
    unsigned pn = 0, ps = 0;  // bit k: chain k has been exposed (N: infection; S: infection or vaccination)
#pragma unroll
    for (int k = 0; k < KC; ++k) {
      inf[k] = 0, T[k] = 0.0, U[k] = 0.0, rho_s[k] = 1.0;
      if (k < nc) {
        const int8_t* col = i_raw + (size_t)(c0 + k) * G * N + n;
        M raw = 0;
        for (int t = 0; t < G; ++t) raw |= (M)(__ldg(col + (size_t)t * N) != 0) << t;
        inf[k] = constrain<M>(raw, pcr, dc.ch);
        if (waner[(size_t)(c0 + k) * N + n] != 0) rho_s[k] = s_th[k][S_RHO];
      }
    }
    for (int t = 0; t < G; ++t) {
      const int vt = (int)((vac >> t) & 1);
      double si = 0.0, sn = 0.0, ss = 0.0;
#pragma unroll
      for (int k = 0; k < KC; ++k) {
        if (k < nc) {
          const int it = (int)((inf[k] >> t) & 1);
          T[k] = T[k] * s_th[k][N_RHO] + it;
          U[k] = U[k] * rho_s[k] + (it + vt);
          if (it) pn |= 1u << k;
          if (it | vt) ps |= 1u << k;
          si += it;
          sn += s_th[k][N_PERM] * (double)((pn >> k) & 1u) + s_th[k][N_TEMP] * T[k] + s_th[k][N_INIT];
          ss += s_th[k][S_PERM] * (double)((ps >> k) & 1u) + U[k] + s_th[k][S_INIT];
        }
      }
      // one reduction-add per element and launch (no other thread touches (t, n)): fire and forget,
      // and the totals do not depend on any ordering between threads
      const size_t o = (size_t)t * N + n;
      if (sum_i && si != 0.0) atomicAdd(sum_i + o, si);
      if (sum_mu_n) atomicAdd(sum_mu_n + o, sn);
      if (sum_mu_s) atomicAdd(sum_mu_s + o, ss);
    }
  }
}

// Pointwise log-likelihood of every OD row of one antigen (what PyMC records in the InferenceData's log_likelihood
// group for the observed nodes it_n_lik / it_s_lik, abd.py:459-469), written in the caller's row order.  One thread per
// (row, chain); a post-processing kernel (recorded draws only), not part of the sampling loop.
template <typename M>
__global__ void __launch_bounds__(256)
k_loglik_rows(const DevCohort dc, const int a, const int R, const double* __restrict__ theta13,
              const int8_t* __restrict__ i_raw, const int8_t* __restrict__ waner, double* __restrict__ out) {
  const int c = blockIdx.y, r = blockIdx.x * blockDim.x + threadIdx.x;
  const int G = dc.G, N = dc.N;
  __shared__ double s_th[16];
  if (threadIdx.x < 13) s_th[threadIdx.x] = theta13[(size_t)c * 13 + threadIdx.x];
  __syncthreads();
  if (r >= R) return;
  const uint32_t mt = dc.meta[a][r];
  const int n = (int)(mt >> kGapBits<M>), t = (int)(mt & kGapMask<M>);
  M raw = 0;
  const int8_t* col = i_raw + (size_t)c * G * N + n;
  for (int g = 0; g < G; ++g) raw |= (M)(col[(size_t)g * N] != 0) << g;   // (the whole column: the constraints are per chunk)
  const M inf = constrain<M>(raw, reinterpret_cast<const M*>(dc.pcr)[n], dc.ch) & low_mask<M>(t);
  const M vac = a ? (reinterpret_cast<const M*>(dc.vac)[n] & low_mask<M>(t)) : (M)0;
  const int w = waner[(size_t)c * N + n] != 0;
  const double rho = a ? (w ? s_th[S_RHO] : 1.0) : s_th[N_RHO];
  double T = 0.0;
  for (int g = 0; g <= t; ++g) T = T * rho + (double)(((inf >> g) & 1) + ((vac >> g) & 1));   // abd.py:277-293
  const double P = (inf | vac) ? 1.0 : 0.0;
  const double m = a ? s_th[S_INIT] + s_th[S_PERM] * P + T : s_th[N_INIT] + s_th[N_PERM] * P + s_th[N_TEMP] * T;
  const double b = s_th[a ? S_B : N_B], d = s_th[a ? S_D : N_D], sg = s_th[a ? S_SIGMA : N_SIGMA];
  const double pred = d / (1.0 + exp(-b * (dc.x[a][r] - m)));
  const double z = (dc.od[a][r] - pred) / sg;
  out[(size_t)c * R + dc.rowperm[a][r]] = -0.5 * z * z - kHalfLog2Pi - log(sg);
}

// int8 boundary state -> packed resident state (see PackedState): one thread per (individual, chain)
template <typename M>
__global__ void __launch_bounds__(128)
k_pack(const DevCohort dc, const int8_t* __restrict__ i_raw, const int8_t* __restrict__ waner,
       PackedState<M>* __restrict__ pack) {
  const int c = blockIdx.y, n = blockIdx.x * blockDim.x + threadIdx.x;
  const int G = dc.G, N = dc.N;
  if (n >= N) return;
  const M raw = load_column<M>(i_raw + (size_t)c * G * N + n, G, N);
  PackedState<M> ps;
  ps.inf = constrain<M>(raw, reinterpret_cast<const M*>(dc.pcr)[n], dc.ch);
  ps.rw = raw | (waner[(size_t)c * N + n] != 0 ? top_bit<M>() : (M)0);
  pack[(size_t)c * N + n] = ps;
}

// pinned host memory -> device memory by the SMs (see copy_state_h2d); n16 16-byte words + rem bytes
__global__ void __launch_bounds__(256)
k_pull(const uint4* __restrict__ src, uint4* __restrict__ dst, const size_t n16, const size_t rem) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (; i + 3 * stride < n16; i += 4 * stride) {  // four independent loads in flight per thread
    const uint4 a = src[i], b = src[i + stride], c = src[i + 2 * stride], d = src[i + 3 * stride];
    dst[i] = a, dst[i + stride] = b, dst[i + 2 * stride] = c, dst[i + 3 * stride] = d;
  }
  for (; i < n16; i += stride) dst[i] = src[i];
  if (blockIdx.x == 0 && threadIdx.x < rem)
    reinterpret_cast<uint8_t*>(dst + n16)[threadIdx.x] = reinterpret_cast<const uint8_t*>(src + n16)[threadIdx.x];
}

__global__ void k_debug_fast_math(const long long n, const double* __restrict__ z, double* __restrict__ out_exp,
                                  double* __restrict__ out_rcp) {
  __shared__ double s_tab[kExpTab];
  fill_exp_table(s_tab, threadIdx.x, blockDim.x);
  __syncthreads();
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    out_exp[i] = fast_exp(z[i], s_tab);
    out_rcp[i] = fast_rcp(1.0 + fabs(z[i]));
  }
}

}  // namespace
