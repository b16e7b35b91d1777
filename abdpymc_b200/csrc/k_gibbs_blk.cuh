// k_gibbs_blk -- ABD_GIBBS_BLOCKED: the Gibbs sweep with one EXACT block draw per time chunk.
//
// BinaryGibbsMetropolis (k_gibbs) flips one raw bit at a time.  With time chunks the constrained
// infections of a chunk are "the first raw 1 of the chunk" (abd.py:792-862), so moving an infection
// by a month takes a specific sequence of single-bit flips through unlikely states, and the
// quantities tied to the infection configuration (ab_n_temp, the rhos, the sigmas, p_waner) mix
// over hundreds of sweeps.  Here the raw bits of one chunk are redrawn TOGETHER from their exact
// full conditional given everything else -- still a Gibbs kernel on (i_raw, ab_s_waner) with the
// same stationary distribution, at the cost of about as many likelihood evaluations as a
// Metropolis sweep makes (G + number of chunks + 1 per individual):
//   * a chunk holding a PCR+ month is replaced by the PCR+ column whatever i_raw says
//     (abd.py:691-697, 722-729): its raw bits only have their Bernoulli(p) prior -> fresh draws;
//   * otherwise the chunk's state is summarised by o = position of its first raw 1 (or none):
//     P(o) ∝ p (1-p)^o exp(loglik_n | infection at o)   /   (1-p)^len exp(loglik_n | none),
//     the bits after the first 1 are marginalised (they do not enter the likelihood) and then
//     redrawn from Bernoulli(p); the bits before it are 0;
//   * ab_s_waner from its exact conditional (as ABD_GIBBS_HEATBATH).
// One warp per (chain, individual), lanes = OD rows for a likelihood evaluation, lanes = options
// for the constraint step and the categorical draw.  G <= 31 and >= 2 chunks (the one-chunk model
// has no "first 1" structure: abd.py:640-649); the host routes everything else to k_gibbs.
#pragma once
#include "k_gibbs.cuh"

namespace {
using namespace abd;

__global__ void __launch_bounds__(kGibbsWarps * 32, ABD_GIBBS_MINB)
k_gibbs_blk(const DevCohort dc, const int* __restrict__ order, const int C,
            const double* __restrict__ theta, const int theta_is_q,
            const double* __restrict__ p_arr, const double* __restrict__ pw_arr,
            int8_t* __restrict__ i_raw, int8_t* __restrict__ waner, PackedState<uint32_t>* __restrict__ pack,
            unsigned* __restrict__ queue, const GibbsCfg cfg) {
  using M = uint32_t;
  constexpr unsigned FULL = 0xffffffffu;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int G = dc.G, N = dc.N;

  __shared__ double s_tab[kExpTab];
  __shared__ double s_th_all[kGibbsWarps][24];            // see gibbs_load_chain
  __shared__ double s_pw_all[kGibbsWarps][3][kGapTab<M>];   // rho_n^k, rho_s^k, ones
  double* s_th = s_th_all[warp];
  const double (*s_pw)[kGapTab<M>] = s_pw_all[warp];

  fill_exp_table(s_tab, tid, kGibbsWarps * 32);
  for (int k = lane; k < kGapTab<M>; k += 32) s_pw_all[warp][2][k] = 1.0;
  __syncthreads();

  ChainQueues q(queue, cfg.stats, C, N, blockIdx.x * kGibbsWarps + warp);
  while (true) {
    int c;
    unsigned item;
    if (!q.claim(lane, c, item)) {
      if (q.done()) break;
      continue;
    }
    const int n = order[item];
    if (q.enter(c, lane)) gibbs_load_chain(theta, theta_is_q, p_arr, pw_arr, c, G, lane, s_th, s_pw_all[warp]);

    // ---- this individual's state, masks, rows ----
    const M pcr = reinterpret_cast<const M*>(dc.pcr)[n];
    M raw, inf;
    int w;
    int8_t* col = i_raw + (size_t)c * G * N + n;
    warp_load_state<M>(dc, pack, col, waner, c, n, pcr, lane, raw, inf, w);
    const M raw_in = raw;
    const int w_in = w;
    const M vac = reinterpret_cast<const M*>(dc.vac)[n];
    GibbsRows<M> rows(dc, n, lane, s_th, s_pw, s_tab);
    const int t_last = rows.t_last, t_last_s = rows.t_last_s;
    rows.set_w(vac, w);
    auto indiv_ll = [&](M inf_, int w_) { return rows.ll(inf_, vac, w_); };

    double ll = indiv_ll(inf, w);

    // ---- random numbers: lane t: fresh Bernoulli(p) draw for gap t (x), categorical uniform of
    //      chunk t (y), waner uniform (lane 0, z) ----
    const uint4 rnd = philox4x32_10(
        make_uint4((uint32_t)lane, (uint32_t)n + dc.ind_offset, (uint32_t)c + dc.chain_offset, (uint32_t)cfg.sweep),
        make_uint2((uint32_t)cfg.seed, (uint32_t)(cfg.seed >> 32) ^ (uint32_t)(cfg.sweep >> 32)));
    const double pv = s_th[TH_P], lp1 = s_th[TH_LOG_P], lp0 = s_th[TH_LOG1M_P];
    const M fresh = __ballot_sync(FULL, lane < G && u01(rnd.x) <= pv);
    const double u_cat = u01(rnd.y);

    for (int k = 0; k < dc.ch.n; ++k) {
      const M cm = (M)dc.ch.mask[k];
      if (cm == 0) continue;
      ++q.n_prop;
      if (pcr & cm) {  // the chunk is the PCR+ column: its raw bits are free
        raw = (raw & ~cm) | (fresh & cm);
        continue;
      }
      const int c0 = ctz(cm), len = popc(cm);  // options o < len: first raw 1 at gap c0 + o; o == len: none
      const M base = raw & ~cm;
      const M inf_own = constrain<M>(base | ((lane < len) ? ((M)1 << (c0 + lane)) : (M)0), pcr, dc.ch);
      const M inf_none = __shfl_sync(FULL, inf_own, len);
      const double ll_none = (inf_none == inf) ? ll : indiv_ll(inf_none, w);
      const double llv = chunk_options_ll<M>(inf_own, len, inf_none, ll_none, inf, w, ll, t_last, lane, indiv_ll);
      // categorical draw over the len + 1 options: inclusive scan of exp(log weight - max)
      double lw = (lane < len) ? llv + (double)lane * lp0 + lp1 : llv + (double)len * lp0;
      if (lane > len || !(lw == lw)) lw = -INFINITY;
      double mx = lw;
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) mx = fmax(mx, __shfl_xor_sync(FULL, mx, off));
      double cum = (lane <= len) ? exp(lw - mx) : 0.0;
#pragma unroll
      for (int off = 1; off < 32; off <<= 1) {
        const double up = __shfl_up_sync(FULL, cum, off);
        if (lane >= off) cum += up;
      }
      const double thr = __shfl_sync(FULL, u_cat, k) * __shfl_sync(FULL, cum, len);
      int pick = popc(__ballot_sync(FULL, lane < len && cum < thr));  // in [0, len]
      if (!(mx > -INFINITY)) pick = len;  // every option impossible (NaN parameters): keep "none"
      const M old_first = (raw & cm) & (~(raw & cm) + 1);
      M newbits = 0;
      if (pick < len) {
        const M bit = (M)1 << (c0 + pick);
        newbits = bit | (fresh & cm & ~((bit << 1) - 1));
      }
      const M new_first = newbits & (~newbits + 1);
      if (new_first != old_first) ++q.n_acc;
      raw = base | newbits;
      inf = __shfl_sync(FULL, inf_own, pick);
      ll = __shfl_sync(FULL, llv, pick);
    }

    // ---- waner: exact conditional ----
    {
      ++q.n_prop;
      double d10, ll2;
      waner_logodds<M>(inf, vac, w, ll, t_last_s, s_th, indiv_ll, d10, ll2);
      const double p1 = 1.0 / (1.0 + exp(-d10));
      const int w_new = (__shfl_sync(FULL, u01(rnd.z), 0) <= p1) ? 1 : 0;
      if (w_new != w) {
        w = w_new;
        rows.set_w(vac, w);
        ll = ll2;
        ++q.n_acc;
      }
    }

    warp_store_state<M>(dc, pack, col, waner, c, n, lane, raw, raw_in, w, w_in, inf);
  }
  q.flush(lane);
}

}  // namespace
