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

  unsigned n_prop = 0, n_acc = 0;
  int cur_c = -1;

  // One work queue per chain (individuals by decreasing OD-row count); a warp starts at the chain its global index
  // points to and moves on when that queue is empty, so it (re)loads chain parameters once or twice per sweep instead
  // of once per chain (a single chain-major queue walked every warp through all C chains: ~6 % of the sweep's instructions).
  int cq = (int)((blockIdx.x * kGibbsWarps + warp) % (unsigned)C), exhausted = 0;
  while (true) {
    unsigned item = 0;
    if (lane == 0) item = atomicAdd(queue + cq, 1u);
    item = __shfl_sync(FULL, item, 0);
    if (item >= (unsigned)N) {
      if (++exhausted >= C) break;
      cq = (cq + 1 == C) ? 0 : cq + 1;
      continue;
    }
    exhausted = 0;
    const int c = cq;
    const int n = order[item];

    if (c != cur_c) {  // (re)load this chain's parameters into the warp's shared-memory slot
      if (cur_c >= 0 && cfg.stats && lane == 0) {
        atomicAdd(&cfg.stats[(size_t)cur_c * 2], (unsigned long long)n_prop);
        atomicAdd(&cfg.stats[(size_t)cur_c * 2 + 1], (unsigned long long)n_acc);
      }
      n_prop = n_acc = 0;
      cur_c = c;
      gibbs_load_chain(theta, theta_is_q, p_arr, pw_arr, c, G, lane, s_th, s_pw_all[warp]);
    }

    // ---- this individual's column of i_raw (lane t reads gap t), waner, masks, rows ----
    int8_t* col = i_raw + (size_t)c * G * N + n;
    const M pcr = reinterpret_cast<const M*>(dc.pcr)[n];
    M raw, inf;
    int w;
    if (pack) {  // resident state: one broadcast load, constraints already applied
      const PackedState<M> ps = pack[(size_t)c * N + n];
      raw = ps.rw & ~top_bit<M>();
      w = (ps.rw & top_bit<M>()) != 0;
      inf = ps.inf;
    } else {
      const int8_t b0 = (lane < G) ? col[(size_t)lane * N] : (int8_t)0;
      raw = __ballot_sync(FULL, b0 != 0);
      w = waner[(size_t)c * N + n] != 0;
      inf = constrain<M>(raw, pcr, dc.ch);
    }
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
    const double pv = s_th[21], lp1 = s_th[19], lp0 = s_th[20];
    const M fresh = __ballot_sync(FULL, lane < G && u01(rnd.x) <= pv);
    const double u_cat = u01(rnd.y);

    for (int k = 0; k < dc.ch.n; ++k) {
      const M cm = (M)dc.ch.mask[k];
      if (cm == 0) continue;
      ++n_prop;
      if (pcr & cm) {  // the chunk is the PCR+ column: its raw bits are free
        raw = (raw & ~cm) | (fresh & cm);
        continue;
      }
      const int c0 = ctz(cm), len = popc(cm);  // options o < len: first raw 1 at gap c0 + o; o == len: none
      const M base = raw & ~cm;
      const M inf_own = constrain<M>(base | ((lane < len) ? ((M)1 << (c0 + lane)) : (M)0), pcr, dc.ch);
      const M inf_none = __shfl_sync(FULL, inf_own, len);
      const double ll_none = (inf_none == inf) ? ll : indiv_ll(inf_none, w);
      double llv = ll_none;  // lane o: log-likelihood under option o
      for (int o = 0; o < len; ++o) {
        const M io = __shfl_sync(FULL, inf_own, o);
        const M diff = io ^ inf_none;
        if (diff != 0 && ctz(diff) <= t_last) {  // otherwise the data cannot tell it from "none"
          const double v = (io == inf) ? ll : indiv_ll(io, w);
          if (lane == o) llv = v;
        }
      }
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
      if (new_first != old_first) ++n_acc;
      raw = base | newbits;
      inf = __shfl_sync(FULL, inf_own, pick);
      ll = __shfl_sync(FULL, llv, pick);
    }

    // ---- waner: exact conditional ----
    {
      ++n_prop;
      const M ex = inf | vac;
      const bool affected = ex != 0 && ctz(ex | top_bit<M>()) < t_last_s;
      double d10 = s_th[16], ll2 = ll;
      if (affected) {
        ll2 = indiv_ll(inf, w ^ 1);
        d10 += w ? (ll - ll2) : (ll2 - ll);  // log-odds of 1 versus 0
      }
      const double p1 = 1.0 / (1.0 + exp(-d10));
      const int w_new = (__shfl_sync(FULL, u01(rnd.z), 0) <= p1) ? 1 : 0;
      if (w_new != w) {
        w = w_new;
        rows.set_w(vac, w);
        ll = ll2;
        ++n_acc;
      }
    }

    {  // write back only what changed
      const M changed = raw ^ raw_in;
      if (lane < G && ((changed >> lane) & 1)) col[(size_t)lane * N] = (int8_t)((raw >> lane) & 1);
      if (lane == 0 && w != w_in) waner[(size_t)c * N + n] = (int8_t)w;
      if (pack && lane == 0 && (changed != 0 || w != w_in)) {
        PackedState<M> ps;
        ps.rw = raw | (w ? top_bit<M>() : (M)0);
        ps.inf = inf;
        pack[(size_t)c * N + n] = ps;
      }
    }
  }
  if (cfg.stats && lane == 0 && cur_c >= 0) {
    atomicAdd(&cfg.stats[(size_t)cur_c * 2], (unsigned long long)n_prop);
    atomicAdd(&cfg.stats[(size_t)cur_c * 2 + 1], (unsigned long long)n_acc);
  }
}

}  // namespace
