// k_infprob_accum -- Rao-Blackwellised posterior infection and waner probabilities (DESIGN.md section 4).
//
// For one recorded state of each chain (theta13, p, p_w from q17, i_raw, waner) the kernel adds, per (gap, individual),
// the exact conditional probability that the constrained infection i[t, n] (abd.py:640-667) is 1 given everything
// outside the block that holds it, and per individual the exact conditional probability of ab_s_waner[n] = 1.
// Averaged over the recorded draws these estimate the same posterior means as the average of the 0/1 draws of i and
// ab_s_waner (E_pi[E[f | rest]] = E_pi[f]) without the per-draw Bernoulli noise.  Every term conditions on the same
// state; nothing is updated, no random number is drawn.  L_n below is individual n's data log-likelihood (both antigens).
//   * time chunks (>= 2 chunks), chunk k = gaps [c0, c0 + len):
//       - a chunk holding a PCR+ month: its constrained bits do not depend on its raw bits -> constrain(current)[t];
//       - otherwise option o < len = "first raw 1 at c0 + o", o = len = "none"; base = raw with the chunk cleared;
//         log w_o = o log(1-p) + log p + L_n(constrain(base | bit c0+o)), log w_len = len log(1-p) + L_n(constrain(base));
//         gap c0 + o gets w_o bit_{c0+o}(constrain(base | bit c0+o)) / sum w  (the 3-gap rule may clear the bit);
//   * one chunk (no splits): bit by bit, E[i_t | raw_-t] = sum_b P(raw_t = b | rest) constrain(raw, raw_t = b)[t];
//   * waner: sigmoid(logit p_w + L_n(w = 1) - L_n(w = 0)), p_w when no S row follows the first exposure.
// A log-likelihood that is NaN counts as -inf; when every option of a block has weight zero the block contributes the
// current state's value (k_gibbs_blk then keeps "none").  Options whose constrained column equals the current one, or
// differs from "none" only after the individual's last sample, reuse that likelihood (k_gibbs_blk's t_last shortcut).
//
// Layout: a CTA of kGibbsWarps warps takes kGibbsWarps consecutive individuals of `order` (decreasing row count, so
// the warps of a CTA have similar work), one warp each, and walks the chains in order; warp 0 loads each chain's
// parameters into shared memory once for the CTA.  Lanes are OD rows during a likelihood pass (GibbsRows) and options
// during the weighting.  Chunks longer than 32 gaps (64- and 128-bit masks) are weighted in groups of 32 options with
// an online log-sum-exp; a lane owns sizeof(M) / 4 gap slots (accumulators and option weights), selected by unrolled
// compares, never by a dynamic index (DESIGN.md section 4: that would put the arrays in local memory).  The sum over
// the chains is formed in registers in chain order and added with one reduction-add per (gap, individual) and per
// individual, so the totals do not depend on the launch geometry or on timing.
#pragma once
#include "k_gibbs.cuh"

namespace {
using namespace abd;

template <int NS>
__device__ __forceinline__ void slot_add(double (&acc)[NS], int s, double v) {
#pragma unroll
  for (int k = 0; k < NS; ++k)
    if (k == s) acc[k] += v;
}

template <typename M>
__global__ void __launch_bounds__(kGibbsWarps * 32)
k_infprob_accum(const DevCohort dc, const int* __restrict__ order, const int C, const double* __restrict__ q17,
                const int8_t* __restrict__ i_raw, const int8_t* __restrict__ waner, const PackedState<M>* __restrict__ pack,
                double* __restrict__ sum_i, double* __restrict__ sum_w) {
  constexpr int NSLOT = sizeof(M) / 4;  // gap slots (and groups of 32 options) per lane
  constexpr unsigned FULL = 0xffffffffu;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int G = dc.G, N = dc.N;

  __shared__ double s_tab[kExpTab];
  __shared__ double s_th[24];                 // see gibbs_load_chain
  __shared__ double s_pw[3][kGapTab<M>];      // rho_n^k, rho_s^k, ones
  fill_exp_table(s_tab, tid, kGibbsWarps * 32);
  for (int k = tid; k < kGapTab<M>; k += kGibbsWarps * 32) s_pw[2][k] = 1.0;

  const int item = blockIdx.x * kGibbsWarps + warp;
  const bool active = item < N;
  const int n = active ? order[item] : 0;
  const M pcr = active ? reinterpret_cast<const M*>(dc.pcr)[n] : (M)0;
  const M vac = active ? reinterpret_cast<const M*>(dc.vac)[n] : (M)0;

  double acc[NSLOT];  // lane l, slot s: gap 32 s + l, summed over the chains in order
#pragma unroll
  for (int s = 0; s < NSLOT; ++s) acc[s] = 0.0;
  double acc_w = 0.0;

  for (int c = 0; c < C; ++c) {
    __syncthreads();  // every warp is done with the previous chain's parameters
    if (warp == 0) gibbs_load_chain<M>(q17, 1, nullptr, nullptr, c, G, lane, s_th, s_pw);
    __syncthreads();
    if (!active) continue;

    M raw, inf;
    int w;
    warp_load_state<M>(dc, pack, i_raw + (size_t)c * G * N + n, waner, c, n, pcr, lane, raw, inf, w);
    GibbsRows<M> rows(dc, n, lane, s_th, s_pw, s_tab);
    const int t_last = rows.t_last;
    rows.set_w(vac, w);
    auto indiv_ll = [&](M inf_, int w_) {
      const double v = rows.ll(inf_, vac, w_);
      return (v == v) ? v : -INFINITY;
    };
    const double ll = indiv_ll(inf, w);

    if (dc.ch.n < 2) {
      // ---- one chunk: the two values of each raw bit, the rest fixed ----
      M alt_own[NSLOT];  // constrained infections with the lane's raw bit flipped
#pragma unroll
      for (int s = 0; s < NSLOT; ++s) {
        const int t = lane + 32 * s;
        alt_own[s] = (t < G) ? constrain<M>(raw ^ ((M)1 << t), pcr, dc.ch) : inf;
      }
      for (int t = 0; t < G; ++t) {
        const M alt = shfl_mask(slot(alt_own, t >> 5), t & 31);
        const M diff = alt ^ inf;
        const double ll_alt = (diff != 0 && ctz(diff) <= t_last) ? indiv_ll(alt, w) : ll;
        const bool cur = (raw >> t) & 1;
        const M inf1 = cur ? inf : alt, inf0 = cur ? alt : inf;
        const int b1 = (int)((inf1 >> t) & 1), b0 = (int)((inf0 >> t) & 1);
        double v = (double)b1;
        if (b1 != b0) {
          const double d = s_th[TH_LOGIT_P] + (cur ? ll - ll_alt : ll_alt - ll);  // log-odds of raw_t = 1 versus 0
          const double p1 = 1.0 / (1.0 + exp(-d));
          v = (p1 == p1) ? (b1 ? p1 : 1.0 - p1) : (double)((inf >> t) & 1);
        }
        if (lane == (t & 31)) slot_add(acc, t >> 5, v);
      }
    } else {
      // ---- time chunks: the position of the chunk's first raw 1, or none ----
      const double lp1 = s_th[TH_LOG_P], lp0 = s_th[TH_LOG1M_P];
      for (int k = 0; k < dc.ch.n; ++k) {
        const M cm = chunk_mask<M>(dc.ch, k);
        if (cm == 0) continue;
        if (pcr & cm) {  // the chunk is the PCR+ column whatever its raw bits
#pragma unroll
          for (int s = 0; s < NSLOT; ++s) {
            const int t = lane + 32 * s;
            if (t < G && ((cm >> t) & 1)) acc[s] += (double)((inf >> t) & 1);
          }
          continue;
        }
        const int c0 = ctz(cm), len = popc(cm);
        const M base = raw & ~cm;
        const M inf_none = constrain<M>(base, pcr, dc.ch);
        const double ll_none = (inf_none == inf) ? ll : indiv_ll(inf_none, w);
        double mx = ll_none + (double)len * lp0;  // running maximum of the log weights ...
        if (!(mx == mx)) mx = -INFINITY;
        double S = (mx > -INFINITY) ? 1.0 : 0.0;  // ... and sum of exp(log weight - mx)
        double num[NSLOT];  // lane l, group g: log weight of option 32 g + l if it infects its gap, else -inf
#pragma unroll
        for (int g = 0; g < NSLOT; ++g) {
          num[g] = -INFINITY;
          if (32 * g >= len) continue;
          const int o_own = 32 * g + lane;
          const M inf_own = (o_own < len) ? constrain<M>(base | ((M)1 << (c0 + o_own)), pcr, dc.ch) : inf_none;
          const double llv =
              chunk_options_ll<M>(inf_own, min(32, len - 32 * g), inf_none, ll_none, inf, w, ll, t_last, lane, indiv_ll);
          double lw = (o_own < len) ? llv + (double)o_own * lp0 + lp1 : -INFINITY;
          if (!(lw == lw)) lw = -INFINITY;
          double gm = lw;
#pragma unroll
          for (int off = 16; off > 0; off >>= 1) gm = fmax(gm, __shfl_xor_sync(FULL, gm, off));
          const double m_new = fmax(mx, gm);
          if (m_new > -INFINITY) {
            double e = exp(lw - m_new);
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) e += __shfl_xor_sync(FULL, e, off);
            S = S * exp(mx - m_new) + e;
            mx = m_new;
          }
          if (o_own < len && ((inf_own >> (c0 + o_own)) & 1)) num[g] = lw;
        }
        // gap c0 + o lives in lane (c0 + o) & 31: every lane takes option 32 g + ((lane - c0) & 31) of each group
        const bool ok = mx > -INFINITY;
        const int src = (lane - c0) & 31;
#pragma unroll
        for (int g = 0; g < NSLOT; ++g) {
          if (32 * g >= len) continue;
          const double v = __shfl_sync(FULL, num[g], src);
          const int o = 32 * g + src;
          if (o < len) {
            const int t = c0 + o;
            slot_add(acc, t >> 5, ok ? exp(v - mx) / S : (double)((inf >> t) & 1));
          }
        }
      }
    }

    // ---- waner ----
    {
      double d10, ll2, p1 = s_th[TH_SIG_PW];
      if (waner_logodds<M>(inf, vac, w, ll, rows.t_last_s, s_th, indiv_ll, d10, ll2)) {
        p1 = 1.0 / (1.0 + exp(-d10));
        if (!(p1 == p1)) p1 = (double)w;
      }
      acc_w += p1;
    }
  }

  if (active) {
#pragma unroll
    for (int s = 0; s < NSLOT; ++s) {
      const int t = lane + 32 * s;
      if (t < G) atomicAdd(sum_i + (size_t)t * N + n, acc[s]);
    }
    if (lane == 0) atomicAdd(sum_w + n, acc_w);
  }
}

}  // namespace
