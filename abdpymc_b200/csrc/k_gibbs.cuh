// k_gibbs -- the Gibbs sweep over i_raw / waner (one warp per (chain, individual)).
#pragma once
#include "abd_kernels_common.cuh"

namespace {
using namespace abd;

// ------------------------------------------------------------------------------------------
// k_gibbs
// ------------------------------------------------------------------------------------------
struct GibbsCfg {
  uint64_t seed, sweep;
  int mode;          // ABD_GIBBS_*; -1 = conditional log-odds only (no update, no RNG)
  double transit_p;
  double* out_i;     // [C][G][N] (mode -1)
  double* out_w;     // [C][N]
  unsigned long long* stats;  // [C][2] proposals, accepted flips (may be null)
};

// One OD row of one individual under a candidate state (value only, times -1/(2 sigma^2)).
// N and S rows share one code path: lanes differ only in their per-lane parameters.
struct RowPar {
  double init, perm, tfac, b, d, nh;
};
template <typename M>
__device__ __forceinline__ double gibbs_row(double x, double od, int t, bool is_s, M inf, M vac, int w,
                                            const RowPar& rp, const double (*s_pw)[kGapTab<M>],
                                            const double* __restrict__ s_tab) {
  const M lm = low_mask<M>(t);
  M e = inf & lm, v = is_s ? (vac & lm) : (M)0;
  const double P = (e | v) ? rp.perm : 0.0;
  const double* pw = is_s ? (w ? s_pw[1] : s_pw[2]) : s_pw[0];  // s_pw[2] = all ones (rho_ind = 1)
  double T = 0.0;
  while (e) {
    T += pw[t - ctz(e)];
    e &= e - 1;
  }
  while (v) {
    T += pw[t - ctz(v)];
    v &= v - 1;
  }
  return rp.nh * row_resid2(x, od, fma(rp.tfac, T, rp.init + P), rp.b, rp.d, s_tab);
}

// The vaccinations' share of an S row's decaying response, sum_{s in vac, s <= t} rho_ind^(t - s): it only changes with
// ab_s_waner, so a lane keeps it for its row instead of re-summing it in every candidate evaluation.
template <typename M>
__device__ __forceinline__ double gibbs_vac_sum(int t, M vac, int w, const double (*s_pw)[kGapTab<M>]) {
  M v = vac & low_mask<M>(t);
  const double* pw = w ? s_pw[1] : s_pw[2];
  double T = 0.0;
  while (v) {
    T += pw[t - ctz(v)];
    v &= v - 1;
  }
  return T;
}
// gibbs_row with the vaccinations' share handed in (tv; any_v: a vaccination at or before t)
template <typename M>
__device__ __forceinline__ double gibbs_row_tv(double x, double od, int t, bool is_s, M inf, double tv, bool any_v, int w,
                                               const RowPar& rp, const double (*s_pw)[kGapTab<M>],
                                               const double* __restrict__ s_tab) {
  M e = inf & low_mask<M>(t);
  const double P = (e != 0 || any_v) ? rp.perm : 0.0;
  const double* pw = is_s ? (w ? s_pw[1] : s_pw[2]) : s_pw[0];  // s_pw[2] = all ones (rho_ind = 1)
  double T = tv;
  while (e) {
    T += pw[t - ctz(e)];
    e &= e - 1;
  }
  return rp.nh * row_resid2(x, od, fma(rp.tfac, T, rp.init + P), rp.b, rp.d, s_tab);
}

// One chain's parameters into a warp's shared-memory slot (all 32 lanes call it):
//   s_th[0..12] theta13, [13], [14] -1/(2 sigma^2) of N / S, [15], [16] logit p / p_waner,
//   [17], [18] sigmoid of those, [19], [20], [21] log p, log(1 - p), p; s_pw[0] = rho_n^k, s_pw[1] = rho_s^k.
__device__ __forceinline__ void gibbs_load_chain(const double* __restrict__ theta, int theta_is_q,
                                                 const double* __restrict__ p_arr, const double* __restrict__ pw_arr,
                                                 int c, int G, int lane, double* s_th, double (*s_pw)[kGapTab<uint32_t>]) {
  __syncwarp();
  fill_pow_warp(load_param(theta, theta_is_q, c, N_RHO), G, lane, s_pw[0], nullptr);
  fill_pow_warp(load_param(theta, theta_is_q, c, S_RHO), G, lane, s_pw[1], nullptr);
  if (lane < 13) s_th[lane] = load_param(theta, theta_is_q, c, lane);
  if (lane == 13 || lane == 14) {
    const double sg = load_param(theta, theta_is_q, c, lane == 13 ? N_SIGMA : S_SIGMA);
    s_th[lane] = -0.5 / (sg * sg);
  }
  if (lane == 15 || lane == 16) {
    const int which = lane - 15;
    double lo, pv;
    if (theta_is_q) {  // logit of a logodds-transformed value is the value itself
      lo = theta[(size_t)c * 17 + (which ? kQ_PW : kQ_P)];
      pv = 1.0 / (1.0 + exp(-lo));
    } else {
      pv = which ? pw_arr[c] : p_arr[c];
      lo = log(pv) - log1p(-pv);
    }
    s_th[lane] = lo;
    s_th[lane + 2] = 1.0 / (1.0 + exp(-lo));  // the heat-bath threshold of a prior-only bit: sigmoid(logit)
    if (!which) {
      s_th[19] = log(pv);
      s_th[20] = log1p(-pv);
      s_th[21] = pv;
    }
  }
  __syncwarp();
}

// The OD rows of one individual as a warp holds them: lane l keeps row l (N rows first, then S
// rows) in registers, rows beyond 32 are read again in every pass; ll() is the individual's
// log-likelihood under a candidate state (butterfly sum: every lane gets the total).
template <typename M>
struct GibbsRows {
  const DevCohort& dc;
  const double* s_th;
  const double (*s_pw)[kGapTab<M>];
  const double* s_tab;
  int lane, rn0, cnt_n, rs0, cnt_s, nrows;
  double x0, od0;
  int t0;
  bool s0;
  RowPar rp0;
  int w_cur;       // the waner state tv0 was summed for
  double tv0;      // the vaccinations' share of the lane's own row (S rows; 0 for N rows)
  bool anyv0;
  M vac_own;
  int t_last, t_last_s;  // latest sampled gap of either antigen / of the S antigen (rows are sorted by gap)

  __device__ __forceinline__ GibbsRows(const DevCohort& dc_, int n, int lane_, const double* s_th_,
                                       const double (*s_pw_)[kGapTab<M>], const double* s_tab_)
      : dc(dc_), s_th(s_th_), s_pw(s_pw_), s_tab(s_tab_), lane(lane_) {
    rn0 = dc.rp[0][n], cnt_n = dc.rp[0][n + 1] - rn0;
    rs0 = dc.rp[1][n], cnt_s = dc.rp[1][n + 1] - rs0;
    nrows = cnt_n + cnt_s;
    load_row(lane, x0, od0, t0, s0);
    rp0 = row_par(s0);
    t_last = t0, t_last_s = s0 ? t0 : -1;
    for (int l = lane + 32; l < nrows; l += 32) {
      const bool is_s = l >= cnt_n;
      const int r = is_s ? rs0 + (l - cnt_n) : rn0 + l;
      const int t = (int)((is_s ? dc.meta[1] : dc.meta[0])[r] & kGapMask<M>);
      t_last = max(t_last, t);
      if (is_s) t_last_s = max(t_last_s, t);
    }
    t_last = __reduce_max_sync(0xffffffffu, t_last);
    t_last_s = __reduce_max_sync(0xffffffffu, t_last_s);
    w_cur = -1, tv0 = 0.0, anyv0 = false, vac_own = 0;
  }
  // (re)sum the vaccinations' share of the lane's own row for waner state w
  __device__ __forceinline__ void set_w(M vac, int w) {
    vac_own = (t0 >= 0 && s0) ? (vac & low_mask<M>(t0)) : (M)0;
    anyv0 = vac_own != 0;
    tv0 = anyv0 ? gibbs_vac_sum<M>(t0, vac_own, w, s_pw) : 0.0;
    w_cur = w;
  }
  __device__ __forceinline__ void load_row(int l, double& x, double& od, int& t, bool& is_s) const {
    is_s = l >= cnt_n;
    const int r = is_s ? rs0 + (l - cnt_n) : rn0 + l;
    if (l < nrows) {
      x = (is_s ? dc.x[1] : dc.x[0])[r];
      od = (is_s ? dc.od[1] : dc.od[0])[r];
      t = (int)((is_s ? dc.meta[1] : dc.meta[0])[r] & kGapMask<M>);
    } else {
      x = 0.0;
      od = 0.0;
      t = -1;
    }
  }
  __device__ __forceinline__ RowPar row_par(bool is_s) const {
    RowPar rp;
    rp.init = s_th[is_s ? S_INIT : N_INIT];
    rp.perm = s_th[is_s ? S_PERM : N_PERM];
    rp.tfac = is_s ? 1.0 : s_th[N_TEMP];
    rp.b = s_th[is_s ? S_B : N_B];
    rp.d = s_th[is_s ? S_D : N_D];
    rp.nh = s_th[is_s ? 14 : 13];
    return rp;
  }
  __device__ __forceinline__ double ll(M inf_, M vac, int w_) const {
    double a = 0.0;
    if (t0 >= 0) {
      const double tv = (w_ == w_cur || !anyv0) ? tv0 : gibbs_vac_sum<M>(t0, vac_own, w_, s_pw);
      a = gibbs_row_tv<M>(x0, od0, t0, s0, inf_, tv, anyv0, w_, rp0, s_pw, s_tab);
    }
    for (int l = lane + 32; l < nrows; l += 32) {  // individuals with more than 32 rows
      double x, od;
      int t;
      bool is_s;
      load_row(l, x, od, t, is_s);
      a += gibbs_row<M>(x, od, t, is_s, inf_, vac, w_, row_par(is_s), s_pw, s_tab);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) a += __shfl_xor_sync(0xffffffffu, a, off);
    return a;
  }
};

// a[i] of a per-lane array of proposal slots (i uniform over the warp), by selects: a dynamic index would put the
// array in local memory
template <int NS, typename T>
__device__ __forceinline__ T slot(const T (&a)[NS], int i) {
  if constexpr (NS <= 2) {
    return (NS > 1 && i) ? a[NS - 1] : a[0];
  } else {
    T v = a[0];
#pragma unroll
    for (int s = 1; s < NS; ++s) v = (i == s) ? a[s] : v;
    return v;
  }
}

// (k_gibbs below keeps its own hand-inlined copy of these two: going through the helpers costs it
// 4 % -- 274 instead of 264 us per sweep, a few more spilled registers under its 64-register cap.)
// Persistent warps: every warp repeatedly claims the next (chain, individual) from a global
// counter.  Items are ordered chain-major and, inside a chain, by decreasing OD-row count
// (longest job first), so the tail at the end of the launch is one short job.
// 4 CTAs/SM (64 registers, a few spills) is 3 % faster than 3 x 80 registers; 5 is slower.  Also
// measured and dropped: patching each row's decaying response for a candidate instead of summing
// it again (no gain: the extra live registers cost what the shorter loops save).
template <typename M>
__global__ void __launch_bounds__(kGibbsWarps * 32, kGibbsMinB<M>)
k_gibbs(const DevCohort dc, const int* __restrict__ order, const int C,
        const double* __restrict__ theta, const int theta_is_q,
        const double* __restrict__ p_arr, const double* __restrict__ pw_arr,
        int8_t* __restrict__ i_raw, int8_t* __restrict__ waner, PackedState<M>* __restrict__ pack,
        unsigned* __restrict__ queue, const GibbsCfg cfg) {
  constexpr int NSLOT = sizeof(M) / 4;  // proposals owned per lane
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int G = dc.G, N = dc.N;

  __shared__ double s_tab[kExpTab];
  __shared__ double s_th_all[kGibbsWarps][20];            // theta13, -1/(2 sigma^2) x 2, logit p / p_w, p / p_w
  __shared__ double s_pw_all[kGibbsWarps][3][kGapTab<M>];   // rho_n^k, rho_s^k, ones
  __shared__ unsigned char s_ord[kGibbsWarps][kGapTab<M>];
  double* s_th = s_th_all[warp];
  const double (*s_pw)[kGapTab<M>] = s_pw_all[warp];

  fill_exp_table(s_tab, tid, kGibbsWarps * 32);
  for (int k = lane; k < kGapTab<M>; k += 32) s_pw_all[warp][2][k] = 1.0;
  __syncthreads();

  const int nprop = G + 1;  // proposal j < G flips i_raw[j, n]; j == G flips waner[n]
  unsigned n_prop = 0, n_acc = 0;
  int cur_c = -1;

  // One work queue per chain (individuals by decreasing OD-row count); a warp starts at the chain its global index
  // points to and moves on when that queue is empty, so it (re)loads chain parameters once or twice per sweep instead
  // of once per chain (a single chain-major queue walked every warp through all C chains: ~6 % of the sweep's instructions).
  int cq = (int)((blockIdx.x * kGibbsWarps + warp) % (unsigned)C), exhausted = 0;
  while (true) {
    unsigned item = 0;
    if (lane == 0) item = atomicAdd(queue + cq, 1u);
    item = __shfl_sync(0xffffffffu, item, 0);
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
      __syncwarp();
      fill_pow_warp(load_param(theta, theta_is_q, c, N_RHO), G, lane, s_pw_all[warp][0], nullptr);
      fill_pow_warp(load_param(theta, theta_is_q, c, S_RHO), G, lane, s_pw_all[warp][1], nullptr);
      if (lane < 13) s_th[lane] = load_param(theta, theta_is_q, c, lane);
      if (lane == 13 || lane == 14) {
        const double sg = load_param(theta, theta_is_q, c, lane == 13 ? N_SIGMA : S_SIGMA);
        s_th[lane] = -0.5 / (sg * sg);
      }
      if (lane == 15 || lane == 16) {
        const int which = lane - 15;
        double lo;
        if (theta_is_q) {  // logit of a logodds-transformed value is the value itself
          lo = theta[(size_t)c * 17 + (which ? kQ_PW : kQ_P)];
        } else {
          const double p = which ? pw_arr[c] : p_arr[c];
          lo = log(p) - log1p(-p);
        }
        s_th[lane] = lo;
        s_th[lane + 2] = 1.0 / (1.0 + exp(-lo));
      }
      __syncwarp();
    }

    // ---- this individual's column of i_raw (lane t reads gap t), waner, masks, rows ----
    int8_t* col = i_raw + (size_t)c * G * N + n;
    const M pcr = reinterpret_cast<const M*>(dc.pcr)[n];
    M raw = 0, inf;
    int w;
    if (pack) {  // resident state: one broadcast load instead of G strided bytes, constraints already applied
      const PackedState<M> ps = pack[(size_t)c * N + n];
      raw = ps.rw & ~top_bit<M>();
      w = (ps.rw & top_bit<M>()) != 0;
      inf = ps.inf;
    } else {
#pragma unroll
      for (int sl = 0; sl < NSLOT; ++sl) {
        const int t = lane + 32 * sl;
        const int8_t b = (t < G) ? col[(size_t)t * N] : (int8_t)0;
        raw |= (M)__ballot_sync(0xffffffffu, b != 0) << (32 * sl);
      }
      w = waner[(size_t)c * N + n] != 0;
      inf = constrain<M>(raw, pcr, dc.ch);
    }
    const M raw_in = raw;
    const int w_in = w;
    const M vac = reinterpret_cast<const M*>(dc.vac)[n];
    const int rn0 = dc.rp[0][n], cnt_n = dc.rp[0][n + 1] - rn0;
    const int rs0 = dc.rp[1][n], cnt_s = dc.rp[1][n + 1] - rs0;
    const int nrows = cnt_n + cnt_s;

    // rows of this individual, one per lane (N rows first, then S rows); kept in registers
    auto load_row = [&](int l, double& x, double& od, int& t, bool& is_s) {
      is_s = l >= cnt_n;
      const int r = is_s ? rs0 + (l - cnt_n) : rn0 + l;
      if (l < nrows) {
        x = (is_s ? dc.x[1] : dc.x[0])[r];
        od = (is_s ? dc.od[1] : dc.od[0])[r];
        t = (int)((is_s ? dc.meta[1] : dc.meta[0])[r] & kGapMask<M>);
      } else {
        x = 0.0;
        od = 0.0;
        t = -1;
      }
    };
    auto row_par = [&](bool is_s) {
      RowPar rp;
      rp.init = s_th[is_s ? S_INIT : N_INIT];
      rp.perm = s_th[is_s ? S_PERM : N_PERM];
      rp.tfac = is_s ? 1.0 : s_th[N_TEMP];
      rp.b = s_th[is_s ? S_B : N_B];
      rp.d = s_th[is_s ? S_D : N_D];
      rp.nh = s_th[is_s ? 14 : 13];
      return rp;
    };
    double x0, od0;
    int t0;
    bool s0;
    load_row(lane, x0, od0, t0, s0);
    const RowPar rp0 = row_par(s0);
    // latest sampled gap of either antigen / of the S antigen (rows are sorted by gap)
    int t_last = t0, t_last_s = s0 ? t0 : -1;
    for (int l = lane + 32; l < nrows; l += 32) {
      const bool is_s = l >= cnt_n;
      const int r = is_s ? rs0 + (l - cnt_n) : rn0 + l;
      const int t = (int)((is_s ? dc.meta[1] : dc.meta[0])[r] & kGapMask<M>);
      t_last = max(t_last, t);
      if (is_s) t_last_s = max(t_last_s, t);
    }
    t_last = __reduce_max_sync(0xffffffffu, t_last);
    t_last_s = __reduce_max_sync(0xffffffffu, t_last_s);

    // (keeping the vaccinations' share of the row in a register, as k_gibbs_blk does through GibbsRows, was measured
    // here too: 245 -> 255 us per sweep -- two more live registers under the 64-register cap cost more than the loop saves)
    auto indiv_ll = [&](M inf_, int w_) {
      double a = (t0 >= 0) ? gibbs_row<M>(x0, od0, t0, s0, inf_, vac, w_, rp0, s_pw, s_tab) : 0.0;
      for (int l = lane + 32; l < nrows; l += 32) {  // individuals with more than 32 rows
        double x, od;
        int t;
        bool is_s;
        load_row(l, x, od, t, is_s);
        a += gibbs_row<M>(x, od, t, is_s, inf_, vac, w_, row_par(is_s), s_pw, s_tab);
      }
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) a += __shfl_xor_sync(0xffffffffu, a, off);
      return a;
    };

    double ll = indiv_ll(inf, w);

    // ---- lane-owned proposals: Philox key (visiting order), transit / accept uniforms ----
    M act = 0;              // steps that are not skipped
    int jp_step[NSLOT];     // lane k (+32 sl): proposal visited at step k
    double acc_u[NSLOT];    // log(u) (Metropolis) or u (heat bath) of the proposals this lane owns
#pragma unroll
    for (int sl = 0; sl < NSLOT; ++sl) acc_u[sl] = 0.0;
    if (cfg.mode >= 0) {
      uint32_t key[NSLOT];
      int rank[NSLOT];
      bool skip[NSLOT];
#pragma unroll
      for (int sl = 0; sl < NSLOT; ++sl) {
        const uint4 r = philox4x32_10(
            make_uint4((uint32_t)(lane + 32 * sl), (uint32_t)n + dc.ind_offset, (uint32_t)c + dc.chain_offset, (uint32_t)cfg.sweep),
            make_uint2((uint32_t)cfg.seed, (uint32_t)(cfg.seed >> 32) ^ (uint32_t)(cfg.sweep >> 32)));
        key[sl] = r.x;
        const double u_t = u01(r.y), u_a = u01(r.z);
        skip[sl] = (cfg.mode == ABD_GIBBS_METROPOLIS) && !(u_t <= cfg.transit_p);
        acc_u[sl] = (cfg.mode == ABD_GIBBS_METROPOLIS) ? log(u_a) : u_a;
        rank[sl] = 0;
      }
      for (int jj = 0; jj < nprop; ++jj) {
        const uint32_t kj = __shfl_sync(0xffffffffu, NSLOT <= 2 ? key[(jj >> 5) & 1] : slot(key, jj >> 5), jj & 31);
#pragma unroll
        for (int sl = 0; sl < NSLOT; ++sl) {
          const int me = lane + 32 * sl;
          rank[sl] += (kj < key[sl]) || (kj == key[sl] && jj < me);
        }
      }
      __syncwarp();
#pragma unroll
      for (int sl = 0; sl < NSLOT; ++sl) {
        const int me = lane + 32 * sl;
        if (me < nprop) s_ord[warp][rank[sl]] = (unsigned char)me;
      }
      __syncwarp();
      // the proposal visited at the step this lane stands for; skipped steps drop out of `act`
#pragma unroll
      for (int sl = 0; sl < NSLOT; ++sl) {
        const int step = lane + 32 * sl;
        const int jp = (step < nprop) ? (int)s_ord[warp][step] : 0;
        jp_step[sl] = jp;
        bool sk = __shfl_sync(0xffffffffu, (int)skip[0], jp & 31);
#pragma unroll
        for (int s2 = 1; s2 < NSLOT; ++s2) {  // (jp >> 5 differs between lanes: every slot is shuffled)
          const bool sk1 = __shfl_sync(0xffffffffu, (int)skip[s2], jp & 31);
          if (NSLOT <= 2 ? (jp >> 5) != 0 : (jp >> 5) == s2) sk = sk1;
        }
        act |= (M)__ballot_sync(0xffffffffu, step < nprop && !sk) << (32 * sl);
      }
    } else {
#pragma unroll
      for (int sl = 0; sl < NSLOT; ++sl) jp_step[sl] = lane + 32 * sl;
      act = low_mask<M>(G);  // every proposal 0..G, in order
    }

    // Everything about a proposal that depends only on the current state lives in the lane that
    // owns it and is refreshed (lane-parallel) after an accepted flip of an infection bit:
    //   inf2  constrained infections if the flip were accepted
    //   code  2: the data term changes, the individual's likelihood must be evaluated;
    //         1 / 0: it cannot change (the constrained infections differ only after the last
    //         sampled gap, or -- waner bit -- there is no S sample after the first exposure), so
    //         logp(prop) - logp(cur) = +-logit(p) and the flip decision (1 / 0) is already known
    M inf2_own[NSLOT];
    int code_own[NSLOT];
    auto refresh = [&]() {
#pragma unroll
      for (int sl = 0; sl < NSLOT; ++sl) {
        const int me = lane + 32 * sl;
        const bool is_w = (me == G);
        const M i2 = (me < G) ? constrain<M>(raw ^ ((M)1 << me), pcr, dc.ch) : inf;
        inf2_own[sl] = i2;
        const int cur_bit = is_w ? w : (int)((raw >> (me < G ? me : 0)) & 1);
        bool affected;
        if (is_w) {
          const M ex = inf | vac;
          affected = ex != 0 && ctz(ex | top_bit<M>()) < t_last_s;
        } else {
          const M diff = inf ^ i2;
          affected = diff != 0 && ctz(diff | top_bit<M>()) <= t_last;
        }
        bool flip0;
        if (cfg.mode == ABD_GIBBS_METROPOLIS) {
          const double lo = s_th[is_w ? 16 : 15];
          const double delta = cur_bit ? -lo : lo;
          flip0 = isfinite(delta) && (acc_u[sl] < delta);
        } else {
          flip0 = ((acc_u[sl] <= s_th[is_w ? 18 : 17]) ? 1 : 0) != cur_bit;  // s_th[17 / 18] = sigmoid(logit)
        }
        code_own[sl] = affected ? 2 : (flip0 ? 1 : 0);
      }
    };
    refresh();

    while (act) {
      const int step = ctz(act);
      act &= act - 1;
      const int jp = __shfl_sync(0xffffffffu, slot(jp_step, step >> 5), step & 31);
      const int owner = jp & 31, jb = jp >> 5;
      const int code = __shfl_sync(0xffffffffu, slot(code_own, jb), owner);
      const bool is_w = (jp == G);
      if (cfg.mode >= 0) {
        ++n_prop;
        if (code == 0) continue;
      }
      const M inf2 = shfl_mask(slot(inf2_own, jb), owner);
      const int w2 = is_w ? (w ^ 1) : w;
      double ll2 = ll;
      bool flip = true;
      if (code == 2 || cfg.mode < 0) {
        const int cur_bit = is_w ? w : (int)((raw >> jp) & 1);
        if (code == 2) ll2 = indiv_ll(inf2, w2);
        const double lo = s_th[is_w ? 16 : 15];
        const double d10 = cur_bit ? (ll - ll2 + lo) : (ll2 - ll + lo);  // log-odds of 1 versus 0
        if (cfg.mode < 0) {
          if (lane == 0) {
            if (is_w) cfg.out_w[(size_t)c * N + n] = d10;
            else cfg.out_i[((size_t)c * G + jp) * N + n] = d10;
          }
          continue;
        }
        const double au = __shfl_sync(0xffffffffu, slot(acc_u, jb), owner);
        if (cfg.mode == ABD_GIBBS_METROPOLIS) {
          const double delta = cur_bit ? -d10 : d10;  // logp(proposed) - logp(current)
          flip = isfinite(delta) && (au < delta);
        } else {
          const double p1 = 1.0 / (1.0 + exp(-d10));
          flip = ((au <= p1) ? 1 : 0) != cur_bit;
        }
      }
      if (flip) {
        ++n_acc;
        ll = ll2;
        if (is_w) {
          w = w2;
        } else {
          raw ^= (M)1 << jp;
          inf = inf2;
          refresh();
        }
      }
    }

    if (cfg.mode >= 0) {  // write back only what changed
      const M changed = raw ^ raw_in;
#pragma unroll
      for (int sl = 0; sl < NSLOT; ++sl) {
        const int t = lane + 32 * sl;
        if (t < G && ((changed >> t) & 1)) col[(size_t)t * N] = (int8_t)((raw >> t) & 1);
      }
      if (lane == 0 && w != w_in) waner[(size_t)c * N + n] = (int8_t)w;
      if (pack && lane == 0 && (changed != 0 || w != w_in)) {
        PackedState<M> ps;
        ps.rw = raw | (w ? top_bit<M>() : (M)0);
        ps.inf = inf;
        pack[(size_t)c * N + n] = ps;
      }
    }
  }
  if (cfg.mode >= 0 && cfg.stats && lane == 0 && cur_c >= 0) {
    atomicAdd(&cfg.stats[(size_t)cur_c * 2], (unsigned long long)n_prop);
    atomicAdd(&cfg.stats[(size_t)cur_c * 2 + 1], (unsigned long long)n_acc);
  }
}

}  // namespace
