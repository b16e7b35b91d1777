// k_sums -- joint logp + gradient sums (one CTA per tile of individuals and chain), k_finalize.
// See DESIGN.md section 4 for the phases, the measured timeline and what was tried.
#pragma once
#include "abd_kernels_common.cuh"
#include "k_nuts.cuh"

namespace {
using namespace abd;

// ------------------------------------------------------------------------------------------
// k_sums
// ------------------------------------------------------------------------------------------
// Parameters of a few chains handed over by value, inside the kernel's parameter space (constant
// bank): the host-pointer calls (abd_logp_dlogp, abd_loglik_grad) then need no host -> device copy
// of q17 / theta13 before the launch.  n = 0: read the `theta` pointer instead.
constexpr int kInlineChains = 8;
constexpr int kMaxChainsPerCta = 32;  // a CTA remembers at most this many chains it finished last
struct ThetaInline {
  int n;
  double v[kInlineChains * 17];
};

struct FinalizeCfg {
  int mode;        // 0: write raw sums only; 1: loglik + grad13; 2: joint logp + dlogp17
  Totals tot;
  double* out_val;   // [C]
  double* out_grad;  // [C][13] or [C][17] (may be null)
};

struct SumsCfg {
  int ntiles;
  int cap_n, cap_s;      // staged doubles per antigen (even)
  int capr_n, capr_s;    // staged row->cell words per antigen (multiple of 4)
  int capk_n, capk_s;    // staged cell-meta words per antigen (multiple of 4)
  int chains_per_cta;
  int C;
};

// Fused all-reduce over NVLink peer memory (individuals sharded over `world` GPUs of one node):
// the CTA that finishes a chain last on each rank stores its 16 raw sums straight into every
// peer's exchange buffer -- as 32 eight-byte words, each half a double plus the 32-bit sequence
// number of the exchange, so that no fence and no separate flag (a second trip over NVLink) is
// needed --, later polls the words the peers store in ITS buffer, adds the `world` contributions
// in rank order (bitwise the same result on every rank) and finalises: compute, exchange and
// finalisation in one launch, no NCCL call.  Buffers are double-buffered on the parity of a
// per-chain sequence number kept on the device (a rank can be at most one exchange ahead of a
// peer: it cannot finish exchange k + 1 before the peer has posted k + 1, i.e. finished k).
constexpr int kMaxPeers = 8;
constexpr unsigned long long kXchTimeoutNs = 10ull * 1000 * 1000 * 1000;  // a peer that is 10 s late is declared lost
struct XchCfg {
  int world, rank, cmax;                 // world == 0: not sharded
  unsigned long long* buf[kMaxPeers];    // peer r's buffer: [2][world][cmax][32] words = 32-bit half | sequence << 32
  unsigned* seq;                         // [cmax] local sequence numbers
  unsigned* err;
  unsigned long long* stat;              // [kMaxPeers + 1]: ns spent waiting for each peer's flag, exchanges done
};

// Trajectory mode (n_steps > 0): the kernel stays resident for n_steps leapfrog steps of
// Hamiltonian dynamics over q17 with the binary state fixed.  Per step every CTA evaluates its
// tile at the current position; the CTA that finishes a chain last finalises logp / gradient,
// advances (q, p) and publishes them with a per-chain generation counter the other CTAs of that
// chain wait on -- no kernel launch, no re-staging of the cohort between evaluations.
struct TrajCfg {
  int n_steps;             // 0 = plain evaluation
  double* q;               // [C][17] in: start position, out: end position
  double* p;               // [C][17] in/out momentum
  double* grad;            // [C][17] in: gradient at q, out: gradient at the end position
  double* logp;            // [C]     out: logp at the end position
  const double* eps;       // [C] step sizes
  const double* inv_mass;  // [17][17] (symmetric) inverse mass matrix, shared by all chains
  double* state;           // [C][34] scratch: position and half-step momentum of the current step
  unsigned* gen;           // [C] generation counters (zeroed before the launch)
  unsigned* err;           // set to 1 if a wait timed out
  NutsLeafArgs nuts;       // single-step launches: fold the new state into the chain's No-U-Turn tree (state == nullptr: no)
};

// tile descriptor (48 bytes, three 16-byte loads): individuals [i0, i1); per antigen the OD rows
// [r0, r1) and the (individual, gap) cells [c0, c1) of those individuals
struct __align__(16) TileDesc {
  int i0, i1, rn0, rn1;
  int rs0, rs1, cn0, cn1;
  int cs0, cs1, pad0, pad1;
};

// trajectory of one cell: titer m, decaying part T (or U) and its rho-derivative; in factored mode
// also Em = exp(b m) (capped so that exp(-b x) * Em <= e^700)
template <bool FX, bool CP>
struct CellValT {
  double m, T, dT;
};
template <>
struct __align__(16) CellValT<true, false> {
  double m, T, dT, Em;
};
// Compact layout (factored mode, tiles too large for the 32-byte cells at full occupancy): 16 bytes per cell plus
// Em = exp(b m) in an array of its own (24 bytes per cell, not 32).  N antigen: m is not kept, sum q (x - m) is formed
// as  sum q x - (init sum q + perm sum q P + temp sum q T)  from sums the rows accumulate anyway; S antigen: the T
// slot holds m (the S rows never need U itself).
template <>
struct __align__(16) CellValT<true, true> {
  double T, dT;
};
constexpr int kMaxXLevels = 32;

#ifdef ABD_PHASE_TIMING
__device__ unsigned long long g_phase[4096][16];
__device__ unsigned long long g_span[256][2];  // per launch: first CTA start, last CTA end
__device__ unsigned g_span_idx, g_span_done;
__device__ __forceinline__ unsigned long long gtime() {
  unsigned long long t_;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));
  return t_;
}
#define SPAN_BEGIN()                                                                      \
  unsigned span_slot_ = 0;                                                                \
  if (threadIdx.x == 0) {                                                                 \
    span_slot_ = *(volatile unsigned*)&g_span_idx & 255u;                                 \
    atomicMin(&g_span[span_slot_][0], gtime());                                           \
  }
#define SPAN_END()                                                                        \
  if (threadIdx.x == 0) {                                                                 \
    atomicMax(&g_span[span_slot_][1], gtime());                                           \
    if (atomicAdd(&g_span_done, 1u) == gridDim.x * gridDim.y - 1) {                       \
      g_span_done = 0;                                                                    \
      __threadfence();                                                                    \
      atomicAdd(&g_span_idx, 1u);                                                         \
    }                                                                                     \
  }
#define PHASE(i)                                                                         \
  do {                                                                                   \
    if (tid == 0 && blockIdx.y * gridDim.x + blockIdx.x < 4096) {                        \
      unsigned long long t_;                                                             \
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));                             \
      g_phase[blockIdx.y * gridDim.x + blockIdx.x][i] = t_;                              \
    }                                                                                    \
  } while (0)
#define PHASEW(i, cond)                                                                  \
  do {                                                                                   \
    if ((cond) && blockIdx.y * gridDim.x + blockIdx.x < 4096) {                          \
      unsigned long long t_;                                                             \
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));                             \
      g_phase[blockIdx.y * gridDim.x + blockIdx.x][i] = t_;                              \
    }                                                                                    \
  } while (0)
#else
#define PHASE(i)
#define PHASEW(i, cond)
#define SPAN_BEGIN()
#define SPAN_END()
#endif

#ifndef ABD_ROW_UNROLL
#define ABD_ROW_UNROLL 1  // measured 1, 2, 3, 4 (and cells 1, 2): within 1.5 %, 1 is the fastest and smallest
#endif
#ifndef ABD_CELL_UNROLL
#define ABD_CELL_UNROLL 1
#endif
constexpr int kRowUnroll = ABD_ROW_UNROLL, kCellUnroll = ABD_CELL_UNROLL;
#ifndef ABD_SUMS_MINB
#define ABD_SUMS_MINB 3
#endif
// XT: how the dilutions reach the row loop.  uint8_t = factored mode: a row carries the index of
// its dilution (packed with its cell index), exp(-b (x - m)) = exp(-b x) * exp(b m) costs one exp
// per CELL plus a per-chain table over the distinct dilutions; double = general fallback, the
// dilutions themselves are staged and every row evaluates its own exp.
template <typename M, typename XT, bool TRAJ, bool CP>
__global__ void __launch_bounds__(kSumsBlock, ABD_SUMS_MINB)
k_sums(const DevCohort dc, const TileDesc* __restrict__ tiles, const SumsCfg cfg,
       const double* __restrict__ theta_ptr, const int theta_is_q,
       const int8_t* __restrict__ i_raw, const int8_t* __restrict__ waner, const PackedState<M>* __restrict__ pack,
       double* __restrict__ partial, unsigned* __restrict__ ticket, double* __restrict__ sums,
       const FinalizeCfg fin, const Priors* __restrict__ priors, double* __restrict__ aux, const TrajCfg traj,
       const XchCfg xch, const __grid_constant__ ThetaInline thin) {
  const double* theta = thin.n ? thin.v : theta_ptr;
  const int tile = blockIdx.x, tid = threadIdx.x;
  const int lane = tid & 31, warp = tid >> 5;
  const int G = dc.G, N = dc.N, ntiles = cfg.ntiles;

  // dynamic shared memory: staged rows (od, x, row->cell), staged cell meta, per-cell values
  extern __shared__ __align__(16) unsigned char dyn_smem[];
  constexpr bool kFX = sizeof(XT) == 1;
  constexpr bool kCP = kFX && CP;  // compact cells (see CellValT)
  using CellVal = CellValT<kFX, kCP>;
  double* s_od_n = reinterpret_cast<double*>(dyn_smem);
  double* s_od_s = s_od_n + cfg.cap_n;
  CellVal* s_cv_n = reinterpret_cast<CellVal*>(s_od_s + cfg.cap_s);
  CellVal* s_cv_s = s_cv_n + cfg.capk_n;
  double* s_em_n = reinterpret_cast<double*>(s_cv_s + cfg.capk_s);  // capk_n + capk_s doubles (compact cells only)
  double* s_em_s = s_em_n + (kCP ? cfg.capk_n : 0);
  double* s_x_n = s_em_s + (kCP ? cfg.capk_s : 0);                  // cap_n doubles (not in factored mode)
  double* s_x_s = s_x_n + (kFX ? 0 : cfg.cap_n);
  uint32_t* s_rc_n = reinterpret_cast<uint32_t*>(s_x_s + (kFX ? 0 : cfg.cap_s));
  uint32_t* s_rc_s = s_rc_n + cfg.capr_n;
  uint32_t* s_cm_n = s_rc_s + cfg.capr_s;
  uint32_t* s_cm_s = s_cm_n + cfg.capk_n;

  __shared__ double s_th[16];
  __shared__ double2 s_pw[2][kGapTab<M>];  // {rho^k, k rho^(k-1)} for rho_n, rho_s
  __shared__ double s_tab[kExpTab];
  __shared__ IndState<M> s_ind[kTileMaxInds];
  __shared__ double s_red[kSumsWarps][kNSums];
  __shared__ double s_fin[kSumsBlock / 16][kNSums];
  __shared__ int s_last;
  __shared__ __align__(8) uint64_t s_bar;
  __shared__ PriorPre s_pre[17];
  __shared__ LikPre s_lik;
  __shared__ double s_q[17], s_ph[17], s_out[18];  // trajectory mode: position, half-step momentum, logp + gradient
  __shared__ double s_im[TRAJ ? 17 * 17 : 1];       // trajectory mode: inverse mass matrix
  __shared__ double2 s_xe[kFX ? 2 : 1][kMaxXLevels];  // factored mode: {x_j, exp(-b x_j)} per antigen
  __shared__ double s_zmax[2];                      // cap on b m so that exp(-b x) exp(b m) <= e^700
  __shared__ int s_direct;                          // |b| x too large to factor: rows take their own exp

  PHASE(0);
  SPAN_BEGIN();
  griddep_launch_dependents();
  const int4 d0 = reinterpret_cast<const int4*>(tiles + tile)[0];
  const int4 d1 = reinterpret_cast<const int4*>(tiles + tile)[1];
  const int2 d2 = reinterpret_cast<const int2*>(tiles + tile)[4];
  const int i0 = d0.x, ni = d0.y - d0.x;
  const int rn0 = d0.z, rn1 = d0.w, rs0 = d1.x, rs1 = d1.y;
  const int cn0 = d1.z, cn1 = d1.w, cs0 = d2.x, cs1 = d2.y;

  // ---- stage this tile's rows and cell table in shared memory: one thread, bulk async copies ----
  const int an0 = rn0 & ~1, as0 = rs0 & ~1;      // 16-byte aligned starts (doubles)
  const int qn0 = rn0 & ~3, qs0 = rs0 & ~3;      // (32-bit words)
  const int kn0 = cn0 & ~3, ks0 = cs0 & ~3;
  if (tid == 0) {
    mbar_init(&s_bar, 1);
    const uint32_t bn = (uint32_t)(((rn1 + 1) & ~1) - an0) * 8u, bs = (uint32_t)(((rs1 + 1) & ~1) - as0) * 8u;
    const uint32_t bqn = (uint32_t)(((rn1 + 3) & ~3) - qn0) * 4u, bqs = (uint32_t)(((rs1 + 3) & ~3) - qs0) * 4u;
    const uint32_t bkn = (uint32_t)(((cn1 + 3) & ~3) - kn0) * 4u, bks = (uint32_t)(((cs1 + 3) & ~3) - ks0) * 4u;
    mbar_expect_tx(&s_bar, (kFX ? bn + bs : 2 * bn + 2 * bs) + bqn + bqs + bkn + bks);
    if (bkn) bulk_g2s(s_cm_n, dc.cmeta[0] + kn0, bkn, &s_bar);
    if (bks) bulk_g2s(s_cm_s, dc.cmeta[1] + ks0, bks, &s_bar);
    if (bn) {
      bulk_g2s(s_od_n, dc.od[0] + an0, bn, &s_bar);
      if (!kFX) bulk_g2s(s_x_n, dc.x[0] + an0, bn, &s_bar);
    }
    if (bs) {
      bulk_g2s(s_od_s, dc.od[1] + as0, bs, &s_bar);
      if (!kFX) bulk_g2s(s_x_s, dc.x[1] + as0, bs, &s_bar);
    }
    if (bqn) bulk_g2s(s_rc_n, (kFX ? dc.rcx[0] : dc.rowcell[0]) + qn0, bqn, &s_bar);
    if (bqs) bulk_g2s(s_rc_s, (kFX ? dc.rcx[1] : dc.rowcell[1]) + qs0, bqs, &s_bar);
  }
  fill_exp_table(s_tab, tid, kSumsBlock);
  // the immutable PCR+ / vaccination masks of this thread's individual (read before the wait)
  M my_pcr = 0, my_vac = 0;
  if (tid < ni) {
    my_pcr = reinterpret_cast<const M*>(dc.pcr)[i0 + tid];
    my_vac = reinterpret_cast<const M*>(dc.vac)[i0 + tid];
  }
  double x_lev = 0.0;  // factored mode, last warp: lane j holds the j-th distinct dilution
  if (kFX && warp == kSumsWarps - 1) x_lev = dc.xlev[lane];
  __syncthreads();  // the exp table is usable from here on (still before the dependency wait)
  // everything above reads only the immutable cohort; parameters, chain state and the reduction
  // scratch may be written by the previous kernel in the stream
  griddep_wait();
  if (TRAJ) {
    for (int k = tid; k < 17 * 17; k += kSumsBlock) s_im[k] = traj.inv_mass[k];
    __syncthreads();
  }
  PHASE(1);

  __shared__ int s_pend[kMaxChainsPerCta], s_npend;   // chains this CTA finished last (queued for the reduction + finaliser)
  __shared__ unsigned s_pend_seq[kMaxChainsPerCta];
  __shared__ unsigned s_xw[kMaxPeers][32];     // sharded: the peers' 16 sums as 32-bit halves
  if (tid == 0) s_npend = 0;
  // the parameter-only part of the finaliser, parked in `aux` by the chain's first tile
  auto load_aux = [&](int c) {
    if (fin.mode && tid < kAuxDoubles) {
      const double v = __ldcg(aux + (size_t)c * kAuxDoubles + tid);
      if (tid < 17 * 7) reinterpret_cast<double*>(s_pre)[tid] = v;
      else if (tid < 17 * 7 + 6) reinterpret_cast<double*>(&s_lik)[tid - 17 * 7] = v;
    }
  };
  // all threads: the chain's totals over the tiles' partials, in a fixed order, into s_red[0] (and `sums`)
  auto sum_partials = [&](int c, bool sharded_) {
    const int k = tid & 15, g = tid >> 4;  // 16 groups of 16 values
    double v = 0.0;
    const double* src = partial + (size_t)c * ntiles * kNSums + k;
    for (int tl = g; tl < ntiles; tl += 8 * (kSumsBlock / 16)) {  // 8 loads in flight, fixed order
      double ld[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {  // unpredicated (clamped) loads, masked afterwards: all in flight
        const int tt = tl + u * (kSumsBlock / 16);
        ld[u] = __ldcg(src + (size_t)min(tt, ntiles - 1) * kNSums);
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) v += (tl + u * (kSumsBlock / 16) < ntiles) ? ld[u] : 0.0;
    }
    s_fin[g][k] = v;
    PHASE(9);
    __syncthreads();
    if (tid < kNSums) {
      double tot = 0.0;
#pragma unroll
      for (int gg = 0; gg < kSumsBlock / 16; ++gg) tot += s_fin[gg][tid];
      s_red[0][tid] = tot;
      if (sums && !sharded_) sums[(size_t)c * kNSums + tid] = tot;
    }
    if (tid == 0) ticket[c] = 0;  // re-arm for the next launch
    __syncthreads();
  };
  // thread 0: the ticket drawn for the previous chain (looked at one chain later, see below)
  unsigned tk_prev = 0;
  int tk_c = 0;
  bool tk_valid = false;
  // warp 0: totals in s_red[0] -> loglik / joint logp and gradient (or, trajectory mode, the end of the step)
  auto finalize_chain = [&](int c, int step, int nsteps) {
    if (fin.mode == 1) {
      if (lane == 0)
        finalize_loglik_post(s_th, s_lik, s_red[0], fin.tot, &fin.out_val[c],
                             fin.out_grad ? &fin.out_grad[(size_t)c * 13] : nullptr);
    } else if (fin.mode == 2 && !TRAJ) {
      finalize_logp_post(lane, s_pre, s_th, s_lik, s_red[0], fin.tot, &fin.out_val[c],
                         fin.out_grad ? &fin.out_grad[(size_t)c * 17] : nullptr);
    } else if (TRAJ && fin.mode == 2) {
      // trajectory mode: finish this leapfrog step and either publish the next position or
      // write the end point
      finalize_logp_post(lane, s_pre, s_th, s_lik, s_red[0], fin.tot, &s_out[0], &s_out[1]);
      __syncwarp();
      const double e = traj.eps[c];
      const double g = lane < 17 ? s_out[1 + lane] : 0.0;
      const double ph = lane < 17 ? s_ph[lane] : 0.0;
      if (step == nsteps - 1) {
        if (lane < 17) {
          traj.q[(size_t)c * 17 + lane] = s_q[lane];
          traj.p[(size_t)c * 17 + lane] = fma(0.5 * e, g, ph);
          traj.grad[(size_t)c * 17 + lane] = g;
        }
        if (lane == 0) traj.logp[c] = s_out[0];
        if (traj.nuts.state) {  // the leaf's tree bookkeeping in the same launch (this warp is the chain's only writer)
          __syncwarp();
          nuts_leaf_chain(traj.nuts, c, lane, traj.q, traj.p, traj.grad, traj.logp, s_im);
        }
      } else {
        const double ph2 = fma(e, g, ph);  // two half steps: end of this step + start of the next
        double dot = 0.0;
        for (int j = 0; j < 17; ++j) {
          const double pj = __shfl_sync(0xffffffffu, ph2, j);
          if (lane < 17) dot = fma(s_im[lane * 17 + j], pj, dot);
        }
        if (lane < 17) {
          traj.state[(size_t)c * 34 + lane] = fma(e, dot, s_q[lane]);
          traj.state[(size_t)c * 34 + 17 + lane] = ph2;
        }
        __threadfence();
        __syncwarp();
        if (lane == 0) {
          const unsigned nxt = (unsigned)step + 1u;
          asm volatile("st.release.gpu.u32 [%0], %1;" ::"l"(traj.gen + c), "r"(nxt) : "memory");
        }
      }
    }
  };

  for (int cc = 0; cc < cfg.chains_per_cta; ++cc) {
    const int c = blockIdx.y * cfg.chains_per_cta + cc;
    if (c >= cfg.C) break;

    const int nsteps = TRAJ ? traj.n_steps : 1;
    double cnt_i = 0.0, cnt_w = 0.0;  // this thread's individual: sum(i_raw), waner
    // ---- phase 0 (state): warps 0-3, one thread per individual, read the int8 column (every load
    //      of the warp is one coalesced 32-byte segment) and apply the infection constraints.  The
    //      binary state is fixed over a trajectory, so this sits OUTSIDE the step loop (inside it
    //      the compiler hoisted and spilled the 31 column addresses of the trajectory variant, and
    //      the spills serialised the loads: 4.9 us instead of 1.9) ----
    if (tid < ni && pack) {
      // resident state, packed (PackedState): one coalesced 8 / 16-byte load per individual, the
      // constraints were applied when the state was written
      const PackedState<M> ps = pack[(size_t)c * N + i0 + tid];
      const M w = ps.waner_bit();
      IndState<M> st;
      st.inf = ps.inf;
      st.vacw = my_vac | w;
      s_ind[tid] = st;
      cnt_i = (double)popc(ps.raw());
      cnt_w = w ? 1.0 : 0.0;
    } else if (tid < ni) {
      // (unpredicated loads, all in flight: see load_column; without them the column costs 5 memory round trips)
      const M raw = load_column<M>(i_raw + (size_t)c * G * N + i0 + tid, G, N);
      const int w = waner[(size_t)c * N + i0 + tid] != 0;
      IndState<M> st;
      st.inf = constrain<M>(raw, my_pcr, dc.ch);
      st.vacw = my_vac | (w ? top_bit<M>() : (M)0);
      s_ind[tid] = st;
      cnt_i = (double)popc(raw);
      cnt_w = (double)w;
    }
    for (int step = 0; step < nsteps; ++step) {
    double acc[kNSums];
#pragma unroll
    for (int k = 0; k < kNSums; ++k) acc[k] = 0.0;
    acc[S_KI] = cnt_i;
    acc[S_KW] = cnt_w;

    // trajectory mode: this step's position.  Step 0: every warp that needs it advances the
    // start point itself (p_half = p + eps/2 g, q' = q + eps Sigma p_half: 17 FMAs per lane);
    // later steps: wait for the chain's previous finaliser to publish (q', p_half).
    double q_lane = 0.0, ph_lane = 0.0;  // lane k < 17: component k
    if (TRAJ) {
      if (step > 0) {
        if (tid == 0) {
          unsigned seen, polls = 0;
          do {
            asm volatile("ld.acquire.gpu.u32 %0, [%1];" : "=r"(seen) : "l"(traj.gen + c) : "memory");
          } while (seen < (unsigned)step && ++polls < (1u << 26));
          if (seen < (unsigned)step) *traj.err = 1u;  // watchdog: never hang the GPU
        }
        __syncthreads();
        if (lane < 17) {
          q_lane = __ldcg(traj.state + (size_t)c * 34 + lane);
          ph_lane = __ldcg(traj.state + (size_t)c * 34 + 17 + lane);
        }
      } else if (warp >= 4) {
        const double e = traj.eps[c];
        double mine = 0.0;
        if (lane < 17) mine = fma(0.5 * e, traj.grad[(size_t)c * 17 + lane], traj.p[(size_t)c * 17 + lane]);
        double dot = 0.0;
        for (int j = 0; j < 17; ++j) {
          const double pj = __shfl_sync(0xffffffffu, mine, j);
          if (lane < 17) dot = fma(s_im[lane * 17 + j], pj, dot);
        }
        ph_lane = mine;
        if (lane < 17) q_lane = fma(e, dot, traj.q[(size_t)c * 17 + lane]);
      }
    }
    // parameter k13 of this chain for the calling warp (uniform over the warp)
    auto param13 = [&](int k13) -> double {
      if (TRAJ) {
        const int j = kQOfTheta[k13];
        return backward(__shfl_sync(0xffffffffu, q_lane, j), kQTransform[j]);
      }
      return load_param(theta, theta_is_q, c, k13);
    };

    // ---- phase 0 (parameters): warps 4-7: parameters, power tables, dilution table, while warps
    //      0-3 wait for their columns (above).  (Fetching the state block as aligned
    //      32-bit words + shared-memory atomics / ballots was measured: slower, the transposition
    //      costs more than the byte loads save; two lanes per individual (even / odd gaps, one
    //      shuffle) was measured too: 12.2 -> 13.4 us per launch.) ----
    if (tid < kTileMaxInds) {
      PHASEW(12, tid == 0);
    } else if (warp == 4) {
      fill_pow2_warp(param13(N_RHO), G, lane, s_pw[0]);
      PHASEW(13, lane == 0);
    } else if (warp == 5) {
      fill_pow2_warp(param13(S_RHO), G, lane, s_pw[1]);
    } else if (warp == 6) {
      if (TRAJ) {
        const int j = kQOfTheta[lane < 13 ? lane : 0];
        const double v = backward(__shfl_sync(0xffffffffu, q_lane, j), kQTransform[j]);
        if (lane < 13) s_th[lane] = v;
      } else if (lane < 13) {
        s_th[lane] = load_param(theta, theta_is_q, c, lane);
      }
      PHASEW(14, lane == 0);
    } else if (warp == kSumsWarps - 1) {
      if (kFX) {
        // per-chain table {x_j, exp(-b x_j)} over the distinct dilutions, both antigens, and the
        // cap on b m that keeps the product <= e^700 (b is not transformed: read it directly)
        const double zn = -param13(N_B) * x_lev, zs = -param13(S_B) * x_lev;
        double mn = (lane < dc.n_xlev) ? fabs(zn) : 0.0, ms = (lane < dc.n_xlev) ? fabs(zs) : 0.0;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
          mn = fmax(mn, __shfl_xor_sync(0xffffffffu, mn, off));
          ms = fmax(ms, __shfl_xor_sync(0xffffffffu, ms, off));
        }
        // NaN / huge |b| x: every row evaluates its own exponential (same arithmetic as the fallback)
        const bool direct = !(mn < 300.0 && ms < 300.0);
        s_xe[0][lane] = make_double2(x_lev, direct ? 0.0 : fast_exp(zn, s_tab));
        s_xe[kFX ? 1 : 0][lane] = make_double2(x_lev, direct ? 0.0 : fast_exp(zs, s_tab));
        if (lane == 0) {
          s_zmax[0] = 700.0 - mn;
          s_zmax[1] = 700.0 - ms;
          s_direct = direct;
        }
      }
      if (TRAJ && lane < 17) {  // keeps (q, p_half) for the finaliser
        s_q[lane] = q_lane;
        s_ph[lane] = ph_lane;
      }
      PHASEW(15, lane == 0);
    }
    __syncthreads();
    PHASE(2);
    // The finaliser's parameter-only part (priors, transforms, logs: ~2 us of cold libm code) is
    // taken off the critical path: warp 7 of the chain's first tile computes it now, instead of
    // processing cells / rows, and parks it in global memory for whichever CTA finishes last.
    // (the row -> thread assignment must not depend on fin.mode: abd_sums_dev + abd_finalize_* has
    // to reproduce the fused launch bit for bit)
    const bool aux_cta = (tile == 0);
    const int nwork = aux_cta ? kSumsBlock - 32 : kSumsBlock;
    if (aux_cta && fin.mode != 0 && warp == kSumsWarps - 1) {
      double* a = aux + (size_t)c * kAuxDoubles;
      if (fin.mode == 2 && lane < 17) {
        const PriorPre pp = prior_pre(lane, TRAJ ? s_q[lane] : theta[(size_t)c * 17 + lane], priors->v[lane]);
        double* o = a + lane * 7;
        o[0] = pp.lpA, o[1] = pp.dA, o[2] = pp.f, o[3] = pp.lx, o[4] = pp.l1mx, o[5] = pp.x, o[6] = pp.omx;
      }
      if (lane == 17) {
        const LikPre lk = lik_pre(s_th[N_SIGMA], s_th[S_SIGMA]);
        double* o = a + 17 * 7;
        o[0] = lk.lsn, o[1] = lk.lss, o[2] = lk.ivn, o[3] = lk.ivs, o[4] = lk.isn, o[5] = lk.iss;
      }
    }
    if (cc == 0 && step == 0) mbar_wait(&s_bar, 0);
    PHASE(3);

    // ---- phase 1: one thread per (individual, gap) cell: titer in closed form from the masks ----
    {
      const double init = s_th[N_INIT], perm = s_th[N_PERM], temp = s_th[N_TEMP];
      const double bn_fx = s_th[N_B], zmax_n = s_zmax[0];
#pragma unroll kCellUnroll
      for (int k = cn0 + tid; k < cn1 && tid < nwork; k += nwork) {
        const uint32_t mt = s_cm_n[k - kn0];
        const int t = mt & kGapMask<M>, li = (int)(mt >> kGapBits<M>) - i0;
        double P, T, dT;
        traj_n<M>(s_ind[li].inf, t, s_pw[0], P, T, dT);
        CellVal cv;
        const double m = init + perm * P + temp * T;
        cv.T = T;
        cv.dT = (P != 0.0) ? dT : -0.0;  // sign bit of dT carries "never exposed" (P = 0)
        if constexpr (!kCP) cv.m = m;
        if constexpr (kFX) {
          const double z = bn_fx * m;
          const double em = fast_exp((z > zmax_n) ? zmax_n : z, s_tab);  // NaN stays NaN
          if constexpr (kCP) s_em_n[k - cn0] = em;
          else cv.Em = em;
        }
        s_cv_n[k - cn0] = cv;
      }
    }
    {
      const double init = s_th[S_INIT], perm = s_th[S_PERM];
      const double bs_fx = s_th[S_B], zmax_s = s_zmax[1];
#pragma unroll kCellUnroll
      for (int k = cs0 + tid; k < cs1 && tid < nwork; k += nwork) {
        const uint32_t mt = s_cm_s[k - ks0];
        const int t = mt & kGapMask<M>, li = (int)(mt >> kGapBits<M>) - i0;
        const IndState<M> st = s_ind[li];
        double P, U, dU;
        traj_s<M>(st.inf, st.vacw & ~top_bit<M>(), (st.vacw & top_bit<M>()) != 0, t, s_pw[1], P, U, dU);
        CellVal cv;
        const double m = init + perm * P + U;
        cv.T = kCP ? m : U;
        cv.dT = (P != 0.0) ? dU : -0.0;
        if constexpr (!kCP) cv.m = m;
        if constexpr (kFX) {
          const double z = bs_fx * m;
          const double em = fast_exp((z > zmax_s) ? zmax_s : z, s_tab);
          if constexpr (kCP) s_em_s[k - cs0] = em;
          else cv.Em = em;
        }
        s_cv_s[k - cs0] = cv;
      }
    }
    __syncthreads();
    PHASE(4);

    // ---- phase 2: one thread per OD row; everything comes from shared memory, no divergence.
    //      P (ever exposed) travels in the sign bit of dT ----
    //      The loops exist twice: `direct` (a chain whose |b| x is too large to factor, or the
    //      fallback kernel) evaluates one exponential per row, the common case only a product ----
    auto rows = [&](auto direct_tag) {
      [[maybe_unused]] constexpr bool kDirect = decltype(direct_tag)::value;
      {
        const double b = s_th[N_B], d = s_th[N_D];
        const uint32_t* rcp = s_rc_n - qn0;
        const double* odp = s_od_n - an0;
        const CellVal* cvp = s_cv_n - cn0;
        [[maybe_unused]] const double* emp = s_em_n - cn0;
#pragma unroll kRowUnroll
        for (int r = rn0 + tid; r < rn1 && tid < nwork; r += nwork) {
          double sg, res, q, xm;
          const uint32_t rc = rcp[r];
          const CellVal cv = cvp[kFX ? (rc >> 5) : rc];
          if constexpr (kCP) {
            const double2 xe = s_xe[0][rc & 31];
            if constexpr (kDirect) {  // (the cell's response again: init + perm P + temp T)
              const double m = s_th[N_INIT] + ((__double2hiint(cv.dT) < 0) ? 0.0 : s_th[N_PERM]) + s_th[N_TEMP] * cv.T;
              row_eval(xe.x, odp[r], m, b, d, s_tab, sg, res, q, xm);
            } else {
              row_eval_E(xe.y * emp[rc >> 5], odp[r], d, sg, res, q);
              xm = xe.x;  // sum q x here; the cells' share  sum q m  is taken off the block's total (below)
            }
          } else if constexpr (kFX) {
            const double2 xe = s_xe[0][rc & 31];
            xm = xe.x - cv.m;
            if constexpr (kDirect) row_eval(xe.x, odp[r], cv.m, b, d, s_tab, sg, res, q, xm);
            else row_eval_E(xe.y * cv.Em, odp[r], d, sg, res, q);
          } else {
            row_eval((s_x_n - an0)[r], odp[r], cv.m, b, d, s_tab, sg, res, q, xm);
          }
          acc[SN_0] = fma(res, res, acc[SN_0]);
          acc[SN_1] = fma(res, sg, acc[SN_1]);
          acc[SN_2] = fma(q, xm, acc[SN_2]);
          acc[SN_QINIT] += q;
          acc[SN_QPERM] += (__double2hiint(cv.dT) < 0) ? 0.0 : q;
          acc[SN_QTEMP] = fma(q, cv.T, acc[SN_QTEMP]);
          acc[SN_QRHO] = fma(q, cv.dT, acc[SN_QRHO]);
        }
      }
      {
        const double b = s_th[S_B], d = s_th[S_D];
        const uint32_t* rcp = s_rc_s - qs0;
        const double* odp = s_od_s - as0;
        const CellVal* cvp = s_cv_s - cs0;
        [[maybe_unused]] const double* emp = s_em_s - cs0;
#pragma unroll kRowUnroll
        for (int r = rs0 + tid; r < rs1 && tid < nwork; r += nwork) {
          double sg, res, q, xm;
          const uint32_t rc = rcp[r];
          const CellVal cv = cvp[kFX ? (rc >> 5) : rc];
          if constexpr (kCP) {  // (the T slot holds m)
            const double2 xe = s_xe[1][rc & 31];
            xm = xe.x - cv.T;
            if constexpr (kDirect) row_eval(xe.x, odp[r], cv.T, b, d, s_tab, sg, res, q, xm);
            else row_eval_E(xe.y * emp[rc >> 5], odp[r], d, sg, res, q);
          } else if constexpr (kFX) {
            const double2 xe = s_xe[1][rc & 31];
            xm = xe.x - cv.m;
            if constexpr (kDirect) row_eval(xe.x, odp[r], cv.m, b, d, s_tab, sg, res, q, xm);
            else row_eval_E(xe.y * cv.Em, odp[r], d, sg, res, q);
          } else {
            row_eval((s_x_s - as0)[r], odp[r], cv.m, b, d, s_tab, sg, res, q, xm);
          }
          acc[SS_0] = fma(res, res, acc[SS_0]);
          acc[SS_1] = fma(res, sg, acc[SS_1]);
          acc[SS_2] = fma(q, xm, acc[SS_2]);
          acc[SS_QINIT] += q;
          acc[SS_QPERM] += (__double2hiint(cv.dT) < 0) ? 0.0 : q;
          acc[SS_QRHO] = fma(q, cv.dT, acc[SS_QRHO]);
        }
      }
    };
    if (!kFX || s_direct) rows(std::true_type{});
    else rows(std::false_type{});

    PHASE(5);
    // ---- block reduction: butterfly inside a warp, shared memory across warps ----
    {
      const double tot = warp_reduce16(acc, lane);
      if ((lane & 1) == 0) s_red[warp][warp_reduce16_index(lane)] = tot;
    }
    __syncthreads();
    if (warp == 0) {
      double v = 0.0;
      if (lane < kNSums) {
#pragma unroll
        for (int wv = 0; wv < kSumsWarps; ++wv) v += s_red[wv][lane];
      }
      if constexpr (kCP) {
        if (!s_direct) {
          // the factored N rows accumulated  sum q x;  sum q (x - m) = sum q x - sum q m  with
          // m = init + perm P + temp T, linear in sums this warp holds
          const double qi = __shfl_sync(0xffffffffu, v, SN_QINIT), qp = __shfl_sync(0xffffffffu, v, SN_QPERM);
          const double qt = __shfl_sync(0xffffffffu, v, SN_QTEMP);
          if (lane == SN_2) v -= s_th[N_INIT] * qi + s_th[N_PERM] * qp + s_th[N_TEMP] * qt;
        }
      }
      if (lane < kNSums) partial[((size_t)c * ntiles + tile) * kNSums + lane] = v;
    }

    PHASE(6);
    // ---- which CTA finishes this chain last?  One thread releases the CTA's partials (barrier, then an
    //      acq_rel ticket) and, if it drew the last ticket, has acquired everybody else's: the grid-sync idiom
    //      with ONE atomic per CTA.  The ticket's answer is not waited for: the CTA goes straight on to its
    //      next chain and thread 0 looks at the answer one chain later (a global atomic round trip is ~1400
    //      cycles during which the whole CTA would sit at a barrier), queueing the chain for the ordered
    //      cross-tile reduction + finalisation after the chain loop.  The persistent multi-step trajectory
    //      mode must finalise in place (the chain's other CTAs wait for the next position). ----
    __syncthreads();
    // (one chain per CTA and no exchange: nothing to overlap the answer with, finalise in place as well)
    if (!((TRAJ && nsteps > 1) || (cfg.chains_per_cta == 1 && xch.world <= 1))) {
      if (tid == 0) {
        if (tk_valid && tk_prev == (unsigned)(ntiles - 1)) s_pend[s_npend++] = tk_c;
        asm volatile("atom.add.acq_rel.gpu.global.u32 %0, [%1], 1;" : "=r"(tk_prev) : "l"(ticket + c) : "memory");
        tk_c = c;
        tk_valid = true;
      }
      PHASE(8);
      continue;  // (the barrier above already separates this chain's shared-memory reads from the next chain's writes)
    }
    if (tid == 0) {
      unsigned prev;
      asm volatile("atom.add.acq_rel.gpu.global.u32 %0, [%1], 1;" : "=r"(prev) : "l"(ticket + c) : "memory");
      s_last = (prev == (unsigned)(ntiles - 1));
    }
    __syncthreads();
    PHASE(7);
    if (s_last) {
      load_aux(c);
      sum_partials(c, false);
      PHASE(10);
      if (warp == 0) finalize_chain(c, step, nsteps);
    }
    if (s_last) PHASE(11);
    PHASE(8);
    __syncthreads();  // shared memory is reused by the next step / chain
    }  // step
  }

  // ---- the chains this CTA finished last: ordered reduction over the tiles' partials, then either the
  //      finaliser, or (individuals sharded over GPUs) the exchange with the peers first ----
  if (tid == 0 && tk_valid && tk_prev == (unsigned)(ntiles - 1)) s_pend[s_npend++] = tk_c;
  __syncthreads();
  const int npend = s_npend;
  const bool sharded = xch.world > 1;
  PHASE(7);
  for (int pi = 0; pi < npend; ++pi) {
    const int c = s_pend[pi];
    if (!sharded) {
      load_aux(c);
      if (!TRAJ && warp == 1 && lane < 13) s_th[lane] = load_param(theta, theta_is_q, c, lane);  // as warp 6 computed it
    }
    sum_partials(c, sharded);
    PHASE(10);
    if (!sharded) {
      if (warp == 0) finalize_chain(c, 0, 1);
      __syncthreads();
      continue;
    }
    // ---- post this rank's 16 sums into every peer's buffer and move on to the next pending chain; the peers'
    //      sums are collected below.  Low-latency protocol: every 8-byte word carries 4 bytes of payload and
    //      the 4-byte sequence number of this exchange, so the words may arrive in any order and no fence /
    //      separate flag (a second NVLink round trip) is needed. ----
    const unsigned seq = xch.seq[c] + 1u;  // every thread reads it before thread 0 writes it back (barrier below)
    if (tid < 32 * xch.world) {
      const int r = tid >> 5, j = tid & 31;
      const double val = s_red[0][j >> 1];
      const unsigned half = (j & 1) ? (unsigned)__double2hiint(val) : (unsigned)__double2loint(val);
      const unsigned long long word = ((unsigned long long)seq << 32) | half;
      unsigned long long* dst = xch.buf[r] + ((((size_t)(seq & 1u) * xch.world + xch.rank) * xch.cmax + c) << 5) + j;
      asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(dst), "l"(word) : "memory");
    }
    __syncthreads();
    if (tid == 0) {
      xch.seq[c] = seq;
      s_pend_seq[pi] = seq;
    }
  }
  if (npend) PHASE(11);

  // ---- sharded: collect the peers' sums, add the `world` contributions in rank order (bitwise the same
  //      total on every rank) and finalise ----
  if (sharded) {
    __syncthreads();
    for (int pi = 0; pi < npend; ++pi) {
      const int c = s_pend[pi];
      const unsigned seq = s_pend_seq[pi];
      load_aux(c);
      if (!TRAJ && warp == 0 && lane < 13) s_th[lane] = load_param(theta, theta_is_q, c, lane);  // as warp 6 computed it
      if (tid < 32 * xch.world) {
        const int r = tid >> 5, j = tid & 31;
        const unsigned long long* mine = xch.buf[xch.rank] + ((((size_t)(seq & 1u) * xch.world + r) * xch.cmax + c) << 5) + j;
        unsigned long long word, t_start, t_now;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_start));
        do {
          asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(word) : "l"(mine) : "memory");
          asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_now));
        } while ((unsigned)(word >> 32) != seq && t_now - t_start < kXchTimeoutNs);
        if ((unsigned)(word >> 32) != seq) *xch.err = 1u;  // watchdog: never hang the GPU
        s_xw[r][j] = (unsigned)word;
        // exchange cost, kept apart from compute: how long this CTA sat waiting for peer r's sums
        if (j == 0) {
          atomicAdd(xch.stat + r, t_now - t_start);
          if (r == 0) atomicAdd(xch.stat + kMaxPeers, 1ull);
        }
      }
      __syncthreads();
      if (tid < kNSums) {
        double tot = 0.0;
        for (int r = 0; r < xch.world; ++r) tot += __hiloint2double((int)s_xw[r][2 * tid + 1], (int)s_xw[r][2 * tid]);
        s_red[0][tid] = tot;
        if (sums) sums[(size_t)c * kNSums + tid] = tot;
      }
      __syncthreads();
      if (warp == 0) finalize_chain(c, 0, 1);
      __syncthreads();
    }
  }
  SPAN_END();
}

// one warp per chain
__global__ void k_finalize(const int C, const double* __restrict__ theta,
                           const double* __restrict__ sums, const FinalizeCfg fin,
                           const Priors* __restrict__ priors) {
  const int c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (c >= C) return;
  if (fin.mode == 1) {
    if (lane == 0)
      finalize_loglik(&theta[(size_t)c * 13], &sums[(size_t)c * kNSums], fin.tot, &fin.out_val[c],
                      fin.out_grad ? &fin.out_grad[(size_t)c * 13] : nullptr);
  } else {
    __shared__ double s_th[4][16];  // 128 threads = 4 chains per CTA
    __shared__ PriorPre s_pre[4][17];
    const int wv = threadIdx.x >> 5;
    if (lane < 13) s_th[wv][lane] = load_param(theta, 1, c, lane);
    if (lane < 17) s_pre[wv][lane] = prior_pre(lane, theta[(size_t)c * 17 + lane], priors->v[lane]);
    __syncwarp();
    finalize_logp_post(lane, s_pre[wv], s_th[wv], lik_pre(s_th[wv][N_SIGMA], s_th[wv][S_SIGMA]),
                       &sums[(size_t)c * kNSums], fin.tot, &fin.out_val[c],
                       fin.out_grad ? &fin.out_grad[(size_t)c * 17] : nullptr);
  }
}

}  // namespace
