// libabd_b200.so -- kernels (sm_100a) and the C ABI declared in include/abd_b200.h.
//
// HBM layout (all built once in abd_create, see DESIGN.md):
//   pcr[N], vac[N]              one bit mask over gaps per individual: uint32 (G <= 31), uint64 (G <= 63) or
//                               128 bits (G <= 127), see with_mask
//   per antigen a in {N, S}:    CSR by individual -- rp_a[N+1] (int32), and row arrays sorted by
//                               (individual, gap): od_a[R_a] f64, x_a[R_a] f64,
//                               meta_a[R_a] u32 = individual << 6 | gap (<< 7 with 128-bit masks)
//   per chain (resident state): i_raw[C][G][N] int8, waner[C][N] int8  (the reference layout), and beside it
//                               PackedState[C][N] (raw bit mask | waner, constrained infections): what the kernels read
//
// Files
//   abd_device.cuh          per-individual building blocks (constraints, trajectories, row likelihood,
//                           finaliser, Philox, fast exp / reciprocal, mbarrier + bulk-copy wrappers)
//   abd_kernels_common.cuh  device view of the cohort, launch configurations
//   k_sums.cuh              k_sums (joint logp + gradient sums, fused finaliser, persistent trajectory
//                           mode, fused peer all-reduce), k_finalize
//   k_gibbs.cuh             k_gibbs (Gibbs sweep, conditional log-odds); k_gibbs_blk.cuh: the per-chunk block draw
//   k_infprob.cuh           k_infprob_accum (Rao-Blackwellised posterior infection and waner probabilities)
//   k_nuts.cuh              the No-U-Turn tree (k_nuts_begin / k_nuts_leaf / k_nuts_end; nuts_leaf_chain is also called by
//                           the finishing warp of k_sums' single-step leapfrog launches)
//   k_misc.cuh              k_hmc_begin / k_hmc_end, k_determ, k_determ_accum, k_loglik_rows, k_pack, k_pull, k_debug_fast_math
//   abd_b200.cu (this file) host side: cohort preprocessing, cache file, tilings and grid plans, the C ABI
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <type_traits>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/abd_b200.h"
#include "abd_device.cuh"

using namespace abd;

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}

#define CU(call)                                                                              \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess)                                                                    \
      return fail(ABD_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));          \
  } while (0)

}  // namespace

#include "abd_kernels_common.cuh"
#include "k_sums.cuh"
#include "k_gibbs.cuh"
#include "k_gibbs_blk.cuh"
#include "k_infprob.cuh"
#include "k_misc.cuh"


// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
namespace {

// Device allocations released together: a handle's cohort arrays, its per-chain buffers, or one call's temporaries
// (cudaFree waits for the device, so temporaries may go out of scope while work that uses them is still queued)
struct DevBufs {
  std::vector<void*> ptrs;
  template <typename T>
  int alloc(T** p, size_t n) {
    void* q = nullptr;
    cudaError_t e = cudaMalloc(&q, std::max<size_t>(n, 1) * sizeof(T));
    if (e != cudaSuccess) return fail(ABD_ERR_ALLOC, std::string("cudaMalloc: ") + cudaGetErrorString(e));
    ptrs.push_back(q);
    *p = (T*)q;
    return ABD_OK;
  }
  void release() {
    for (void* p : ptrs) cudaFree(p);
    ptrs.clear();
  }
  ~DevBufs() { release(); }
};

// Preprocessed-cohort cache file (SURVEY 8f-4: TiterData -> device upload format).  Its header is also the
// description of the cohort every handle is built from (new_handle), whether abd_create derived it or a file carried it.
struct CacheHeader {
  char magic[8];           // "ABDB200\0"
  int32_t version, G, N, n_chunks;
  uint64_t chunk_mask[3];
  int32_t wide, fx, n_xlev, has_pcr;   // wide: mask layout, 0 = 32, 1 = 64, 2 = 128 bits
  int64_t R[2], K[2];      // OD rows / (individual, gap) cells per antigen (N, S)
  double tot[4];
  uint32_t ind_offset, pad;
  double xlev[kMaxXLevels];
};
// Version 2: 32- and 64-bit masks.  Version 3 (128-bit masks): the same header, then the chunk masks' high words
// (gaps 64..127) before the arrays.
constexpr int kCacheVersion = 2, kCacheVersionWide = 3;

struct CohortDesc {
  CacheHeader hd;
  uint64_t mask_hi[3];  // the chunk masks' high words
};

}  // namespace

struct abd_handle {
  int device = 0;
  int G = 0, N = 0;
  int mask_bits = 32;  // gap-mask layout (32, 64 or 128 bits): read through with_mask only
  int64_t R[2] = {0, 0};
  Totals tot{};
  DevCohort dc{};
  CohortDesc desc{};          // what the handle was built from (abd_save_cache writes it)
  DevBufs owned;              // cohort arrays and other allocations that live as long as the handle
  std::vector<int> h_rp[2];   // host copy of the row CSR pointers (for tilings)
  std::vector<int> h_cp[2];   // host copy of the cell CSR pointers
  cudaStream_t stream = nullptr;
  Priors* d_priors = nullptr;
  int64_t launches = 0;

  struct Tiling {
    int ntiles = 0;
    void* d_tiles = nullptr;   // TileDesc[ntiles]
    int cap_n = 0, cap_s = 0, capr_n = 0, capr_s = 0, capk_n = 0, capk_s = 0;  // staging capacities (elements)
    size_t smem = 0;                                     // dynamic shared memory per CTA (0 = does not fit at all)
    int occ = 0;                                         // resident CTAs per SM (0 = not queried yet)
    size_t smem_cp = 0;                                  // the same with the compact cell layout (factored mode; 0 = none)
    int occ_cp = 0;
  };
  std::map<int, Tiling> tilings;  // keyed by number of tiles requested
  int last_plan[6] = {0, 0, 0, 0, 0, 0};  // abd_last_plan
  bool force_compact = false;
  int tile_rows_override = 0;     // 0 = automatic
  int chains_per_cta_override = 0;
  int n_sms = 148;
  size_t smem_optin = 0;
  int* d_order = nullptr;       // individuals by decreasing OD-row count (Gibbs work queue)
  int gibbs_ctas = 0;
  int gibbs_blk_ctas = 0;
  ThetaInline thin{};           // parameters passed by value with the next k_sums launch (n = 0: none)
  // peer exchange (individual sharding over NVLink)
  XchCfg xch{};
  void* xch_local = nullptr;
  void* xch_peer[kMaxPeers] = {};
  bool fx = false;              // factored mode: rows carry (cell, dilution index), see k_sums

  // per-chain buffers for cap_chains chains: allocated by ensure_chains, released by free_chains
  int cap_chains = 0;
  DevBufs chain_bufs;
  int8_t* d_iraw = nullptr;
  int8_t* d_waner = nullptr;
  void* d_pack = nullptr;      // PackedState<M>[C][N] beside the int8 state (see abd_kernels_common.cuh)
  int pack_valid = 0;          // leading chains whose packed entries mirror d_iraw / d_waner
  bool lazy_pack = true;       // a launch on the resident state may (re)build the packed copy first
  double* d_theta = nullptr;   // [C][17]
  double* d_p = nullptr;       // [C][2]
  double* d_sums = nullptr;    // [C][16]
  double* d_out = nullptr;     // [C][18]
  unsigned* d_ticket = nullptr;
  double* d_aux = nullptr;     // [C][kAuxDoubles] finaliser inputs that depend on parameters only
  double* d_traj = nullptr;    // [C][34] trajectory-mode scratch (position, half-step momentum)
  unsigned* d_gen = nullptr;   // [C + 1] generation counters + error flag
  unsigned long long* d_stats = nullptr;
  unsigned* d_queue = nullptr; // Gibbs work queues: one counter per chain
  double* h_pin = nullptr;     // pinned staging [C][40]
  double* h_pin_dev = nullptr; // the same buffer as the device sees it
  // k_sums' partial sums, sized by the grid plan
  DevBufs partial_buf;
  double* d_partial = nullptr;
  size_t cap_partial = 0;
};

namespace {

// The one place that turns a handle's mask layout into the kernels' mask type: returns f(M{}) for M = uint32_t,
// uint64_t or u128.
template <typename F>
auto with_mask(const abd_handle* h, F&& f) {
  if (h->mask_bits == 128) return f(u128{});
  if (h->mask_bits == 64) return f(uint64_t{});
  return f(uint32_t{});
}
// mask layout for a cohort of G gaps, as the cache header's `wide` field: the narrowest that holds G gaps and the waner
// bit (new_handle turns it into mask_bits)
int wide_for(int G) { return G <= 31 ? 0 : (G <= 63 ? 1 : 2); }

template <typename T>
int upload(abd_handle* h, T** dptr, const std::vector<T>& v) {
  int rc = h->owned.alloc(dptr, v.size());
  if (rc) return rc;
  if (!v.empty()) CU(cudaMemcpy(*dptr, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
  return ABD_OK;
}

Priors default_priors(int G) {
  // abd.py:424 p ~ Beta(1, G-1); :329-340 N response; :367-388 S response; :464-467 sigmoids
  auto normal = [](double mu, double sd) { return PriorSpec{0, mu, sd, -kHalfLog2Pi - std::log(sd)}; };
  auto gamma = [](double mu, double sd) {
    const double a = mu * mu / (sd * sd), b = mu / (sd * sd);
    return PriorSpec{1, a, b, -std::lgamma(a) + a * std::log(b)};
  };
  auto beta = [](double a, double b) {
    return PriorSpec{2, a, b, -(std::lgamma(a) + std::lgamma(b) - std::lgamma(a + b))};
  };
  auto expo = [](double lam) { return PriorSpec{3, lam, 0.0, std::log(lam)}; };
  Priors p;
  p.v[0] = beta(1.0, (double)(G - 1));
  p.v[1] = gamma(2.0, 0.5);
  p.v[2] = gamma(1.0, 0.5);
  p.v[3] = beta(10.0, 1.0);
  p.v[4] = normal(-2.0, 1.0);
  p.v[5] = gamma(2.0, 0.5);
  p.v[6] = beta(10.0, 1.0);
  p.v[7] = beta(1.0, 1.0);
  p.v[8] = gamma(1.0, 0.5);
  p.v[9] = gamma(1.0, 0.5);
  p.v[10] = normal(-2.0, 1.0);
  p.v[11] = normal(-1.0, 0.5);
  p.v[12] = normal(2.0, 0.5);
  p.v[13] = expo(1.0);
  p.v[14] = normal(-1.0, 0.5);
  p.v[15] = normal(2.0, 0.5);
  p.v[16] = expo(1.0);
  return p;
}

// CSR by individual for one antigen (counting sort by individual, then by gap inside)
int build_rows(abd_handle* h, int a, int64_t R, const double* x, const double* od, const int32_t* gap,
               const int32_t* ind) {
  const int N = h->N, G = h->G;
  const int gap_bits = with_mask(h, [](auto m) { return kGapBits<decltype(m)>; });
  if (R > 0 && (!x || !od || !gap || !ind)) return fail(ABD_ERR_INVALID, "NULL row array");
  if (R >= (int64_t)1 << 31) return fail(ABD_ERR_INVALID, "too many OD rows for int32 CSR");
  std::vector<int>& rp = h->h_rp[a];
  rp.assign((size_t)N + 1, 0);
  for (int64_t r = 0; r < R; ++r) {
    if (ind[r] < 0 || ind[r] >= N) return fail(ABD_ERR_INVALID, "individual index out of range");
    if (gap[r] < 0 || gap[r] >= G) return fail(ABD_ERR_INVALID, "gap index out of range");
    rp[(size_t)ind[r] + 1]++;
  }
  for (int n = 0; n < N; ++n) rp[n + 1] += rp[n];
  std::vector<int64_t> order((size_t)R);
  {
    std::vector<int> cur(rp.begin(), rp.end() - 1);
    for (int64_t r = 0; r < R; ++r) order[(size_t)cur[ind[r]]++] = r;
  }
  for (int n = 0; n < N; ++n)
    std::stable_sort(order.begin() + rp[n], order.begin() + rp[n + 1],
                     [&](int64_t p, int64_t q) { return gap[p] < gap[q]; });
  // padded so that the 16-byte-aligned bulk copies of k_sums may read past the last row
  std::vector<double> xs((size_t)R + 2, 0.0), ods((size_t)R + 2, 0.0);
  std::vector<uint32_t> meta((size_t)R + 4, 0u);
  // cells: the distinct (individual, gap) pairs, in row order; every row points at its cell
  std::vector<uint32_t> rowcell((size_t)R + 4, 0u), cmeta;
  std::vector<int>& cp = h->h_cp[a];
  cp.assign((size_t)N + 1, 0);
  std::vector<int> perm((size_t)R);
  for (int64_t k = 0; k < R; ++k) {
    const int64_t r = order[(size_t)k];
    perm[(size_t)k] = (int)r;
    xs[(size_t)k] = x[r];
    ods[(size_t)k] = od[r];
    const uint32_t m = ((uint32_t)ind[r] << gap_bits) | (uint32_t)gap[r];
    meta[(size_t)k] = m;
    if (cmeta.empty() || cmeta.back() != m) {
      cmeta.push_back(m);
      cp[(size_t)ind[r] + 1]++;
    }
    rowcell[(size_t)k] = (uint32_t)cmeta.size() - 1;
  }
  for (int n = 0; n < N; ++n) cp[n + 1] += cp[n];
  cmeta.resize(cmeta.size() + 4, 0u);
  int rc;
  int* d_rp;
  double *d_x, *d_od;
  uint32_t *d_meta, *d_rowcell, *d_cmeta;
  if ((rc = upload(h, &d_rp, rp))) return rc;
  if ((rc = upload(h, &d_x, xs))) return rc;
  if ((rc = upload(h, &d_od, ods))) return rc;
  if ((rc = upload(h, &d_meta, meta))) return rc;
  if ((rc = upload(h, &d_rowcell, rowcell))) return rc;
  if ((rc = upload(h, &d_cmeta, cmeta))) return rc;
  {
    int* d_perm;
    if ((rc = upload(h, &d_perm, perm))) return rc;
    h->dc.rowperm[a] = d_perm;
  }
  h->dc.rcx[a] = nullptr;
  if (h->fx) {
    std::vector<uint32_t> rcx((size_t)R + 4, 0u);
    for (int64_t k = 0; k < R; ++k) {
      const double* lv = h->desc.hd.xlev;
      const int xi = (int)(std::lower_bound(lv, lv + h->desc.hd.n_xlev, xs[(size_t)k]) - lv);
      rcx[(size_t)k] = (rowcell[(size_t)k] << 5) | (uint32_t)xi;
    }
    uint32_t* d_rcx;
    if ((rc = upload(h, &d_rcx, rcx))) return rc;
    h->dc.rcx[a] = d_rcx;
  }
  h->dc.rp[a] = d_rp;
  h->dc.x[a] = d_x;
  h->dc.od[a] = d_od;
  h->dc.meta[a] = d_meta;
  h->dc.rowcell[a] = d_rowcell;
  h->dc.cmeta[a] = d_cmeta;
  return ABD_OK;
}

// Split the individuals into `want` contiguous tiles of (nearly) equal OD-row count, at most
// kTileMaxInds individuals each, and size the shared-memory staging buffers for the largest.
int get_tiling(abd_handle* h, int want, abd_handle::Tiling** out) {
  auto it = h->tilings.find(want);
  if (it == h->tilings.end()) {
    const int N = h->N;
    const std::vector<int>&rn = h->h_rp[0], &rs = h->h_rp[1];
    const double total = (double)rn[N] + (double)rs[N];
    std::vector<int> ti{0};
    int inds = 0;
    for (int n = 0; n < N; ++n) {
      // boundary before individual n if the running row count passed the next multiple of total/want
      const double before = (double)rn[n] + (double)rs[n];
      const double target = total * (double)ti.size() / (double)want;
      if (inds > 0 && (inds == kTileMaxInds || (before >= target && (int)ti.size() < want))) {
        ti.push_back(n);
        inds = 0;
      }
      ++inds;
    }
    ti.push_back(N);
    abd_handle::Tiling t;
    t.ntiles = (int)ti.size() - 1;
    const std::vector<int>&cn = h->h_cp[0], &cs = h->h_cp[1];
    auto span = [](int lo, int hi, int al) { return ((hi + al - 1) & ~(al - 1)) - (lo & ~(al - 1)); };
    for (int k = 0; k < t.ntiles; ++k) {
      const int a = ti[k], b = ti[k + 1];
      t.cap_n = std::max(t.cap_n, span(rn[a], rn[b], 2));
      t.cap_s = std::max(t.cap_s, span(rs[a], rs[b], 2));
      t.capr_n = std::max(t.capr_n, span(rn[a], rn[b], 4));
      t.capr_s = std::max(t.capr_s, span(rs[a], rs[b], 4));
      t.capk_n = std::max(t.capk_n, span(cn[a], cn[b], 4));
      t.capk_s = std::max(t.capk_s, span(cs[a], cs[b], 4));
    }
    t.cap_n = std::max(t.cap_n, 2);
    t.cap_s = std::max(t.cap_s, 2);
    t.capr_n = std::max(t.capr_n, 4);
    t.capr_s = std::max(t.capr_s, 4);
    t.capk_n = std::max(t.capk_n, 4);
    t.capk_s = std::max(t.capk_s, 4);
    const size_t rows_b = (size_t)(t.cap_n + t.cap_s) * 8 + (size_t)(t.capr_n + t.capr_s) * 4, cells = (size_t)(t.capk_n + t.capk_s);
    t.smem = rows_b + (h->fx ? cells * (sizeof(CellValT<true, false>) + 4)
                             : cells * (sizeof(CellValT<false, false>) + 4) + (size_t)(t.cap_n + t.cap_s) * 8);
    t.smem_cp = h->fx ? rows_b + cells * (sizeof(CellValT<true, true>) + 8 + 4) : 0;
    if (t.smem_cp && t.smem_cp + 12 * 1024 > h->smem_optin) t.smem_cp = 0;
    if (t.smem + 12 * 1024 > h->smem_optin) t.smem = 0;
    if (!t.smem && !t.smem_cp)
      return fail(ABD_ERR_INVALID, "an individual tile does not fit in shared memory (too many OD rows per 128 individuals)");
    std::vector<TileDesc> desc((size_t)t.ntiles);
    for (int k = 0; k < t.ntiles; ++k) {
      const int a = ti[k], b = ti[k + 1];
      desc[(size_t)k] = TileDesc{a, b, rn[a], rn[b], rs[a], rs[b], cn[a], cn[b], cs[a], cs[b], 0, 0};
    }
    TileDesc* d_desc = nullptr;
    int rc = upload(h, &d_desc, desc);
    if (rc) return rc;
    t.d_tiles = d_desc;
    it = h->tilings.emplace(want, t).first;
  }
  *out = &it->second;
  return ABD_OK;
}

void free_chains(abd_handle* h) {
  h->chain_bufs.release();
  if (h->h_pin) cudaFreeHost(h->h_pin);
  h->h_pin = h->h_pin_dev = nullptr;
  h->cap_chains = h->pack_valid = 0;
}

int ensure_chains(abd_handle* h, int C) {
  if (C <= 0) return fail(ABD_ERR_INVALID, "n_chains must be positive");
  if (C > 65535) return fail(ABD_ERR_INVALID, "n_chains must be <= 65535");
  if (C <= h->cap_chains) return ABD_OK;
  CU(cudaStreamSynchronize(h->stream));
  const int oldC = h->cap_chains;
  const size_t gn = (size_t)h->G * h->N;
  int rc;
  // the chain state moves to the larger buffers; everything else starts afresh
  DevBufs next;
  int8_t *ni, *nw;
  if ((rc = next.alloc(&ni, (size_t)C * gn)) || (rc = next.alloc(&nw, (size_t)C * h->N))) return rc;
  CU(cudaMemset(ni, 0, (size_t)C * gn));
  CU(cudaMemset(nw, 0, (size_t)C * h->N));
  if (oldC) {
    CU(cudaMemcpy(ni, h->d_iraw, (size_t)oldC * gn, cudaMemcpyDeviceToDevice));
    CU(cudaMemcpy(nw, h->d_waner, (size_t)oldC * h->N, cudaMemcpyDeviceToDevice));
  }
  free_chains(h);
  std::swap(h->chain_bufs.ptrs, next.ptrs);
  h->d_iraw = ni;
  h->d_waner = nw;
  DevBufs& b = h->chain_bufs;
  char* pk = nullptr;
  const size_t entry = with_mask(h, [](auto m) { return sizeof(PackedState<decltype(m)>); });
  if ((rc = b.alloc(&pk, (size_t)C * h->N * entry))) return rc;
  h->d_pack = pk;
  if ((rc = b.alloc(&h->d_theta, (size_t)C * 17)) || (rc = b.alloc(&h->d_p, (size_t)C * 2)) ||
      (rc = b.alloc(&h->d_sums, (size_t)C * kNSums)) || (rc = b.alloc(&h->d_out, (size_t)C * 18)) ||
      (rc = b.alloc(&h->d_ticket, (size_t)C)) || (rc = b.alloc(&h->d_aux, (size_t)C * kAuxDoubles)) ||
      (rc = b.alloc(&h->d_traj, (size_t)C * 34)) || (rc = b.alloc(&h->d_gen, (size_t)C + 1)) ||
      (rc = b.alloc(&h->d_stats, (size_t)C * 2)) || (rc = b.alloc(&h->d_queue, (size_t)C)))
    return rc;
  CU(cudaMemset(h->d_ticket, 0, (size_t)C * sizeof(unsigned)));
  CU(cudaMemset(h->d_gen, 0, ((size_t)C + 1) * sizeof(unsigned)));
  CU(cudaMallocHost((void**)&h->h_pin, (size_t)C * 40 * sizeof(double)));
  {
    void* dp = nullptr;
    if (cudaHostGetDevicePointer(&dp, h->h_pin, 0) == cudaSuccess) h->h_pin_dev = (double*)dp;
    else cudaGetLastError();
  }
  h->cap_chains = C;
  return ABD_OK;
}

// Grid plan: CTAs = tiles x chain groups.  Up to a few waves' worth of work the grid is sized
// to exactly `waves` full waves of resident CTAs (n_sms x CTAs-per-SM), so every SM gets the
// same number of equally sized tiles and there is no partial last wave; beyond that the tail is
// negligible and tiles simply hold ~`target` OD rows (a handful per thread).
// `one_wave_rows`: tiles may grow to this many OD rows if that lets the whole grid run as ONE wave (12 500 individuals x
// 4 chains -- an eighth of the 100k cohort -- is 1.25 waves of 2 200-row tiles: two waves, 18.4 us, against one wave of
// 2 650-row tiles); 0 = the ordinary limit.  The caller falls back to 0 when such tiles do not fit in shared memory.
// `cpc_fixed`: chains per CTA (0 = the planner's choice).
constexpr int kTileRowsOneWave = 2750;
void plan_grid(const abd_handle* h, int C, int ctas_per_sm, int cpc_fixed, int one_wave_rows, int* want_tiles,
               int* chains_per_cta) {
  const double rows = (double)(h->R[0] + h->R[1]);
  const int target = h->tile_rows_override > 0 ? h->tile_rows_override : 2200;
  const int min_tiles = (h->N + kTileMaxInds - 1) / kTileMaxInds;
  const int resident = h->n_sms * ctas_per_sm;
  // tiles for `cpc` chains per CTA; returns the number of waves the grid then takes
  auto tiles_for = [&](int cpc, int* tiles_out) -> double {
    const int groups = (C + cpc - 1) / cpc;
    int tiles = std::max(min_tiles, (int)std::ceil(rows / target));
    double waves = std::ceil((double)tiles * groups / resident);
    if ((long)tiles * groups <= 6L * resident) {
      for (int w = 1; w <= 6; ++w) {
        const int t = (resident * w) / groups;
        const double limit = (w == 1 && one_wave_rows > target && h->tile_rows_override == 0) ? (double)one_wave_rows : target * 1.02;
        if (t >= min_tiles && t >= 1 && rows / t <= limit) {
          tiles = t;
          waves = w;
          break;
        }
      }
    }
    *tiles_out = std::max(1, std::min(tiles, h->N));
    return waves;
  };
  // chains looped over inside one CTA (the staged tile is reused): measured at 10k / 12.5k individuals, 32 chains run
  // 4 - 11 % faster with 2 per CTA than with 4 (twice the waves: shorter start-up and drain), 128 chains 5 % faster
  // with 4 than with 2, and 8 / 16 per CTA are 10 / 25 % slower than 4 (tools/tune.py sums)
  int cpc = cpc_fixed > 0 ? cpc_fixed : (C >= 64 ? 4 : (C >= 32 ? 2 : 1));
  cpc = std::min(cpc, C);
  cpc = std::min(cpc, kMaxChainsPerCta);  // a CTA remembers at most this many chains it finished last (k_sums: s_pend)
  int tiles;
  const double waves1 = tiles_for(cpc, &tiles);
  if (cpc_fixed == 0 && cpc == 1 && waves1 >= 3.0) {
    // Few chains on a cohort of several waves: a wave of one-chain CTAs costs ~9.3 us whatever its tile size, a CTA
    // that loops over k chains ~1 + 8.3 k us per wave (measured, 4 chains: 25 000 individuals 28.3 us as 3 waves
    // against 21.2 as ONE wave of two-chain CTAs; 50 000 individuals 47.1 as 5 waves against 35.8 as one wave of
    // four-chain CTAs).  Taken only when the estimate wins by 15 %: e.g. not at 100 000 individuals (82.7 against 85.7).
    double best = 9.3 * waves1;
    for (int k = 2; k <= 4 && k <= C; k *= 2) {
      if (C % k) continue;
      int tk;
      const double cost = tiles_for(k, &tk) * (1.0 + 8.3 * k);
      if (cost < 0.85 * 9.3 * waves1 && cost < best) best = cost, cpc = k, tiles = tk;
    }
  }
  *want_tiles = tiles;
  *chains_per_cta = cpc;
}

// One k_sums instantiation, as a type (its shared-memory setting is remembered per instantiation)
template <typename M, typename XT, bool TRAJ, bool CP>
struct SumsKernel {
  using Mask = M;
  static auto fn() { return k_sums<M, XT, TRAJ, CP>; }
};

// The one place that picks the k_sums instantiation for a launch: returns f(SumsKernel<...>{}) for the handle's mask
// layout and dilution mode (fx), the compact cell layout or not, and trajectory mode or not.
template <typename F>
auto with_sums(const abd_handle* h, bool compact, bool traj, F&& f) {
  return with_mask(h, [&](auto m) {
    using M = decltype(m);
    if (compact) return traj ? f(SumsKernel<M, uint8_t, true, true>{}) : f(SumsKernel<M, uint8_t, false, true>{});
    if (h->fx) return traj ? f(SumsKernel<M, uint8_t, true, false>{}) : f(SumsKernel<M, uint8_t, false, false>{});
    return traj ? f(SumsKernel<M, double, true, false>{}) : f(SumsKernel<M, double, false, false>{});
  });
}

// The dynamic shared-memory limit of a kernel is a per-device function attribute shared by every
// handle of the process: only ever raise it (a small cohort must not lower it under a large one).
template <typename K>
cudaError_t sums_smem_attr(K, int device, size_t smem) {
  static size_t configured[64] = {};
  const int d = (device >= 0 && device < 64) ? device : 0;
  const size_t want = std::max<size_t>(smem, 48 * 1024);
  if (want <= configured[d]) return cudaSuccess;
  cudaError_t e = cudaFuncSetAttribute(K::fn(), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)want);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(K::fn(), cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  if (e != cudaSuccess) return e;
  configured[d] = want;
  return cudaSuccess;
}

// resident CTAs per SM of the plain-evaluation kernel for this handle's mask width / dilution mode
cudaError_t sums_occupancy(const abd_handle* h, bool compact, size_t smem, int* occ) {
  return with_sums(h, compact, false, [&](auto k) {
    cudaError_t e = sums_smem_attr(k, h->device, smem);
    if (e != cudaSuccess) return e;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(occ, decltype(k)::fn(), kSumsBlock, smem);
  });
}

// A launch configuration that lets the kernel start while the previous one on the stream drains (programmatic
// dependent launch); `attr` is the caller's storage for the one launch attribute
cudaLaunchConfig_t pdl_config(dim3 grid, dim3 block, size_t smem, cudaStream_t st, cudaLaunchAttribute* attr) {
  cudaLaunchConfig_t lc{};
  lc.gridDim = grid;
  lc.blockDim = block;
  lc.dynamicSmemBytes = smem;
  lc.stream = st;
  attr->id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr->val.programmaticStreamSerializationAllowed = 1;
  lc.attrs = attr;
  lc.numAttrs = 1;
  return lc;
}

// The packed copy of the resident chain state for a launch that reads (i_raw, waner): non-null only
// when those ARE the handle's resident buffers.  If the copy is stale it is rebuilt first (one small
// launch on the same stream) unless the caller has just staged fresh host state for a single use.
int resident_pack(abd_handle* h, int C, const int8_t* i_raw, const int8_t* waner, cudaStream_t st, void** out) {
  *out = nullptr;
  if (i_raw != h->d_iraw || waner != h->d_waner || !h->d_pack) return ABD_OK;
  if (h->pack_valid < C) {
    if (!h->lazy_pack) return ABD_OK;
    dim3 grid((h->N + 127) / 128, C);
    with_mask(h, [&](auto m) {
      using M = decltype(m);
      k_pack<M><<<grid, 128, 0, st>>>(h->dc, h->d_iraw, h->d_waner, (PackedState<M>*)h->d_pack);
    });
    CU(cudaGetLastError());
    h->launches++;
    h->pack_valid = C;
  }
  *out = h->d_pack;
  return ABD_OK;
}

// `sharded`: the fused launch that all-reduces the sums with the peers of the exchange (see abd_xch_connect)
int launch_sums(abd_handle* h, int C, const double* theta, int theta_is_q, const int8_t* i_raw,
                const int8_t* waner, double* sums, const FinalizeCfg& fin, cudaStream_t st,
                const TrajCfg* traj_in = nullptr, bool sharded = false) {
  TrajCfg traj{};
  if (traj_in) traj = *traj_in;
  const ThetaInline thin = h->thin;  // consumed by this call whatever happens below
  h->thin.n = 0;
  // a single leapfrog step waits on nothing inside the grid: the ordinary plan with one chain per CTA (the trajectory
  // variant keeps a chain's position in shared memory), any number of waves
  const int cpc_fixed = traj.n_steps == 1 ? 1 : h->chains_per_cta_override;
  // plan for the kernel's register-limited occupancy first; if the tiles that plan needs do not
  // fit that many CTAs per SM (shared memory), plan again for what actually fits
  int want, cpc, rc;
  bool compact = false;
  abd_handle::Tiling* tl = nullptr;
  for (int attempt = 0; attempt < 2 * ABD_SUMS_MINB; ++attempt) {
    const int occ = ABD_SUMS_MINB - attempt / 2;
    const int one_wave_rows = (attempt & 1) ? 0 : kTileRowsOneWave;  // first with the larger one-wave tiles, then without
    plan_grid(h, C, occ, cpc_fixed, one_wave_rows, &want, &cpc);
    if (traj.n_steps > 1 && cpc != 1) {  // persistent trajectory: re-plan with one chain per CTA, exactly one wave
      cpc = 1;
      want = std::max((h->N + kTileMaxInds - 1) / kTileMaxInds, (h->n_sms * occ) / C);
      want = std::max(1, std::min(want, h->N));
    }
    if ((rc = get_tiling(h, want, &tl))) return rc;
    // the 32-byte cells if the tile fits `occ` CTAs per SM with them (two shared-memory loads per row), else the
    // compact cells (three narrower loads per row: 2 % slower at equal tiles, but 12 500 individuals x 4 chains -- an
    // eighth of the 100k cohort -- then run as one wave: 18.5 -> 11.6 us per launch)
    if (tl->smem && !tl->occ) {
      int o = 0;
      CU(sums_occupancy(h, false, tl->smem, &o));
      tl->occ = std::max(o, 1);
    }
    compact = false;
    if (tl->smem && tl->occ >= occ && !(h->force_compact && tl->smem_cp)) break;
    if (tl->smem_cp && !tl->occ_cp) {
      int o = 0;
      CU(sums_occupancy(h, true, tl->smem_cp, &o));
      tl->occ_cp = std::max(o, 1);
    }
    compact = tl->smem_cp != 0;
    if (compact && tl->occ_cp >= occ) break;
  }  // (the last attempts ask for one CTA per SM, which any tiling get_tiling accepted provides: the loop always breaks)
  const int tl_occ = compact ? tl->occ_cp : tl->occ;
  if (traj.n_steps > 1) {
    // persistent mode: one chain per CTA and every CTA resident at once
    if (cpc != 1 || (long)tl->ntiles * C > (long)h->n_sms * tl_occ)
      return fail(ABD_ERR_INVALID, "abd_leapfrog_dev: too many chains for one resident grid on this cohort; "
                                   "use abd_logp_dlogp_dev per step");
  }
  const size_t need = (size_t)C * tl->ntiles * kNSums;
  if (need > h->cap_partial) {
    CU(cudaStreamSynchronize(st));
    h->partial_buf.release();
    h->cap_partial = 0;
    if ((rc = h->partial_buf.alloc(&h->d_partial, need))) return rc;
    h->cap_partial = need;
  }
  SumsCfg cfg{tl->ntiles, tl->cap_n, tl->cap_s, tl->capr_n, tl->capr_s, tl->capk_n, tl->capk_s, cpc, C};
  dim3 grid(tl->ntiles, (C + cpc - 1) / cpc);
  const size_t smem = compact ? tl->smem_cp : tl->smem;
  h->last_plan[0] = tl->ntiles, h->last_plan[1] = (int)grid.y, h->last_plan[2] = cpc;
  h->last_plan[3] = (int)smem, h->last_plan[4] = compact ? 1 : 0, h->last_plan[5] = tl_occ;
  void* pack = nullptr;
  if ((rc = resident_pack(h, C, i_raw, waner, st, &pack))) return rc;
  const bool tj = traj.n_steps > 0;
  rc = with_sums(h, compact, tj, [&](auto k) -> int {
    using K = decltype(k);
    CU(sums_smem_attr(k, h->device, smem));
    cudaLaunchAttribute attr;
    cudaLaunchConfig_t lc = pdl_config(grid, dim3(kSumsBlock), smem, st, &attr);
    if (traj.n_steps > 1) {  // CTAs wait on one another: they must all be resident
      int occ = 0;
      CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, K::fn(), kSumsBlock, smem));
      if ((long)grid.x * grid.y > (long)occ * h->n_sms)
        return fail(ABD_ERR_INVALID, "abd_leapfrog_dev: the grid does not fit on the device at once");
      attr.id = cudaLaunchAttributeCooperative;
      attr.val.cooperative = 1;
    }
    CU(cudaLaunchKernelEx(&lc, K::fn(), h->dc, reinterpret_cast<const TileDesc*>(tl->d_tiles), cfg, theta, theta_is_q, i_raw,
                          waner, reinterpret_cast<const PackedState<typename K::Mask>*>(pack), h->d_partial, h->d_ticket, sums,
                          fin, h->d_priors, h->d_aux, traj, sharded ? h->xch : XchCfg{}, tj ? ThetaInline{} : thin));
    return ABD_OK;
  });
  if (rc) return rc;
  CU(cudaGetLastError());
  h->launches++;
  return ABD_OK;
}

int launch_gibbs(abd_handle* h, int C, const double* theta, int theta_is_q, const double* p,
                 const double* pw, int8_t* i_raw, int8_t* waner, const GibbsCfg& cfg, cudaStream_t st) {
  const bool blk = cfg.mode == ABD_GIBBS_BLOCKED;
  if (blk && (h->mask_bits > 32 || h->dc.ch.n < 2)) {
    // no "first raw 1 of the chunk" structure (one chunk) or more options than lanes (masks wider than 32 bits):
    // single-site exact conditionals instead
    GibbsCfg c2 = cfg;
    c2.mode = ABD_GIBBS_HEATBATH;
    return launch_gibbs(h, C, theta, theta_is_q, p, pw, i_raw, waner, c2, st);
  }
  return with_mask(h, [&](auto m) -> int {
    using M = decltype(m);
    auto kernel = k_gibbs<M>;
    if constexpr (std::is_same_v<M, uint32_t>)
      if (blk) kernel = k_gibbs_blk;
    int& ctas = blk ? h->gibbs_blk_ctas : h->gibbs_ctas;  // one persistent wave
    if (!ctas) {
      int occ = 0;
      CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, kGibbsWarps * 32, 0));
      ctas = h->n_sms * std::max(occ, 1);
    }
    const long items = (long)C * h->N;
    const int grid = (int)std::min<long>(ctas, (items + kGibbsWarps - 1) / kGibbsWarps);
    CU(cudaMemsetAsync(h->d_queue, 0, (size_t)C * sizeof(unsigned), st));
    void* pack = nullptr;
    if (int rc = resident_pack(h, C, i_raw, waner, st, &pack)) return rc;
    kernel<<<grid, kGibbsWarps * 32, 0, st>>>(h->dc, h->d_order, C, theta, theta_is_q, p, pw, i_raw, waner,
                                              (PackedState<M>*)pack, h->d_queue, cfg);
    CU(cudaGetLastError());
    h->launches++;
    return ABD_OK;
  });
}

int set_device(const abd_handle* h) {
  CU(cudaSetDevice(h->device));
  return ABD_OK;
}

// Copy of a chain-state array between the host and the device (`dir`).  A copy-engine transfer of ~1 MB from pinned
// memory takes ~60 us on a B200 host (PCIe gen5, measured, whatever the stream count); when the host side is pinned
// (page-locked, hence mapped into the device's address space under UVA) and 16-byte aligned, the SMs move it
// themselves with 16-byte loads and stores -- every byte of the transfer is in flight at once and the copy runs at the
// link's bandwidth (device -> host: posted PCIe writes).  Pageable host memory takes cudaMemcpyAsync.
int copy_state(abd_handle* h, void* dst, const void* src, size_t bytes, cudaMemcpyKind dir) {
  const bool h2d = dir == cudaMemcpyHostToDevice;
  const void* host = h2d ? src : dst;
  if (bytes >= (4u << 10) && (reinterpret_cast<uintptr_t>(host) & 15u) == 0) {
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, host) == cudaSuccess && at.type == cudaMemoryTypeHost && at.devicePointer) {
      const size_t n16 = bytes / 16, rem = bytes - n16 * 16;
      const int grid = (int)std::min<size_t>((size_t)h->n_sms * 4, (n16 + 255) / 256);
      k_pull<<<grid, 256, 0, h->stream>>>(reinterpret_cast<const uint4*>(h2d ? at.devicePointer : src),
                                          reinterpret_cast<uint4*>(h2d ? dst : at.devicePointer), n16, rem);
      CU(cudaGetLastError());
      h->launches++;
      return ABD_OK;
    }
    cudaGetLastError();  // not a CUDA-known pointer: clear the sticky-free error and copy the ordinary way
  }
  CU(cudaMemcpyAsync(dst, src, bytes, dir, h->stream));
  return ABD_OK;
}

int stage_state(abd_handle* h, int C, const int8_t* i_raw, const int8_t* waner) {
  const size_t gn = (size_t)h->G * h->N;
  int rc;
  // fresh host state for (usually) a single use: the kernels of this call read the int8 arrays and the
  // packed copy goes stale; a call on the resident state (NULL pointers) rebuilds it on first use
  h->lazy_pack = !(i_raw || waner);
  if (i_raw || waner) h->pack_valid = 0;
  if (i_raw && (rc = copy_state(h, h->d_iraw, i_raw, (size_t)C * gn, cudaMemcpyHostToDevice))) return rc;
  if (waner && (rc = copy_state(h, h->d_waner, waner, (size_t)C * h->N, cudaMemcpyHostToDevice))) return rc;
  return ABD_OK;
}

// A handle for the cohort `d` describes: its device facts, stream and priors, and every field the description fixes.
// The cohort arrays follow (built by abd_create, read by abd_create_from_cache).
int new_handle(abd_handle** out, int device, const CohortDesc& d) {
  abd_handle* h = new abd_handle();
  h->device = device;
  if (const char* e = std::getenv("ABD_B200_COMPACT_CELLS")) h->force_compact = (e[0] == '1');  // tests: compact cells wherever they exist
  {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && v > 0) h->n_sms = v;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, device) == cudaSuccess) h->smem_optin = (size_t)v;
  }
  const CacheHeader& hd = d.hd;
  h->desc = d;
  h->G = h->dc.G = hd.G;
  h->N = h->dc.N = hd.N;
  h->mask_bits = 32 << hd.wide;
  h->R[0] = hd.R[0], h->R[1] = hd.R[1];
  h->tot = Totals{hd.tot[0], hd.tot[1], hd.tot[2], hd.tot[3]};
  h->dc.ind_offset = hd.ind_offset;
  h->dc.chain_offset = 0;
  h->dc.ch.n = hd.n_chunks;
  for (int k = 0; k < 3; ++k) h->dc.ch.mask[k] = hd.chunk_mask[k], h->dc.ch.mask_hi[k] = d.mask_hi[k];
  h->fx = hd.fx != 0;
  h->dc.n_xlev = hd.n_xlev;
  int rc = ABD_OK;
  double* d_lv = nullptr;
  if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) rc = fail(ABD_ERR_CUDA, "cudaStreamCreate failed");
  if (!rc) rc = upload(h, &d_lv, std::vector<double>(hd.xlev, hd.xlev + kMaxXLevels));
  if (!rc) rc = upload(h, &h->d_priors, std::vector<Priors>{default_priors(hd.G)});
  if (rc) {
    abd_destroy(h);
    return rc;
  }
  h->dc.xlev = d_lv;
  *out = h;
  return ABD_OK;
}

// ---- preprocessed-cohort cache file ---------------------------------------------------------------------
// Everything abd_create derives from the cohort (bit masks, CSR row / cell tables sorted by individual and
// gap, packed row -> cell / dilution words, the Gibbs work order) as one binary file: the header (CacheHeader), then
// the arrays in a fixed order, each padded to 16 bytes.  Loading it is reading + uploading.
struct CacheIo {
  FILE* f = nullptr;
  bool writing = false, ok = true;
  ~CacheIo() {
    if (f) std::fclose(f);
  }
  void raw(void* p, size_t bytes) {
    if (!ok || !bytes) return;
    ok = writing ? std::fwrite(p, 1, bytes, f) == bytes : std::fread(p, 1, bytes, f) == bytes;
    const size_t padn = (16 - bytes % 16) % 16;
    char z[16] = {};
    if (ok && padn) ok = writing ? std::fwrite(z, 1, padn, f) == padn : std::fread(z, 1, padn, f) == padn;
  }
};

// one device array <-> the file (through a host bounce buffer)
template <typename T>
int cache_array(abd_handle* h, CacheIo& io, T** dptr, size_t n, std::vector<T>* keep = nullptr) {
  std::vector<T> host(n);
  if (io.writing) {
    if (n) CU(cudaMemcpy(host.data(), *dptr, n * sizeof(T), cudaMemcpyDeviceToHost));
    io.raw(host.data(), n * sizeof(T));
  } else {
    io.raw(host.data(), n * sizeof(T));
    if (!io.ok) return fail(ABD_ERR_INVALID, "cache file truncated");
    int rc = upload(h, dptr, host);
    if (rc) return rc;
    if (keep) *keep = host;
  }
  return io.ok ? ABD_OK : fail(ABD_ERR_INVALID, "cache file I/O error");
}

// the cohort arrays of a handle, in file order (shared by save and load)
int cache_body(abd_handle* h, CacheIo& io) {
  const CacheHeader& hd = h->desc.hd;
  int rc;
  const size_t N = (size_t)hd.N;
  rc = with_mask(h, [&](auto m) {
    using M = decltype(m);
    M *p = (M*)h->dc.pcr, *v = (M*)h->dc.vac;
    const int r = cache_array(h, io, &p, N);
    if (r) return r;
    h->dc.pcr = p;
    const int r2 = cache_array(h, io, &v, N);
    h->dc.vac = v;
    return r2;
  });
  if (rc) return rc;
  for (int a = 0; a < 2; ++a) {
    const size_t R = (size_t)hd.R[a], K = (size_t)hd.K[a];
    int* rp = (int*)h->dc.rp[a];
    double *x = (double*)h->dc.x[a], *od = (double*)h->dc.od[a];
    uint32_t *meta = (uint32_t*)h->dc.meta[a], *rowcell = (uint32_t*)h->dc.rowcell[a], *cmeta = (uint32_t*)h->dc.cmeta[a];
    uint32_t* rcx = (uint32_t*)h->dc.rcx[a];
    int* perm = (int*)h->dc.rowperm[a];
    if ((rc = cache_array(h, io, &perm, R))) return rc;
    h->dc.rowperm[a] = perm;
    if ((rc = cache_array(h, io, &rp, N + 1, &h->h_rp[a]))) return rc;
    if ((rc = cache_array(h, io, &x, R + 2)) || (rc = cache_array(h, io, &od, R + 2))) return rc;
    if ((rc = cache_array(h, io, &meta, R + 4)) || (rc = cache_array(h, io, &rowcell, R + 4))) return rc;
    if ((rc = cache_array(h, io, &cmeta, K + 4))) return rc;
    if (hd.fx && (rc = cache_array(h, io, &rcx, R + 4))) return rc;
    // the cell CSR pointers only live on the host
    if (io.writing) {
      io.raw(h->h_cp[a].data(), (N + 1) * sizeof(int));
    } else {
      h->h_cp[a].assign(N + 1, 0);
      io.raw(h->h_cp[a].data(), (N + 1) * sizeof(int));
    }
    h->dc.rp[a] = rp, h->dc.x[a] = x, h->dc.od[a] = od, h->dc.meta[a] = meta, h->dc.rowcell[a] = rowcell;
    h->dc.cmeta[a] = cmeta, h->dc.rcx[a] = hd.fx ? rcx : nullptr;
  }
  if ((rc = cache_array(h, io, &h->d_order, N))) return rc;
  return io.ok ? ABD_OK : fail(ABD_ERR_INVALID, "cache file I/O error");
}

// Results that finishing warps write straight into pinned host memory, each 8-byte slot exactly once: the host can
// watch the slots fill instead of asking the driver for the end of the stream (tools/e2e_probe.py: 25.1 -> 19.6 us per
// resident-state call of 4 chains, 61.6 -> 56.4 us with the state upload).  Every slot starts as a signalling-NaN
// pattern no result can equal; slots that do not fill within the spin budget (long launches, a faulted kernel) send
// the caller back to cudaStreamSynchronize, which also reports errors.
constexpr uint64_t kSlotUnset = 0x7FF4A5A5DEADBEEFull;
constexpr size_t kMaxPolledSlots = 18 * 64;
void unset_slots(double* ho, size_t n) {
  volatile uint64_t* slots = reinterpret_cast<volatile uint64_t*>(ho);
  for (size_t k = 0; k < n; ++k) slots[k] = kSlotUnset;
}
bool wait_slots(const double* ho, size_t n) {
  const volatile uint64_t* slots = reinterpret_cast<const volatile uint64_t*>(ho);
  const auto t0 = std::chrono::steady_clock::now();
  size_t k = 0;
  for (unsigned spins = 0; k < n; ++spins) {
    if (slots[k] != kSlotUnset) {
      ++k;
      continue;
    }
    if ((spins & 63u) == 63u && std::chrono::steady_clock::now() - t0 > std::chrono::microseconds(150)) return false;
  }
  std::atomic_thread_fence(std::memory_order_acquire);
  return true;
}

// the first C x k doubles of `v` into the pinned staging buffer and on to d_theta
int stage_params(abd_handle* h, int C, const double* v, int k) {
  std::memcpy(h->h_pin, v, (size_t)C * k * sizeof(double));
  CU(cudaMemcpyAsync(h->d_theta, h->h_pin, (size_t)C * k * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  return ABD_OK;
}

// A host-pointer evaluation on the resident state: k = 13 parameters per chain (log-likelihood and its gradient) or 17
// (joint logp and its gradient).  The finishing warps write the C values and C x k gradients straight into the pinned
// staging buffer (posted PCIe writes cost the kernel nothing), behind the parameters; the host watches those slots
// fill when there are few enough, else synchronises the stream.  Where the device cannot address the pinned buffer,
// the results take a device -> host copy.  `counts`: also read back the Bernoulli counts of every chain.
int eval_to_host(abd_handle* h, int C, const double* params, int k, double* out_val, double* out_grad, int64_t* counts) {
  int rc;
  if (C <= kInlineChains) {  // by value, inside the launch (no host -> device copy)
    h->thin.n = C * k;
    std::memcpy(h->thin.v, params, (size_t)C * k * sizeof(double));
  } else if ((rc = stage_params(h, C, params, k))) {
    return rc;
  }
  double* ho = h->h_pin + (size_t)C * 17;
  double* dout = h->h_pin_dev ? h->h_pin_dev + (size_t)C * 17 : h->d_out;
  const FinalizeCfg fin{k == 17 ? 2 : 1, h->tot, dout, dout + C};
  const size_t nres = (size_t)C * (1 + k);
  const bool poll = h->h_pin_dev && !counts && nres <= kMaxPolledSlots;
  if (poll) unset_slots(ho, nres);
  if ((rc = launch_sums(h, C, h->d_theta, k == 17, h->d_iraw, h->d_waner, h->d_sums, fin, h->stream))) return rc;
  if (!h->h_pin_dev) CU(cudaMemcpyAsync(ho, h->d_out, nres * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  // (the sums go where the parameters were staged: the launch has read those)
  if (counts)
    CU(cudaMemcpyAsync(h->h_pin, h->d_sums, (size_t)C * kNSums * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  if (!(poll && wait_slots(ho, nres))) CU(cudaStreamSynchronize(h->stream));
  std::memcpy(out_val, ho, (size_t)C * sizeof(double));
  if (out_grad) std::memcpy(out_grad, ho + C, (size_t)C * k * sizeof(double));
  if (counts)
    for (int c = 0; c < C; ++c) {
      counts[2 * c] = (int64_t)h->h_pin[(size_t)c * kNSums + S_KI];
      counts[2 * c + 1] = (int64_t)h->h_pin[(size_t)c * kNSums + S_KW];
    }
  return ABD_OK;
}

// Fused sharded launches need the exchange allocated and connected, with room for C chains
int check_xch(const abd_handle* h, int C, const char* fn) {
  if (!h->xch_local || !h->xch.buf[h->xch.world - 1] || !h->xch.buf[0])
    return fail(ABD_ERR_INVALID, std::string(fn) + ": call abd_xch_alloc and abd_xch_connect first");
  if (C > h->xch.cmax) return fail(ABD_ERR_INVALID, "more chains than abd_xch_alloc reserved");
  return ABD_OK;
}

#define PROLOGUE(h, C)                                         \
  if (!(h)) return fail(ABD_ERR_INVALID, "NULL handle");       \
  {                                                            \
    int rc_ = set_device(h);                                   \
    if (rc_) return rc_;                                       \
    rc_ = ensure_chains(h, C);                                 \
    if (rc_) return rc_;                                       \
  }

}  // namespace

extern "C" {

const char* abd_last_error(void) { return g_err.c_str(); }
int abd_version(void) { return 100; }

int abd_create(abd_handle** out, const abd_cohort* co, int device) {
  if (!out || !co) return fail(ABD_ERR_INVALID, "NULL argument");
  *out = nullptr;
  const int G = co->n_gaps, N = co->n_inds;
  if (G < 1 || G > ABD_MAX_GAPS) return fail(ABD_ERR_INVALID, "n_gaps must be in [1, 127]");
  if (N < 1 || N >= (1 << 26)) return fail(ABD_ERR_INVALID, "n_inds must be in [1, 2^26)");
  CohortDesc d{};
  CacheHeader& hd = d.hd;
  // ABD_B200_MASK_BITS=128 (tests, measurements): the 128-bit layout whatever G
  const char* mb = std::getenv("ABD_B200_MASK_BITS");
  hd.wide = (mb && std::strcmp(mb, "128") == 0) ? 2 : wide_for(G);
  if (hd.wide == 2 && N >= (1 << 25))
    return fail(ABD_ERR_INVALID, "n_inds must be < 2^25 with more than 63 gaps (128-bit masks)");
  if (!co->vacs) return fail(ABD_ERR_INVALID, "vacs is NULL");
  // check_splits, abd.py:604-622
  if (co->n_splits < 0 || co->n_splits > 2)
    return fail(ABD_ERR_INVALID, "only implemented 1-3 time chunks (0-2 splits)");  // abd.py:882
  for (int k = 0; k < co->n_splits; ++k) {
    if (co->splits[k] < 0) return fail(ABD_ERR_INVALID, "split indexes must be positive");
    if (co->splits[k] > G) return fail(ABD_ERR_INVALID, "largest split must be less than n_gaps - 1");
  }
  if (co->n_splits == 2 && co->splits[0] == co->splits[1]) return fail(ABD_ERR_INVALID, "splits not unique");
  if (co->n_splits == 2 && co->splits[0] > co->splits[1])
    return fail(ABD_ERR_INVALID, "splits must be in ascending order");

  std::memcpy(hd.magic, "ABDB200", 8);
  hd.version = hd.wide == 2 ? kCacheVersionWide : kCacheVersion;
  hd.G = G, hd.N = N;
  // time chunks, abd.py:865-882
  hd.n_chunks = co->n_splits + 1;
  {
    int edges[4] = {0, 0, 0, 0};
    for (int k = 0; k < co->n_splits; ++k) edges[k + 1] = co->splits[k];
    edges[co->n_splits + 1] = G;
    for (int k = 0; k <= co->n_splits; ++k)
      for (int t = edges[k]; t < edges[k + 1]; ++t) (t < 64 ? hd.chunk_mask[k] : d.mask_hi[k]) |= 1ull << (t & 63);
  }
  // distinct dilutions over both antigens: <= 32 of them (and no NaN) enables the factored mode
  {
    std::vector<double> lv;
    bool ok = std::getenv("ABD_B200_NO_FACTORED") == nullptr;
    for (int a = 0; a < 2 && ok; ++a) {
      const double* xa = a ? co->x_s : co->x_n;
      const int64_t Ra = a ? co->n_rows_s : co->n_rows_n;
      if (Ra > 0 && !xa) break;  // build_rows reports the NULL
      double last = std::nan("");
      for (int64_t r = 0; r < Ra && ok; ++r) {
        const double v = xa[r];
        if (v == last) continue;
        last = v;
        auto it = std::lower_bound(lv.begin(), lv.end(), v);
        if (it != lv.end() && *it == v) continue;
        if (!(v == v) || (int)lv.size() == kMaxXLevels) ok = false;
        else lv.insert(it, v);
      }
    }
    // a row packs its cell index in 27 bits
    hd.fx = ok && (co->n_rows_n < ((int64_t)1 << 27)) && (co->n_rows_s < ((int64_t)1 << 27));
    if (hd.fx) {
      hd.n_xlev = (int)lv.size();
      std::copy(lv.begin(), lv.end(), hd.xlev);
    }
  }
  hd.has_pcr = co->pcrpos != nullptr;
  hd.R[0] = co->n_rows_n, hd.R[1] = co->n_rows_s;
  const double tn = co->total_inds > 0 ? (double)co->total_inds : (double)N;
  hd.tot[0] = co->total_rows_n > 0 ? (double)co->total_rows_n : (double)co->n_rows_n;
  hd.tot[1] = co->total_rows_s > 0 ? (double)co->total_rows_s : (double)co->n_rows_s;
  hd.tot[2] = tn * G;
  hd.tot[3] = tn;
  hd.ind_offset = (uint32_t)co->ind_offset;

  int ndev = 0;
  CU(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return fail(ABD_ERR_CUDA, "no such CUDA device");
  CU(cudaSetDevice(device));

  abd_handle* h = nullptr;
  int rc = new_handle(&h, device, d);
  if (rc) return rc;
  auto bail = [&](int r) {
    abd_destroy(h);
    return r;
  };

  // bit masks per individual
  std::vector<u128> pcr((size_t)N, 0), vac((size_t)N, 0);
  for (int t = 0; t < G; ++t)
    for (int n = 0; n < N; ++n) {
      if (co->pcrpos && co->pcrpos[(size_t)t * N + n]) pcr[n] |= (u128)1 << t;
      if (co->vacs[(size_t)t * N + n]) vac[n] |= (u128)1 << t;
    }
  rc = with_mask(h, [&](auto m) {
    using M = decltype(m);
    std::vector<M> pm(pcr.begin(), pcr.end()), vm(vac.begin(), vac.end());
    M *dp, *dv;
    int r;
    if ((r = upload(h, &dp, pm)) || (r = upload(h, &dv, vm))) return r;
    h->dc.pcr = dp;
    h->dc.vac = dv;
    return ABD_OK;
  });
  if (rc) return bail(rc);
  if ((rc = build_rows(h, 0, co->n_rows_n, co->x_n, co->od_n, co->gap_n, co->ind_n))) return bail(rc);
  if ((rc = build_rows(h, 1, co->n_rows_s, co->x_s, co->od_s, co->gap_s, co->ind_s))) return bail(rc);
  for (int a = 0; a < 2; ++a) h->desc.hd.K[a] = h->h_cp[a][N];

  {
    std::vector<int> order((size_t)N);
    for (int n = 0; n < N; ++n) order[(size_t)n] = n;
    auto nrows = [&](int n) {
      return (h->h_rp[0][n + 1] - h->h_rp[0][n]) + (h->h_rp[1][n + 1] - h->h_rp[1][n]);
    };
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return nrows(a) > nrows(b); });
    if ((rc = upload(h, &h->d_order, order))) return bail(rc);
  }
  *out = h;
  return ABD_OK;
}

int abd_save_cache(abd_handle* h, const char* path) {
  if (!h || !path) return fail(ABD_ERR_INVALID, "NULL argument");
  int rc = set_device(h);
  if (rc) return rc;
  CU(cudaStreamSynchronize(h->stream));
  CacheIo io;
  io.writing = true;
  io.f = std::fopen(path, "wb");
  if (!io.f) return fail(ABD_ERR_INVALID, std::string("cannot write ") + path);
  io.raw(&h->desc.hd, sizeof(h->desc.hd));
  if (h->desc.hd.version == kCacheVersionWide) io.raw(h->desc.mask_hi, sizeof(h->desc.mask_hi));
  if ((rc = cache_body(h, io))) return rc;
  return io.ok ? ABD_OK : fail(ABD_ERR_INVALID, "cache file I/O error");
}

int abd_create_from_cache(abd_handle** out, const char* path, int device) {
  if (!out || !path) return fail(ABD_ERR_INVALID, "NULL argument");
  *out = nullptr;
  CacheIo io;
  io.f = std::fopen(path, "rb");
  if (!io.f) return fail(ABD_ERR_INVALID, std::string("cannot read ") + path);
  CohortDesc d{};
  CacheHeader& hd = d.hd;
  io.raw(&hd, sizeof(hd));
  if (!io.ok || std::memcmp(hd.magic, "ABDB200", 8) != 0) return fail(ABD_ERR_INVALID, "not an abd_b200 cache file");
  if (hd.version != kCacheVersion && hd.version != kCacheVersionWide)
    return fail(ABD_ERR_INVALID, "cache file of another version: rebuild it");
  const bool v3 = hd.version == kCacheVersionWide;
  if (v3) io.raw(d.mask_hi, sizeof(d.mask_hi));
  if (!io.ok || hd.G < 1 || hd.G > ABD_MAX_GAPS || hd.N < 1 || hd.N >= (v3 ? (1 << 25) : (1 << 26)) ||
      hd.n_chunks < 1 || hd.n_chunks > 3 || hd.wide != (v3 ? 2 : (hd.G > 31 ? 1 : 0)) || (!v3 && hd.G > 63) ||
      hd.R[0] < 0 || hd.R[1] < 0 || hd.K[0] < 0 || hd.K[1] < 0 || hd.n_xlev < 0 || hd.n_xlev > kMaxXLevels)
    return fail(ABD_ERR_INVALID, "corrupt cache header");
  int ndev = 0;
  CU(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return fail(ABD_ERR_CUDA, "no such CUDA device");
  CU(cudaSetDevice(device));
  abd_handle* h = nullptr;
  int rc = new_handle(&h, device, d);
  if (rc) return rc;
  if ((rc = cache_body(h, io))) {
    abd_destroy(h);
    return rc;
  }
  *out = h;
  return ABD_OK;
}

int abd_cohort_info(const abd_handle* h, int32_t* n_splits, int32_t* splits, int32_t* has_pcrpos) {
  if (!h) return fail(ABD_ERR_INVALID, "NULL handle");
  const int ns = h->dc.ch.n - 1;
  if (n_splits) *n_splits = ns;
  if (splits)
    for (int k = 0; k < ns; ++k) {
      const uint64_t lo = h->dc.ch.mask[k + 1], hi = h->dc.ch.mask_hi[k + 1];
      splits[k] = lo ? __builtin_ctzll(lo) : (hi ? 64 + __builtin_ctzll(hi) : h->G);
    }
  if (has_pcrpos) *has_pcrpos = h->desc.hd.has_pcr ? 1 : 0;
  return ABD_OK;
}

int abd_destroy(abd_handle* h) {
  if (!h) return ABD_OK;
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  for (void* p : h->xch_peer)
    if (p) cudaIpcCloseMemHandle(p);
  h->owned.release();
  free_chains(h);
  h->partial_buf.release();
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
  return ABD_OK;
}

int abd_sizes(const abd_handle* h, int32_t* g, int32_t* n, int64_t* rs, int64_t* rn) {
  if (!h) return fail(ABD_ERR_INVALID, "NULL handle");
  if (g) *g = h->G;
  if (n) *n = h->N;
  if (rs) *rs = h->R[1];
  if (rn) *rn = h->R[0];
  return ABD_OK;
}

// SURVEY.md section 8d: B_const = 2 G N + 20 R + 8 (N + 1); B_chain = G N + N + 13*8 + 14*8
int64_t abd_algorithmic_bytes_logp(const abd_handle* h, int C) {
  if (!h) return 0;
  const int64_t G = h->G, N = h->N, R = h->R[0] + h->R[1];
  return (int64_t)C * (G * N + N + 216) + 2 * G * N + 20 * R + 8 * (N + 1);
}
int64_t abd_algorithmic_bytes_gibbs(const abd_handle* h, int C) {
  if (!h) return 0;
  const int64_t G = h->G, N = h->N, R = h->R[0] + h->R[1];
  return (int64_t)C * (2 * (G * N + N) + 120) + 2 * G * N + 20 * R + 8 * (N + 1);
}
int64_t abd_launch_count(const abd_handle* h) { return h ? h->launches : 0; }

int abd_last_plan(const abd_handle* h, int32_t* out6) {
  if (!h || !out6) return fail(ABD_ERR_INVALID, "NULL argument");
  for (int k = 0; k < 6; ++k) out6[k] = h->last_plan[k];
  return ABD_OK;
}

int abd_set_tuning(abd_handle* h, int rows_per_tile, int chains_per_cta) {
  if (!h) return fail(ABD_ERR_INVALID, "NULL handle");
  if (rows_per_tile < 0 || chains_per_cta < 0) return fail(ABD_ERR_INVALID, "tuning values must be >= 0");
  h->tile_rows_override = rows_per_tile;
  h->chains_per_cta_override = chains_per_cta;
  return ABD_OK;
}

int abd_upload_state(abd_handle* h, int C, const int8_t* i_raw, const int8_t* waner) {
  PROLOGUE(h, C);
  if (!i_raw || !waner) return fail(ABD_ERR_INVALID, "NULL state");
  int rc = stage_state(h, C, i_raw, waner);
  if (rc) return rc;
  // state uploaded to stay: build its packed copy now (every later evaluation / sweep reads that)
  h->lazy_pack = true;
  void* pk = nullptr;
  if ((rc = resident_pack(h, C, h->d_iraw, h->d_waner, h->stream, &pk))) return rc;
  CU(cudaStreamSynchronize(h->stream));
  return ABD_OK;
}

int abd_state_touch(abd_handle* h) {
  if (!h) return fail(ABD_ERR_INVALID, "NULL handle");
  h->pack_valid = 0;
  return ABD_OK;
}

int abd_set_chain_offset(abd_handle* h, int64_t chain_offset) {
  if (!h) return fail(ABD_ERR_INVALID, "NULL handle");
  if (chain_offset < 0 || chain_offset > 0x7fffffffLL) return fail(ABD_ERR_INVALID, "chain_offset must be in [0, 2^31)");
  h->dc.chain_offset = (unsigned)chain_offset;
  return ABD_OK;
}

int abd_download_state(abd_handle* h, int C, int8_t* i_raw, int8_t* waner) {
  PROLOGUE(h, C);
  const size_t gn = (size_t)h->G * h->N;
  int rc;
  if (i_raw && (rc = copy_state(h, i_raw, h->d_iraw, (size_t)C * gn, cudaMemcpyDeviceToHost))) return rc;
  if (waner && (rc = copy_state(h, waner, h->d_waner, (size_t)C * h->N, cudaMemcpyDeviceToHost))) return rc;
  CU(cudaStreamSynchronize(h->stream));
  return ABD_OK;
}

int abd_state_dev(abd_handle* h, int C, int8_t** i_raw, int8_t** waner) {
  PROLOGUE(h, C);
  if (i_raw) *i_raw = h->d_iraw;
  if (waner) *waner = h->d_waner;
  return ABD_OK;
}

int abd_loglik_grad(abd_handle* h, int C, const double* theta13, const int8_t* i_raw, const int8_t* waner,
                    double* out_loglik, double* out_grad, int64_t* out_counts) {
  PROLOGUE(h, C);
  if (!theta13 || !out_loglik) return fail(ABD_ERR_INVALID, "NULL argument");
  int rc = stage_state(h, C, i_raw, waner);
  if (rc) return rc;
  return eval_to_host(h, C, theta13, 13, out_loglik, out_grad, out_counts);
}

int abd_logp_dlogp(abd_handle* h, int C, const double* q17, const int8_t* i_raw, const int8_t* waner,
                   double* out_logp, double* out_dlogp) {
  PROLOGUE(h, C);
  if (!q17 || !out_logp) return fail(ABD_ERR_INVALID, "NULL argument");
  int rc = stage_state(h, C, i_raw, waner);
  if (rc) return rc;
  // (Letting the kernel read the 17 scalars in place in the pinned staging buffer over PCIe was measured: 81 us per
  // call instead of 41 -- every CTA pays sysmem latency for its parameter loads.)
  return eval_to_host(h, C, q17, 17, out_logp, out_dlogp, nullptr);
}

static int stage_gibbs_params(abd_handle* h, int C, const double* theta13, const double* p, const double* pw) {
  double* hp = h->h_pin;
  for (int c = 0; c < C; ++c) {
    hp[(size_t)C * 13 + c] = p[c];
    hp[(size_t)C * 14 + c] = pw[c];
  }
  CU(cudaMemcpyAsync(h->d_p, hp + (size_t)C * 13, (size_t)C * 2 * sizeof(double), cudaMemcpyHostToDevice,
                     h->stream));
  return stage_params(h, C, theta13, 13);
}

int abd_cond_logodds(abd_handle* h, int C, const double* theta13, const double* p, const double* p_w,
                     const int8_t* i_raw, const int8_t* waner, double* out_i, double* out_w) {
  PROLOGUE(h, C);
  if (!theta13 || !p || !p_w || !out_i || !out_w) return fail(ABD_ERR_INVALID, "NULL argument");
  int rc = stage_state(h, C, i_raw, waner);
  if (rc) return rc;
  if ((rc = stage_gibbs_params(h, C, theta13, p, p_w))) return rc;
  const size_t gn = (size_t)h->G * h->N;
  DevBufs tmp;
  double *d_oi, *d_ow;
  if ((rc = tmp.alloc(&d_oi, (size_t)C * gn)) || (rc = tmp.alloc(&d_ow, (size_t)C * h->N))) return rc;
  GibbsCfg cfg{0, 0, -1, 1.0, d_oi, d_ow, nullptr};
  if ((rc = launch_gibbs(h, C, h->d_theta, 0, h->d_p, h->d_p + C, h->d_iraw, h->d_waner, cfg, h->stream))) return rc;
  CU(cudaMemcpyAsync(out_i, d_oi, (size_t)C * gn * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemcpyAsync(out_w, d_ow, (size_t)C * h->N * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return ABD_OK;
}

int abd_gibbs_sweep(abd_handle* h, int C, const double* theta13, const double* p, const double* p_w,
                    int8_t* i_raw, int8_t* waner, uint64_t seed, uint64_t sweep_idx, int mode,
                    double transit_p, int64_t* out_stats) {
  PROLOGUE(h, C);
  if (!theta13 || !p || !p_w) return fail(ABD_ERR_INVALID, "NULL argument");
  if (mode != ABD_GIBBS_METROPOLIS && mode != ABD_GIBBS_HEATBATH && mode != ABD_GIBBS_BLOCKED)
    return fail(ABD_ERR_INVALID, "bad mode");
  if (!(transit_p >= 0.0 && transit_p <= 1.0)) return fail(ABD_ERR_INVALID, "transit_p must be in [0, 1]");
  int rc = stage_state(h, C, i_raw, waner);
  if (rc) return rc;
  if ((rc = stage_gibbs_params(h, C, theta13, p, p_w))) return rc;
  CU(cudaMemsetAsync(h->d_stats, 0, (size_t)C * 2 * sizeof(unsigned long long), h->stream));
  GibbsCfg cfg{seed, sweep_idx, mode, transit_p, nullptr, nullptr, h->d_stats};
  if ((rc = launch_gibbs(h, C, h->d_theta, 0, h->d_p, h->d_p + C, h->d_iraw, h->d_waner, cfg, h->stream)))
    return rc;
  const size_t gn = (size_t)h->G * h->N;
  if (i_raw && (rc = copy_state(h, i_raw, h->d_iraw, (size_t)C * gn, cudaMemcpyDeviceToHost))) return rc;
  if (waner && (rc = copy_state(h, waner, h->d_waner, (size_t)C * h->N, cudaMemcpyDeviceToHost))) return rc;
  if (out_stats)
    CU(cudaMemcpyAsync(h->h_pin, h->d_stats, (size_t)C * 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost,
                       h->stream));
  CU(cudaStreamSynchronize(h->stream));
  if (out_stats) std::memcpy(out_stats, h->h_pin, (size_t)C * 2 * sizeof(int64_t));
  return ABD_OK;
}

int abd_deterministics(abd_handle* h, int C, const double* theta13, const int8_t* i_raw, const int8_t* waner,
                       int8_t* out_i, double* out_mu_n, double* out_mu_s) {
  PROLOGUE(h, C);
  if (!theta13) return fail(ABD_ERR_INVALID, "NULL argument");
  int rc = stage_state(h, C, i_raw, waner);
  if (rc) return rc;
  if ((rc = stage_params(h, C, theta13, 13))) return rc;
  const size_t gn = (size_t)h->G * h->N * C;
  DevBufs tmp;
  int8_t* d_i = nullptr;
  double *d_n = nullptr, *d_s = nullptr;
  if ((out_i && (rc = tmp.alloc(&d_i, gn))) || (out_mu_n && (rc = tmp.alloc(&d_n, gn))) ||
      (out_mu_s && (rc = tmp.alloc(&d_s, gn))))
    return rc;
  if ((rc = abd_deterministics_dev(h, C, h->d_theta, h->d_iraw, h->d_waner, d_i, d_n, d_s, h->stream))) return rc;
  if (out_i) CU(cudaMemcpyAsync(out_i, d_i, gn, cudaMemcpyDeviceToHost, h->stream));
  if (out_mu_n) CU(cudaMemcpyAsync(out_mu_n, d_n, gn * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  if (out_mu_s) CU(cudaMemcpyAsync(out_mu_s, d_s, gn * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return ABD_OK;
}

int abd_loglik_rows(abd_handle* h, int C, const double* theta13, const int8_t* i_raw, const int8_t* waner, double* out_s,
                    double* out_n) {
  PROLOGUE(h, C);
  if (!theta13) return fail(ABD_ERR_INVALID, "NULL argument");
  int rc = stage_state(h, C, i_raw, waner);
  if (rc) return rc;
  if ((rc = stage_params(h, C, theta13, 13))) return rc;
  DevBufs tmp;
  double *d_s = nullptr, *d_n = nullptr;
  if ((out_s && (rc = tmp.alloc(&d_s, (size_t)C * h->R[1]))) || (out_n && (rc = tmp.alloc(&d_n, (size_t)C * h->R[0]))))
    return rc;
  if ((rc = abd_loglik_rows_dev(h, C, h->d_theta, h->d_iraw, h->d_waner, d_s, d_n, h->stream))) return rc;
  if (out_s) CU(cudaMemcpyAsync(out_s, d_s, (size_t)C * h->R[1] * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  if (out_n) CU(cudaMemcpyAsync(out_n, d_n, (size_t)C * h->R[0] * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return ABD_OK;
}

// ---- device-pointer variants ----------------------------------------------------------------
int abd_loglik_rows_dev(abd_handle* h, int C, const double* theta13, const int8_t* i_raw, const int8_t* waner, double* out_s,
                        double* out_n, void* stream) {
  PROLOGUE(h, C);
  if (!theta13 || !i_raw || !waner) return fail(ABD_ERR_INVALID, "NULL argument");
  const cudaStream_t st = (cudaStream_t)stream;
  for (int a = 0; a < 2; ++a) {
    double* out = a ? out_s : out_n;
    if (!out || h->R[a] == 0) continue;
    dim3 grid((unsigned)((h->R[a] + 255) / 256), C);
    with_mask(h, [&](auto m) {
      k_loglik_rows<decltype(m)><<<grid, 256, 0, st>>>(h->dc, a, (int)h->R[a], theta13, i_raw, waner, out);
    });
    CU(cudaGetLastError());
    h->launches++;
  }
  return ABD_OK;
}

int abd_sums_dev(abd_handle* h, int C, const double* theta, int theta_is_q17, const int8_t* i_raw,
                 const int8_t* waner, double* sums, void* stream) {
  PROLOGUE(h, C);
  h->lazy_pack = true;
  if (!theta || !i_raw || !waner || !sums) return fail(ABD_ERR_INVALID, "NULL argument");
  FinalizeCfg fin{0, h->tot, nullptr, nullptr};
  return launch_sums(h, C, theta, theta_is_q17, i_raw, waner, sums, fin, (cudaStream_t)stream);
}

int abd_finalize_loglik_dev(abd_handle* h, int C, const double* theta13, const double* sums, double* out_loglik,
                            double* out_grad, void* stream) {
  PROLOGUE(h, C);
  if (!theta13 || !sums || !out_loglik) return fail(ABD_ERR_INVALID, "NULL argument");
  FinalizeCfg fin{1, h->tot, out_loglik, out_grad};
  k_finalize<<<(C + 3) / 4, 128, 0, (cudaStream_t)stream>>>(C, theta13, sums, fin, h->d_priors);
  CU(cudaGetLastError());
  h->launches++;
  return ABD_OK;
}

int abd_finalize_logp_dev(abd_handle* h, int C, const double* q17, const double* sums, double* out_logp,
                          double* out_dlogp, void* stream) {
  PROLOGUE(h, C);
  if (!q17 || !sums || !out_logp) return fail(ABD_ERR_INVALID, "NULL argument");
  FinalizeCfg fin{2, h->tot, out_logp, out_dlogp};
  k_finalize<<<(C + 3) / 4, 128, 0, (cudaStream_t)stream>>>(C, q17, sums, fin, h->d_priors);
  CU(cudaGetLastError());
  h->launches++;
  return ABD_OK;
}

int abd_loglik_grad_dev(abd_handle* h, int C, const double* theta13, const int8_t* i_raw, const int8_t* waner,
                        double* out_loglik, double* out_grad, void* stream) {
  PROLOGUE(h, C);
  h->lazy_pack = true;
  if (!theta13 || !i_raw || !waner || !out_loglik) return fail(ABD_ERR_INVALID, "NULL argument");
  FinalizeCfg fin{1, h->tot, out_loglik, out_grad};
  return launch_sums(h, C, theta13, 0, i_raw, waner, h->d_sums, fin, (cudaStream_t)stream);
}

int abd_logp_dlogp_dev(abd_handle* h, int C, const double* q17, const int8_t* i_raw, const int8_t* waner,
                       double* out_logp, double* out_dlogp, void* stream) {
  PROLOGUE(h, C);
  h->lazy_pack = true;
  if (!q17 || !i_raw || !waner || !out_logp) return fail(ABD_ERR_INVALID, "NULL argument");
  FinalizeCfg fin{2, h->tot, out_logp, out_dlogp};
  return launch_sums(h, C, q17, 1, i_raw, waner, h->d_sums, fin, (cudaStream_t)stream);
}

int abd_gibbs_sweep_dev(abd_handle* h, int C, const double* theta, int theta_is_q17, const double* p,
                        const double* p_w, int8_t* i_raw, int8_t* waner, uint64_t seed, uint64_t sweep_idx,
                        int mode, double transit_p, unsigned long long* stats, void* stream) {
  PROLOGUE(h, C);
  h->lazy_pack = true;
  if (!theta || !i_raw || !waner) return fail(ABD_ERR_INVALID, "NULL argument");
  if (!theta_is_q17 && (!p || !p_w)) return fail(ABD_ERR_INVALID, "p / p_w required with theta13");
  if (mode != ABD_GIBBS_METROPOLIS && mode != ABD_GIBBS_HEATBATH && mode != ABD_GIBBS_BLOCKED)
    return fail(ABD_ERR_INVALID, "bad mode");
  GibbsCfg cfg{seed, sweep_idx, mode, transit_p, nullptr, nullptr, stats};
  return launch_gibbs(h, C, theta, theta_is_q17, p, p_w, i_raw, waner, cfg, (cudaStream_t)stream);
}

int abd_deterministics_dev(abd_handle* h, int C, const double* theta13, const int8_t* i_raw, const int8_t* waner,
                           int8_t* out_i, double* out_mu_n, double* out_mu_s, void* stream) {
  PROLOGUE(h, C);
  if (!theta13 || !i_raw || !waner) return fail(ABD_ERR_INVALID, "NULL argument");
  dim3 grid((h->N + 127) / 128, C);
  const cudaStream_t st = (cudaStream_t)stream;
  const bool big = (size_t)C * 17 * h->G * h->N > ((size_t)64 << 20);  // outputs beyond half the L2: stream them
  with_mask(h, [&](auto m) {
    using M = decltype(m);
    if (big) k_determ<M, true><<<grid, 128, 0, st>>>(h->dc, theta13, i_raw, waner, out_i, out_mu_n, out_mu_s);
    else k_determ<M, false><<<grid, 128, 0, st>>>(h->dc, theta13, i_raw, waner, out_i, out_mu_n, out_mu_s);
  });
  CU(cudaGetLastError());
  h->launches++;
  return ABD_OK;
}

int abd_deterministics_accum_dev(abd_handle* h, int C, const double* theta, int theta_is_q17, const int8_t* i_raw,
                                 const int8_t* waner, double* sum_i, double* sum_mu_n, double* sum_mu_s, void* stream) {
  PROLOGUE(h, C);
  if (!theta || !i_raw || !waner) return fail(ABD_ERR_INVALID, "NULL argument");
  const int grid = (h->N + 127) / 128;
  const cudaStream_t st = (cudaStream_t)stream;
  with_mask(h, [&](auto m) {
    k_determ_accum<decltype(m)><<<grid, 128, 0, st>>>(h->dc, C, theta, theta_is_q17, i_raw, waner, sum_i, sum_mu_n, sum_mu_s);
  });
  CU(cudaGetLastError());
  h->launches++;
  return ABD_OK;
}

int abd_infection_probs_accum_dev(abd_handle* h, int C, const double* q17, const int8_t* i_raw, const int8_t* waner,
                                  double* sum_i, double* sum_w, void* stream) {
  PROLOGUE(h, C);
  if (!q17 || !i_raw || !waner || !sum_i || !sum_w) return fail(ABD_ERR_INVALID, "NULL argument");
  const cudaStream_t st = (cudaStream_t)stream;
  void* pack = nullptr;
  int rc = resident_pack(h, C, i_raw, waner, st, &pack);
  if (rc) return rc;
  const int grid = (h->N + kGibbsWarps - 1) / kGibbsWarps;
  with_mask(h, [&](auto m) {
    using M = decltype(m);
    k_infprob_accum<M><<<grid, kGibbsWarps * 32, 0, st>>>(h->dc, h->d_order, C, q17, i_raw, waner,
                                                          (const PackedState<M>*)pack, sum_i, sum_w);
  });
  CU(cudaGetLastError());
  h->launches++;
  return ABD_OK;
}

int abd_leapfrog_dev(abd_handle* h, int C, int n_steps, double* q17, double* p17, double* grad17, double* logp,
                     const double* eps, const double* inv_mass, const int8_t* i_raw, const int8_t* waner, void* stream) {
  PROLOGUE(h, C);
  h->lazy_pack = true;
  if (!q17 || !p17 || !grad17 || !logp || !eps || !inv_mass || !i_raw || !waner) return fail(ABD_ERR_INVALID, "NULL argument");
  if (n_steps < 1 || n_steps > 4096) return fail(ABD_ERR_INVALID, "n_steps must be in [1, 4096]");
  cudaStream_t st = (cudaStream_t)stream;
  if (n_steps > 1) CU(cudaMemsetAsync(h->d_gen, 0, ((size_t)C + 1) * sizeof(unsigned), st));
  TrajCfg traj{n_steps, q17, p17, grad17, logp, eps, inv_mass, h->d_traj, h->d_gen, h->d_gen + C, NutsLeafArgs{}};
  FinalizeCfg fin{2, h->tot, nullptr, nullptr};
  return launch_sums(h, C, q17, 1, i_raw, waner, nullptr, fin, st, &traj);
}

int abd_leapfrog_status(abd_handle* h, int C) {
  PROLOGUE(h, C);
  unsigned err = 0;
  CU(cudaMemcpy(&err, h->d_gen + C, sizeof(unsigned), cudaMemcpyDeviceToHost));
  return err ? fail(ABD_ERR_CUDA, "abd_leapfrog_dev: a CTA timed out waiting for its chain (grid not co-resident?)") : ABD_OK;
}

int abd_hmc_begin_dev(abd_handle* h, int C, const double* q17, const double* grad17, const double* logp,
                      const double* linv_t, uint64_t seed, uint64_t iter, double* qw, double* pw, double* gw, double* h0,
                      void* stream) {
  PROLOGUE(h, C);
  if (!q17 || !grad17 || !logp || !linv_t || !qw || !pw || !gw || !h0) return fail(ABD_ERR_INVALID, "NULL argument");
  k_hmc_begin<<<(C + 3) / 4, 128, 0, (cudaStream_t)stream>>>(C, q17, grad17, logp, linv_t, seed, iter, qw, pw, gw, h0,
                                                              h->dc.chain_offset);
  CU(cudaGetLastError());
  h->launches++;
  return ABD_OK;
}

int abd_hmc_end_dev(abd_handle* h, int C, double* q17, double* grad17, double* logp, const double* qw, const double* pw,
                    const double* gw, const double* lpw, const double* inv_mass, const double* h0, uint64_t seed,
                    uint64_t iter, double* accept_out, double* da, double* eps, int adapt, double target_accept,
                    void* stream) {
  PROLOGUE(h, C);
  if (!q17 || !grad17 || !logp || !qw || !pw || !gw || !lpw || !inv_mass || !h0 || !accept_out)
    return fail(ABD_ERR_INVALID, "NULL argument");
  if (adapt && (!da || !eps)) return fail(ABD_ERR_INVALID, "adapt needs the dual-averaging state and eps");
  k_hmc_end<<<(C + 3) / 4, 128, 0, (cudaStream_t)stream>>>(C, q17, grad17, logp, qw, pw, gw, lpw, inv_mass, h0, seed, iter,
                                                            accept_out, da, eps, adapt, target_accept, h->dc.chain_offset);
  CU(cudaGetLastError());
  h->launches++;
  return ABD_OK;
}

int64_t abd_nuts_state_doubles(int max_depth) {
  if (max_depth < 1 || max_depth > kNutsMaxDepth) return 0;
  return NutsLayout{max_depth}.size();
}

int abd_nuts_begin_dev(abd_handle* h, int C, int max_depth, const double* q17, const double* grad17, const double* logp,
                       const double* linv_t, const double* eps, uint64_t seed, uint64_t iter, double* state, double* qw,
                       double* pw, double* gw, double* eps_signed, int* any_active, void* stream) {
  PROLOGUE(h, C);
  if (!q17 || !grad17 || !logp || !linv_t || !eps || !state || !qw || !pw || !gw || !eps_signed || !any_active)
    return fail(ABD_ERR_INVALID, "NULL argument");
  if (max_depth < 1 || max_depth > kNutsMaxDepth) return fail(ABD_ERR_INVALID, "max_depth must be in [1, 10]");
  k_nuts_begin<<<(C + 3) / 4, 128, 0, (cudaStream_t)stream>>>(C, NutsLayout{max_depth}, q17, grad17, logp, linv_t, eps, seed, iter,
                                                              h->dc.chain_offset, state, qw, pw, gw, eps_signed, any_active);
  CU(cudaGetLastError());
  h->launches++;
  return ABD_OK;
}

int abd_nuts_leaf_dev(abd_handle* h, int C, int max_depth, int depth, int leaf, double* qw, double* pw, double* gw,
                      const double* lpw, const double* inv_mass, const double* eps, uint64_t seed, uint64_t iter, double* state,
                      double* eps_signed, int* any_active, void* stream) {
  PROLOGUE(h, C);
  if (!qw || !pw || !gw || !lpw || !inv_mass || !eps || !state || !eps_signed || !any_active)
    return fail(ABD_ERR_INVALID, "NULL argument");
  if (max_depth < 1 || max_depth > kNutsMaxDepth || depth < 0 || depth >= max_depth || leaf < 0 || leaf >= (1 << depth))
    return fail(ABD_ERR_INVALID, "bad depth / leaf");
  cudaLaunchAttribute attr;
  const cudaLaunchConfig_t lc = pdl_config(dim3((C + 3) / 4), dim3(128), 0, (cudaStream_t)stream, &attr);
  const NutsLeafArgs a{state, NutsLayout{max_depth}, depth, leaf, max_depth, eps, seed, iter, h->dc.chain_offset, eps_signed,
                       any_active};
  CU(cudaLaunchKernelEx(&lc, k_nuts_leaf, C, a, qw, pw, gw, lpw, inv_mass));
  CU(cudaGetLastError());
  h->launches++;
  return ABD_OK;
}

// all 2^depth leaves of one doubling in ONE call: per leaf a single-step leapfrog launch and the tree launch
int abd_nuts_extend_dev(abd_handle* h, int C, int max_depth, int depth, double* qw, double* pw, double* gw, double* lpw,
                        const double* inv_mass, const double* eps, uint64_t seed, uint64_t iter, double* state,
                        double* eps_signed, int* any_active, const int8_t* i_raw, const int8_t* waner, void* stream) {
  if (depth < 0 || depth >= max_depth) return fail(ABD_ERR_INVALID, "bad depth");
  PROLOGUE(h, C);
  h->lazy_pack = true;
  if (!qw || !pw || !gw || !lpw || !inv_mass || !eps || !state || !eps_signed || !any_active || !i_raw || !waner)
    return fail(ABD_ERR_INVALID, "NULL argument");
  if (max_depth < 1 || max_depth > kNutsMaxDepth) return fail(ABD_ERR_INVALID, "max_depth must be in [1, 10]");
  const bool sharded = h->xch_local != nullptr;
  int rc;
  if (sharded && (rc = check_xch(h, C, "abd_nuts_extend_dev"))) return rc;
  for (int n = 0; n < (1 << depth); ++n) {
    // the leaf's leapfrog step and its tree bookkeeping in ONE launch (the finishing warp of each chain does both)
    TrajCfg traj{1, qw, pw, gw, lpw, eps_signed, inv_mass, h->d_traj, h->d_gen, h->d_gen + C,
                 NutsLeafArgs{state, NutsLayout{max_depth}, depth, n, max_depth, eps, seed, iter, h->dc.chain_offset, eps_signed,
                              any_active}};
    FinalizeCfg fin{2, h->tot, nullptr, nullptr};
    if ((rc = launch_sums(h, C, qw, 1, i_raw, waner, nullptr, fin, (cudaStream_t)stream, &traj, sharded))) return rc;
  }
  return ABD_OK;
}

int abd_nuts_end_dev(abd_handle* h, int C, int max_depth, double* q17, double* grad17, double* logp, const double* state,
                     double* accept_out, double* depth_out, double* diverged_out, double* da, double* eps, int adapt,
                     double target_accept, void* stream) {
  PROLOGUE(h, C);
  if (!q17 || !grad17 || !logp || !state || !accept_out) return fail(ABD_ERR_INVALID, "NULL argument");
  if (max_depth < 1 || max_depth > kNutsMaxDepth) return fail(ABD_ERR_INVALID, "max_depth must be in [1, 10]");
  if (adapt && (!da || !eps)) return fail(ABD_ERR_INVALID, "adapt needs the dual-averaging state and eps");
  k_nuts_end<<<(C + 3) / 4, 128, 0, (cudaStream_t)stream>>>(C, NutsLayout{max_depth}, q17, grad17, logp, state, accept_out, depth_out,
                                                            diverged_out, da, eps, adapt, target_accept);
  CU(cudaGetLastError());
  h->launches++;
  return ABD_OK;
}

int abd_xch_alloc(abd_handle* h, int world, int rank, int max_chains, void* out_ipc_handle) {
  if (!h) return fail(ABD_ERR_INVALID, "NULL handle");
  if (world < 2 || world > kMaxPeers || rank < 0 || rank >= world || max_chains < 1 || !out_ipc_handle)
    return fail(ABD_ERR_INVALID, "abd_xch_alloc: need 2 <= world <= 8, 0 <= rank < world, max_chains >= 1");
  if (world * kNSums > kSumsBlock) return fail(ABD_ERR_INVALID, "world too large");
  int rc = set_device(h);
  if (rc) return rc;
  if (h->xch_local) return fail(ABD_ERR_INVALID, "abd_xch_alloc: already allocated");
  const size_t bytes = (size_t)2 * world * max_chains * 32 * sizeof(unsigned long long);
  char* local;
  if ((rc = h->owned.alloc(&local, bytes))) return rc;
  h->xch_local = local;
  CU(cudaMemset(h->xch_local, 0, bytes));
  unsigned* seq;
  if ((rc = h->owned.alloc(&seq, (size_t)max_chains + 1))) return rc;
  CU(cudaMemset(seq, 0, ((size_t)max_chains + 1) * sizeof(unsigned)));
  unsigned long long* stat;
  if ((rc = h->owned.alloc(&stat, (size_t)kMaxPeers + 1))) return rc;
  CU(cudaMemset(stat, 0, ((size_t)kMaxPeers + 1) * sizeof(unsigned long long)));
  h->xch = XchCfg{};
  h->xch.world = world;
  h->xch.rank = rank;
  h->xch.cmax = max_chains;
  h->xch.seq = seq;
  h->xch.err = seq + max_chains;
  h->xch.stat = stat;
  cudaIpcMemHandle_t ipc;
  CU(cudaIpcGetMemHandle(&ipc, h->xch_local));
  static_assert(sizeof(ipc) == ABD_IPC_HANDLE_BYTES, "IPC handle size");
  std::memcpy(out_ipc_handle, &ipc, sizeof(ipc));
  return ABD_OK;
}

int abd_xch_connect(abd_handle* h, const void* all_ipc_handles) {
  if (!h || !all_ipc_handles) return fail(ABD_ERR_INVALID, "NULL argument");
  if (!h->xch_local) return fail(ABD_ERR_INVALID, "abd_xch_connect: call abd_xch_alloc first");
  int rc = set_device(h);
  if (rc) return rc;
  const int world = h->xch.world;
  for (int r = 0; r < world; ++r) {
    void* base = h->xch_local;
    if (r != h->xch.rank) {
      cudaIpcMemHandle_t ipc;
      std::memcpy(&ipc, (const char*)all_ipc_handles + (size_t)r * sizeof(ipc), sizeof(ipc));
      CU(cudaIpcOpenMemHandle(&base, ipc, cudaIpcMemLazyEnablePeerAccess));
      h->xch_peer[r] = base;
    }
    h->xch.buf[r] = (unsigned long long*)base;
  }
  return ABD_OK;
}

int abd_logp_dlogp_sharded_dev(abd_handle* h, int C, const double* q17, const int8_t* i_raw, const int8_t* waner,
                               double* out_logp, double* out_dlogp, void* stream) {
  PROLOGUE(h, C);
  h->lazy_pack = true;
  if (!q17 || !i_raw || !waner || !out_logp) return fail(ABD_ERR_INVALID, "NULL argument");
  if (int rc = check_xch(h, C, "abd_logp_dlogp_sharded_dev")) return rc;
  FinalizeCfg fin{2, h->tot, out_logp, out_dlogp};
  return launch_sums(h, C, q17, 1, i_raw, waner, h->d_sums, fin, (cudaStream_t)stream, nullptr, true);
}

int abd_leapfrog_sharded_dev(abd_handle* h, int C, double* q17, double* p17, double* grad17, double* logp, const double* eps,
                             const double* inv_mass, const int8_t* i_raw, const int8_t* waner, void* stream) {
  PROLOGUE(h, C);
  h->lazy_pack = true;
  if (!q17 || !p17 || !grad17 || !logp || !eps || !inv_mass || !i_raw || !waner) return fail(ABD_ERR_INVALID, "NULL argument");
  if (int rc = check_xch(h, C, "abd_leapfrog_sharded_dev")) return rc;
  TrajCfg traj{1, q17, p17, grad17, logp, eps, inv_mass, h->d_traj, h->d_gen, h->d_gen + C, NutsLeafArgs{}};
  FinalizeCfg fin{2, h->tot, nullptr, nullptr};
  return launch_sums(h, C, q17, 1, i_raw, waner, nullptr, fin, (cudaStream_t)stream, &traj, true);
}

int abd_xch_stats(abd_handle* h, uint64_t* out, int reset) {
  if (!h || !h->xch_local || !out) return fail(ABD_ERR_INVALID, "no exchange buffer");
  int rc = set_device(h);
  if (rc) return rc;
  static_assert(sizeof(unsigned long long) == sizeof(uint64_t), "");
  CU(cudaMemcpy(out, h->xch.stat, (kMaxPeers + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost));
  if (reset) CU(cudaMemset(h->xch.stat, 0, (kMaxPeers + 1) * sizeof(uint64_t)));
  return ABD_OK;
}

int abd_xch_status(abd_handle* h) {
  if (!h || !h->xch_local) return fail(ABD_ERR_INVALID, "no exchange buffer");
  int rc = set_device(h);
  if (rc) return rc;
  unsigned err = 0;
  CU(cudaMemcpy(&err, h->xch.err, sizeof(unsigned), cudaMemcpyDeviceToHost));
  return err ? fail(ABD_ERR_CUDA, "a peer's contribution did not arrive (timeout)") : ABD_OK;
}

int abd_debug_fast_math(int device, int64_t n, const double* z, double* out_exp, double* out_rcp) {
  if (n < 0 || !z || !out_exp || !out_rcp) return fail(ABD_ERR_INVALID, "bad argument");
  CU(cudaSetDevice(device));
  DevBufs tmp;
  double *dz, *de, *dr;
  const size_t n1 = (size_t)std::max<int64_t>(n, 1);
  int rc;
  if ((rc = tmp.alloc(&dz, n1)) || (rc = tmp.alloc(&de, n1)) || (rc = tmp.alloc(&dr, n1))) return rc;
  CU(cudaMemcpy(dz, z, (size_t)n * sizeof(double), cudaMemcpyHostToDevice));
  k_debug_fast_math<<<296, 256>>>(n, dz, de, dr);
  CU(cudaGetLastError());
  CU(cudaMemcpy(out_exp, de, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost));
  CU(cudaMemcpy(out_rcp, dr, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost));
  return ABD_OK;
}

#ifdef ABD_PHASE_TIMING
int abd_debug_spans(unsigned long long* out, int reset) {
  if (reset) {
    unsigned long long init[256][2];
    for (auto& r : init) { r[0] = ~0ull; r[1] = 0; }
    unsigned z = 0;
    CU(cudaMemcpyToSymbol(g_span, init, sizeof(init)));
    CU(cudaMemcpyToSymbol(g_span_idx, &z, sizeof(z)));
    CU(cudaMemcpyToSymbol(g_span_done, &z, sizeof(z)));
    return ABD_OK;
  }
  CU(cudaMemcpyFromSymbol(out, g_span, sizeof(unsigned long long) * 512));
  return ABD_OK;
}
int abd_debug_phase_times(unsigned long long* out, int n_ctas) {
  CU(cudaMemcpyFromSymbol(out, g_phase, sizeof(unsigned long long) * 16 * (size_t)n_ctas));
  return ABD_OK;
}
#endif

}  // extern "C"
