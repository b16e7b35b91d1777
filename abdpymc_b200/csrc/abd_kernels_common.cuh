// Types and helpers shared by the kernels of libabd_b200.so and the host side that launches them
// (device view of the cohort, launch configurations, warp-level power tables).
#pragma once
#include "abd_device.cuh"

namespace {
using namespace abd;

// ------------------------------------------------------------------------------------------
// device-side view of the cohort
// ------------------------------------------------------------------------------------------
// The (individual, gap) words meta / cmeta: individual << kGapBits<M> | gap.  Six gap bits leave 26 for the individual;
// the 128-bit layout needs seven (individuals < 2^25).
template <typename M>
constexpr int kGapBits = sizeof(M) > 8 ? 7 : 6;
template <typename M>
constexpr uint32_t kGapMask = (1u << kGapBits<M>) - 1u;

struct DevCohort {
  int G, N;
  unsigned ind_offset;       // global index of this shard's first individual (RNG streams)
  unsigned chain_offset;     // global index of this handle's first chain (RNG streams; abd_set_chain_offset)
  const void* pcr;
  const void* vac;
  const int* rp[2];          // [0] = N antigen, [1] = S antigen
  const double* od[2];
  const double* x[2];
  // factored mode (the cohort has <= 32 distinct log_dilution values, the usual case):
  const uint32_t* rcx[2];      // per row: cell index << 5 | index of its dilution in xlev
  const double* xlev;          // [32] the distinct dilutions, ascending (padded with 0)
  int n_xlev;                  // 0: not available (k_sums stages the dilutions as doubles)
  const uint32_t* meta[2];     // per row: individual << kGapBits<M> | gap
  const uint32_t* rowcell[2];  // per row: index of its (individual, gap) cell
  const uint32_t* cmeta[2];    // per cell: individual << kGapBits<M> | gap
  const int* rowperm[2];       // per (sorted) row: its index among the antigen's rows as the caller passed them
  Chunks ch;
};

constexpr int kSumsBlock = 256;
constexpr int kSumsWarps = kSumsBlock / 32;
constexpr int kAuxDoubles = 128;  // 17 x PriorPre (7) + LikPre (6), padded
constexpr int kTileMaxInds = 128;
#ifndef ABD_GIBBS_WARPS
#define ABD_GIBBS_WARPS 8
#endif
#ifndef ABD_GIBBS_MINB
#define ABD_GIBBS_MINB 4
#endif
constexpr int kGibbsWarps = ABD_GIBBS_WARPS;  // warps per CTA of the Gibbs kernels; ABD_GIBBS_MINB CTAs per SM
// k_gibbs on 128-bit masks: four proposal slots per lane (two for 64-bit masks) do not fit the 64 registers that 4 CTAs
// per SM leave (see DESIGN.md section 4)
#ifndef ABD_GIBBS_MINB128
#define ABD_GIBBS_MINB128 2
#endif
template <typename M>
constexpr int kGibbsMinB = sizeof(M) > 8 ? ABD_GIBBS_MINB128 : ABD_GIBBS_MINB;

// per-individual state staged in shared memory: constrained infections, vaccinations, waner
// (packed in the top bit of the vaccination mask; usable gaps <= width - 1)
template <typename M>
struct IndState {
  M inf, vacw;
};
template <typename M>
__device__ __forceinline__ M top_bit() { return (M)1 << (sizeof(M) * 8 - 1); }

// Packed resident chain state, one entry per (chain, individual), kept beside the int8 boundary
// arrays by every library call that writes the resident state (abd_upload_state, the Gibbs sweeps):
//   rw  = the individual's i_raw column as a bit mask over gaps | ab_s_waner in the top bit
//   inf = constrain(raw, pcr, chunks), the constrained infections (abd.py:640-667)
// so that an evaluation reads 8 (16) bytes per individual and chain instead of G + 1 strided bytes
// and does not repeat the integer prologue: the binary state only changes once per Gibbs sweep.
template <typename M>
struct __align__(2 * sizeof(M)) PackedState {
  M rw, inf;
};

// One thread's i_raw column (gaps 0..G-1, stride N) as a bit mask.  Unpredicated loads along an address chain that
// stops at the last row, masked afterwards: every load in flight at once, and the compiler cannot precompute (and
// spill) one 64-bit address per gap.  (A load guarded by `t < G` needs a predicate register each, and there are only
// seven: the compiler then keeps ~6 loads in flight.)  The 128-bit layout loads in blocks of 32 gaps, skipping the
// blocks beyond the last gap: 128 bytes in flight per thread would not fit in registers.
template <typename M>
__device__ __forceinline__ M load_column(const int8_t* col, int G, int N) {
  M raw = 0;
  if constexpr (sizeof(M) > 8) {
#pragma unroll 1
    for (int b = 0; b * 32 < G; ++b) {
      const int8_t* p = col + (size_t)b * 32 * N;
      int8_t bytes[32];
#pragma unroll
      for (int t = 0; t < 32; ++t) {
        bytes[t] = __ldg(p);
        p += (b * 32 + t + 1 < G) ? (size_t)N : (size_t)0;
      }
      uint32_t bits = 0;
#pragma unroll
      for (int t = 0; t < 32; ++t) bits |= (uint32_t)(bytes[t] != 0) << t;
      raw |= (M)bits << (32 * b);
    }
  } else {
    int8_t bytes[sizeof(M) * 8];
#pragma unroll
    for (int t = 0; t < (int)sizeof(M) * 8; ++t) {
      bytes[t] = __ldg(col);
      col += (t + 1 < G) ? (size_t)N : (size_t)0;
    }
#pragma unroll
    for (int t = 0; t < (int)sizeof(M) * 8; ++t) raw |= (M)(bytes[t] != 0) << t;
  }
  return raw & low_mask<M>(G - 1);
}

__device__ __forceinline__ double load_param(const double* theta, int theta_is_q, int c, int k13) {
  if (theta_is_q) {
    const int j = kQOfTheta[k13];
    return backward(theta[(size_t)c * 17 + j], kQTransform[j]);
  }
  return theta[(size_t)c * 13 + k13];
}

// One warp: pw[k] = rho^k and (optionally) dpw[k] = k rho^(k-1) for k < G by a shuffle scan.
__device__ __forceinline__ void fill_pow_warp(double rho, int G, int lane, double* pw, double* dpw) {
  double v = rho;  // inclusive prefix product: rho^(lane+1)
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    const double u = __shfl_up_sync(0xffffffffu, v, off);
    if (lane >= off) v *= u;
  }
  const double r32 = __shfl_sync(0xffffffffu, v, 31);  // rho^32
  double prev = __shfl_up_sync(0xffffffffu, v, 1);      // rho^lane
  if (lane == 0) prev = 1.0;
  if (lane == 0) {
    pw[0] = 1.0;
    if (dpw) dpw[0] = 0.0;
  }
  double scale = 1.0;  // rho^(32 blk)
  for (int blk = 0; blk * 32 < G; ++blk) {
    const int k = blk * 32 + lane + 1;
    if (k < G) {
      pw[k] = v * scale;
      if (dpw) dpw[k] = (double)k * prev * scale;
    }
    scale *= r32;
  }
}

// The same, interleaved: tab[k] = {rho^k, k rho^(k-1)}.
__device__ __forceinline__ void fill_pow2_warp(double rho, int G, int lane, double2* tab) {
  double v = rho;  // inclusive prefix product: rho^(lane+1)
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    const double u = __shfl_up_sync(0xffffffffu, v, off);
    if (lane >= off) v *= u;
  }
  const double r32 = __shfl_sync(0xffffffffu, v, 31);  // rho^32
  double prev = __shfl_up_sync(0xffffffffu, v, 1);      // rho^lane
  if (lane == 0) {
    prev = 1.0;
    tab[0] = make_double2(1.0, 0.0);
  }
  double scale = 1.0;  // rho^(32 blk)
  for (int blk = 0; blk * 32 < G; ++blk) {
    const int k = blk * 32 + lane + 1;
    if (k < G) tab[k] = make_double2(v * scale, (double)k * prev * scale);
    scale *= r32;
  }
}

}  // namespace
