"""Rao-Blackwellised posterior infection and waner probabilities, restated in NumPy -- TEST INFRASTRUCTURE.

What ``abd_infection_probs_accum_dev`` (include/abd_b200.h, k_infprob_accum) adds for one chain state, written as the
estimator reads (DESIGN.md section 4, k_infprob_accum) and evaluated with the oracle's whole-cohort per-individual
log-likelihood, one candidate column per option for every individual at once.  No shortcut of the kernel (reused likelihoods) is restated:
they do not change the result.
"""

from __future__ import annotations

import numpy as np

from .abd_oracle import chunk_bounds


def _ll(o, theta13, i_raw, w):
    """Per-individual log-likelihood; NaN counts as -inf (a NaN option has weight zero)."""
    v = o.loglik_per_individual(theta13, i_raw, w)
    return np.where(np.isnan(v), -np.inf, v)


def infection_probs(o, theta13, p, p_w, i_raw, w):
    """For one state (theta13, p, p_w, i_raw (G, N), w (N,)) of the model ``o`` (an ``abd_oracle.Oracle``):
    (E[i[t, n] | the state outside t's block] (G, N), E[ab_s_waner[n] | theta, i_raw] (N,)).

    * time chunks: per chunk and individual, the chunk's raw bits are summarised by the position o of their first 1
      (or none, o = len); log w_o = o log(1-p) + log p + L_n(constrain(base | bit c0+o)), log w_len = len log(1-p) +
      L_n(constrain(base)), base = raw with the chunk cleared; gap c0 + o gets w_o i_{c0+o}(option o) / sum w.  A chunk
      holding a PCR+ month contributes constrain(current), whatever its raw bits.
    * no splits: per bit, the two values of raw_t with the rest fixed.
    * waner: sigmoid(logit p_w + L_n(w = 1) - L_n(w = 0)).
    When every option of a block has weight zero (or the log-odds is undefined) the block contributes the current state.
    """
    G, N = o.G, o.N
    i_raw = (np.asarray(i_raw).reshape(G, N) != 0).astype(np.int64)
    w = (np.asarray(w) != 0).astype(np.int64)
    inf = o.constrain(i_raw)
    out = np.zeros((G, N))
    with np.errstate(all="ignore"):
        if not o.splits:
            lo = np.log(p) - np.log1p(-p)
            for t in range(G):
                hi, lw_ = i_raw.copy(), i_raw.copy()
                hi[t], lw_[t] = 1, 0
                b1, b0 = o.constrain(hi)[t], o.constrain(lw_)[t]
                ll1, ll0 = _ll(o, theta13, hi, w), _ll(o, theta13, lw_, w)
                p1 = 1.0 / (1.0 + np.exp(-(lo + np.where(ll1 == ll0, 0.0, ll1 - ll0))))
                v = np.where(b1 == 1, p1, 1.0 - p1)
                v = np.where(np.isnan(v), inf[t], v)
                out[t] = np.where(b1 == b0, b1, v)
        else:
            lp1, lp0 = np.log(p), np.log1p(-p)
            for a, b in chunk_bounds(G, o.splits):
                if a == b:
                    continue
                n_opt = b - a
                base = i_raw.copy()
                base[a:b] = 0
                lw = np.empty((n_opt + 1, N))
                bit = np.zeros((n_opt, N))
                for k in range(n_opt + 1):
                    cand = base.copy()
                    if k < n_opt:
                        cand[a + k] = 1
                        bit[k] = o.constrain(cand)[a + k]
                    lw[k] = _ll(o, theta13, cand, w) + (k * lp0 + lp1 if k < n_opt else n_opt * lp0)
                lw = np.where(np.isnan(lw), -np.inf, lw)
                mx = lw.max(axis=0)
                ok = mx > -np.inf
                e = np.exp(lw - np.where(ok, mx, 0.0))
                val = np.where(ok, e[:n_opt] * bit / e.sum(axis=0), inf[a:b])
                out[a:b] = np.where(o.pcr[a:b].any(axis=0), inf[a:b], val)
        ll1, ll0 = _ll(o, theta13, i_raw, np.ones(N)), _ll(o, theta13, i_raw, np.zeros(N))
        d10 = np.log(p_w) - np.log1p(-p_w) + np.where(ll1 == ll0, 0.0, ll1 - ll0)
        pw = 1.0 / (1.0 + np.exp(-d10))
    return out, np.where(np.isnan(pw), w, pw)
