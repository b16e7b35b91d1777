"""The device HMC and NUTS transitions restated in float64, one chain at a time, drawing the same Philox words.

``k_hmc_begin`` / ``k_hmc_end`` (csrc/k_misc.cuh) and ``k_nuts_begin`` / ``nuts_leaf_chain`` / ``k_nuts_end``
(csrc/k_nuts.cuh) make their random decisions from counter-based Philox4x32-10 streams.  Given the same leaves, this
module makes the same decisions, so a CUDA transition can be checked decision by decision instead of statistically.

Every decision is recorded with its *margin*: the signed distance of the compared quantity from its threshold,
relative to the scale of the numbers it was computed from (positive: the decision is the one recorded).  The kernels
round differently (fused multiply-adds, warp-shuffle reductions, CUDA ``log`` / ``cospi``), so only decisions whose
margin exceeds that rounding can be required to agree.

The NUTS sub-tree U-turn checks come in two formulations: the kernel's O(depth) momentum checkpoints, and a direct one
that keeps every leaf's momentum and sums each balanced span from them (``direct=True``).  They must agree.
"""

from __future__ import annotations

import math
from dataclasses import dataclass, field

import numpy as np

from .abd_oracle import _u01, philox4x32_10

_M32 = 0xFFFFFFFF
HMC_BEGIN = 0x484D4331   # "HMC1": counter (lane, chain, iter, HMC_BEGIN), the momentum refresh (also k_nuts_begin)
HMC_END = 0x41434331     # "ACC1": counter (0, chain, iter, HMC_END), the accept decision
NUTS = 0x4E555453        # "NUTS": counter (tag, chain, iter, NUTS), every decision of the tree
U_SHIFT = 2.0**-32       # u01 is in (0, 1]; minus 2^-32 it is in [0, 1)
DIVERGENCE = 1000.0      # |H0 - H| above this ends the sub-tree


def tag_direction(j):
    return 0x10000 + j


def tag_leaf(j, n):
    return 0x20000 + (j << 11) + n


def tag_merge(j):
    return 0x30000 + j


def key(seed, it):
    """The Philox key of iteration ``it``: (seed lo, seed hi ^ iter hi)."""
    return (seed & _M32, ((seed >> 32) ^ (it >> 32)) & _M32)


def counter(word0, chain, it, stream):
    return (word0 & _M32, chain & _M32, it & _M32, stream)


def uniform(seed, it, chain, word0, stream):
    """The first Philox word of counter (word0, chain, iter, stream) as a uniform in [0, 1)."""
    return _u01(philox4x32_10(counter(word0, chain, it, stream), key(seed, it))[0]) - U_SHIFT


def cospi(x):
    """cos(pi x) for x in [0, 2] with a relative error of a few ulp, zeros included (the reductions are exact)."""
    if x > 1.0:
        x = 2.0 - x
    sign = 1.0
    if x > 0.5:
        x, sign = 1.0 - x, -1.0
    return sign * (math.sin(math.pi * (0.5 - x)) if x > 0.25 else math.cos(math.pi * x))


# ------------------------------------------------------------------------------------------ decisions
@dataclass
class Decision:
    kind: str        # "direction", "divergent", "take", "turned" (sub-tree span), "merge", "uturn" (whole tree), "accept"
    j: int           # tree depth (-1 for HMC)
    n: int           # leaf of the depth-j sub-tree (-1: not a leaf decision)
    size: int        # "turned": the span's number of leaves; else 0
    value: bool
    margin: float
    x: float = 0.0   # the compared quantity (dh for "divergent")

    def key(self):
        return (self.kind, self.j, self.n, self.size, self.value)


def _log_margin(log_a, u, scale):
    """margin of ``u < exp(log_a)`` in log space, relative to the energy scale the log-weights carry."""
    if log_a >= 0.0 or u == 0.0:   # exp(0) = 1 > u exactly
        return math.inf if log_a > -math.inf else -math.inf
    if log_a == -math.inf:
        return -math.inf
    return (log_a - math.log(u)) / scale


def _turning(inv_mass, pa, pb, rho):
    """The kernel's criterion: either end of the span moves against its momentum sum.  Returns (turned, margin)."""
    adj = rho - 0.5 * (pa + pb)
    sa = inv_mass @ adj
    da, db = float(pa @ sa), float(pb @ sa)
    scale = max(float(np.abs(pa) @ np.abs(sa)), float(np.abs(pb) @ np.abs(sa)),
                float(np.abs(pa) @ (np.abs(inv_mass) @ np.abs(adj))), 1e-300)
    f = min(da, db)
    turned = f <= 0.0
    return turned, (-f if turned else f) / scale


def _logaddexp(a, b):
    m = max(a, b)
    if not m > -math.inf:
        return -math.inf
    return m + math.log(math.exp(a - m) + math.exp(b - m))


# ------------------------------------------------------------------------------------------ HMC
def momentum(seed, it, chain, linv_t):
    """k_hmc_begin / k_nuts_begin: z by Box-Muller on Philox words x, y of counter (lane, chain, iter, HMC1);
    p = linv_t z ~ N(0, M); returns (z, p, z.z)."""
    k = key(seed, it)
    z = np.empty(17)
    for lane in range(17):
        r = philox4x32_10(counter(lane, chain, it, HMC_BEGIN), k)
        z[lane] = math.sqrt(-2.0 * math.log(_u01(r[0]))) * cospi(2.0 * _u01(r[1]))
    return z, np.asarray(linv_t) @ z, float(z @ z)


def hmc_end(h0, lpw, pw, inv_mass, seed, it, chain):
    """k_hmc_end's decision: dh = h0 - (-lpw + p.M^-1 p / 2), non-finite -> -inf, take iff u < exp(min(dh, 0)).
    Returns (take, acceptance statistic, Decision)."""
    h1 = -lpw + 0.5 * float(pw @ (np.asarray(inv_mass) @ pw))
    dh = h0 - h1
    if not math.isfinite(dh):
        dh = -math.inf
    acc = math.exp(min(dh, 0.0))
    u = uniform(seed, it, chain, 0, HMC_END)
    take = u < acc
    scale = max(1.0, abs(h0), abs(h1) if math.isfinite(h1) else 0.0)
    m = _log_margin(min(dh, 0.0), u, scale)
    return take, acc, Decision("accept", -1, -1, 0, take, m if take else -m, dh)


def dual_averaging(da, acc, target, gamma=0.05, t0=10.0, kappa=0.75):
    """Nesterov dual averaging of log(step size), as k_hmc_end / k_nuts_end update it.  ``da`` = (mu, hbar, log_avg,
    t).  Returns (new da, new step size)."""
    mu, hbar, log_avg, t = (float(v) for v in da)
    t += 1.0
    eta = 1.0 / (t + t0)
    hbar = (1.0 - eta) * hbar + eta * (target - acc)
    log_eps = mu - math.sqrt(t) / gamma * hbar
    w = t ** (-kappa)
    return np.array([mu, hbar, w * log_eps + (1.0 - w) * log_avg, t]), math.exp(log_eps)


# ------------------------------------------------------------------------------------------ NUTS
@dataclass
class Tree:
    q: np.ndarray            # the proposal
    grad: np.ndarray
    logp: float
    accept: float            # mean of exp(min(dh, 0)) over the leaves built
    depth: int               # depths built
    diverged: bool
    eps_signed: list         # the signed step of every depth built
    decisions: list = field(default_factory=list)
    counters: list = field(default_factory=list)   # every Philox counter drawn

    @property
    def min_margin(self):
        return min((d.margin for d in self.decisions), default=math.inf)


def nuts_tree(q, grad, logp, p0, h0, eps, inv_mass, seed, it, chain, max_depth, leapfrog, direct=False):
    """One No-U-Turn transition of one chain as k_nuts_begin (after the momentum), k_nuts_leaf per leaf and k_nuts_end
    build it.  ``leapfrog(q, p, g, signed_eps) -> (q, p, g, logp)`` integrates one leaf.  ``direct``: check the
    sub-tree U-turns from the stored leaves instead of the checkpoints."""
    inv_mass = np.asarray(inv_mass)
    ql = qr = qprop = np.asarray(q, dtype=np.float64)
    gl = gr = gprop = np.asarray(grad, dtype=np.float64)
    pl = pr = np.asarray(p0, dtype=np.float64)
    lpprop, log_w, rho = float(logp), 0.0, pl.copy()
    sum_acc = n_acc = 0.0
    depth, diverged = 0, False
    escale = max(1.0, abs(h0))
    out = Tree(qprop, gprop, lpprop, 0.0, 0, False, [])
    dec, ctrs = out.decisions, out.counters

    def draw(word0):
        ctrs.append(counter(word0, chain, it, NUTS))
        return uniform(seed, it, chain, word0, NUTS)

    for j in range(max_depth):
        u = draw(tag_direction(j))
        fwd = u < 0.5
        dec.append(Decision("direction", j, -1, 0, fwd, abs(0.5 - u)))
        e = eps if fwd else -eps
        out.eps_signed.append(e)
        qw, pw, gw = (qr, pr, gr) if fwd else (ql, pl, gl)
        s_log_w, s_lp, s_rho, s_stop = -math.inf, lpprop, np.zeros(17), False
        sq = sg = None
        pck, rck = {}, {}           # checkpoints: momentum and running sum at the even leaf that opened a span
        leaves_p = []               # direct formulation: every leaf's momentum
        for n in range(1 << j):
            qw, pw, gw, lpw = leapfrog(qw, pw, gw, e)
            lpw = float(lpw)
            h = -lpw + 0.5 * float(pw @ (inv_mass @ pw))
            dh = h0 - h
            if not math.isfinite(dh):
                dh = -math.inf
            div = abs(dh) > DIVERGENCE
            scale = max(escale, abs(h) if math.isfinite(h) else 0.0)
            dec.append(Decision("divergent", j, n, 0, div, abs(abs(dh) - DIVERGENCE) / scale, dh))
            sum_acc += math.exp(min(dh, 0.0))
            n_acc += 1.0
            if div:
                diverged = s_stop = True
                break
            new_w = _logaddexp(s_log_w, dh)
            u = draw(tag_leaf(j, n))
            m = _log_margin(dh - new_w, u, scale)
            take = m > 0
            dec.append(Decision("take", j, n, 0, take, abs(m)))
            if take:
                sq, sg, s_lp = qw, gw, lpw
            s_rho = s_rho + pw
            s_log_w = new_w
            if j > 0:
                if direct:
                    leaves_p.append(pw)
                    size = 2
                    while (n + 1) % size == 0:   # every balanced span of >= 2 leaves that ends at leaf n
                        span = leaves_p[n + 1 - size:n + 1]
                        turned, m = _turning(inv_mass, span[0], pw, np.sum(span, axis=0))
                        dec.append(Decision("turned", j, n, size, turned, m))
                        s_stop |= turned
                        size *= 2
                else:
                    idx_max = bin(n >> 1).count("1")
                    if n % 2 == 0:
                        pck[idx_max], rck[idx_max] = pw, s_rho
                    else:
                        trailing = (n ^ (n + 1)).bit_length() - 1
                        for i in range(idx_max, idx_max - trailing, -1):
                            turned, m = _turning(inv_mass, pck[i], pw, s_rho - rck[i] + pck[i])
                            dec.append(Decision("turned", j, n, 1 << (idx_max - i + 1), turned, m))
                            s_stop |= turned
            if s_stop:
                break
        depth += 1
        if s_stop:
            break
        # merge the finished sub-tree: biased progressive sampling
        u = draw(tag_merge(j))
        m = _log_margin(min(s_log_w - log_w, 0.0), u, escale)
        take = m > 0
        dec.append(Decision("merge", j, -1, 0, take, abs(m)))
        if take:
            qprop, gprop, lpprop = sq, sg, s_lp
        rho = rho + s_rho
        if fwd:
            qr, pr, gr = qw, pw, gw
        else:
            ql, pl, gl = qw, pw, gw
        log_w = _logaddexp(log_w, s_log_w)
        if j + 1 == max_depth:
            break
        turned, m = _turning(inv_mass, pl, pr, rho)
        dec.append(Decision("uturn", j, -1, 0, turned, m))
        if turned:
            break
    out.q, out.grad, out.logp = qprop, gprop, lpprop
    out.accept = sum_acc / max(n_acc, 1.0)
    out.depth, out.diverged = depth, diverged
    return out
