"""CPU checks of the Rao-Blackwellised infection / waner probabilities' restatement (oracle/infection_probs.py), which
the GPU kernel k_infprob_accum is compared against in tests/test_gpu_infection_probs.py:
  * against a brute force that sums over ALL raw configurations of each block (2^len per time chunk, both values of a
    bit without splits) with the rest of the state fixed -- an independent check of the "first raw 1" reduction;
  * unbiasedness, exactly: on an enumerable model sum_x pi(x) h(x) = sum_x pi(x) f(x) (the tower property)."""
import numpy as np
import pytest

from oracle import abd_oracle as ora
from oracle.infection_probs import infection_probs


def small_cohort(rng, G, N, p_pcr=0.15):
    from abdpymc_b200.cohort import CohortArrays

    counts = rng.poisson(5, size=N)
    counts[0] = 0                       # an individual without rows
    ind = np.repeat(np.arange(N), counts)
    r = len(ind)
    pcr = rng.random((N, G)) < p_pcr
    pcr[1] = False
    pcr[1, G // 2] = True               # at least one PCR+ month
    return CohortArrays(vacs=rng.random((N, G)) < 0.1, pcrpos=pcr, ind=ind, gap=rng.integers(0, G, size=r),
                        antigen=rng.integers(0, 2, size=r), x=rng.integers(0, 8, size=r).astype(float),
                        od=rng.normal(0.9, 0.4, size=r))


def point(rng, G):
    v = ora.sample_prior(rng, G)
    v.update(it_n_sigma=0.7, it_s_sigma=0.7, p=0.3, ab_s_p_waner=0.4)
    return np.array([v[n] for n in ora.THETA13]), v["p"], v["ab_s_p_waner"]


def brute_force(o, th, p, pw, i_raw, w):
    """Every raw configuration of each block (a time chunk, or one bit without splits), the rest fixed."""
    G, N = o.G, o.N
    blocks = ora.chunk_bounds(G, o.splits) if o.splits else [(t, t + 1) for t in range(G)]
    out = np.zeros((G, N))
    for a, b in blocks:
        n = b - a
        lw, cols = [], []
        for x in range(2 ** n):
            bits = np.array([(x >> j) & 1 for j in range(n)])
            cand = i_raw.copy()
            cand[a:b] = bits[:, None]
            k = bits.sum()
            lw.append(o.loglik_per_individual(th, cand, w) + k * np.log(p) + (n - k) * np.log1p(-p))
            cols.append(o.constrain(cand)[a:b])
        lw = np.array(lw)
        e = np.exp(lw - lw.max(axis=0))
        out[a:b] = (e[:, None, :] * np.array(cols)).sum(axis=0) / e.sum(axis=0)
    l1, l0 = o.loglik_per_individual(th, i_raw, np.ones(N)), o.loglik_per_individual(th, i_raw, np.zeros(N))
    lw1, lw0 = l1 + np.log(pw), l0 + np.log1p(-pw)
    m = np.maximum(lw1, lw0)
    return out, np.exp(lw1 - m) / (np.exp(lw1 - m) + np.exp(lw0 - m))


@pytest.mark.parametrize("ignore_pcrpos", [False, True])
@pytest.mark.parametrize("G,splits", [(5, ()), (6, (2,)), (8, (2, 4)), (7, (2, 4))])
def test_oracle_matches_brute_force_over_block_configurations(G, splits, ignore_pcrpos):
    rng = np.random.default_rng(G * 10 + len(splits) + 2 * ignore_pcrpos)
    N = 7
    co = small_cohort(rng, G, N)
    o = ora.Oracle(co, splits=splits, ignore_pcrpos=ignore_pcrpos, dense=False)
    for rep in range(3):
        th, p, pw = point(rng, G)
        i_raw = (rng.random((G, N)) < (0.1, 0.3, 0.6)[rep]).astype(np.int64)
        w = (rng.random(N) < 0.5).astype(np.int64)
        got_i, got_w = infection_probs(o, th, p, pw, i_raw, w)
        ref_i, ref_w = brute_force(o, th, p, pw, i_raw, w)
        np.testing.assert_allclose(got_i, ref_i, rtol=0, atol=1e-12)
        np.testing.assert_allclose(got_w, ref_w, rtol=0, atol=1e-12)
        assert np.all((got_i >= 0) & (got_i <= 1))
        # the individual without rows: the prior alone
        np.testing.assert_allclose(got_w[0], pw, rtol=1e-14)


@pytest.mark.parametrize("with_pcr", [False, True])
@pytest.mark.parametrize("splits", [(), (2,), (2, 4)])
def test_estimator_is_unbiased_on_an_enumerable_model(splits, with_pcr):
    """sum_x pi(x) h(x) = sum_x pi(x) f(x) over all 2^(G+1) states (i_raw column, waner) of each individual at fixed
    theta: h = the Rao-Blackwellised probabilities, f = the constrained infections and the waner bit."""
    rng = np.random.default_rng(31 + len(splits) + with_pcr)
    G, N = 5, 4
    co = small_cohort(rng, G, N, p_pcr=0.2 if with_pcr else 0.0)
    if not with_pcr:
        co.pcrpos[:] = 0
    th, p, pw = point(rng, G)
    for n in range(N):
        sub = ora.Oracle(co.take(np.array([n])), splits=splits, dense=False)
        lp, hs, fs, hw, fw = [], [], [], [], []
        for s in range(2 ** (G + 1)):
            col, wn = np.array([(s >> t) & 1 for t in range(G)]).reshape(G, 1), np.array([(s >> G) & 1])
            k = col.sum()
            lp.append(sub.loglik(th, col, wn) + k * np.log(p) + (G - k) * np.log1p(-p)
                      + (np.log(pw) if wn[0] else np.log1p(-pw)))
            h_i, h_w = infection_probs(sub, th, p, pw, col, wn)
            hs.append(h_i[:, 0])
            fs.append(sub.constrain(col)[:, 0])
            hw.append(h_w[0])
            fw.append(wn[0])
        pi = np.exp(np.array(lp) - max(lp))
        pi /= pi.sum()
        np.testing.assert_allclose(pi @ np.array(hs), pi @ np.array(fs), rtol=0, atol=1e-12)
        assert abs(pi @ np.array(hw) - pi @ np.array(fw)) < 1e-12
