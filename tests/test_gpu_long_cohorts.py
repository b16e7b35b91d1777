"""Cohorts of 64 to 127 gaps: the 128-bit gap-mask layout, through every layer, against the oracles.

ABD_B200_MASK_BITS=128 forces that layout on any cohort, so the reference goldens (G = 26, 31) drive the
same kernels too.  Tolerances as in test_gpu_parity.py.
"""
import ctypes
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from oracle import abd_oracle as ora

ROOT = Path(__file__).resolve().parent.parent
RTOL = 1e-10


def grad_ok(g, ref, rtol=RTOL):
    scale = np.maximum(np.abs(ref), 1e-3 * np.abs(ref).max(axis=-1, keepdims=True))
    return np.all(np.abs(g - ref) <= rtol * scale + 1e-300)


@pytest.fixture(scope="module")
def Engine():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from abdpymc_b200 import build

    build.build()
    from abdpymc_b200.engine import AbdEngine

    return AbdEngine


@pytest.fixture
def wide128(monkeypatch):
    monkeypatch.setenv("ABD_B200_MASK_BITS", "128")


def random_cohort(rng, G, N, rows_per_ind=6, p_empty=0.2):
    from abdpymc_b200.cohort import CohortArrays

    counts = rng.poisson(rows_per_ind, size=N) * (rng.random(N) > p_empty)
    ind = np.repeat(np.arange(N), counts)
    r = len(ind)
    perm = rng.permutation(r)  # rows need not be sorted at the boundary
    return CohortArrays(
        vacs=rng.random((N, G)) < 0.05, pcrpos=rng.random((N, G)) < 0.03, ind=ind[perm],
        gap=rng.integers(0, G, size=r), antigen=rng.integers(0, 2, size=r),
        x=rng.integers(0, 8, size=r).astype(float) + rng.random(r) * (rng.random(r) < 0.2),
        od=rng.normal(0.8, 0.5, size=r),
    )


def draw_points(rng, G, N, n_points):
    q = np.stack([ora.forward(ora.sample_prior(rng, G)) for _ in range(n_points)])
    dens = np.where(rng.random(n_points) < 0.5, 0.05, 1.0 / G)
    i_raw = (rng.random((n_points, G, N)) < dens[:, None, None]).astype(np.int8)
    w = (rng.random((n_points, N)) < 0.5).astype(np.int8)
    if n_points >= 6:  # adversarial points (SURVEY.md section 8d)
        i_raw[0] = 0
        i_raw[1] = 1
        w[2] = 0
        q[3, 3] = 18.0   # ab_n_rho -> 1
        q[3, 6] = 25.0   # ab_s_rho -> 1
        q[4, 11] = 1e-9  # it_n_b ~ 0
        q[5, 13] = np.log(0.02)  # small sigma
    return q, i_raw, w


def theta_of(q):
    vals = [ora.backward(q[k])[0] for k in range(len(q))]
    th = np.array([[v[n] for n in ora.THETA13] for v in vals])
    return th, np.array([v["p"] for v in vals]), np.array([v["ab_s_p_waner"] for v in vals])


# ------------------------------------------------------------------------------ reference known answers
@pytest.mark.gpu
@pytest.mark.parametrize("forced", [False, True])
def test_constrained_infections_vs_reference_kats(Engine, kats, monkeypatch, forced):
    """K1 -> K2 -> K3 through the deterministics kernel: the G = 64 reference cases on their own layout, and every
    constraint case with the 128-bit layout forced."""
    from abdpymc_b200.cohort import CohortArrays

    if forced:
        monkeypatch.setenv("ABD_B200_MASK_BITS", "128")
    th = np.array([2.0, 1.0, 0.9, -2.0, 2.0, 0.9, -2.0, -1.0, 2.0, 1.0, -1.0, 2.0, 1.0])
    done = 0
    for k in kats["constrain"]:
        i_raw, pcr, want = np.array(k["i_raw"]), np.array(k["pcrpos"]), np.array(k["out"])
        g, n = i_raw.shape
        if not forced and g <= 63:
            continue
        co = CohortArrays(vacs=np.zeros((n, g)), pcrpos=pcr.T, ind=[0], gap=[0], antigen=[0], x=[0.0], od=[0.0])
        with Engine(co, splits=tuple(k["splits"])) as eng:
            i, _, _ = eng.deterministics(th, i_raw, np.zeros(n))
        assert np.array_equal(i, want), k["splits"]
        done += 1
    assert done >= (47 if forced else 7)


# ------------------------------------------------------------------------------ reference goldens, 128-bit layout
def group_cases(cases):
    groups = {}
    for c in cases:
        groups.setdefault((c["cohort"], tuple(c["splits"]), c["ignore_pcrpos"]), []).append(c)
    return groups


@pytest.mark.gpu
def test_reference_goldens_on_the_128_bit_layout(Engine, goldens, cohorts, wide128):
    """The reference goldens (G = 26, 31) through the 128-bit kernels: logp and gradient, the Deterministics and
    the conditional log-odds."""
    z, cases = goldens
    for _, cs in group_cases(cases).items():
        c0 = cs[0]
        with Engine(cohorts[c0["cohort"]], splits=c0["splits"], ignore_pcrpos=c0["ignore_pcrpos"]) as eng:
            q = np.stack([z[f"{c['key']}/q"] for c in cs])
            i_raw = np.stack([z[f"{c['key']}/i_raw"] for c in cs])
            w = np.stack([z[f"{c['key']}/w"] for c in cs])
            ref = np.array([float(z[f"{c['key']}/logp"]) for c in cs])
            gref = np.stack([z[f"{c['key']}/grad"] for c in cs])
            lp, g = eng.logp_dlogp(q, i_raw, w)
            assert np.all(np.abs(lp - ref) <= RTOL * np.abs(ref)), (lp - ref) / ref
            assert grad_ok(g, gref), np.abs(g - gref).max()
            for c in cs:
                k = c["key"]
                vals = ora.backward(z[f"{k}/q"])[0]
                th = np.array([vals[m] for m in ora.THETA13])
                i, mu_n, mu_s = eng.deterministics(th, z[f"{k}/i_raw"], z[f"{k}/w"])
                assert int(i.sum()) == int(z[f"{k}/i_sum"])
                np.testing.assert_allclose(mu_n.sum(), float(z[f"{k}/mu_n_sum"]), rtol=1e-12)
                np.testing.assert_allclose(mu_s.sum(), float(z[f"{k}/mu_s_sum"]), rtol=1e-12)
                if f"{k}/i" in z:
                    assert np.array_equal(i, z[f"{k}/i"])
                    np.testing.assert_allclose(mu_n, z[f"{k}/mu_n"], rtol=1e-12, atol=1e-12)
                    np.testing.assert_allclose(mu_s, z[f"{k}/mu_s"], rtol=1e-12, atol=1e-12)
                if f"{k}/cond" in z:
                    lo, lo_w = eng.cond_logodds(th, vals["p"], vals["ab_s_p_waner"], z[f"{k}/i_raw"], z[f"{k}/w"])
                    ref_c, ref_w = z[f"{k}/cond"], z[f"{k}/cond_w"]
                    assert np.all(np.abs(lo - ref_c) <= 3e-9 * np.maximum(1, np.abs(ref_c)))
                    assert np.all(np.abs(lo_w - ref_w) <= 3e-9 * np.maximum(1, np.abs(ref_w)))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1])
def test_reference_cohort_gibbs_on_the_128_bit_layout(Engine, cohorts, wide128, mode):
    """Gibbs sweeps on the bundled test cohort with the 128-bit layout forced, bit for bit against the restated sweep."""
    co = cohorts["test_cohort"]
    splits = (14, 20)
    rng = np.random.default_rng(31 + mode)
    C = 2
    vals = [ora.sample_prior(rng, co.n_gaps) for _ in range(C)]
    th = np.array([[v[n] for n in ora.THETA13] for v in vals])
    p, pw = np.array([v["p"] for v in vals]), np.array([v["ab_s_p_waner"] for v in vals])
    i_raw = (rng.random((C, co.n_gaps, co.n_inds)) < 0.05).astype(np.int8)
    w = (rng.random((C, co.n_inds)) < 0.5).astype(np.int8)
    with Engine(co, splits=splits) as eng:
        gi, gw, st = eng.gibbs_sweep(th, p, pw, i_raw, w, seed=17, sweep=2, mode=mode, transit_p=0.8)
    for c in range(C):
        ri, rw, rst = ora.device_gibbs_sweep(co, splits, False, th[c], p[c], pw[c], i_raw[c], w[c], 17, 2, c, mode=mode)
        assert np.array_equal(gi[c], ri) and np.array_equal(gw[c], rw) and list(st[c]) == rst


# ------------------------------------------------------------------------------ random long cohorts
@pytest.mark.gpu
@pytest.mark.parametrize("G,N,splits", [(64, 60, (63, 64)), (65, 50, (30, 65)), (96, 70, ()), (96, 40, (64,)),
                                        (127, 45, (100,)), (127, 30, (30, 70))])
def test_long_ragged_cohorts_against_the_oracle(Engine, G, N, splits):
    """logp + gradient against the dense oracle, Deterministics, conditional log-odds, pointwise log-likelihood and
    the streaming posterior sums, on ragged cohorts with splits on both sides of gap 64, PCR+ and vaccination months
    after it and individuals without rows."""
    import torch

    rng = np.random.default_rng(G * 1000 + N + sum(splits))
    co = random_cohort(rng, G, N)
    late = min(64, G - 1)
    assert co.pcrpos[:, late:].any() and co.vacs[:, late:].any() and (np.bincount(co.ind, minlength=N) == 0).any()
    q, i_raw, w = draw_points(rng, G, N, 8)
    o = ora.Oracle(co, splits=splits, dense=True)
    th, p, pw = theta_of(q)
    with Engine(co, splits=splits) as eng:
        lp, g = eng.logp_dlogp(q, i_raw, w)
        for k in range(len(q)):
            rl, rg = o.logp_dlogp(q[k], i_raw[k], w[k])
            assert abs(lp[k] - rl) <= RTOL * abs(rl), (k, lp[k], rl)
            assert grad_ok(g[k], rg), (k, g[k] - rg)
        for k in (5, 6):
            i, mu_n, mu_s = eng.deterministics(th[k], i_raw[k], w[k])
            ri, rn, rs = o.deterministics(th[k], i_raw[k], w[k])
            assert np.array_equal(i, ri)
            np.testing.assert_allclose(mu_n, rn, rtol=1e-12, atol=1e-12)
            np.testing.assert_allclose(mu_s, rs, rtol=1e-12, atol=1e-12)
            lo, lo_w = eng.cond_logodds(th[k], p[k], pw[k], i_raw[k], w[k])
            rlo, rlo_w = o.cond_logodds(th[k], p[k], pw[k], i_raw[k], w[k])
            assert np.all(np.abs(lo - rlo) <= 1e-9 * np.maximum(1, np.abs(rlo)))
            assert np.all(np.abs(lo_w - rlo_w) <= 1e-9 * np.maximum(1, np.abs(rlo_w)))
        ls, ln = eng.loglik_rows(th[:3], i_raw[:3], w[:3])
        for c in range(3):
            ref = o.loglik_rows(th[c], i_raw[c], w[c])
            np.testing.assert_allclose(ls[c], ref["s"], rtol=1e-10, atol=1e-10)
            np.testing.assert_allclose(ln[c], ref["n"], rtol=1e-10, atol=1e-10)
        # streaming posterior sums over 5 chains, straight from q17
        C = 5
        eng.upload_state(i_raw[:C], w[:C])
        di, dw = eng.state_dev(C)
        sums = [torch.zeros(G, N, dtype=torch.float64, device="cuda") for _ in range(3)]
        tq = torch.from_numpy(q[:C].copy()).cuda()
        eng.deterministics_accum_dev(C, tq.data_ptr(), 1, di, dw, sums[0].data_ptr(), sums[1].data_ptr(), sums[2].data_ptr())
        torch.cuda.synchronize()
        want = [np.zeros((G, N)) for _ in range(3)]
        for c in range(C):
            for acc, v in zip(want, o.deterministics(th[c], i_raw[c], w[c])):
                acc += v
        got = [t.cpu().numpy() for t in sums]
        assert np.array_equal(got[0], want[0])
        np.testing.assert_allclose(got[1], want[1], rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(got[2], want[2], rtol=1e-12, atol=1e-12)


# ------------------------------------------------------------------------------ Gibbs at G = 96
@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_gibbs_sweeps_at_96_gaps_bit_exact(Engine, mode):
    """Three sweeps with a chain offset, bit for bit against the restated device sweep (mode 2 runs as mode 1 on
    masks wider than 32 bits)."""
    G, N, C, splits = 96, 24, 2, (30, 70)
    rng = np.random.default_rng(96 + mode)
    co = random_cohort(rng, G, N, rows_per_ind=12, p_empty=0.1)
    vals = [ora.sample_prior(rng, G) for _ in range(C)]
    th = np.array([[v[n] for n in ora.THETA13] for v in vals])
    p, pw = np.array([v["p"] for v in vals]), np.array([v["ab_s_p_waner"] for v in vals])
    i_raw = (rng.random((C, G, N)) < 0.04).astype(np.int8)
    w = (rng.random((C, N)) < 0.5).astype(np.int8)
    seed, off = 0xDEAD_BEEF_0123_4567, 3
    with Engine(co, splits=splits) as eng:
        eng.set_chain_offset(off)
        gi, gw = i_raw, w
        ri, rw = i_raw.copy(), w.copy()
        for sweep in range(3):
            gi, gw, st = eng.gibbs_sweep(th, p, pw, gi, gw, seed=seed, sweep=sweep, mode=mode, transit_p=0.8)
            for c in range(C):
                ri[c], rw[c], rst = ora.device_gibbs_sweep(co, splits, False, th[c], p[c], pw[c], ri[c], rw[c], seed, sweep,
                                                           off + c, mode=min(mode, 1), transit_p=0.8)
                assert list(st[c]) == rst, (sweep, c)
            assert np.array_equal(gi, ri) and np.array_equal(gw, rw), sweep
        assert not np.array_equal(gi, i_raw) and (gi[:, 64:] != i_raw[:, 64:]).any()


@pytest.mark.gpu
def test_packed_resident_state_matches_the_int8_path_at_96_gaps(Engine):
    """The packed resident state (two 128-bit masks per chain and individual) against the int8 route, kept in step
    by the sweeps, and rebuilt after abd_state_touch."""
    import torch

    G, N, C, splits = 96, 41, 3, (64,)
    rng = np.random.default_rng(961)
    co = random_cohort(rng, G, N, rows_per_ind=7)
    q, i_raw, w = draw_points(rng, G, N, C)
    th, p, pw = theta_of(q)
    with Engine(co, splits=splits) as eng:
        lp_h, g_h = eng.logp_dlogp(q, i_raw, w)
        eng.upload_state(i_raw, w)
        lp_r, g_r = eng.logp_dlogp(q)
        assert np.array_equal(lp_h, lp_r) and np.array_equal(g_h, g_r)
        for mode in (0, 1, 2):
            a_i, a_w = i_raw.copy(), w.copy()
            _, _, st_a = eng.gibbs_sweep(th, p, pw, a_i, a_w, seed=3, sweep=mode, mode=mode, inplace=True)
            b_i, b_w, st_b = eng.gibbs_sweep(th, p, pw, i_raw, w, seed=3, sweep=mode, mode=mode)
            assert np.array_equal(a_i, b_i) and np.array_equal(a_w, b_w) and np.array_equal(st_a, st_b)
            lp_res, g_res = eng.logp_dlogp(q)
            lp_dl, g_dl = eng.logp_dlogp(q, b_i, b_w)
            assert np.array_equal(lp_res, lp_dl) and np.array_equal(g_res, g_dl)
            assert not np.array_equal(b_i, i_raw)
        eng.upload_state(i_raw, w)
        d_i, _ = eng.state_dev(C)
        new_i = (rng.random((C, G, N)) < 0.1).astype(np.int8)
        ti = torch.from_numpy(new_i).cuda()
        cudart = ctypes.CDLL("libcudart.so.12")  # already loaded by torch
        cudart.cudaMemcpy.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int]
        assert cudart.cudaMemcpy(d_i, ti.data_ptr(), new_i.nbytes, 3) == 0  # device to device
        torch.cuda.synchronize()
        eng.state_touch()
        lp_t, g_t = eng.logp_dlogp(q)
        lp_n, g_n = eng.logp_dlogp(q, new_i, w)
        assert np.array_equal(lp_t, lp_n) and np.array_equal(g_t, g_n)


# ------------------------------------------------------------------------------ grid planner variants, C oracle
@pytest.mark.gpu
def test_planner_variants_at_96_gaps_against_the_c_oracle(Engine, monkeypatch):
    """A few thousand individuals at G = 96: 4, 32 and 128 chains (multi-chain CTAs), the compact cell layout, and a
    2 000 x 4-chain Gibbs sweep whose decisions match the C oracle's."""
    from oracle import c_oracle

    G, N, splits = 96, 3000, (30, 70)
    rng = np.random.default_rng(9600)
    co = random_cohort(rng, G, N, rows_per_ind=8, p_empty=0.05)
    co.x[:] = np.floor(co.x)  # integer dilutions: the factored mode, which has the compact cell layout
    o = c_oracle.COracle(co, splits=splits)
    q, i_raw, w = draw_points(rng, G, N, 128)
    ref = {}

    def check(lp, g, ks):
        for k in ks:
            if k not in ref:
                ref[k] = o.logp_dlogp(q[k], i_raw[k], w[k])
            rl, rg = ref[k]
            assert abs(lp[k] - rl) <= RTOL * abs(rl), k
            assert grad_ok(g[k], rg), k

    with Engine(co, splits=splits) as eng:
        for C in (4, 32, 128):
            lp, g = eng.logp_dlogp(q[:C], i_raw[:C], w[:C])
            plan = eng.last_plan()
            assert C < 32 or plan["chains_per_cta"] > 1, plan
            check(lp, g, [0, 1, 3, C - 1])
    monkeypatch.setenv("ABD_B200_COMPACT_CELLS", "1")
    with Engine(co, splits=splits) as eng:
        lp, g = eng.logp_dlogp(q[:8], i_raw[:8], w[:8])
        assert eng.last_plan()["compact_cells"] == 1
        check(lp, g, range(8))
    monkeypatch.delenv("ABD_B200_COMPACT_CELLS")
    sub = co.take(np.arange(2000))
    o2 = c_oracle.COracle(sub, splits=splits)
    C = 4
    th, p, pw = theta_of(q[:C])
    si, sw = i_raw[:C, :, :2000], w[:C, :2000]
    with Engine(sub, splits=splits) as eng:
        gi, gw, st = eng.gibbs_sweep(th, p, pw, si, sw, seed=77, sweep=5, mode=0)
    for c in range(C):
        ri, rw, rst = o2.gibbs_sweep(th[c], p[c], pw[c], si[c], sw[c], 77, 5, c, mode=0)
        assert np.array_equal(gi[c], ri) and np.array_equal(gw[c], rw) and list(st[c]) == rst, c


# ------------------------------------------------------------------------------ cache file
@pytest.mark.gpu
def test_cache_round_trip_at_96_gaps(Engine, cohorts, tmp_path):
    """A 128-bit handle writes a version-3 cache file; read back it is the same engine bit for bit.  A handle of at
    most 63 gaps still writes version 2."""
    G, N, splits = 96, 50, (30, 70)
    rng = np.random.default_rng(3)
    co = random_cohort(rng, G, N, rows_per_ind=9)
    q, i_raw, w = draw_points(rng, G, N, 2)
    th, p, pw = theta_of(q)
    path = tmp_path / "c.abdcache"
    with Engine(co, splits=splits) as eng:
        eng.save_cache(path)
        lp, g = eng.logp_dlogp(q, i_raw, w)
        gi, gw, st = eng.gibbs_sweep(th, p, pw, i_raw, w, seed=4, sweep=2)
    assert int(np.frombuffer(path.read_bytes()[8:12], np.int32)[0]) == 3
    with Engine.from_cache(path) as e2:
        assert (e2.G, e2.N, e2.R_s + e2.R_n) == (G, N, co.n_rows)
        assert e2.splits == splits
        lp2, g2 = e2.logp_dlogp(q, i_raw, w)
        gi2, gw2, st2 = e2.gibbs_sweep(th, p, pw, i_raw, w, seed=4, sweep=2)
    assert np.array_equal(lp, lp2) and np.array_equal(g, g2)
    assert np.array_equal(gi, gi2) and np.array_equal(gw, gw2) and np.array_equal(st, st2)
    path.write_bytes(path.read_bytes()[:300])
    with pytest.raises(Exception, match="cache"):
        Engine.from_cache(path)
    p2 = tmp_path / "t.abdcache"
    with Engine(cohorts["test_cohort"], splits=(14, 20)) as eng:
        eng.save_cache(p2)
    assert int(np.frombuffer(p2.read_bytes()[8:12], np.int32)[0]) == 2


# ------------------------------------------------------------------------------ sampler and CLI
@pytest.mark.gpu
@pytest.mark.parametrize("kernel", ["hmc", "nuts"])
def test_sampler_recovers_the_priors_on_a_96_gap_cohort_without_data(Engine, kernel):
    """HMC / NUTS + Gibbs at G = 96 without OD rows: the posterior of the 17 scalars is their prior (p ~ Beta(1, G - 1))."""
    import torch
    from scipy import stats

    from abdpymc_b200 import diagnostics as dg
    from abdpymc_b200.cohort import CohortArrays
    from abdpymc_b200.engine import Q17_RV, backward, forward
    from abdpymc_b200.sampler import AbdTarget, SamplerConfig, sample

    rng = np.random.default_rng(1)
    G, N, C = 96, 6, 8
    empty = np.zeros(0)
    co = CohortArrays(vacs=rng.random((N, G)) < 0.1, pcrpos=np.zeros((N, G)), ind=empty.astype(int), gap=empty.astype(int),
                      antigen=empty.astype(int), x=empty, od=empty)

    def gam(mu, sigma):
        return stats.gamma(a=mu * mu / sigma**2, scale=sigma**2 / mu)

    prior = {"p": stats.beta(1, G - 1), "ab_n_perm": gam(2, .5), "ab_n_temp": gam(1, .5), "ab_n_rho": stats.beta(10, 1),
             "ab_n_init": stats.norm(-2, 1), "ab_s_perm": gam(2, .5), "ab_s_rho": stats.beta(10, 1),
             "ab_s_p_waner": stats.beta(1, 1), "ab_s_tempinf": gam(1, .5), "ab_s_tempvac": gam(1, .5),
             "ab_s_init": stats.norm(-2, 1), "it_n_b": stats.norm(-1, .5), "it_n_d": stats.norm(2, .5),
             "it_n_sigma": stats.expon(), "it_s_b": stats.norm(-1, .5), "it_s_d": stats.norm(2, .5), "it_s_sigma": stats.expon()}
    with Engine(co, splits=(70,)) as eng:
        tgt = AbdTarget(eng, C, np.zeros((C, G, N), np.int8), np.zeros((C, N), np.int8), seed=3, gibbs_mode=0)
        x0 = np.array([1.0 / G, 2, 1, 10 / 11, -2, 2, 10 / 11, 0.5, 1, 1, -2, -1, 2, 1, -1, 2, 1], dtype=np.float64)
        q0 = forward(x0)[None, :] + rng.uniform(-1, 1, size=(C, 17))
        cfg = SamplerConfig(tune=1000, draws=6000, seed=3, kernel=kernel, persistent_trajectories=True)
        res = sample(tgt, torch.from_numpy(q0).to("cuda:0"), cfg)
        i_raw, waner = tgt.state()
    x = backward(res.q)
    summ = dg.summary({name: x[:, :, k] for k, (name, _) in enumerate(Q17_RV)})
    for name, dist in prior.items():
        v = summ[name]
        se = dist.std() / np.sqrt(max(v["ess_bulk"], 50.0))
        assert v["rhat"] < 1.05, (name, v)
        assert abs(v["mean"] - dist.mean()) < 5 * se + 0.01 * dist.std(), (name, v, dist.mean())
        assert abs(v["sd"] / dist.std() - 1.0) < 0.15, (name, v, dist.std())
        draws = x[:, :, [k for k, (n_, _) in enumerate(Q17_RV) if n_ == name][0]].ravel()
        for qq in (0.1, 0.5, 0.9):
            assert abs((draws < dist.ppf(qq)).mean() - qq) < 0.05, (name, qq)
    assert set(np.unique(i_raw)) <= {0, 1} and set(np.unique(waner)) <= {0, 1}


@pytest.mark.gpu
def test_cli_on_a_96_gap_cohort(Engine, tmp_path):
    """abdpymc-infer on a cohort followed for 96 months."""
    from abdpymc_b200 import abd

    if abd.HAVE_PYMC:
        pytest.skip("PyMC present: the CLI takes the pm.sample path")
    co = random_cohort(np.random.default_rng(8), 96, 40, rows_per_ind=10)
    co.to_disk(tmp_path / "cohort_data")
    out = tmp_path / "post.npz"
    abd.main(["--tune", "40", "--draws", "20", "--ititers_data", str(tmp_path / "cohort_data"), "--split_delta",
              "--split_omicron", "--netcdf", str(out), "--chains", "2", "--thinned", "4"])
    z = np.load(out)
    assert z["p"].shape == (2, 20) and np.isfinite(z["sample_stats_lp"]).all()
    assert z["mean_i"].shape == (96, 40) and z["last_i_raw"].shape == (2, 96, 40) and z["i"].shape == (2, 4, 96, 40)


# ------------------------------------------------------------------------------ two GPUs
XCH_SCRIPT = r"""
import json, os, sys
import numpy as np
import torch
import torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from abdpymc_b200.cohort import CohortArrays
from abdpymc_b200.distributed import ShardedEngine
from abdpymc_b200.engine import AbdEngine
from oracle import abd_oracle as ora

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
rng = np.random.default_rng(96)
G, N, C = 96, 3000, 4
counts = rng.poisson(8, size=N)
ind = np.repeat(np.arange(N), counts)
r = len(ind)
co = CohortArrays(vacs=rng.random((N, G)) < 0.05, pcrpos=rng.random((N, G)) < 0.03, ind=ind, gap=rng.integers(0, G, size=r),
                  antigen=rng.integers(0, 2, size=r), x=rng.integers(0, 8, size=r).astype(float), od=rng.normal(0.8, 0.5, size=r))
i_raw = (rng.random((C, G, N)) < 0.04).astype(np.int8)
w = (rng.random((C, N)) < 0.5).astype(np.int8)
q = np.stack([ora.forward(ora.sample_prior(rng, G)) for _ in range(C)])
se = ShardedEngine(co, splits=(30, 70), device_index=local, rank=rank, world=world, fused=True, max_chains=C)
se.upload_state(i_raw, w)
lp, g = (t.clone() for t in se.logp_dlogp(torch.from_numpy(q).to(dev)))
torch.cuda.synchronize()
se.engine.xch_status()
both = torch.cat([lp, g.reshape(-1)])
gathered = [torch.empty_like(both) for _ in range(world)]
dist.all_gather(gathered, both)
ok = all(torch.equal(gathered[0], t) for t in gathered)
if rank == 0:
    with AbdEngine(co, splits=(30, 70), device=local) as eng:
        lp1, g1 = eng.logp_dlogp(q, i_raw, w)
    rel = float(np.max(np.abs(lp.cpu().numpy() - lp1) / np.abs(lp1)))
    scale = np.maximum(np.abs(g1), 1e-3 * np.abs(g1).max(axis=-1, keepdims=True))
    rel_g = float(np.max(np.abs(g.cpu().numpy() - g1) / scale))
    print(json.dumps({"ok": bool(ok), "rel_err": rel, "rel_err_grad": rel_g}))
se.close()
dist.destroy_process_group()
"""


@pytest.mark.gpu
def test_fused_sharded_evaluation_at_96_gaps_equals_one_gpu(tmp_path):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = tmp_path / "xch96.py"
    script.write_text(XCH_SCRIPT)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29599", str(script), str(ROOT)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=str(ROOT))
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    line = json.loads([ln for ln in res.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["ok"] and line["rel_err"] < 1e-11 and line["rel_err_grad"] < 1e-9, line


# ------------------------------------------------------------------------------ host-side limits (no GPU needed)
def _create(lib_path, G, N):
    from abdpymc_b200 import _lib

    lib = _lib.load(lib_path)
    d = _lib.AbdCohort()
    d.n_gaps, d.n_inds = G, N
    h = ctypes.c_void_p()
    rc = lib.abd_create(ctypes.byref(h), ctypes.byref(d), 0)
    return rc, lib.abd_last_error().decode()


@pytest.fixture(scope="module")
def lib_path():
    from abdpymc_b200 import _lib

    if not _lib.LIB_PATH.exists():
        pytest.skip("libabd_b200.so not built")
    return _lib.LIB_PATH


def test_gap_and_individual_limits_are_checked_before_anything_else(lib_path):
    """abd_create checks sizes before it reads an array or touches a device: G = 128 and G = 0 are refused, and with
    more than 63 gaps (7 gap bits in the row words) so are 2^25 individuals."""
    from abdpymc_b200 import _lib

    assert _lib.MAX_GAPS == 127
    for G in (0, 128, 200):
        rc, msg = _create(lib_path, G, 10)
        assert rc == -1 and msg == "n_gaps must be in [1, 127]", (G, msg)
    rc, msg = _create(lib_path, 64, 1 << 25)
    assert rc == -1 and "2^25" in msg, msg
    rc, msg = _create(lib_path, 127, (1 << 25) - 1)
    assert rc == -1 and msg == "vacs is NULL", msg   # past the size checks
    rc, msg = _create(lib_path, 63, 1 << 25)
    assert rc == -1 and msg == "vacs is NULL", msg
