"""GPU tests of the Rao-Blackwellised posterior infection and waner probabilities (abd_infection_probs_accum_dev,
k_infprob_accum): per-state sums against the NumPy restatement (oracle/infection_probs.py, itself checked against a
brute force in tests/test_infection_probs_oracle.py), reproducibility, no effect on the chain, agreement with the
posterior goldens, sharding, and the Python / CLI front ends."""
import numpy as np
import pytest

from oracle import abd_oracle as ora
from oracle.infection_probs import infection_probs

pytestmark = pytest.mark.gpu

ATOL = 1e-10


@pytest.fixture(scope="module")
def Engine():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from abdpymc_b200 import build

    build.build()
    from abdpymc_b200.engine import AbdEngine

    return AbdEngine


def ragged_cohort(rng, G, N, rows_per_ind=6, p_empty=0.2):
    from abdpymc_b200.cohort import CohortArrays

    counts = rng.poisson(rows_per_ind, size=N) * (rng.random(N) > p_empty)
    ind = np.repeat(np.arange(N), counts)
    r = len(ind)
    return CohortArrays(
        vacs=rng.random((N, G)) < 0.05, pcrpos=rng.random((N, G)) < 0.01, ind=ind[rng.permutation(r)],
        gap=rng.integers(0, G, size=r), antigen=rng.integers(0, 2, size=r),
        x=rng.integers(0, 8, size=r).astype(float), od=rng.normal(0.8, 0.5, size=r),
    )


def draw_states(rng, G, N, C):
    q = np.stack([ora.forward(ora.sample_prior(rng, G)) for _ in range(C)])
    q[:, 13] = q[:, 16] = np.log(0.6)   # sigmas of a fitted model: the conditionals are neither flat nor degenerate
    dens = np.where(rng.random(C) < 0.5, 0.05, 3.0 / G)
    i_raw = (rng.random((C, G, N)) < dens[:, None, None]).astype(np.int8)
    w = (rng.random((C, N)) < 0.5).astype(np.int8)
    return q, i_raw, w


def oracle_sums(co, splits, ignore_pcrpos, q, i_raw, w):
    o = ora.Oracle(co, splits=splits, ignore_pcrpos=ignore_pcrpos, dense=False)
    si, sw = np.zeros((co.n_gaps, co.n_inds)), np.zeros(co.n_inds)
    for c in range(len(q)):
        vals = ora.backward(q[c])[0]
        th = np.array([vals[n] for n in ora.THETA13])
        a, b = infection_probs(o, th, vals["p"], vals["ab_s_p_waner"], i_raw[c], w[c])
        si += a
        sw += b
    return si, sw


def gpu_sums(eng, q, i_raw, w, resident):
    """One accumulation into zeroed totals, from the resident (packed) state or from freshly uploaded int8 arrays."""
    import torch

    dev = torch.device("cuda", eng.device)
    C = len(q)
    qd = torch.from_numpy(np.ascontiguousarray(q)).to(dev)
    if resident:
        eng.upload_state(i_raw, w)
        d_i, d_w = eng.state_dev(C)
    else:
        ti, tw = torch.from_numpy(i_raw).to(dev), torch.from_numpy(w).to(dev)
        d_i, d_w = ti.data_ptr(), tw.data_ptr()
    si = torch.zeros(eng.G, eng.N, dtype=torch.float64, device=dev)
    sw = torch.zeros(eng.N, dtype=torch.float64, device=dev)
    eng.infection_probs_accum_dev(C, qd.data_ptr(), d_i, d_w, si.data_ptr(), sw.data_ptr(),
                                  torch.cuda.current_stream(dev).cuda_stream)
    torch.cuda.synchronize(dev)
    return si.cpu().numpy(), sw.cpu().numpy()


def check_case(Engine, co, splits, ignore_pcrpos, C, seed, chain_offset=0):
    rng = np.random.default_rng(seed)
    q, i_raw, w = draw_states(rng, co.n_gaps, co.n_inds, C)
    ref_i, ref_w = oracle_sums(co, splits, ignore_pcrpos, q, i_raw, w)
    with Engine(co, splits=splits, ignore_pcrpos=ignore_pcrpos) as eng:
        if chain_offset:
            eng.set_chain_offset(chain_offset)   # keys random streams only: no effect here
        for resident in (False, True):
            gi, gw = gpu_sums(eng, q, i_raw, w, resident)
            np.testing.assert_allclose(gi, ref_i, rtol=0, atol=ATOL)
            np.testing.assert_allclose(gw, ref_w, rtol=0, atol=ATOL)
    return gi, gw


@pytest.mark.parametrize("splits,ignore_pcrpos,C", [((14, 20), False, 3), ((14,), False, 1), ((), False, 3),
                                                    ((14, 20), True, 33), ((), True, 1)])
def test_test_cohort_against_the_oracle(Engine, cohorts, splits, ignore_pcrpos, C):
    check_case(Engine, cohorts["test_cohort"], splits, ignore_pcrpos, C, seed=len(splits) + C, chain_offset=5 * (C > 1))


@pytest.mark.parametrize("splits", [(14, 20), ()])
def test_simulated_1k_cohort_against_the_oracle(Engine, splits):
    from abdpymc_b200.cohort import synthetic_cohort

    check_case(Engine, synthetic_cohort(1000), splits, False, 2, seed=41 + len(splits))


@pytest.mark.parametrize("G,N,splits", [(45, 40, (5,)), (64, 50, (20, 50)), (96, 40, (20,)), (96, 30, ()), (127, 30, (20, 93)),
                                        (127, 20, (60,))])
def test_long_ragged_cohorts_against_the_oracle(Engine, G, N, splits):
    """Chunks of 33 to 96 gaps on the 64- and 128-bit layouts: options weighted in groups of 32 with the online
    log-sum-exp; and one-chunk models of 96 gaps."""
    rng = np.random.default_rng(G + N)
    check_case(Engine, ragged_cohort(rng, G, N), splits, False, 3, seed=G)


@pytest.mark.parametrize("splits", [(14, 20), ()])
def test_forced_128_bit_layout_against_the_oracle(Engine, cohorts, monkeypatch, splits):
    monkeypatch.setenv("ABD_B200_MASK_BITS", "128")
    check_case(Engine, cohorts["test_cohort"], splits, False, 3, seed=7)


def test_reproducible_and_read_only(Engine, cohorts):
    """Two calls give bitwise-identical sums; the resident int8 state and its packed copy are unchanged afterwards
    (the download, and the log-density evaluated from the packed copy, are bitwise what they were)."""
    import torch

    co = cohorts["test_cohort"]
    rng = np.random.default_rng(3)
    C = 4
    q, i_raw, w = draw_states(rng, co.n_gaps, co.n_inds, C)
    with Engine(co, splits=(14, 20)) as eng:
        a = gpu_sums(eng, q, i_raw, w, resident=True)
        lp0, g0 = eng.logp_dlogp(q)
        dev = torch.device("cuda", eng.device)
        qd = torch.from_numpy(q).to(dev)
        d_i, d_w = eng.state_dev(C)
        st = torch.cuda.current_stream(dev).cuda_stream
        again = []
        for _ in range(2):   # on the state the first call left, without a new upload
            si = torch.zeros(eng.G, eng.N, dtype=torch.float64, device=dev)
            sw = torch.zeros(eng.N, dtype=torch.float64, device=dev)
            eng.infection_probs_accum_dev(C, qd.data_ptr(), d_i, d_w, si.data_ptr(), sw.data_ptr(), st)
            eng.infection_probs_accum_dev(C, qd.data_ptr(), d_i, d_w, si.data_ptr(), sw.data_ptr(), st)
            again.append((si.cpu().numpy(), sw.cpu().numpy()))
        for si, sw in again:   # each call adds exactly what the first one did
            assert np.array_equal(si, 2 * a[0]) and np.array_equal(sw, 2 * a[1])
        di, dw = eng.download_state(C)
        assert np.array_equal(di, i_raw) and np.array_equal(dw, w)
        lp1, g1 = eng.logp_dlogp(q)
        assert np.array_equal(lp0, lp1) and np.array_equal(g0, g1)


def test_shard_blocks_concatenate_to_the_whole_cohort(Engine, cohorts):
    """Individual-local: every block of individuals adds exactly its own entries (bitwise), no collective."""
    from abdpymc_b200.distributed import shard_cohort

    co = cohorts["test_cohort"]
    rng = np.random.default_rng(12)
    C = 5
    q, i_raw, w = draw_states(rng, co.n_gaps, co.n_inds, C)
    with Engine(co, splits=(14, 20)) as eng:
        whole = gpu_sums(eng, q, i_raw, w, resident=True)
    parts = []
    for rank in range(3):
        shard, totals, offset, sl = shard_cohort(co, rank, 3)
        with Engine(shard, splits=(14, 20), totals=totals, ind_offset=offset) as eng:
            parts.append(gpu_sums(eng, q, np.ascontiguousarray(i_raw[..., sl]), np.ascontiguousarray(w[..., sl]), True))
    assert np.array_equal(np.concatenate([p[0] for p in parts], axis=1), whole[0])
    assert np.array_equal(np.concatenate([p[1] for p in parts]), whole[1])


def test_rb_average_matches_exact_marginals_with_smaller_error(Engine):
    """G = 5 enumerable model at fixed theta (test_gibbs_stationary_distribution_small_model's setup): over Gibbs sweeps,
    the average of the Rao-Blackwellised probabilities matches the exact posterior marginals of i and ab_s_waner, and
    its chain-to-chain standard error (16 groups of 16 chains) is below that of the plain average of the draws.
    Observed on a B200: median ratio of standard errors (RB / plain) 0.170 over the infections with probability in
    (0.01, 0.99), 0.001 over the waner bits (for individuals without an S row after their first exposure the RB value is
    p_w in every draw)."""
    import torch

    from abdpymc_b200.cohort import CohortArrays

    rng = np.random.default_rng(2024)
    G, N, C, sweeps, groups = 5, 6, 256, 400, 16
    co = ragged_cohort(rng, G, N, rows_per_ind=5, p_empty=0.0)
    pcrpos = np.zeros((N, G))
    pcrpos[0, 1] = pcrpos[1, 3] = 1
    co = CohortArrays(vacs=co.vacs, pcrpos=pcrpos, ind=co.ind, gap=co.gap, antigen=co.antigen, x=co.x,
                      od=rng.normal(0.9, 0.4, size=co.n_rows))
    v = ora.sample_prior(rng, G)
    v.update(it_n_sigma=0.8, it_s_sigma=0.8, p=0.3, ab_s_p_waner=0.4)
    th = np.array([v[n] for n in ora.THETA13])
    splits = (2,)
    # exact marginals per individual
    exact_i, exact_w = np.zeros((G, N)), np.zeros(N)
    for n in range(N):
        sub = ora.Oracle(co.take(np.array([n])), splits=splits, dense=False)
        lp, cols, ws = [], [], []
        for s in range(2 ** (G + 1)):
            col, wn = np.array([(s >> t) & 1 for t in range(G)]), (s >> G) & 1
            k = col.sum()
            lp.append(sub.loglik(th, col.reshape(G, 1), np.array([wn])) + k * np.log(v["p"]) + (G - k) * np.log1p(-v["p"])
                      + (np.log(v["ab_s_p_waner"]) if wn else np.log1p(-v["ab_s_p_waner"])))
            cols.append(sub.constrain(col.reshape(G, 1))[:, 0])
            ws.append(wn)
        pi = np.exp(np.array(lp) - max(lp))
        pi /= pi.sum()
        exact_i[:, n], exact_w[n] = pi @ np.array(cols), pi @ np.array(ws)

    o = ora.Oracle(co, splits=splits, dense=False)
    thC = np.tile(th, (C, 1))
    pC, pwC = np.full(C, v["p"]), np.full(C, v["ab_s_p_waner"])
    dev = torch.device("cuda", 0)
    qd = torch.from_numpy(np.tile(ora.forward(v), (C, 1))).to(dev)
    per = C // groups
    rb_i = torch.zeros(groups, G, N, dtype=torch.float64, device=dev)
    rb_w = torch.zeros(groups, N, dtype=torch.float64, device=dev)
    plain_i, plain_w = np.zeros((groups, G, N)), np.zeros((groups, N))
    with Engine(co, splits=splits) as eng:
        eng.upload_state(np.zeros((C, G, N), np.int8), np.zeros((C, N), np.int8))
        st = torch.cuda.current_stream(dev).cuda_stream
        for sweep in range(sweeps + 50):
            gi, gw, _ = eng.gibbs_sweep(thC, pC, pwC, seed=99, sweep=sweep, mode=2)
            if sweep < 50:
                continue
            d_i, d_w = eng.state_dev(C)
            for g in range(groups):   # one launch per group of chains: pointers into the resident state
                c0 = g * per
                eng.infection_probs_accum_dev(per, qd[c0:].data_ptr(), d_i + c0 * G * N, d_w + c0 * N,
                                              rb_i[g].data_ptr(), rb_w[g].data_ptr(), st)
            for c in range(C):
                plain_i[c // per] += o.constrain(gi[c])
            plain_w += gw.reshape(groups, per, N).sum(axis=1)
        torch.cuda.synchronize(dev)
    rb_i = rb_i.cpu().numpy() / (sweeps * per)
    rb_w = rb_w.cpu().numpy() / (sweeps * per)
    plain_i /= sweeps * per
    plain_w /= sweeps * per
    se = lambda a: a.std(axis=0, ddof=1) / np.sqrt(groups)  # noqa: E731
    assert np.all(np.abs(rb_i.mean(axis=0) - exact_i) < 5 * se(rb_i) + 2e-3), np.abs(rb_i.mean(axis=0) - exact_i).max()
    assert np.all(np.abs(rb_w.mean(axis=0) - exact_w) < 5 * se(rb_w) + 2e-3), np.abs(rb_w.mean(axis=0) - exact_w).max()
    sel = (exact_i > 0.01) & (exact_i < 0.99)
    ratio_i = float(np.median(se(rb_i)[sel] / se(plain_i)[sel]))
    ratio_w = float(np.median(se(rb_w) / se(plain_w)))
    print(f"median standard-error ratio RB / plain: i {ratio_i:.3f}, waner {ratio_w:.3f}")
    assert ratio_i < 1.0 and ratio_w < 1.0, (ratio_i, ratio_w)


def _run(gpu_cohort, rao_blackwell, kernel="hmc"):
    import torch

    from abdpymc_b200.abd import make_engine
    from abdpymc_b200.sampler import AbdTarget, SamplerConfig, sample

    co = gpu_cohort
    C = 4
    rng = np.random.default_rng(0)
    q0 = torch.from_numpy(np.stack([ora.forward(ora.sample_prior(rng, co.n_gaps)) for _ in range(C)])).to("cuda:0")
    eng = make_engine(co, splits=(14, 20))
    target = AbdTarget(eng, C, np.zeros((C, co.n_gaps, co.n_inds), np.int8), np.zeros((C, co.n_inds), np.int8), seed=4)
    cfg = SamplerConfig(tune=80, draws=60, seed=4, record_deterministics_every=1, thinned_deterministics=5, kernel=kernel,
                        rao_blackwell=rao_blackwell)
    res = sample(target, q0, cfg)
    last = target.state()
    eng.close()
    return res, last


@pytest.mark.parametrize("kernel", ["hmc", "nuts"])
def test_sampler_chain_is_unchanged_by_rao_blackwell(Engine, cohorts, kernel):
    """Same seed with and without the flag: every SamplerResult field but the wall-clock times and the two new keys is
    bitwise identical, and so is the final binary state."""
    a, la = _run(cohorts["test_cohort"], False, kernel)
    b, lb = _run(cohorts["test_cohort"], True, kernel)
    assert set(b.means) == set(a.means) | {"i_rb", "ab_s_waner_rb"}
    assert b.means["i_rb"].shape == a.means["i"].shape and b.means["ab_s_waner_rb"].shape == (a.means["i"].shape[1],)
    for f in ("q", "logp", "accept", "step_size", "inv_mass"):
        assert np.array_equal(getattr(a, f), getattr(b, f)), f
    assert a.n_grad_evals == b.n_grad_evals and a.n_grad_evals_tune == b.n_grad_evals_tune
    for d in ("means", "thinned", "stats"):
        x, y = getattr(a, d), getattr(b, d)
        for k in x:
            assert np.array_equal(x[k], y[k]), (d, k)
    assert np.array_equal(la[0], lb[0]) and np.array_equal(la[1], lb[1])


def test_rb_means_agree_with_the_posterior_goldens(Engine):
    """``means["i_rb"]`` against the reference algorithm's posterior infection probabilities
    (tests/golden/posterior_goldens.npz, test_cohort/mean_i) under test_posterior_agrees_with_the_reference_algorithm's
    tolerance, and against this run's plain ``means["i"]`` within the same Monte-Carlo error; the waner probabilities
    against the goldens' mean_w."""
    import json
    from pathlib import Path

    from abdpymc_b200.abd import infer_builtin
    from abdpymc_b200.cohort import CohortArrays

    z = np.load(Path(__file__).resolve().parent / "golden" / "posterior_goldens.npz")
    case = "test_cohort"
    meta = json.loads(str(z["meta"]))[case]
    co = CohortArrays.load(case)
    res, _, _ = infer_builtin(co, tuple(meta["splits"]), False, tune=1500, draws=6000, chains=8, seed=3, rao_blackwell=True)
    ref_i, by_chain = z[f"{case}/mean_i"], z[f"{case}/mean_i_by_chain"]
    mc = by_chain.std(axis=0, ddof=1) / np.sqrt(by_chain.shape[0])
    rb = res.means["i_rb"]
    assert np.all(np.abs(rb - ref_i) < 5 * mc + 0.03), float(np.abs(rb - ref_i).max())
    assert np.all(np.abs(rb - res.means["i"]) < 5 * mc + 0.03), float(np.abs(rb - res.means["i"]).max())
    assert np.all(np.abs(res.means["ab_s_waner_rb"] - z[f"{case}/mean_w"]) < 0.15)


def test_cli_writes_the_rb_keys_only_with_the_flag(Engine, tmp_path):
    from abdpymc_b200 import abd
    from abdpymc_b200.cohort import CohortArrays

    if abd.HAVE_PYMC:
        pytest.skip("PyMC present: the CLI takes the pm.sample path")
    CohortArrays.load("test_cohort").to_disk(tmp_path / "cohort_data")
    args = ["--tune", "40", "--draws", "20", "--ititers_data", str(tmp_path / "cohort_data"), "--split_delta",
            "--split_omicron", "--chains", "2", "--thinned", "5"]
    abd.main(args + ["--netcdf", str(tmp_path / "a.npz")])
    abd.main(args + ["--netcdf", str(tmp_path / "b.npz"), "--rao_blackwell"])
    za, zb = np.load(tmp_path / "a.npz"), np.load(tmp_path / "b.npz")
    assert set(zb.files) == set(za.files) | {"mean_i_rb", "mean_ab_s_waner_rb"}
    assert "mean_i_rb" not in za.files
    assert zb["mean_i_rb"].shape == (26, 10) and zb["mean_ab_s_waner_rb"].shape == (10,)
    assert np.all((zb["mean_i_rb"] >= 0) & (zb["mean_i_rb"] <= 1)) and np.all((zb["mean_ab_s_waner_rb"] >= 0))
    assert np.array_equal(za["p"], zb["p"]) and np.array_equal(za["mean_i"], zb["mean_i"])


def test_infection_probabilities_of_a_posterior_dict(Engine, cohorts):
    """The post-hoc helper for PyMC / InferenceData users: (chain, draw, ...) arrays in, averages out."""
    from abdpymc_b200 import abd
    from abdpymc_b200.engine import Q17_RV

    co = cohorts["test_cohort"]
    rng = np.random.default_rng(5)
    n_c, n_d = 2, 5
    q, i_raw, w = draw_states(rng, co.n_gaps, co.n_inds, n_c * n_d)
    vals = np.stack([[ora.backward(q[k])[0][n] for n, _ in Q17_RV] for k in range(len(q))])
    post = {n: vals[:, j].reshape(n_c, n_d) for j, (n, _) in enumerate(Q17_RV)}
    post.update(i_raw=i_raw.astype(np.int64).reshape(n_c, n_d, co.n_gaps, co.n_inds),
                ab_s_waner=w.astype(np.int64).reshape(n_c, n_d, co.n_inds))
    splits = (14, 20)
    with Engine(co, splits=splits) as eng:
        out = abd.infection_probabilities(eng, post, batch=3)
    ref_i, ref_w = oracle_sums(co, splits, False, q, i_raw, w)
    np.testing.assert_allclose(out["i_rb"], ref_i / len(q), rtol=0, atol=ATOL)
    np.testing.assert_allclose(out["ab_s_waner_rb"], ref_w / len(q), rtol=0, atol=ATOL)


def test_sharded_cli_run_on_two_gpus(Engine, tmp_path):
    """--shard individuals: each rank adds its own block; the gathered means have the whole cohort's shapes."""
    import torch

    from abdpymc_b200 import abd
    from abdpymc_b200.cohort import CohortArrays

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    if abd.HAVE_PYMC:
        pytest.skip("PyMC present: the CLI takes the pm.sample path")
    CohortArrays.load("test_cohort").to_disk(tmp_path / "cohort_data")
    out = tmp_path / "post.npz"
    abd.main(["--tune", "40", "--draws", "20", "--ititers_data", str(tmp_path / "cohort_data"), "--split_delta",
              "--split_omicron", "--chains", "2", "--devices", "0,1", "--shard", "individuals", "--rao_blackwell",
              "--netcdf", str(out)])
    z = np.load(out)
    assert z["mean_i_rb"].shape == (26, 10) and z["mean_ab_s_waner_rb"].shape == (10,)
    assert np.all((z["mean_i_rb"] >= 0) & (z["mean_i_rb"] <= 1))
