"""The device HMC and NUTS transitions decision by decision against their fp64 restatement (oracle/transitions.py).

The kernels draw from counter-based Philox streams, so given the same leaves the restatement makes the same random
decisions.  A decision is compared only where its restated margin exceeds ``TIE`` (relative to the scale of the numbers
it was computed from): below that, rounding may legitimately flip it.  A near-tie is reported and the chain is not
compared for the rest of that iteration; the seeds below produce none.
"""
import math

import numpy as np
import pytest

from oracle import abd_oracle as ora
from oracle import transitions as tr

TIE = 1e-9
SEED = 0x9E37_79B9_7F4A_7C15           # above 2^32: the key's high word is seed hi ^ iter hi
IT = (5 << 32) + 17                    # likewise for the iteration index
X0 = np.array([1.0 / 26, 2, 1, 10 / 11, -2, 2, 10 / 11, 0.5, 1, 1, -2, -1, 2, 1, -1, 2, 1], dtype=np.float64)


class Tally:
    """Decisions compared and near-ties skipped, printed at the end of each GPU test."""

    def __init__(self, name):
        self.name, self.compared, self.ties = name, 0, []

    def ok(self, decisions, where):
        m = min((d.margin for d in decisions), default=math.inf)
        if m <= TIE:
            bad = min(decisions, key=lambda d: d.margin)
            self.ties.append((where, bad))
            print(f"{self.name}: near-tie at {where}: {bad}")
            return False
        self.compared += len(decisions)
        return True

    def report(self):
        print(f"{self.name}: {self.compared} decisions compared, {len(self.ties)} near-ties skipped")
        assert self.compared > 0


def metric(rng, D=17):
    a = rng.normal(size=(D, D))
    inv_mass = a @ a.T / D + np.eye(D)
    chol = np.linalg.cholesky(inv_mass)
    return inv_mass, np.linalg.inv(chol.T)


def gaussian(rng, D=17, stiff=0.0, box=None):
    """logp of N(mu, A^-1) with a dense precision A; ``stiff``: one direction's precision raised by that much;
    ``box``: logp = -inf where any |q - mu| exceeds it (the cliff)."""
    a = rng.normal(size=(D, D))
    A = a @ a.T / D + 0.5 * np.eye(D)
    if stiff:
        v = rng.normal(size=D)
        v /= np.linalg.norm(v)
        A = A + stiff * np.outer(v, v)
    mu = rng.normal(size=D)

    def f(q):
        d = q - mu
        g = -(A @ d)
        lp = 0.5 * float(d @ g)
        if box is not None and np.any(np.abs(d) > box):
            lp = -np.inf
        return lp, g

    return f, mu, A


def leapfrog_of(f, inv_mass):
    """One leaf: the same NumPy arithmetic for the device driver and the restatement, so both see the same bits."""

    def lf(q, p, g, e):
        with np.errstate(all="ignore"):
            ph = p + 0.5 * e * g
            qn = q + e * (inv_mass @ ph)
            lp, gn = f(qn)
            return qn, ph + 0.5 * e * gn, gn, lp

    return lf


# ------------------------------------------------------------------------------------------ CPU
def _trees(kind, max_depth, n_chains=6):
    rng = np.random.default_rng(max_depth * 10 + len(kind))
    inv_mass, linv_t = metric(rng)
    f, mu, A = gaussian(rng, stiff=1e4 if kind == "stiff" else 0.0, box=1.0 if kind == "cliff" else None)
    inv_mass = np.linalg.inv(A) if kind != "stiff" else inv_mass
    linv_t = np.linalg.inv(np.linalg.cholesky(inv_mass).T)
    lf = leapfrog_of(f, inv_mass)
    eps = {"gauss": 0.35, "cliff": 0.5, "stiff": 0.05, "tiny": 1e-3}[kind]
    for c in range(n_chains):
        q = mu + 0.3 * rng.normal(size=17)
        lp, g = f(q)
        for it in (IT, IT + 1):
            z, p0, zz = tr.momentum(SEED, it, c, linv_t)
            args = (q, g, lp, p0, -lp + 0.5 * zz, eps * (1 + 0.1 * c), inv_mass, SEED, it, c, max_depth, lf)
            yield tr.nuts_tree(*args), tr.nuts_tree(*args, direct=True)


@pytest.mark.parametrize("kind,max_depth", [("gauss", 1), ("gauss", 4), ("cliff", 4), ("stiff", 4), ("gauss", 10),
                                            ("tiny", 10), ("cliff", 10)])
def test_checkpoints_and_direct_spans_make_the_same_decisions(kind, max_depth):
    """The kernel's O(depth) checkpoint scheme for the sub-tree U-turn checks (indices popc(n >> 1) and trailing-one
    counts) against every balanced span summed directly from the stored leaves: the same checks in the same order,
    the same outcome, the same tree."""
    seen = {"fwd": 0, "bwd": 0, "div": 0, "turned": 0, "depth": 0}
    for a, b in _trees(kind, max_depth):
        assert [d.key() for d in a.decisions] == [d.key() for d in b.decisions]
        np.testing.assert_allclose([d.margin for d in a.decisions], [d.margin for d in b.decisions], rtol=1e-6, atol=1e-12)
        assert a.min_margin > TIE
        assert np.array_equal(a.q, b.q) and a.depth == b.depth and a.diverged == b.diverged and a.accept == b.accept
        for d in a.decisions:
            seen["fwd"] += d.kind == "direction" and d.value
            seen["bwd"] += d.kind == "direction" and not d.value
            seen["div"] += d.kind == "divergent" and d.value
            seen["turned"] += d.kind == "turned" and d.value
        seen["depth"] = max(seen["depth"], a.depth)
    assert seen["fwd"] and seen["bwd"]
    if max_depth > 1:
        assert seen["turned"] or kind in ("tiny", "stiff") or seen["div"]
    if kind in ("cliff", "stiff"):
        assert seen["div"]
    if kind == "tiny":
        assert seen["depth"] == 10


def test_no_two_draws_of_an_iteration_share_a_philox_counter():
    """Every counter a transition may draw at max_depth 10 -- the 17 momentum lanes, the HMC accept, and every NUTS
    direction, leaf and merge -- is distinct, per chain and across chains; a depth-10 tree draws only from that set."""
    D, chains = 10, (0, 1, 7)
    tags = [tr.tag_direction(j) for j in range(D)] + [tr.tag_merge(j) for j in range(D)]
    tags += [tr.tag_leaf(j, n) for j in range(D) for n in range(1 << j)]
    assert len(set(tags)) == len(tags) and all(0 <= t < 2**32 for t in tags)
    ctrs = set()
    for c in chains:
        mine = [tr.counter(lane, c, IT, tr.HMC_BEGIN) for lane in range(17)] + [tr.counter(0, c, IT, tr.HMC_END)]
        mine += [tr.counter(t, c, IT, tr.NUTS) for t in tags]
        assert ctrs.isdisjoint(mine)
        ctrs.update(mine)
    assert len(ctrs) == len(chains) * (18 + len(tags))
    tree = next(t for t, _ in _trees("tiny", D, n_chains=1))
    assert tree.depth == D and len(set(tree.counters)) == len(tree.counters) == 2 * D + 2**D - 1
    assert set(tree.counters) <= ctrs


def test_restated_dual_averaging_matches_the_host_sampler():
    import torch

    from abdpymc_b200.sampler import _DualAveraging

    rng = np.random.default_rng(4)
    eps0 = rng.uniform(0.01, 0.5, size=6)
    ref = _DualAveraging(torch.from_numpy(eps0.copy()), 0.8, "cpu")
    da = np.zeros((6, 4))
    da[:, 0] = np.log(10 * eps0)
    for _ in range(40):
        acc = rng.random(6)
        want = ref.update(torch.from_numpy(acc)).numpy()
        for c in range(6):
            da[c], e = tr.dual_averaging(da[c], acc[c], 0.8)
            assert abs(e - want[c]) <= 1e-12 * want[c]
    np.testing.assert_allclose(np.exp(da[:, 2]), ref.final().numpy(), rtol=1e-12)


# ------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def gpu():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from abdpymc_b200 import build

    build.build()
    return torch.device("cuda:0")


def _dev(a, gpu):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(gpu)


def _engine(co=None, splits=(14, 20)):
    from abdpymc_b200.cohort import CohortArrays
    from abdpymc_b200.engine import AbdEngine

    return AbdEngine(co if co is not None else CohortArrays.load("test_cohort"), splits=splits)


@pytest.mark.gpu
@pytest.mark.parametrize("C,offset", [(1, 0), (5, 3), (4097, 1000)])
def test_hmc_kernels_match_the_restatement(gpu, C, offset):
    """k_hmc_begin: the momenta to 1e-13 and h0 to 1e-12 of the restated Box-Muller draws (several blocks, the last one
    partly empty, a chain offset, seed and iteration above 2^32, a dense metric).  k_hmc_end over three adapting calls:
    every accept decision, the chains' q / grad / logp bit for bit, NaN and +-inf energies rejected, the acceptance
    statistic, the step size and the dual-averaging state to 1e-12."""
    import torch

    tally = Tally(f"hmc C={C}")
    rng = np.random.default_rng(C)
    inv_mass, linv_t = metric(rng)
    q, grad = rng.normal(size=(C, 17)), rng.normal(size=(C, 17))
    logp = 10 * rng.normal(size=C)
    f64 = dict(dtype=torch.float64, device=gpu)
    d_q, d_g, d_lp, d_im, d_lt = (_dev(a, gpu) for a in (q, grad, logp, inv_mass, linv_t))
    qw, pw, gw, h0 = torch.empty(C, 17, **f64), torch.empty(C, 17, **f64), torch.empty(C, 17, **f64), torch.empty(C, **f64)
    with _engine() as eng:
        if offset:
            eng.set_chain_offset(offset)
        eng.hmc_begin_dev(C, d_q.data_ptr(), d_g.data_ptr(), d_lp.data_ptr(), d_lt.data_ptr(), SEED, IT, qw.data_ptr(),
                          pw.data_ptr(), gw.data_ptr(), h0.data_ptr())
        torch.cuda.synchronize()
        P, H0 = pw.cpu().numpy(), h0.cpu().numpy()
        assert np.array_equal(qw.cpu().numpy(), q) and np.array_equal(gw.cpu().numpy(), grad)
        for c in range(C):
            z, p, zz = tr.momentum(SEED, IT, offset + c, linv_t)
            assert np.all(np.abs(P[c] - p) <= 1e-13 * (np.abs(linv_t) @ np.abs(z))), c
            assert abs(H0[c] - (-logp[c] + 0.5 * zz)) <= 1e-12 * (abs(logp[c]) + zz), c

        # proposals with known energy errors dh in (-3, 3), and non-finite energies
        kin = 0.5 * np.einsum("ci,ij,cj->c", P, inv_mass, P)
        dh = np.linspace(-3, 3, C) if C > 1 else np.array([-0.4])
        lpw = -(H0 - dh) + kin
        if C > 3:
            lpw[1::4], lpw[2::4], lpw[3::8] = np.nan, np.inf, -np.inf
        q_new, g_new = q + 1.0, grad - 1.0
        eps0 = rng.uniform(0.05, 0.2, size=C)
        da = np.zeros((C, 4))
        da[:, 0] = np.log(10 * eps0)
        d_qn, d_gn, d_lpw, d_da, d_eps = (_dev(a, gpu) for a in (q_new, g_new, lpw, da, eps0))
        acc = torch.empty(C, **f64)
        want_q, want_g, want_lp, eps = q.copy(), grad.copy(), logp.copy(), eps0.copy()
        live = np.ones(C, bool)
        for k in range(3):
            it = IT + 10 + k
            eng.hmc_end_dev(C, d_q.data_ptr(), d_g.data_ptr(), d_lp.data_ptr(), d_qn.data_ptr(), pw.data_ptr(), d_gn.data_ptr(),
                            d_lpw.data_ptr(), d_im.data_ptr(), h0.data_ptr(), SEED, it, acc.data_ptr(), d_da.data_ptr(),
                            d_eps.data_ptr(), 1, 0.8)
            torch.cuda.synchronize()
            got_q, got_g, got_lp, got_acc = d_q.cpu().numpy(), d_g.cpu().numpy(), d_lp.cpu().numpy(), acc.cpu().numpy()
            got_da, got_eps = d_da.cpu().numpy(), d_eps.cpu().numpy()
            for c in range(C):
                take, a, dec = tr.hmc_end(H0[c], lpw[c], P[c], inv_mass, SEED, it, offset + c)
                if not np.isfinite(lpw[c]):
                    assert not take and a == 0.0
                assert abs(got_acc[c] - a) <= 1e-12 * a, (c, got_acc[c], a)
                da[c], eps[c] = tr.dual_averaging(da[c], a, 0.8)
                np.testing.assert_allclose(got_da[c], da[c], rtol=1e-12, atol=1e-15)
                assert abs(got_eps[c] - eps[c]) <= 1e-12 * eps[c]
                if not (live[c] and tally.ok([dec], (k, c))):
                    live[c] = False
                    continue
                if take:
                    want_q[c], want_g[c], want_lp[c] = q_new[c], g_new[c], lpw[c]
                assert np.array_equal(got_q[c], want_q[c]) and np.array_equal(got_g[c], want_g[c]), (k, c, take)
                assert got_lp[c] == want_lp[c], (k, c)
    if C > 3:
        taken = np.array([np.array_equal(want_q[c], q_new[c]) for c in range(C)])
        assert taken.any() and not taken.all()
    tally.report()


def _state_view(eng, state, D):
    """PL (the initial momentum right after k_nuts_begin) and H0 of every chain's tree state (NutsLayout)."""
    S = state.cpu().numpy()
    scal = (12 + 2 * D) * 17
    assert S.shape[1] == eng.nuts_state_doubles(D) == scal + 16
    return S[:, 17:34].copy(), S[:, scal + 4].copy()


def _any_active(trees, D):
    return [1] + [int(any(t.depth >= k + 1 for t in trees)) for k in range(1, D + 1)]


B_CASES = [("gauss", 131, 6, 0), ("gauss", 1, 1, 0), ("gauss", 5, 10, 11), ("cliff", 131, 6, 7), ("cliff", 5, 1, 0),
           ("stiff", 131, 6, 0), ("stiff", 5, 10, 0), ("tiny", 5, 10, 3), ("tiny", 1, 6, 0)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,C,D,offset", B_CASES)
def test_nuts_tree_bookkeeping_matches_the_restatement(gpu, kind, C, D, offset):
    """k_nuts_begin, one k_nuts_leaf launch per leaf, k_nuts_end, with the leaves integrated in NumPy on an analytic
    17-dimensional target: a correlated Gaussian with a dense metric, the same behind a cliff (divergences through
    non-finite energies), a stiff direction (finite |dH| > 1000), a tiny step (trees reach max_depth).  The kernel and
    the restatement see the same leaves, so the proposal must be bitwise the restated leaf, and the signed steps, the
    any-active words, depth, divergence, acceptance statistic and dual averaging must match."""
    import torch

    tally = Tally(f"tree {kind} C={C} D={D}")
    rng = np.random.default_rng(C * 100 + D)
    f, mu, A = gaussian(rng, stiff=1e6 if kind == "stiff" else 0.0, box=1.0 if kind == "cliff" else None)
    inv_mass = np.eye(17) if kind == "stiff" else np.linalg.inv(A + 0.1 * metric(rng)[0])
    linv_t = np.linalg.inv(np.linalg.cholesky(inv_mass).T)
    lf = leapfrog_of(f, inv_mass)
    eps = {"gauss": rng.uniform(0.2, 0.6, C), "cliff": rng.uniform(0.3, 0.7, C), "stiff": rng.uniform(0.001, 0.03, C),
           "tiny": np.full(C, 1e-3)}[kind]
    q = mu + 0.3 * rng.normal(size=(C, 17))
    lg = [f(x) for x in q]
    logp, grad = np.array([v[0] for v in lg]), np.array([v[1] for v in lg])
    da = np.zeros((C, 4))
    da[:, 0] = np.log(10 * eps)
    f64 = dict(dtype=torch.float64, device=gpu)
    d_q, d_g, d_lp, d_eps, d_da, d_im, d_lt = (_dev(a, gpu) for a in (q, grad, logp, eps, da, inv_mass, linv_t))
    qw, pw, gw, lpw = torch.empty(C, 17, **f64), torch.empty(C, 17, **f64), torch.empty(C, 17, **f64), torch.empty(C, **f64)
    acc, dep, div, es = (torch.empty(C, **f64) for _ in range(4))
    any_active = torch.zeros(D + 1, dtype=torch.int32, device=gpu)
    seen = {"div_inf": 0, "div_finite": 0, "max_depth": 0}
    with _engine() as eng:
        if offset:
            eng.set_chain_offset(offset)
        state = torch.zeros(C, eng.nuts_state_doubles(D), **f64)
        for k in range(2 if D == 10 else 3):
            it = IT + k
            q0, g0, lp0, eps0 = d_q.cpu().numpy(), d_g.cpu().numpy(), d_lp.cpu().numpy(), d_eps.cpu().numpy()
            eng.nuts_begin_dev(C, D, d_q.data_ptr(), d_g.data_ptr(), d_lp.data_ptr(), d_lt.data_ptr(), d_eps.data_ptr(), SEED,
                               it, state.data_ptr(), qw.data_ptr(), pw.data_ptr(), gw.data_ptr(), es.data_ptr(),
                               any_active.data_ptr())
            torch.cuda.synchronize()
            p0, h0 = _state_view(eng, state, D)
            trees = []
            for c in range(C):
                z, p, zz = tr.momentum(SEED, it, offset + c, linv_t)
                assert np.all(np.abs(p0[c] - p) <= 1e-13 * (np.abs(linv_t) @ np.abs(z)))
                assert abs(h0[c] - (-lp0[c] + 0.5 * zz)) <= 1e-12 * (abs(lp0[c]) + zz)
                trees.append(tr.nuts_tree(q0[c], g0[c], lp0[c], p0[c], h0[c], eps0[c], inv_mass, SEED, it, offset + c, D, lf))
            live = [tally.ok(t.decisions, (k, c)) for c, t in enumerate(trees)]
            for j in range(D):
                for n in range(1 << j):
                    Q, Pm, G, E = qw.cpu().numpy(), pw.cpu().numpy(), gw.cpu().numpy(), es.cpu().numpy()
                    leaves = [lf(Q[c], Pm[c], G[c], E[c]) for c in range(C)]
                    qw.copy_(_dev([v[0] for v in leaves], gpu))
                    pw.copy_(_dev([v[1] for v in leaves], gpu))
                    gw.copy_(_dev([v[2] for v in leaves], gpu))
                    lpw.copy_(_dev([v[3] for v in leaves], gpu))
                    eng.nuts_leaf_dev(C, D, j, n, qw.data_ptr(), pw.data_ptr(), gw.data_ptr(), lpw.data_ptr(), d_im.data_ptr(),
                                      d_eps.data_ptr(), SEED, it, state.data_ptr(), es.data_ptr(), any_active.data_ptr())
                E = es.cpu().numpy()
                for c, t in enumerate(trees):       # the signed step of the depth each chain opens next (or its last)
                    if live[c]:
                        assert E[c] == t.eps_signed[min(j + 1, t.depth - 1)], (k, j, c)
                if j + 1 < D and any_active[j + 1].item() == 0:
                    break
            assert any_active.cpu().tolist() == _any_active([t for t, ok in zip(trees, live) if ok], D) or not all(live)
            eng.nuts_end_dev(C, D, d_q.data_ptr(), d_g.data_ptr(), d_lp.data_ptr(), state.data_ptr(), acc.data_ptr(),
                             dep.data_ptr(), div.data_ptr(), d_da.data_ptr(), d_eps.data_ptr(), 1, 0.8)
            torch.cuda.synchronize()
            Q, G, LP, ACC, DEP, DIV = (t.cpu().numpy() for t in (d_q, d_g, d_lp, acc, dep, div))
            DA, EPS = d_da.cpu().numpy(), d_eps.cpu().numpy()
            for c, t in enumerate(trees):
                da[c], e = tr.dual_averaging(da[c], t.accept, 0.8)
                seen["max_depth"] = max(seen["max_depth"], t.depth)
                for d in t.decisions:
                    if d.kind == "divergent" and d.value:
                        seen["div_finite" if np.isfinite(d.x) else "div_inf"] += 1
                if not live[c]:
                    continue
                assert np.array_equal(Q[c], t.q) and np.array_equal(G[c], t.grad) and LP[c] == t.logp, (k, c)
                assert DEP[c] == t.depth and bool(DIV[c]) == t.diverged, (k, c, DEP[c], t.depth)
                assert abs(ACC[c] - t.accept) <= 1e-12, (k, c)
                np.testing.assert_allclose(DA[c], da[c], rtol=1e-12, atol=1e-15)
                assert abs(EPS[c] - e) <= 1e-12 * e
            da = DA.copy()
    if kind == "cliff":
        assert seen["div_inf"]
    if kind == "stiff":
        assert seen["div_finite"]
    if kind == "tiny" and D == 10:
        assert seen["max_depth"] == 10
    tally.report()


def random_cohort(rng, G, N, rows_per_ind=6, p_empty=0.2):
    from abdpymc_b200.cohort import CohortArrays

    counts = rng.poisson(rows_per_ind, size=N) * (rng.random(N) > p_empty)
    ind = np.repeat(np.arange(N), counts)
    r = len(ind)
    return CohortArrays(
        vacs=rng.random((N, G)) < 0.05, pcrpos=rng.random((N, G)) < 0.03, ind=ind[rng.permutation(r)],
        gap=rng.integers(0, G, size=r), antigen=rng.integers(0, 2, size=r),
        x=rng.integers(0, 8, size=r).astype(float), od=rng.normal(0.8, 0.5, size=r),
    )


def _start(rng, G, N, C):
    q = ora.forward(dict(zip([n for n, _ in ora.VALUE_VARS], X0)))[None, :] + rng.uniform(-0.3, 0.3, size=(C, 17))
    q[:, 0] = np.log(1.0 / G) - np.log1p(-1.0 / G) + rng.uniform(-0.3, 0.3, size=C)
    i_raw = (rng.random((C, G, N)) < 0.03).astype(np.int8)
    w = (rng.random((C, N)) < 0.5).astype(np.int8)
    return q, i_raw, w


@pytest.mark.gpu
@pytest.mark.parametrize("name,C", [("test_cohort", 3), ("test_cohort", 5), ("synthetic_1000", 5), ("synthetic_60000", 3),
                                    ("random_96_gaps", 5)])
def test_fused_nuts_leaf_equals_the_standalone_leaf(gpu, name, C):
    """abd_nuts_extend_dev runs each leaf's leapfrog step and its tree bookkeeping in ONE k_sums launch (the finishing
    warp of the chain calls nuts_leaf_chain).  The same iterations as one single-step abd_leapfrog_dev launch plus one
    k_nuts_leaf launch per leaf must leave the whole tree state, q / grad / logp, the statistics, the step size and the
    dual-averaging state identical bit for bit: on the bundled cohort, 1000 and 60 000 individuals (a grid of several
    waves), and a 96-gap cohort (128-bit gap masks)."""
    import torch

    from abdpymc_b200.cohort import CohortArrays, synthetic_cohort

    rng = np.random.default_rng(len(name) + C)
    if name == "test_cohort":
        co, splits = CohortArrays.load("test_cohort"), (14, 20)
    elif name.startswith("synthetic"):
        co, splits = synthetic_cohort(int(name.split("_")[1])), (14, 20)
    else:
        co, splits = random_cohort(rng, 96, 300), (30, 70)
    D = 6
    q, i_raw, w = _start(rng, co.n_gaps, co.n_inds, C)
    inv_mass, linv_t = metric(rng)
    inv_mass, linv_t = 0.01 * inv_mass, 10.0 * linv_t
    f64 = dict(dtype=torch.float64, device=gpu)
    with _engine(co, splits) as eng:
        eng.upload_state(i_raw, w)
        d_i, d_w = eng.state_dev(C)
        d_q = _dev(q, gpu)
        d_lp, d_g = torch.empty(C, **f64), torch.empty(C, 17, **f64)
        eng.logp_dlogp_dev(C, d_q.data_ptr(), d_i, d_w, d_lp.data_ptr(), d_g.data_ptr())
        eps = _dev(rng.uniform(0.05, 0.15, C) * np.sqrt(10 / co.n_inds), gpu)   # the posterior narrows as 1 / sqrt(N)
        da = torch.zeros(C, 4, **f64)
        da[:, 0] = torch.log(10 * eps)
        d_im, d_lt = _dev(inv_mass, gpu), _dev(linv_t, gpu)
        depths = []
        for k in range(3):
            out = []
            for fused in (True, False):
                st = [t.clone() for t in (d_q, d_g, d_lp, eps, da)]
                qq, gg, ll, ee, dd = st
                state = torch.zeros(C, eng.nuts_state_doubles(D), **f64)
                qw, pw, gw = torch.empty(C, 17, **f64), torch.empty(C, 17, **f64), torch.empty(C, 17, **f64)
                lpw, es, acc, dep, div = (torch.empty(C, **f64) for _ in range(5))
                act = torch.zeros(D + 1, dtype=torch.int32, device=gpu)
                ptr = lambda t: t.data_ptr()  # noqa: E731
                eng.nuts_begin_dev(C, D, ptr(qq), ptr(gg), ptr(ll), ptr(d_lt), ptr(ee), SEED, IT + k, ptr(state), ptr(qw),
                                   ptr(pw), ptr(gw), ptr(es), ptr(act))
                for j in range(D):
                    if fused:
                        eng.nuts_extend_dev(C, D, j, ptr(qw), ptr(pw), ptr(gw), ptr(lpw), ptr(d_im), ptr(ee), SEED, IT + k,
                                            ptr(state), ptr(es), ptr(act), d_i, d_w)
                    else:
                        for n in range(1 << j):
                            eng.leapfrog_dev(C, 1, ptr(qw), ptr(pw), ptr(gw), ptr(lpw), ptr(es), ptr(d_im), d_i, d_w)
                            eng.nuts_leaf_dev(C, D, j, n, ptr(qw), ptr(pw), ptr(gw), ptr(lpw), ptr(d_im), ptr(ee), SEED,
                                              IT + k, ptr(state), ptr(es), ptr(act))
                eng.nuts_end_dev(C, D, ptr(qq), ptr(gg), ptr(ll), ptr(state), ptr(acc), ptr(dep), ptr(div), ptr(dd), ptr(ee),
                                 1, 0.8)
                torch.cuda.synchronize()
                eng.leapfrog_status(C)
                out.append([t.cpu().numpy() for t in (state, qq, gg, ll, ee, dd, acc, dep, div, es, act, qw, pw, gw, lpw)])
            for a, b in zip(*out):
                assert np.array_equal(a, b, equal_nan=True), k
            depths.extend(out[0][7].tolist())
            d_q, d_g, d_lp, eps, da = (_dev(a, gpu) for a in out[0][1:6])
    assert max(depths) >= 2


@pytest.mark.gpu
def test_fused_nuts_on_the_posterior_matches_the_restatement(gpu):
    """The fused device tree on the bundled cohort's posterior against the restatement with leaves from
    Oracle.logp_dlogp: 8 chains, 4 iterations, each from the device's state after the previous one (so that rounding
    does not compound into different trajectories).  q within 1e-8, depth and divergence exact."""
    import torch

    from abdpymc_b200.cohort import CohortArrays

    tally = Tally("posterior")
    co, splits = CohortArrays.load("test_cohort"), (14, 20)
    C, D = 8, 8
    rng = np.random.default_rng(8)
    q, i_raw, w = _start(rng, co.n_gaps, co.n_inds, C)
    o = ora.Oracle(co, splits=splits, dense=False)
    inv_mass, linv_t = np.eye(17), np.eye(17)
    f64 = dict(dtype=torch.float64, device=gpu)
    with _engine(co, splits) as eng:
        eng.upload_state(i_raw, w)
        d_i, d_w = eng.state_dev(C)
        d_q, d_lp, d_g = _dev(q, gpu), torch.empty(C, **f64), torch.empty(C, 17, **f64)
        eng.logp_dlogp_dev(C, d_q.data_ptr(), d_i, d_w, d_lp.data_ptr(), d_g.data_ptr())
        d_eps, d_im, d_lt = _dev(np.full(C, 0.08), gpu), _dev(inv_mass, gpu), _dev(linv_t, gpu)
        state = torch.zeros(C, eng.nuts_state_doubles(D), **f64)
        qw, pw, gw = torch.empty(C, 17, **f64), torch.empty(C, 17, **f64), torch.empty(C, 17, **f64)
        lpw, es, acc, dep, div = (torch.empty(C, **f64) for _ in range(5))
        act = torch.zeros(D + 1, dtype=torch.int32, device=gpu)
        depths = []
        for k in range(4):
            it = IT + k
            Q0, G0, LP0, EPS = (t.cpu().numpy() for t in (d_q, d_g, d_lp, d_eps))
            eng.nuts_begin_dev(C, D, d_q.data_ptr(), d_g.data_ptr(), d_lp.data_ptr(), d_lt.data_ptr(), d_eps.data_ptr(), SEED,
                               it, state.data_ptr(), qw.data_ptr(), pw.data_ptr(), gw.data_ptr(), es.data_ptr(), act.data_ptr())
            for j in range(D):
                eng.nuts_extend_dev(C, D, j, qw.data_ptr(), pw.data_ptr(), gw.data_ptr(), lpw.data_ptr(), d_im.data_ptr(),
                                    d_eps.data_ptr(), SEED, it, state.data_ptr(), es.data_ptr(), act.data_ptr(), d_i, d_w)
                if j + 1 < D and act[j + 1].item() == 0:
                    break
            eng.nuts_end_dev(C, D, d_q.data_ptr(), d_g.data_ptr(), d_lp.data_ptr(), state.data_ptr(), acc.data_ptr(),
                             dep.data_ptr(), div.data_ptr(), None, None, 0, 0.8)
            torch.cuda.synchronize()
            Q, DEP, DIV, ACC = (t.cpu().numpy() for t in (d_q, dep, div, acc))
            for c in range(C):
                def lf(x, p, g, e, c=c):
                    ph = p + 0.5 * e * g
                    xn = x + e * (inv_mass @ ph)
                    lp, gn = o.logp_dlogp(xn, i_raw[c], w[c])
                    return xn, ph + 0.5 * e * gn, gn, lp

                z, p0, zz = tr.momentum(SEED, it, c, linv_t)
                t = tr.nuts_tree(Q0[c], G0[c], LP0[c], p0, -LP0[c] + 0.5 * zz, EPS[c], inv_mass, SEED, it, c, D, lf)
                depths.append(t.depth)
                if not tally.ok(t.decisions, (k, c)):
                    continue
                assert np.all(np.abs(Q[c] - t.q) <= 1e-8 * np.maximum(1.0, np.abs(t.q))), (k, c, Q[c] - t.q)
                assert DEP[c] == t.depth and bool(DIV[c]) == t.diverged, (k, c, DEP[c], t.depth)
                assert abs(ACC[c] - t.accept) <= 1e-8, (k, c)
    assert max(depths) >= 3
    tally.report()


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", ["hmc", "nuts"])
def test_sampler_iteration_matches_the_restatement(gpu, kernel):
    """One iteration as ``sample`` composes it -- _DeviceLoop.transition(it), target.gibbs(q, it), refresh -- against
    the restated iteration: the trajectory length from np.random.default_rng(cfg.seed), the transition with the
    target's seed and the iteration index, the Gibbs sweep (oracle.device_gibbs_sweep) with the same seed and
    sweep = it.  Each iteration starts from the device's state: q within 1e-9, the binaries bit for bit, the
    acceptance statistic within 1e-8 and the adapted step size (from the device's statistic) within 1e-12."""
    import torch

    from abdpymc_b200.cohort import CohortArrays
    from abdpymc_b200.sampler import AbdTarget, SamplerConfig, _DeviceLoop

    tally = Tally(f"sampler {kernel}")
    co, splits = CohortArrays.load("test_cohort"), (14, 20)
    C, tseed = 5, 0x0123_4567_89AB_CDEF
    rng = np.random.default_rng(9)
    q, i_raw, w = _start(rng, co.n_gaps, co.n_inds, C)
    o = ora.Oracle(co, splits=splits, dense=False)
    cfg = SamplerConfig(tune=100, draws=10, seed=21, kernel=kernel, max_treedepth=6)
    L_rng = np.random.default_rng(cfg.seed)
    with _engine(co, splits) as eng:
        tgt = AbdTarget(eng, C, i_raw, w, seed=tseed, gibbs_mode=0, transit_p=0.8)
        run = _DeviceLoop(tgt, torch.from_numpy(q).to(gpu), cfg)
        im = run.inv_mass.cpu().numpy()
        lt = run.linv_t.cpu().numpy()
        for it in range(4):
            torch.cuda.synchronize()
            Q0, G0, LP0 = run.q.cpu().numpy(), run.grad.cpu().numpy(), run.logp.cpu().numpy()
            EPS0, DA0 = run.eps.cpu().numpy(), run.da.cpu().numpy()
            I0, W0 = tgt.state()
            L = max(1, int(round(cfg.n_leapfrog * (cfg.jitter[0] + (cfg.jitter[1] - cfg.jitter[0]) * L_rng.random()))))
            run.transition(it)
            torch.cuda.synchronize()
            Q1, ACC, EPS1, DA1 = run.q.cpu().numpy(), run.acc.cpu().numpy(), run.eps.cpu().numpy(), run.da.cpu().numpy()
            for c in range(C):
                def lf(x, p, g, e, c=c):
                    ph = p + 0.5 * e * g
                    xn = x + e * (im @ ph)
                    lp, gn = o.logp_dlogp(xn, I0[c], W0[c])
                    return xn, ph + 0.5 * e * gn, gn, lp

                z, p0, zz = tr.momentum(tseed, it, c, lt)
                h0 = -LP0[c] + 0.5 * zz
                if kernel == "hmc":
                    x, p, g, lp = Q0[c], p0, G0[c], LP0[c]
                    for _ in range(L):
                        x, p, g, lp = lf(x, p, g, EPS0[c])
                    take, a, dec = tr.hmc_end(h0, lp, p, im, tseed, it, c)
                    want, decisions = (x if take else Q0[c]), [dec]
                else:
                    t = tr.nuts_tree(Q0[c], G0[c], LP0[c], p0, h0, EPS0[c], im, tseed, it, c, run.TD, lf)
                    want, a, decisions = t.q, t.accept, t.decisions
                da, e = tr.dual_averaging(DA0[c], ACC[c], cfg.target_accept)
                np.testing.assert_allclose(DA1[c], da, rtol=1e-12, atol=1e-15)
                assert abs(EPS1[c] - e) <= 1e-12 * e
                if not tally.ok(decisions, (it, c)):
                    continue
                assert np.all(np.abs(Q1[c] - want) <= 1e-9 * np.maximum(1.0, np.abs(want))), (it, c)
                assert abs(ACC[c] - a) <= 1e-8, (it, c, ACC[c], a)
                if kernel == "nuts":
                    assert run.depth[c].item() == t.depth and bool(run.div[c].item()) == t.diverged, (it, c)
            tgt.gibbs(run.q, it)
            run.refresh()
            I1, W1 = tgt.state()
            LP1 = run.logp.cpu().numpy()
            for c in range(C):
                vals = ora.backward(Q1[c])[0]
                th = np.array([vals[n] for n in ora.THETA13])
                ri, rw, _ = ora.device_gibbs_sweep(co, splits, False, th, vals["p"], vals["ab_s_p_waner"], I0[c], W0[c],
                                                   tseed, it, c, mode=0, transit_p=0.8)
                assert np.array_equal(I1[c], ri) and np.array_equal(W1[c], rw), (it, c)
                rl, _ = o.logp_dlogp(Q1[c], ri, rw)
                assert abs(LP1[c] - rl) <= 1e-10 * abs(rl)
    tally.report()
