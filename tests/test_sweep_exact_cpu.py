"""The extended-precision check of theta, values, flags, block ids and summary (tests/sweep_exact.py) on the CPU
oracle: it accepts every sweep of the oracle's chains for all four samplers, it rejects states drawn with a wrong
conditional or the wrong uniforms, and it catches the value draw of a cluster whose binary64 weights overflow."""
import numpy as np
import pytest
from scipy import stats

from helpers import agreeing_cluster, oracle_setup, random_state, synth_problem
from link_exact import snapshot, tables_of
import sweep_exact as S

SAMPLERS = ["PCG-I", "PCG-II", "Gibbs", "Gibbs-Sequential"]


def test_numpy_philox_matches_the_oracle_stream(oracle):
    rng = np.random.default_rng(1)
    ids, subs = rng.integers(0, 2 ** 32, 64), rng.integers(0, 2 ** 32, 64)
    for seed, ph, it in [(0, 3, 1), (0xC0FFEE123456789A, 4, 77), (31, 1, 0xFFFFFFFF)]:
        u0, u1 = S.uniform2(seed, ph, it, ids, subs)
        for i in range(64):
            assert (u0[i], u1[i]) == oracle.uniform2(seed, ph, it, int(ids[i]), int(subs[i]))


def _check_chain(O, m, st, tables, x, file, seed, sampler, tree, n):
    for _ in range(n):
        before = snapshot(st)
        assert st.sweep(O.SAMPLERS[sampler]) == 0
        out = S.check_sweep(before, snapshot(st), st.summary(), tables, x, file, seed, sampler, m.alpha, m.beta, tree)
        S.assert_sweep_ok(out, f"oracle {sampler}")
        assert out["values"]["checked"] == st.E * m.A


@pytest.mark.parametrize("sampler", SAMPLERS)
def test_checker_accepts_oracle_chains(oracle, sampler):
    """three files, missing values, four k-d blocks; from the initial state and from a random valid state"""
    g = synth_problem(seed=13, R=900, n_files=3, missing=0.08, distortion=0.15)
    m, st, tree, x, file = oracle_setup(oracle, g, 31, 2, (2, 3))
    tables = tables_of(m.indexes)
    _check_chain(oracle, m, st, tables, x, file, 31, sampler, tree, 3)
    rng = np.random.default_rng(5)
    y, link, z = random_state(rng, x, 700, [ix.V for ix in m.indexes])
    st = oracle.State.from_arrays(m, x, file, z, link, y, rng.uniform(0.005, 0.3, (len(m.indexes), 3)), 17)
    _check_chain(oracle, m, st, tables, x, file, 31, sampler, tree, 2)


@pytest.mark.parametrize("sampler", ["PCG-II", "Gibbs"])
def test_checker_accepts_clusters_beyond_the_cached_powers(oracle, sampler):
    """kmax = 2: clusters of up to 25 records take the uncached base distribution"""
    g = synth_problem(seed=31, R=300, dup=0.0)
    m, st, tree, x, file = oracle_setup(oracle, g, 17, 0, (), kmax=2)
    rng = np.random.default_rng(5)
    y, link, z = random_state(rng, x, 12, [ix.V for ix in m.indexes])
    st = oracle.State.from_arrays(m, x, file, z, link, y, np.full((len(m.indexes), 1), 0.05), 0)
    _check_chain(oracle, m, st, tables_of(m.indexes), x, file, 17, sampler, tree, 2)


@pytest.fixture(scope="module")
def chain(oracle):
    """one PCG-II and one Gibbs sweep of the oracle from a random valid state with three files and distinct theta"""
    g = synth_problem(seed=13, R=900, n_files=3, missing=0.08, distortion=0.15)
    m, st0, tree, x, file = oracle_setup(oracle, g, 31, 2, (2, 3))
    rng = np.random.default_rng(12)
    y, link, z = random_state(rng, x, 700, [ix.V for ix in m.indexes])
    theta = rng.uniform(0.005, 0.3, (len(m.indexes), 3))
    out = {"m": m, "x": x, "file": file, "tree": tree, "tables": tables_of(m.indexes)}
    for sampler in ("PCG-II", "Gibbs"):
        st = oracle.State.from_arrays(m, x, file, z, link, y, theta, 40)
        before = snapshot(st)
        assert st.sweep(oracle.SAMPLERS[sampler]) == 0
        out[sampler] = (before, snapshot(st), st.summary())
    return out


def _values(c, sampler, after, **kw):
    before = c[sampler][0]
    return S.check_values(before, after, c["tables"], c["x"], c["file"], 31, sampler, verbose=0, **kw)


def test_negative_control_value_moved_to_another_id(chain):
    before, after, _ = chain["PCG-II"]
    ok = _values(chain, "PCG-II", after)
    assert ok["mismatches"] == 0
    band = set(ok["band_cells"])
    bad = dict(after, y=after["y"].copy())
    cells = [(e, a) for e in range(0, len(bad["y"]), 37) for a in range(bad["y"].shape[1]) if (e, a) not in band][:20]
    for e, a in cells:
        bad["y"][e, a] = (bad["y"][e, a] + 1) % chain["tables"][a]["phi"].size
    out = _values(chain, "PCG-II", bad)
    assert out["mismatches"] >= 15 and set(out["bad"]) <= set(cells)


def test_negative_control_theta_of_two_files_swapped(chain):
    before, after, _ = chain["PCG-II"]
    out = _values(chain, "PCG-II", dict(after, theta=after["theta"][:, [1, 0, 2]]))
    assert out["mismatches"] >= 5


@pytest.mark.parametrize("variant,sampler", [("drop_theta_term", "PCG-II"), ("ignore_forced", "Gibbs")])
def test_negative_control_wrong_value_conditional(chain, variant, sampler):
    """values drawn without the (1/theta - 1) term of GU:557/560, or ignoring the value a z = 0 record forces"""
    before, after, _ = chain[sampler]
    wrong = S.exact_values(before, after, chain["tables"], chain["x"], chain["file"], 31, sampler, variant=variant)
    assert (wrong != after["y"]).sum() >= 5
    out = _values(chain, sampler, dict(after, y=wrong))
    assert out["mismatches"] >= 5


def test_exact_values_agree_with_the_oracle(chain):
    for sampler in ("PCG-II", "Gibbs"):
        before, after, _ = chain[sampler]
        band = set(_values(chain, sampler, after)["band_cells"])
        y = S.exact_values(before, after, chain["tables"], chain["x"], chain["file"], 31, sampler)
        diff = {tuple(map(int, c)) for c in np.argwhere(y != after["y"])}
        assert diff <= band


def test_negative_control_value_uniform_of_the_next_iteration(chain):
    before, after, _ = chain["PCG-II"]
    out = S.check_values(dict(before, iteration=before["iteration"] + 1), after, chain["tables"], chain["x"],
                         chain["file"], 31, "PCG-II", verbose=0)
    assert out["mismatches"] >= 50


def test_negative_control_flags_without_the_diagonal_similarity(chain):
    """flags drawn with P(z = 1 | x = y) missing its factor E(x, x)"""
    c = chain
    for sampler in ("PCG-II", "Gibbs"):
        before, after, _ = c[sampler]
        assert S.check_dist(before, after, c["tables"], c["x"], c["file"], 31)["mismatches"] == 0
        wrong = S.exact_dist(before, after, c["tables"], c["x"], c["file"], 31, with_diag=False)
        assert (wrong != after["z"]).sum() >= 20
        out = S.check_dist(before, dict(after, z=wrong), c["tables"], c["x"], c["file"], 31, verbose=0)
        assert out["mismatches"] >= 20


def test_negative_control_theta_of_wrong_counts(chain):
    c = chain
    before, after, _ = c["PCG-II"]
    assert S.check_theta(before, after, c["file"], 31, c["m"].alpha, c["m"].beta)[0]
    z = before["z"].copy()
    z[np.flatnonzero(c["file"] == 1)[0], 2] ^= 1
    assert not S.check_theta(dict(before, z=z), after, c["file"], 31, c["m"].alpha, c["m"].beta)[0]


def test_negative_control_summary_with_one_flag_flipped(chain):
    c = chain
    before, after, summ = c["PCG-II"]
    assert S.check_summary(summ, after, c["tables"], c["x"], c["file"], c["m"].alpha, c["m"].beta) == []
    agg = summ["agg_dist"].copy()
    agg[1, 2] += 1
    bad = S.check_summary(dict(summ, agg_dist=agg), after, c["tables"], c["x"], c["file"], c["m"].alpha, c["m"].beta)
    assert bad == ["agg_dist"]
    ll = S.check_summary(dict(summ, log_likelihood=summ["log_likelihood"] * (1 + 1e-9)), after, c["tables"], c["x"],
                         c["file"], c["m"].alpha, c["m"].beta)
    assert ll == ["log_likelihood"]


def test_negative_control_block_ids(chain):
    c = chain
    before, after, _ = c["PCG-II"]
    blk = S.leaf_ids(c["tree"], after["y"])
    assert np.array_equal(blk, after["block"]) and len(np.unique(blk)) == 4
    e = int(np.flatnonzero(blk == 0)[0])
    y = after["y"].copy()
    y[e] = after["y"][int(np.flatnonzero(blk == 3)[0])]
    assert S.leaf_ids(c["tree"], y)[e] == 3


def test_theta_draw_follows_the_beta_conditional():
    """PIT values of the protocol's theta draw (the host build of the device's draw) under scipy's Beta CDF, pooled
    over iterations and (attribute, file) pairs with shapes from 0.3 to 60 000"""
    alpha = np.array([0.3, 2.0, 10.0, 0.7])
    beta = np.array([0.5, 30.0, 1000.0, 5.0])
    fs = np.array([0, 7, 400, 60000])
    agg = np.array([[0, 0, 3, 100], [0, 7, 200, 30000], [0, 1, 0, 59990], [0, 3, 390, 12]])
    s1 = agg + alpha[:, None]
    s2 = fs[None, :] - agg + beta[:, None]
    assert s1.min() < 1 and s2.min() < 1 and max(s1.max(), s2.max()) > 20000
    pit = [stats.beta.cdf(S.draw_theta(alpha, beta, 0xBEEF, agg, fs, it), s1, s2) for it in range(1, 401)]
    pit = np.array(pit).reshape(400, -1)
    for j in range(pit.shape[1]):  # each pair alone, then all pooled
        assert stats.kstest(pit[:, j], "uniform").pvalue > 1e-4, j
    assert stats.kstest(pit.ravel(), "uniform").pvalue > 1e-3


def _cluster(oracle, K, theta, distorted=(), seed=1):
    """the default model (R = 600, alpha = 10, beta = 1000) with a cluster of K records agreeing on every attribute:
    value 7 of s0 (E(x,x) = e^10, phi = 0.26, n = 1.7e-4: at theta = 0.05 each record multiplies the weight of x by
    ~4e5), constants no other entity shares; the other flags set at a rate that draws theta within a factor 2 of
    `theta`"""
    g = synth_problem()
    m, st, tree, x, file = oracle_setup(oracle, g, seed)
    x = x.copy()
    x[0] = [5, 17, 7, x[0, 3] if x[0, 3] >= 0 else 0]
    rate = max(0.0, (theta * (len(x) + 1010) - 10 - K * len(distorted)) / len(x))
    x, y, link, z = agreeing_cluster(np.random.default_rng(seed), x, st.y, st.link, st.z, K, distorted, rate)
    assert (y[1:] == y[0]).all(axis=1).sum() == 0
    return m, oracle.State.from_arrays(m, x, file, z, link, y, np.full((m.A, 1), theta), 0), x, file, tree


@pytest.mark.parametrize("K", [55, 60])
def test_value_draw_of_a_cluster_whose_weights_overflow(oracle, K):
    """the product of the K factors of x passes DBL_MAX: every uniform must still draw x, whose conditional
    probability is 1 to double precision (without the log-domain redo the draw fell through to the last value of
    positive weight of the support, another value)"""
    m, st, x, file, _ = _cluster(oracle, K, 0.05)
    pmf = st.ref_value_pmf(0, 2, oracle.PCG_II)
    assert np.isfinite(pmf).all() and pmf[7] > 1 - 1e-12
    for s in ("PCG-I", "PCG-II"):
        for u0 in (0.1, 0.5, 0.9):
            for u1 in (0.1, 0.5, 0.9):
                assert st.value_draw(0, 2, oracle.SAMPLERS[s], u0, u1) == 7, (s, u0, u1)


@pytest.mark.parametrize("sampler", SAMPLERS)
@pytest.mark.parametrize("K,theta", [(40, 0.05), (64, 0.3), (120, 0.05)])
def test_sweep_of_a_large_cluster(oracle, sampler, K, theta):
    """a whole sweep with a cluster of K agreeing records (distorted in s0 for the non-collapsed samplers), checked
    value by value; at K = 120 the binary64 weights overflow (and n(v)^120 underflows) in every sampler"""
    distorted = (2,) if sampler in ("Gibbs", "Gibbs-Sequential") else ()
    m, st, x, file, tree = _cluster(oracle, K, theta, distorted)
    before = snapshot(st)
    assert st.sweep(oracle.SAMPLERS[sampler]) == 0
    after = snapshot(st)
    assert theta / 2 < after["theta"][2, 0] < 2 * theta
    out = S.check_sweep(before, after, st.summary(), tables_of(m.indexes), x, file, 1, sampler, m.alpha, m.beta,
                        tree)
    S.assert_sweep_ok(out, f"oracle cluster K={K} theta={theta} {sampler}")
    if K == 120:
        assert (after["link"][:K] == 0).sum() >= 100
        assert out["values"]["overflow"] >= 1 and after["y"][0, 2] == 7
