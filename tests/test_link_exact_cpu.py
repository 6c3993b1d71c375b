"""The extended-precision link-draw check (tests/link_exact.py) on the CPU oracle: it accepts every draw of the
oracle's chains for all four samplers, and it rejects a state whose links were drawn with a wrong record, wrong theta,
a wrong weight factor or the wrong uniform."""
import numpy as np
import pytest

from helpers import oracle_setup, random_state, synth_problem
from link_exact import check_link_draws, exact_draws, snapshot, tables_of

SAMPLERS = ["PCG-I", "PCG-II", "Gibbs", "Gibbs-Sequential"]


def _sweep_and_check(O, st, tables, x, file, seed, sampler, n=1):
    out = []
    for _ in range(n):
        before = snapshot(st)
        assert st.sweep(O.SAMPLERS[sampler]) == 0
        res = check_link_draws(before, snapshot(st), tables, x, file, seed, sampler)
        assert res["mismatches"] == 0, res["bad"][:10]
        assert res["checked"] == len(x)
        assert res["band"] <= 0.005 * res["checked"]
        out.append(res)
    return out


@pytest.mark.parametrize("sampler", SAMPLERS)
def test_checker_accepts_oracle_chains(oracle, sampler):
    """several files, missing values, four k-d blocks: from the initial state and from a random valid state"""
    g = synth_problem(seed=13, R=900, n_files=3, missing=0.08, distortion=0.15)
    m, st, tree, x, file = oracle_setup(oracle, g, 31, 2, (2, 3))
    assert tree.n_leaves == 4
    assert (x < 0).any(axis=0)[2:].all()  # missing string values
    tables = tables_of(m.indexes)
    _sweep_and_check(oracle, st, tables, x, file, 31, sampler, 3)
    rng = np.random.default_rng(5)
    y, link, z = random_state(rng, x, 700, [ix.V for ix in m.indexes])
    theta = rng.uniform(0.005, 0.3, (len(m.indexes), 3))
    st = oracle.State.from_arrays(m, x, file, z, link, y, theta, 17)
    assert len(np.unique(st.block)) == 4
    _sweep_and_check(oracle, st, tables, x, file, 31, sampler, 2)


@pytest.mark.parametrize("sampler", ["PCG-II", "PCG-I"])
def test_checker_accepts_a_block_beyond_32_tiles(oracle, sampler):
    """one block of 4 500 entities (36 tiles of 128: draw chunks of two tiles), records without a must-match
    attribute included"""
    g = synth_problem(seed=3, R=500, n_files=2, missing=0.05)
    m, st, tree, x, file = oracle_setup(oracle, g, 8, pop=4500)
    assert st.E == 4500 and tree.n_leaves == 1
    tables = tables_of(m.indexes)
    _sweep_and_check(oracle, st, tables, x, file, 8, sampler, 2)
    rng = np.random.default_rng(9)
    y, link, z = random_state(rng, x, 4500, [ix.V for ix in m.indexes])
    z[rng.choice(len(x), 40, replace=False)] = 1
    st = oracle.State.from_arrays(m, x, file, z, link, y, rng.uniform(0.01, 0.3, (len(m.indexes), 2)), 4)
    _sweep_and_check(oracle, st, tables, x, file, 8, sampler, 1)


@pytest.fixture(scope="module")
def pcg2_sweep(oracle):
    """one PCG-II sweep of the oracle from a random valid state with three files, distinct theta per file and
    missing string values; the check passes on it"""
    g = synth_problem(seed=13, R=900, n_files=3, missing=0.08, distortion=0.15)
    m, st0, tree, x, file = oracle_setup(oracle, g, 31, 2, (2, 3))
    rng = np.random.default_rng(12)
    y, link, z = random_state(rng, x, 700, [ix.V for ix in m.indexes])
    theta = rng.uniform(0.005, 0.3, (len(m.indexes), 3))
    st = oracle.State.from_arrays(m, x, file, z, link, y, theta, 40)
    before = snapshot(st)
    assert st.sweep(oracle.PCG_II) == 0
    after = snapshot(st)
    tables = tables_of(m.indexes)
    res = check_link_draws(before, after, tables, x, file, 31, "PCG-II")
    assert res["mismatches"] == 0
    return before, after, tables, x, file, res


def test_negative_control_link_moved_to_the_next_candidate(pcg2_sweep):
    before, after, tables, x, file, res = pcg2_sweep
    block = before["block"]
    band = set(res["band_records"])
    r = next(r for r in range(len(x)) if r not in band and (block == block[before["link"][r]]).sum() > 1)
    cand = np.flatnonzero(block == block[before["link"][r]])
    p = int(np.searchsorted(cand, after["link"][r]))
    bad = dict(after, link=after["link"].copy())
    bad["link"][r] = cand[p + 1] if p + 1 < len(cand) else cand[p - 1]
    out = check_link_draws(before, bad, tables, x, file, 31, "PCG-II")
    assert out["mismatches"] == 1 and out["bad"] == [r]


def test_negative_control_theta_of_two_files_swapped(pcg2_sweep):
    before, after, tables, x, file, res = pcg2_sweep
    bad = dict(after, theta=after["theta"][:, [1, 0, 2]])
    out = check_link_draws(before, bad, tables, x, file, 31, "PCG-II", verbose=0)
    assert out["mismatches"] >= 5
    assert set(out["bad"]) <= set(np.flatnonzero(file <= 1).tolist())  # file 2 keeps its theta


def test_negative_control_missing_attribute_factor_dropped(pcg2_sweep):
    """links drawn as a kernel would draw them that omitted the 1/n(y) factor of a missing non-constant attribute
    (k_link_pcg2 running the loop body without the missing-attribute gather for such a record)"""
    before, after, tables, x, file, res = pcg2_sweep
    miss = np.flatnonzero(np.array([(x[:, a] < 0) & (not t["is_const"]) for a, t in enumerate(tables)]).any(axis=0))
    assert len(miss) > 50
    wrong = exact_draws(before, after["theta"], tables, x, file, 31, "PCG-II", records=miss, missing_norm=False)
    bad = dict(after, link=after["link"].copy())
    for r, e in wrong.items():
        bad["link"][r] = e
    assert (bad["link"] != after["link"]).sum() >= 3
    out = check_link_draws(before, bad, tables, x, file, 31, "PCG-II", verbose=0)
    assert out["mismatches"] >= 3 and set(out["bad"]) <= set(miss.tolist())


def test_negative_control_uniform_of_the_next_iteration(pcg2_sweep):
    """the draws checked as if they had used the uniform of iteration + 2 instead of iteration + 1"""
    before, after, tables, x, file, res = pcg2_sweep
    out = check_link_draws(dict(before, iteration=before["iteration"] + 1), after, tables, x, file, 31, "PCG-II",
                           verbose=0)
    assert out["mismatches"] >= 50


def test_exact_draws_agree_with_the_oracle(pcg2_sweep):
    """outside the rounding band the extended-precision inverse CDF picks what the oracle picked"""
    before, after, tables, x, file, res = pcg2_sweep
    draws = exact_draws(before, after["theta"], tables, x, file, 31, "PCG-II")
    band = set(res["band_records"])
    assert all(after["link"][r] == e for r, e in draws.items() if r not in band)
