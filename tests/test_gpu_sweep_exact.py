"""Every sweep of the value, distortion, theta, block-id and summary kernels against the literal conditionals of
tests/sweep_exact.py, which share nothing with the kernels but the Philox stream and the orders that decide which value
a uniform picks.  Each case first asserts the path it is named after (the k_values variant by its dispatch rule,
similarity-row lengths, cluster sizes, theta); where the oracle is cheap the state is also compared with it bit for
bit."""
import numpy as np
import pytest

from helpers import agreeing_cluster, oracle_setup, product_setup, random_state, synth_problem
from link_exact import snapshot, tables_of
import sweep_exact as S
from test_gpu_parity import assert_same_state

pytestmark = pytest.mark.gpu

SAMPLERS = ["PCG-I", "PCG-II", "Gibbs", "Gibbs-Sequential"]


def _values_threshold():
    """k_values<8> runs while E * A <= sm_count * 8192 (value_update's dispatch), k_values<2> beyond"""
    import torch

    return torch.cuda.get_device_properties(0).multi_processor_count * 8192


def _sweep(label, eng, tables, x, file, sampler, tree, st=None, oracle=None, entities=None):
    """one sweep, all five checks, and (st not None) the oracle's sweep compared bit for bit -> check results"""
    before = snapshot(eng)
    eng.sweep(sampler, 1)
    after = snapshot(eng)
    out = S.check_sweep(before, after, eng.summary(), tables, x, file, eng.seed, sampler, eng.alpha, eng.beta, tree,
                        entities)
    S.assert_sweep_ok(out, f"{label} {sampler}")
    if st is not None:
        assert st.sweep(oracle.SAMPLERS[sampler]) == 0
        assert_same_state(eng, st)
    return out


@pytest.mark.parametrize("sampler", SAMPLERS)
def test_chain_small_values_kernel(oracle, sampler):
    """the default model with two files, missing values and four blocks: three sweeps from the initial state, one
    from a random valid state (Gibbs: values forced by z = 0 records)"""
    g = synth_problem(seed=41, R=1200, n_files=2, missing=0.05)
    eng, rc, x, file = product_setup(g, 99, 2, (2, 3))
    m, st, tree, ox, ofile = oracle_setup(oracle, g, 99, 2, (2, 3))
    np.testing.assert_array_equal(x, ox)
    assert eng.num_entities * eng.A <= _values_threshold()
    tables = tables_of(rc.indexes)
    ptree = eng.partitioner.export()
    for _ in range(3):
        _sweep("default k_values<8>", eng, tables, x, file, sampler, ptree, st, oracle)
    rng = np.random.default_rng(7)
    y, link, z = random_state(rng, x, 900, [ix.num_values for ix in rc.indexes])
    theta = rng.uniform(0.005, 0.3, (eng.A, 2))
    eng.upload_state(x, file, z, link, y, theta, iteration=20)
    st = oracle.State.from_arrays(m, x, file, z, link, y, theta, 20)
    out = _sweep("random state k_values<8>", eng, tables, x, file, sampler, ptree, st, oracle)
    assert out["values"]["checked"] == 900 * eng.A


@pytest.mark.parametrize("sampler", ["PCG-II", "Gibbs"])
def test_large_values_kernel(sampler):
    """320 000 records on as many entities: E * A above the threshold, so k_values<2> runs; every flag, theta, block
    id and the summary are checked, the values of 6 000 entities (all the multi-record ones among them)"""
    g = synth_problem(seed=3, R=320000, n_files=2)
    eng, rc, x, file = product_setup(g, 5, 3, (2, 3))
    assert eng.num_entities * eng.A > _values_threshold()
    tables = tables_of(rc.indexes)
    ptree = eng.partitioner.export()
    eng.sweep(sampler, 2)
    rng = np.random.default_rng(1)
    for _ in range(2):
        link = eng.links()[0]
        cnt = np.bincount(link, minlength=eng.num_entities)
        ents = np.union1d(rng.choice(eng.num_entities, 4000, replace=False), np.flatnonzero(cnt > 1)[:2000])
        out = _sweep("k_values<2>", eng, tables, x, file, sampler, ptree, entities=ents)
        assert out["dist"]["checked"] == x.size


def _clique_index(D, O, sizes, kmax, rng):
    """a string-like attribute whose similarity rows have exactly the given lengths: cliques of those sizes (each
    value similar to every value of its clique, itself included), E in (e^0.5, e^10]"""
    V = int(sum(sizes))
    rows, cols, vals = [], [], []
    start = 0
    for s in sizes:
        ids = np.arange(start, start + s)
        e = np.exp(rng.uniform(0.5, 10.0, (s, s)))
        e = np.triu(e) + np.triu(e, 1).T
        np.fill_diagonal(e, np.exp(10.0))
        rows.append(np.repeat(ids, s))
        cols.append(np.tile(ids, s))
        vals.append(e.ravel())
        start += s
    rows, cols, vals = np.concatenate(rows), np.concatenate(cols), np.concatenate(vals)
    rowptr = np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=V))]).astype(np.int32)
    probs = rng.uniform(0.2, 1.0, V)
    probs /= probs.sum()
    prod = D.AttributeIndex.from_tables(probs, rowptr, cols.astype(np.int32), vals, constant=False,
                                        expected_max_cluster_size=kmax)
    orc = O.Index.from_tables(probs, rowptr, cols, vals, False, kmax)
    return prod, orc


@pytest.mark.parametrize("sampler", SAMPLERS)
@pytest.mark.parametrize("per_entity", [1, 8])
def test_similarity_row_lengths(oracle, sampler, per_entity):
    """rows of 1, 7, 8, 9, 16, 17 and 260 values (the UB-batched single-record loop ends at every remainder; 260 is
    past the PCG-II row limit), a constant attribute, kmax = 2.  per_entity = 1: single linked records, isolated
    entities and entities whose records are all missing; 8: the multi-record path with agreeing duplicates (the
    `repeated` skip and the x_j == x_r shortcut), overlapping rows of different values and k > kmax"""
    import dblink_b200 as D

    rng = np.random.default_rng(11 + per_entity)
    sizes = [1, 7, 8, 9, 16, 17, 260]
    sp, so = _clique_index(D, oracle, sizes, 2, rng)
    cp = D.AttributeIndex.from_tables(np.full(6, 1 / 6), constant=True, expected_max_cluster_size=2)
    co = oracle.Index.from_tables(np.full(6, 1 / 6), [0] * 7, [], [], True, 2)
    lens = np.diff(sp.tables()["rowptr"])
    assert set(lens.tolist()) == set(sizes)
    R, F = 1600, 2
    E = R // per_entity
    x = np.stack([rng.integers(0, 6, R), rng.integers(0, int(sum(sizes)), R)], axis=1).astype(np.int32)
    x[rng.random((R, 2)) < 0.05] = -1
    file = (np.arange(R) % F).astype(np.int32)
    y, link, z = random_state(rng, x, E, [6, int(sum(sizes))])
    if per_entity == 1:  # entities E-50.. hold only records whose string value is missing
        miss = x[:, 1] < 0
        link[miss] = rng.integers(E - 50, E, miss.sum())
        link[~miss & (link >= E - 50)] = rng.integers(0, E - 50, (~miss & (link >= E - 50)).sum())
        z |= ((x >= 0) & (x != y[link])).astype(np.uint8)
    theta = rng.uniform(0.01, 0.3, (2, F))
    eng = D.GibbsEngine([cp, sp], [1.0, 1.0], [50.0, 50.0], None, 3, F)
    eng.upload_state(x, file, z, link, y, theta, iteration=0)
    m = oracle.Model([co, so], [1.0, 1.0], [50.0, 50.0], None, 3, F)
    st = oracle.State.from_arrays(m, x, file, z, link, y, theta, 0)
    cnt = np.bincount(link, minlength=E)
    assert (cnt > 2).any() if per_entity == 8 else ((cnt == 1).sum() > E // 4 and (cnt == 0).any())
    tables = tables_of([cp, sp])
    for _ in range(2):
        _sweep(f"rows {sizes} x{per_entity}", eng, tables, x, file, sampler, None, st, oracle)


@pytest.mark.parametrize("sampler", SAMPLERS)
@pytest.mark.parametrize("level", ["low", "high"])
def test_theta_at_the_extremes(oracle, sampler, level):
    """priors that put theta below 1e-4 (no flags, alpha = 0.05, beta = 2000) or near 0.9 (every flag set,
    alpha = 9000, beta = 1000): the collapsed factor (1/theta - 1) at both ends.  Every record on an entity of its
    own values, so that no flag is forced"""
    import dblink_b200 as D

    g = synth_problem(seed=21, R=800, n_files=2, missing=0.05)
    rc = D.RecordsCache.build(g["values"], g["files"], g["attributes"], 10)
    x, file = rc.transform_records(g["values"], g["files"])
    alpha, beta = ([0.05] * 4, [2000.0] * 4) if level == "low" else ([9000.0] * 4, [1000.0] * 4)
    eng = D.GibbsEngine(rc.indexes, alpha, beta, None, 8, 2)
    y, link = np.where(x >= 0, x, 0).astype(np.int32), np.arange(len(x), dtype=np.int32)
    z = np.full(x.shape, 0 if level == "low" else 1, np.uint8)
    eng.upload_state(x, file, z, link, y, np.full((4, 2), 0.5), iteration=0)
    out = _sweep(f"theta {level}", eng, tables_of(rc.indexes), x, file, sampler, None)
    th = snapshot(eng)["theta"]
    assert (th < 1e-2).all() if level == "low" else ((th > 0.85) & (th < 0.95)).all()
    assert out["values"]["checked"] == len(x) * 4


@pytest.mark.parametrize("sampler", SAMPLERS)
@pytest.mark.parametrize("theta", [0.05, 0.3])
@pytest.mark.parametrize("K", [40, 55, 64, 120])
def test_large_cluster(oracle, sampler, theta, K):
    """a cluster of K records agreeing on every attribute (distorted in s0 for the non-collapsed samplers): from
    K = 55 (theta = 0.05) or 64 (theta = 0.3) the binary64 product of the similarity factors overflows and the kernel
    redoes the draw in the log domain; at K = 120 n(v)^K underflows as well"""
    g = synth_problem()
    eng, rc, x0, file = product_setup(g, 1)
    m, st0, tree, ox, ofile = oracle_setup(oracle, g, 1)
    x = ox.copy()
    x[0] = [5, 17, 7, x[0, 3] if x[0, 3] >= 0 else 0]
    distorted = (2,) if sampler in ("Gibbs", "Gibbs-Sequential") else ()
    rate = max(0.0, (theta * (len(x) + 1010) - 10 - K * len(distorted)) / len(x))
    x, y, link, z = agreeing_cluster(np.random.default_rng(K), x, st0.y, st0.link, st0.z, K, distorted, rate)
    th = np.full((4, 1), theta)
    eng.upload_state(x, file, z, link, y, th, iteration=0)
    st = oracle.State.from_arrays(m, x, file, z, link, y, th, 0)
    out = _sweep(f"cluster K={K} theta={theta}", eng, tables_of(rc.indexes), x, file, sampler, None, st, oracle)
    after = snapshot(eng)
    assert theta / 2 < after["theta"][2, 0] < 2 * theta
    assert (after["link"][:K] == 0).sum() >= 0.8 * K
    if K == 120:
        assert out["values"]["overflow"] >= 1 and after["y"][0, 2] == 7


@pytest.mark.parametrize("sampler", ["PCG-II", "Gibbs"])
def test_two_ranks(oracle, sampler):
    """two contexts of one device (LocalShards): the summary reduced across the ranks"""
    import dblink_b200 as D
    from dblink_b200.distributed import LocalShards

    g = synth_problem(seed=5, R=1500, n_files=2)
    rc = D.RecordsCache.build(g["values"], g["files"], g["attributes"])
    x, file = rc.transform_records(g["values"], g["files"])
    alpha, beta = [a.alpha for a in g["attributes"]], [a.beta for a in g["attributes"]]
    sh = LocalShards(rc.indexes, alpha, beta, seed=99, num_files=2, levels=3, split_attrs=(2, 3), world=2)
    sh.init_state(x, file)
    m, st, tree, ox, ofile = oracle_setup(oracle, g, 99, 3, (2, 3))
    tables = tables_of(rc.indexes)
    try:
        for _ in range(3):
            before = snapshot(sh)
            sh.sweep(sampler, 1)
            after = snapshot(sh)
            out = S.check_sweep(before, after, sh.summary(), tables, x, file, 99, sampler, alpha, beta, tree)
            S.assert_sweep_ok(out, f"two ranks {sampler}")
            assert st.sweep(oracle.SAMPLERS[sampler]) == 0
            for k in ("theta", "link", "y", "z", "block"):
                np.testing.assert_array_equal(after[k], getattr(st, k), err_msg=k)
    finally:
        sh.close()


def test_device_theta_follows_the_beta_conditional():
    """PIT of the device's theta draws under scipy's Beta CDF, pooled over 4 attributes x 3 files and 60 uploads at
    different iterations; shapes from 0.3 (the U^(1/a) boost) to 40 000"""
    from scipy import stats

    import dblink_b200 as D

    g = synth_problem(seed=2, R=90000, n_files=3, dup=0.0)
    rc = D.RecordsCache.build(g["values"], g["files"], g["attributes"], 10)
    x, file = rc.transform_records(g["values"], g["files"])
    alpha, beta = np.array([0.3, 2.0, 10.0, 0.7]), np.array([0.5, 30.0, 1000.0, 5.0])
    eng = D.GibbsEngine(rc.indexes, alpha, beta, None, 77, 3)
    y, link = np.where(x >= 0, x, 0).astype(np.int32), np.arange(len(x), dtype=np.int32)
    rng = np.random.default_rng(3)
    pits, shapes = [], []
    for i in range(60):
        z = (rng.random(x.shape) < [0.0, 0.5, 0.001, 1.0][i % 4]).astype(np.uint8)  # any flags: every x = y
        eng.upload_state(x, file, z, link, y, np.full((4, 3), 0.1), iteration=1000 + 37 * i)
        before = snapshot(eng)
        eng.sweep("PCG-II", 1)
        after = snapshot(eng)
        ok, expect = S.check_theta(before, after, file, 77, alpha, beta)
        assert ok
        agg, fs = S.literal_counts(z, file, 3)
        s1, s2 = agg + alpha[:, None], fs[None, :] - agg + beta[:, None]
        shapes += [s1.min(), s2.min(), s1.max(), s2.max()]
        pits.append(stats.beta.cdf(after["theta"], s1, s2).ravel())
    assert min(shapes) < 1 and max(shapes) > 20000
    pit = np.concatenate(pits)
    p = stats.kstest(pit, "uniform").pvalue
    print(f"theta PIT: {len(pit)} draws, KS p = {p:.3g}")
    assert p > 1e-3
