"""Every link-kernel family and dispatch path against an extended-precision inverse CDF of the literal link
conditional (tests/link_exact.py), which shares nothing with the kernels but the Philox stream and the candidate
order of the draw.  Each case first asserts that the model really takes the path it is named after (kernel name, hash
size, record classes counted on the host), so that a change of a dispatch threshold fails here instead of quietly
testing something else.  Where the oracle costs seconds, the state is also compared with it bit for bit."""
import numpy as np
import pytest

from helpers import oracle_setup, product_setup, random_state, synth_problem
from link_exact import check_link_draws, snapshot, tables_of
from test_gpu_parity import assert_same_state

pytestmark = pytest.mark.gpu


def _lowered(g, thresholds):
    """g with the Levenshtein thresholds of the named attributes replaced"""
    from dblink_b200.records import Attribute, SimilarityFn

    g = dict(g)
    g["attributes"] = [Attribute(a.name, SimilarityFn("LevenshteinSimilarityFn", thresholds[a.name], 10.0), a.alpha,
                                 a.beta) if a.name in thresholds else a for a in g["attributes"]]
    return g


def _check(case, eng, before, tables, x, file, sampler, records=None):
    res = check_link_draws(before, snapshot(eng), tables, x, file, eng.seed, sampler, records)
    print(f"link_exact {case} {sampler} {eng.link_kernel(sampler)}: {res['checked']} records checked, "
          f"{res['band']} in the rounding band, {res['mismatches']} mismatches")
    assert res["mismatches"] == 0, res["bad"][:10]
    assert res["checked"] == (len(x) if records is None else len(records))
    assert res["band"] <= 0.005 * res["checked"]
    return res


def _sweeps(case, oracle, eng, st, tables, x, file, sampler, n):
    """n single sweeps, each checked against the inverse CDF and (st not None) against the oracle"""
    for _ in range(n):
        before = snapshot(eng)
        eng.sweep(sampler, 1)
        _check(case, eng, before, tables, x, file, sampler)
        if st is not None:
            assert st.sweep(oracle.SAMPLERS[sampler]) == 0
            assert_same_state(eng, st)


def _chain_and_random_state(case, oracle, g, seed, sampler, expect, levels=0, attr_ids=(), pop=0, n=3, E=None):
    """n sweeps from the initial state, then one from a random valid state with several files and missing values"""
    eng, rc, x, file = product_setup(g, seed, levels, attr_ids, pop)
    m, st, tree, ox, ofile = oracle_setup(oracle, g, seed, levels, attr_ids, pop)
    np.testing.assert_array_equal(x, ox)
    assert eng.link_kernel(sampler) == expect
    tables = tables_of(rc.indexes)
    _sweeps(case, oracle, eng, st, tables, x, file, sampler, n)
    F = len(rc.file_ids)
    assert F >= 2 and (x < 0).any()
    rng = np.random.default_rng(seed)
    E = E or eng.num_entities
    y, link, z = random_state(rng, x, E, [ix.num_values for ix in rc.indexes])
    theta = rng.uniform(0.005, 0.3, (len(rc.indexes), F))
    eng.upload_state(x, file, z, link, y, theta, iteration=20)
    st = oracle.State.from_arrays(m, x, file, z, link, y, theta, 20)
    assert eng.link_kernel(sampler) == expect
    _sweeps(case, oracle, eng, st, tables, x, file, sampler, 1)
    return eng, rc, x, file


def test_pcg2_two_records_per_warp(oracle):
    """the default model: 32-slot tables, byte-packed constants, two records per warp -- the baseline of the check"""
    g = synth_problem(seed=41, R=1200, n_files=2, missing=0.05)
    _chain_and_random_state("pcg2-HC32-PK1", oracle, g, 99, "PCG-II", "k_link_pcg2<A=4,NS=2,HC=32,PK=1>", 2, (2, 3))


@pytest.mark.parametrize("V", [255, 256])
def test_pcg2_constant_packing_boundary(oracle, V):
    """a constant attribute with exactly 255 values used packs into a byte; with 256 it does not"""
    from dblink_b200 import synth

    attrs = [synth.SynthAttr("c0", "constant", V, 0.5), synth.SynthAttr("c1", "constant", 20, 0.5),
             synth.SynthAttr("s0", "levenshtein", 120, 1.0), synth.SynthAttr("s1", "levenshtein", 160, 1.0)]
    g = synth.generate(43, 1500, attrs, dup=0.3, distortion=0.1, missing=0.03, n_files=2)
    for r in range(V):  # every value of c0 used
        g["values"][r][0] = f"{r:03d}"
    eng, rc, x, file = _chain_and_random_state(f"pcg2-V{V}", oracle, g, 5, "PCG-II",
                                               "k_link_pcg2<A=4,NS=2,HC=32,PK=%d>" % (1 if V <= 255 else 0), 1, (3,))
    assert rc.indexes[0].num_values == V


@pytest.mark.parametrize("n_const,n_str", [(0, 9), (2, 10)])
def test_pcg2_one_record_per_warp(oracle, n_const, n_str):
    """32-slot shapes with 9..16 non-constant attributes run one record per warp"""
    from dblink_b200 import synth

    attrs = [synth.SynthAttr(f"c{i}", "constant", 5 + 3 * i, 0.5) for i in range(n_const)]
    attrs += [synth.SynthAttr(f"s{i}", "levenshtein", 60 + 10 * i, 1.0) for i in range(n_str)]
    g = synth.generate(47 + n_str, 700, attrs, dup=0.3, distortion=0.15, missing=0.05, n_files=2)
    A = n_const + n_str
    _chain_and_random_state(f"pcg2-NS{n_str}", oracle, g, 13, "PCG-II",
                            "k_link_pcg2<A=%d,NS=%d,HC=32,PK=%d>" % (A, n_str, 1 if n_const else 0), 1, (A - 1,))


@pytest.mark.parametrize("slots,vocab,thresholds", [(64, 200, {"s0": 3.5, "s1": 3.5}), (128, 200, {"s0": 3.0}),
                                                    (256, 400, {"s0": 3.0, "s1": 3.0})])
def test_pcg2_runtime_hash_size(oracle, slots, vocab, thresholds):
    """rows longer than 31 values: the PCG-II kernel whose table size (64, 128 or 256 slots) is a run-time parameter;
    with one attribute lowered the other is re-hashed from 32 slots to the model-wide size"""
    from dblink_b200 import synth

    attrs = [synth.SynthAttr("c0", "constant", 8, 0.5), synth.SynthAttr("c1", "constant", 20, 0.5),
             synth.SynthAttr("s0", "levenshtein", vocab, 1.0), synth.SynthAttr("s1", "levenshtein", vocab, 1.0)]
    g = _lowered(synth_problem(seed=7, R=900, attrs=attrs, n_files=2), thresholds)
    eng, rc, x, file = _chain_and_random_state(f"pcg2-HC0-{slots}", oracle, g, 17, "PCG-II",
                                               "k_link_pcg2<A=4,NS=2,HC=0,PK=0>", 1, (2,))
    hs = [ix.hash_slots for ix in rc.indexes]
    assert max(hs) == slots and (hs[3] == 32) == ("s1" not in thresholds)
    assert ((x[:, 2] < 0) | (x[:, 3] < 0)).sum() >= 20  # records with a missing string attribute


@pytest.mark.parametrize("why", ["row-longer-than-256", "shared-memory"])
def test_pcg2_falls_back_to_the_generic_kernel(oracle, why):
    """PCG-II in automatic mode takes k_link_generic when a similarity row does not hash into 256 slots, or when the
    PCG-II kernel would need more than 100 KB of shared memory (4 string attributes at 256 slots)"""
    from dblink_b200 import synth

    if why == "row-longer-than-256":
        attrs = [synth.SynthAttr("c0", "constant", 8, 0.5), synth.SynthAttr("c1", "constant", 20, 0.5),
                 synth.SynthAttr("s0", "levenshtein", 1600, 0.3), synth.SynthAttr("s1", "levenshtein", 200, 1.0)]
        g = _lowered(synth_problem(seed=7, R=1500, attrs=attrs, n_files=2), {"s0": 3.0})
    else:
        attrs = [synth.SynthAttr("c0", "constant", 8, 0.5), synth.SynthAttr("c1", "constant", 20, 0.5)]
        attrs += [synth.SynthAttr(f"s{i}", "levenshtein", 400, 1.0) for i in range(4)]
        g = _lowered(synth_problem(seed=7, R=900, attrs=attrs, n_files=2), {f"s{i}": 3.0 for i in range(4)})
    eng, rc, x, file = _chain_and_random_state(f"pcg2-fallback-{why}", oracle, g, 19, "PCG-II", "k_link_generic",
                                               1, (0,), n=2)
    hs = [ix.hash_slots for ix in rc.indexes]
    if why == "row-longer-than-256":
        assert hs[2] == 0 and np.diff(rc.indexes[2].tables()["rowptr"]).max() > 256
    else:
        assert max(hs) == 256 and min(hs[2:]) >= 32  # every string attribute hashes; the tables need 256 slots


def _survivor_classes(d, x, A):
    """per record, from the state before a sweep: (number of candidates agreeing on every observed non-distorted
    attribute, has such an attribute, size of its block)"""
    link, y, z, block = d["link"], d["y"], d["z"], d["block"]
    rb = block[link]
    surv = np.zeros(len(x), np.int64)
    must = (x >= 0) & (z == 0)
    for b in np.unique(rb):
        cand = np.flatnonzero(block == b)
        rs = np.flatnonzero(rb == b)
        ok = np.ones((len(rs), len(cand)), bool)
        for a in range(A):
            ok &= ~must[rs, a][:, None] | (x[rs, a][:, None] == y[cand, a][None, :])
        surv[rs] = ok.sum(axis=1)
    return surv, must.any(axis=1), np.bincount(block)[rb]


def _pruned_state(rng, eng, x, E, small, Vs):
    """a valid state with one block of `small` entities and one of E - small (the tree splits on attribute 1), records
    with many survivors (only attribute 0 must match) and records with nothing to match (every attribute distorted)"""
    R, A = x.shape
    side = np.array([eng.partitioner.get_partition_id(np.array([0, v, 0, 0], np.int32)) for v in range(Vs[1])])
    assert set(side) == {0, 1}
    y = np.stack([rng.integers(0, Vs[a], E) for a in range(A)], axis=1).astype(np.int32)
    y[:small, 1] = rng.choice(np.flatnonzero(side == 0), small)
    y[small:, 1] = rng.choice(np.flatnonzero(side == 1), E - small)
    link = rng.integers(0, E, R).astype(np.int32)
    for r in range(R):
        if rng.random() < 0.7:
            for a in (0, 2, 3):
                if x[r, a] >= 0 and rng.random() < 0.8:
                    y[link[r], a] = x[r, a]
    recs = rng.permutation(R)
    heavy, many = recs[:400], recs[400:560]
    for r in many:
        if x[r, 0] >= 0:
            y[link[r], 0] = x[r, 0]
    yl = y[link]
    z = np.where(x < 0, rng.random((R, A)) < 0.1, (x != yl) | (rng.random((R, A)) < 0.2)).astype(np.uint8)
    z[heavy] = 1
    z[many] = 1
    z[many, 0] = np.where((x[many, 0] >= 0) & (x[many, 0] == yl[many, 0]), 0, 1)
    return y, link, z


@pytest.mark.parametrize("sampler", ["PCG-I", "Gibbs"])
def test_pruned_heavy_match_generic_kernels(oracle, sampler, monkeypatch):
    """k_link_pruned with more than 48 survivors (pass 2 walks the postings again) and with exactly one (the shortcut),
    records with nothing to match in a block of <= 256 entities (scored by the pruned kernel) and in one of > 256
    (k_link_heavy); then the same state through k_link_generic (mode 1), k_link_match (mode 2) and the pruned kernel
    without the dense posting pointers"""
    g = synth_problem(seed=21, R=1500, n_files=2, missing=0.05, distortion=0.2)
    m, st0, tree, ox, ofile = oracle_setup(oracle, g, 5, 1, (1,))
    rng = np.random.default_rng(33)
    state = None
    for mode, kernel, sparse in ((0, "k_link_pruned", False), (1, "k_link_generic", False),
                                 (2, "k_link_match", False), (0, "k_link_pruned", True)):
        if sparse:
            monkeypatch.setenv("DBL_INV_DENSE_MAX", "0")
        eng, rc, x, file = product_setup(g, 5, 1, (1,))
        eng.set_link_mode(mode)
        assert eng.num_partitions == 2 and eng.link_kernel(sampler) == kernel
        Vs = [ix.num_values for ix in rc.indexes]
        if state is None:
            y, link, z = _pruned_state(rng, eng, x, 1400, 200, Vs)
            state = (y, link, z, rng.uniform(0.01, 0.3, (len(Vs), 2)))
        y, link, z, theta = state
        eng.upload_state(x, file, z, link, y, theta, iteration=7)
        before = snapshot(eng)
        surv, has_must, bsize = _survivor_classes(before, x, len(Vs))
        assert sorted(np.bincount(before["block"])) == [200, 1200]
        classes = {">48 survivors": has_must & (surv > 48), "1 survivor": has_must & (surv == 1),
                   "nothing to match, block <= 256": ~has_must & (bsize <= 256),
                   "nothing to match, block > 256": ~has_must & (bsize > 256)}
        for k, v in classes.items():
            assert v.sum() >= 20, (k, int(v.sum()))
        st = oracle.State.from_arrays(m, x, file, z, link, y, theta, 7)
        eng.sweep(sampler, 1)
        res = _check(f"link-mode{mode}{'-sparse' if sparse else ''}", eng, before, tables_of(rc.indexes), x, file,
                     sampler)
        for k, v in classes.items():
            assert not set(np.flatnonzero(v)) & set(res["bad"]), k
        assert st.sweep(oracle.SAMPLERS[sampler]) == 0
        assert_same_state(eng, st)
        _sweeps(f"link-mode{mode}", oracle, eng, st, tables_of(rc.indexes), x, file, sampler, 2)
        eng.close()


@pytest.mark.parametrize("E", [4096, 4097, 9000])
def test_chunks_of_several_tiles(oracle, E):
    """one block of 32 tiles (one tile per chunk), 33 (two per chunk, the last chunk one tile) and 71 (three per
    chunk): PCG-II, and PCG-I with records that have nothing to match (k_link_heavy)"""
    g = synth_problem(seed=51, R=500, n_files=2, missing=0.05)
    assert (E + 127) // 128 == {4096: 32, 4097: 33, 9000: 71}[E]
    _chain_and_random_state(f"tiles-E{E}", oracle, g, 3, "PCG-II", "k_link_pcg2<A=4,NS=2,HC=32,PK=1>", pop=E, n=2)
    eng, rc, x, file = product_setup(g, 3, 0, (), E)
    m, st0, tree, ox, ofile = oracle_setup(oracle, g, 3, 0, (), E)
    assert eng.num_entities == E and eng.link_kernel("PCG-I") == "k_link_pruned"
    rng = np.random.default_rng(E)
    y, link, z = random_state(rng, x, E, [ix.num_values for ix in rc.indexes])
    z[rng.choice(len(x), 40, replace=False)] = 1  # nothing to match in a block of > 256 entities: k_link_heavy
    theta = rng.uniform(0.01, 0.3, (len(rc.indexes), 2))
    eng.upload_state(x, file, z, link, y, theta, iteration=5)
    st = oracle.State.from_arrays(m, x, file, z, link, y, theta, 5)
    assert (((x < 0) | (z == 1)).all(axis=1)).sum() >= 40
    _sweeps(f"tiles-E{E}", oracle, eng, st, tables_of(rc.indexes), x, file, "PCG-I", 2)


def test_full_size_benchmarked_model():
    """BASELINE.json configs[3] (1M records / 10 attributes / 64 blocks, the model bench.py times): one PCG-II sweep,
    a fixed seeded sample of 4 096 records checked (no oracle run)"""
    import dblink_b200 as D
    from dblink_b200 import synth

    enc = synth.generate_encoded(2, 1_000_000, synth.config_attrs(4), dup=0.10, distortion=0.05, missing=0.01,
                                 n_files=2)
    indexes, x, file, F = synth.build_encoded(enc)
    eng = D.GibbsEngine(indexes, [a.alpha for a in enc["attributes"]], [a.beta for a in enc["attributes"]], None, 2024, F)
    eng.init_state(x, file)
    part = D.KDTreePartitioner(6, [4, 5, 6, 7, 8, 9]).fit(eng.download_state()["y"])
    eng.set_partitioner(part)
    assert eng.num_partitions == 64
    assert eng.link_kernel("PCG-II") == "k_link_pcg2<A=10,NS=6,HC=32,PK=1>"
    before = snapshot(eng)
    eng.sweep("PCG-II", 1)
    sample = np.random.default_rng(4096).choice(len(x), 4096, replace=False)
    _check("full-size", eng, before, tables_of(indexes), x, file, "PCG-II", sample)
    eng.close()
