"""BASELINE.json's full size (1M records / 10 attributes / 64 blocks) on the GPU, where the oracle is too slow:
size-independent properties of a sweep -- state invariants, summary identities, determinism, and agreement of the
two independent link-kernel implementations (TMA/hash kernels vs generic fallback), which share only the draw
protocol."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def big():
    import dblink_b200 as D
    from dblink_b200 import synth

    enc = synth.generate_encoded(2, 1_000_000, synth.config_attrs(4), dup=0.10, distortion=0.05, missing=0.01, n_files=2)
    indexes, x, file, F = synth.build_encoded(enc)
    alpha = [a.alpha for a in enc["attributes"]]
    beta = [a.beta for a in enc["attributes"]]

    def make():
        eng = D.GibbsEngine(indexes, alpha, beta, None, 2024, F)
        eng.init_state(x, file)
        part = D.KDTreePartitioner(6, [4, 5, 6, 7, 8, 9]).fit(eng.download_state()["y"])
        eng.set_partitioner(part)
        eng._keep = part
        return eng

    return make, x, file


def check_invariants(eng, x, prev_block_of_record=None):
    d = eng.download_state()
    s = eng.summary()
    R, A = x.shape
    y_of = d["y"][d["link"]]
    # GU:262-263: a non-distorted observed attribute always agrees with the linked entity
    assert not ((d["z"] == 0) & (x >= 0) & (x != y_of)).any()
    # observed and different => distorted (GU:352-354)
    assert (d["z"][(x >= 0) & (x != y_of)] == 1).all()
    # summary identities (GU:219-301)
    assert s["rec_dist"].sum() == R
    assert (s["rec_dist"] * np.arange(A + 1)).sum() == s["agg_dist"].sum() == int(d["z"].sum())
    assert s["num_isolates"] == eng.num_entities - len(np.unique(d["link"]))
    assert np.isfinite(s["log_likelihood"])
    assert ((s["theta"] > 0) & (s["theta"] < 1)).all()
    assert d["block"].min() >= 0 and d["block"].max() < eng.num_partitions
    return d, s


@pytest.mark.parametrize("sampler", ["PCG-II", "PCG-I"])
def test_full_size_properties(big, sampler):
    make, x, file = big
    a, b = make(), make()
    b.set_link_mode(1)  # generic fallback kernel
    check_invariants(a, x)
    blk_before = a.download_state()["block"]
    link_before = a.download_state()["link"]
    for it in range(2):
        a.sweep(sampler, 1)
        b.sweep(sampler, 1)
        da, sa = check_invariants(a, x)
        db = b.download_state()
        for k in ("link", "y", "z", "theta", "block"):
            assert np.array_equal(da[k], db[k]), (sampler, it, k)  # two kernel implementations, identical draws
        sb = b.summary()
        assert np.array_equal(sa["agg_dist"], sb["agg_dist"]) and np.array_equal(sa["rec_dist"], sb["rec_dist"])
        assert sa["log_likelihood"] == pytest.approx(sb["log_likelihood"], rel=1e-9)
        if it == 0:
            # a record can only link to an entity of the block it was in (GU:137, 192-198)
            assert np.array_equal(blk_before[da["link"]], blk_before[link_before])
    if sampler == "PCG-II":
        assert sa["pairs_scored"] == sb["pairs_scored"] > 3e10  # dense scoring: every entity of the block, every record
    else:  # the pruned kernel reports the postings it walked, the generic one every pair
        assert sb["pairs_scored"] > 3e10 and 0 < sa["pairs_scored"] < sb["pairs_scored"] / 100
    # determinism: a fresh engine replays the same chain (here through the dense TMA kernels, mode 2)
    c = make()
    c.set_link_mode(2)
    c.sweep(sampler, 2)
    dc = c.download_state()
    for k in ("link", "y", "z", "theta"):
        assert np.array_equal(da[k], dc[k])
    for e in (a, b, c):
        e.close()


def _full_config_against_oracle(monkeypatch, config, records, levels, split, samplers, seed=2024):
    """A BASELINE.json configuration at full size, sweep by sweep against the oracle: its link update runs on the
    host threads this process may use (ORC_THREADS; the split does not change the draws).  Bit-exact links, values,
    flags, theta, block ids after every sweep, and the state fingerprint bench.py prints (`state_hash`)."""
    import os
    import sys

    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench
    import dblink_b200 as D
    from dblink_b200 import synth
    from dblink_b200.engine import combine_state_hash
    from helpers import host_threads, state_hash_numpy
    from oracle import oracle as O

    monkeypatch.setenv("ORC_THREADS", str(host_threads()))
    enc = synth.generate_encoded(2 if config != 3 else 1, records, synth.config_attrs(config), dup=0.10,
                                 distortion=0.30 if config == 5 else 0.05, missing=0.01, n_files=1 if config == 3 else 2)
    indexes, x, file, F = synth.build_encoded(enc)
    eng = D.GibbsEngine(indexes, [a.alpha for a in enc["attributes"]], [a.beta for a in enc["attributes"]], None, seed, F)
    eng.init_state(x, file)
    eng.set_partitioner(D.KDTreePartitioner(levels, split).fit(eng.download_state()["y"]))
    st, tree = bench.cpu_prepare(enc, levels, split)  # the oracle's own tables, initial state and tree, same seed
    assert tree.n_leaves == eng.num_partitions == 1 << levels
    # the fast kernels, not a silent fall-back to the generic one (an order of magnitude slower)
    assert eng.link_kernel("PCG-II").startswith("k_link_pcg2<") and "HC=32" in eng.link_kernel("PCG-II")
    assert eng.link_kernel("PCG-I") == "k_link_pruned"
    d = eng.download_state()
    for k in ("link", "y", "z", "theta", "block"):
        np.testing.assert_array_equal(d[k], getattr(st, k), err_msg="initial " + k)
    for sampler in samplers:
        eng.sweep(sampler, 1)
        assert st.sweep(O.SAMPLERS[sampler]) == 0
        d = eng.download_state()
        for k in ("theta", "link", "y", "z", "block"):
            np.testing.assert_array_equal(d[k], getattr(st, k), err_msg=f"{sampler} {k}")
        s = eng.summary()
        he, hr = eng.state_hash()
        assert combine_state_hash(he, hr, s["theta"], s["iteration"]) == \
            combine_state_hash(*state_hash_numpy(st.y, st.link, st.z), st.theta, st.iteration)
    eng.close()
    return d


def test_baseline_config3_bit_parity_with_the_oracle(monkeypatch):
    """BASELINE.json configs[2]: 100k records / 8 string attributes / 16 blocks of 6 250 entities."""
    _full_config_against_oracle(monkeypatch, 3, 100_000, 4, [0, 1, 2, 3], ("PCG-II", "PCG-I", "PCG-II"))


def test_baseline_config4_bit_parity_with_the_oracle(monkeypatch):
    """BASELINE.json configs[3], the configuration bench.py times: 1M records / 10 attributes / 64 blocks.  One
    PCG-II and one PCG-I sweep; the oracle scores 1.6e10 pairs per sweep on the host threads (tens of seconds)."""
    _full_config_against_oracle(monkeypatch, 4, 1_000_000, 6, [4, 5, 6, 7, 8, 9], ("PCG-II", "PCG-I"))


def test_baseline_config5_bit_parity_with_the_oracle(monkeypatch):
    """BASELINE.json configs[4]: 1M records, distortion 0.30, Zipf(1.5) on the first two split attributes, so the 64
    k-d leaves are unbalanced and clusters carry many distorted attributes.  One PCG-II and one PCG-I sweep."""
    d = _full_config_against_oracle(monkeypatch, 5, 1_000_000, 6, [4, 5, 6, 7, 8, 9], ("PCG-II", "PCG-I"))
    sizes = np.bincount(d["block"], minlength=64)
    assert sizes.max() > 1.3 * sizes.mean()  # the skew the configuration is about


def test_bench_dump_outputs_follow_the_timed_steps(tmp_path):
    """bench.py --dump-outputs: the state after warmup + steps sweeps, the same on a repeated run with the same
    arguments (same inputs, same chain; the log-likelihood up to rounding), another one when --steps changes; nothing
    written into the tree"""
    import json
    import os
    import subprocess
    import sys

    from helpers import tree_files

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

    def run(steps, name):
        before = tree_files(root)
        out = tmp_path / name
        res = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--records", "20000", "--steps", str(steps),
                              "--warmup", "2", "--no-cpu", "--no-small", "--no-e2e", "--dump-outputs", str(out)],
                             capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, res.stderr[-3000:]
        assert tree_files(root) == before
        line = json.loads(res.stdout.strip().splitlines()[-1])
        assert line["steps"] == steps and line["state_hash_iteration"] == 2 + steps
        dump = {p.name[:-4]: np.load(p) for p in out.iterdir()}
        assert dump["iteration"][0] == 2 + steps and len(dump["link"]) == len(dump["record_ids"]) == 20000
        assert all(a.dtype in (np.float32, np.float64) for a in dump.values())
        return line["state_hash"], dump

    h1, d1 = run(3, "a")
    h2, d2 = run(3, "b")
    h3, d3 = run(4, "c")
    assert h1 == h2 and d1.keys() == d2.keys()
    for k in d1:
        if k == "log_likelihood":  # a sum of double atomics: its rounding depends on the order of the additions
            np.testing.assert_allclose(d1[k], d2[k], rtol=1e-9)
        else:
            np.testing.assert_array_equal(d1[k], d2[k], err_msg=k)
    assert h3 != h1 and not np.array_equal(d1["theta"], d3["theta"])
