"""CPU-only tests of the host layer around the sweep: HOCON surface, posterior summaries, output formats,
project/step parsing (SURVEY.md section 8f).  No GPU compute."""
import os

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

CONF = """
dblink : {
    // hyper-parameters (referenced below)
    lowDistortion : {alpha : 0.5, beta : 50.0}
    constSimFn : { name : "ConstantSimilarityFn", }
    levSimFn : {
        name : "LevenshteinSimilarityFn",
        parameters : {
            threshold : 7.0
            maxSimilarity : 10.0
        }
    }
    data : {
        path : "%s"
        recordIdentifier : "rec_id",
        # fileIdentifier : null,
        entityIdentifier : "ent_id" // optional
        nullValue : "NA"
        matchingAttributes : [
            {name : "by", similarityFunction : ${dblink.constSimFn}, distortionPrior : ${dblink.lowDistortion}},
            {name : "bm", similarityFunction : ${dblink.constSimFn}, distortionPrior : ${dblink.lowDistortion}},
            {name : "bd", similarityFunction : ${dblink.constSimFn}, distortionPrior : ${dblink.lowDistortion}},
            {name : "fname_c1", similarityFunction : ${dblink.levSimFn}, distortionPrior : ${dblink.lowDistortion}},
            {name : "lname_c1", similarityFunction : ${dblink.levSimFn}, distortionPrior : ${dblink.lowDistortion}}
        ]
    }
    randomSeed : 319158
    expectedMaxClusterSize : 10
    partitioner : {
        name : "KDTreePartitioner",
        parameters : {
            numLevels : %d, // zero = no partitioning
            matchingAttributes : %s
        }
    }
    outputPath : "%s"
    checkpointPath : "/tmp/spark_checkpoint/"
    steps : [
        {name : "sample", parameters : {
            sampleSize : %d,
            burninInterval : 0,
            thinningInterval : %d,
            resume : false,
            sampler : "%s"
        }},
        {name : "summarize", parameters : {
            lowerIterationCutoff : 0,
            quantities : ["cluster-size-distribution", "partition-sizes"]
        }},
        {name : "evaluate", parameters : {
            lowerIterationCutoff : %d,
            metrics : ["pairwise", "cluster"],
            useExistingSMPC : false
        }}
    ]
}
"""


def make_conf(data, out, levels=0, attrs="[]", sample_size=100, thinning=10, sampler="PCG-I", cutoff=100):
    return CONF % (data, levels, attrs, out, sample_size, thinning, sampler, cutoff)


def test_hocon_subset():
    from dblink_b200 import config

    c = config.parse_string(make_conf("d.csv", "out/"))
    assert c.get_string("dblink.data.path") == "d.csv"
    assert c.get_int("dblink.randomSeed") == 319158
    ma = c.get_list("dblink.data.matchingAttributes")
    assert [a["name"] for a in ma] == ["by", "bm", "bd", "fname_c1", "lname_c1"]
    assert ma[3]["similarityFunction"] == {"name": "LevenshteinSimilarityFn",
                                           "parameters": {"threshold": 7.0, "maxSimilarity": 10.0}}
    assert ma[0]["distortionPrior"] == {"alpha": 0.5, "beta": 50.0}
    assert not c.has("dblink.data.fileIdentifier")      # commented out
    assert c.get("dblink.populationSize", None) is None  # optional key (Project.scala:194)
    assert c.get_list("dblink.steps")[0]["parameters"]["resume"] is False
    # other HOCON features: '=' separator, object without separator, dotted keys, merge, optional substitution
    d = config.parse_string('a { b = 1 }\na.c : "x"\nd = ${a.b}\ne = ${?nope}\nf = [1, 2,\n 3,]\n')
    assert d.tree == {"a": {"b": 1, "c": "x"}, "d": 1, "e": None, "f": [1, 2, 3]}
    with pytest.raises(config.ConfigError):
        config.parse_string("a = ${missing}")
    with pytest.raises(config.ConfigError):
        config.parse_string("a { b : 1")
    with pytest.raises(config.ConfigError):
        c.get_string("dblink.nope")


def test_project_parsing_and_data(tmp_path):
    import dblink_b200 as D
    from dblink_b200 import config
    from dblink_b200.project import Project

    data = os.path.join(GOLDEN, "RLdata500.csv.gz")
    p = Project(config.parse_string(make_conf(data, str(tmp_path) + "/", 1, '["fname_c1"]')), base_dir="")
    assert [a.name for a in p.matching_attributes] == ["by", "bm", "bd", "fname_c1", "lname_c1"]
    assert [a.is_constant for a in p.matching_attributes] == [True, True, True, False, False]
    assert p.num_levels == 1 and p.partition_attribute_ids == [3] and p.expected_max_cluster_size == 10
    steps = p.steps()
    assert [s[0] for s in steps] == ["sample", "summarize", "evaluate"]
    assert steps[0][1] == dict(sample_size=100, burnin_interval=0, thinning_interval=10, resume=False, sampler="PCG-I")
    d = p.load()
    assert d["x"].shape == (500, 5) and (d["x"] >= 0).all()
    assert [ix.num_values for ix in d["cache"].indexes] == [86, 12, 31, 146, 108]  # SURVEY.md appendix B
    assert [ix.nnz for ix in d["cache"].indexes][3:] == [236, 236]
    truth = p.true_clusters()
    assert len(truth) == 450 and sum(len(c) == 2 for c in truth) == 50
    bad = make_conf(data, str(tmp_path) + "/").replace('"KDTreePartitioner"', '"SimplePartitioner"')
    with pytest.raises(config.ConfigError):
        Project(config.parse_string(bad), base_dir="")
    bad = make_conf(data, str(tmp_path) + "/").replace('["pairwise", "cluster"]', '["accuracy"]')
    with pytest.raises(ValueError):
        Project(config.parse_string(bad), base_dir="").steps()


def test_analysis_metrics():
    from dblink_b200 import analysis as an

    truth = [frozenset("ab"), frozenset("cd"), frozenset("e"), frozenset("fgh")]
    pred = [frozenset("ab"), frozenset("c"), frozenset("de"), frozenset("fg"), frozenset("h")]
    m = an.pairwise_metrics(pred, truth)
    assert (m["TP"], m["FP"], m["FN"]) == (2, 1, 3)
    assert m["precision"] == pytest.approx(2 / 3) and m["recall"] == pytest.approx(2 / 5)
    assert m["f1score"] == pytest.approx(2 * (2 / 3) * (2 / 5) / (2 / 3 + 2 / 5))
    assert an.adjusted_rand_index(truth, truth) == pytest.approx(1.0)
    from sklearn.metrics import adjusted_rand_score

    recs = sorted("abcdefgh")
    lab = lambda cl: [next(i for i, c in enumerate(cl) if r in c) for r in recs]  # noqa: E731
    assert an.adjusted_rand_index(pred, truth) == pytest.approx(adjusted_rand_score(lab(truth), lab(pred)))
    chain = [(10, {0: [["a", "b"], ["c"]], 1: [["d", "e"]]}), (20, {0: [["a", "b"], ["c", "d"]], 1: [["e"]]}),
             (30, {0: [["a", "b", "c"]], 1: [["d", "e"]]})]
    mpc = an.most_probable_clusters(chain)
    assert mpc["a"][0] == frozenset("ab") and mpc["a"][1] == pytest.approx(2 / 3)
    assert mpc["d"][0] == frozenset("de")
    assert set(an.shared_most_probable_clusters(chain)) == {frozenset("ab"), frozenset("c"), frozenset("de")}
    assert an.cluster_size_distribution(chain)[30] == {3: 1, 2: 1}
    assert an.partition_sizes(chain)[20] == {0: 2, 1: 1}


def test_writers_roundtrip(tmp_path):
    import pyarrow.parquet as pq

    from dblink_b200 import analysis as an, writers as w

    link = np.array([3, 0, 3, 2, 0, 4], np.int32)
    blk = np.array([0, 1, 1, 0, 0], np.int32)  # entity 1 is isolated
    ids = ["r%d" % i for i in range(6)]
    parts = w.linkage_structure(link, blk, ids)
    assert parts == {0: [["r1", "r4"], ["r0", "r2"], ["r5"]], 1: [["r3"]]}
    path = os.path.join(tmp_path, "linkage-chain.parquet")
    lw = w.LinkageChainWriter(path, write_buffer_size=2)
    for it in (0, 10, 20):
        lw.append(it, parts)
    lw.close()
    assert sorted(os.listdir(path)) == ["partitionId=0", "partitionId=1"]  # hive partitioning (BufferedRDDWriter:49)
    t = pq.ParquetFile(os.path.join(path, "partitionId=0", sorted(os.listdir(os.path.join(path, "partitionId=0")))[0])).read()
    assert t.schema.names == ["iteration", "linkageStructure"]
    assert str(t.schema.field("iteration").type) == "int64"
    assert str(t.schema.field("linkageStructure").type).startswith("list<") and "string" in str(t.schema.field("linkageStructure").type)
    chain = w.read_linkage_chain(path, lower_iteration_cutoff=10)
    assert [c[0] for c in chain] == [10, 20] and chain[0][1] == parts
    dw = w.DiagnosticsWriter(os.path.join(tmp_path, "diagnostics.csv"), ["by", "fname_c1"])
    dw.write_row({"iteration": 7, "num_isolates": 2, "log_likelihood": -123.456, "agg_dist": np.array([[1, 2], [3, 4]]),
                  "rec_dist": np.array([5, 1, 0])}, 10)
    dw.close()
    lines = open(os.path.join(tmp_path, "diagnostics.csv")).read().splitlines()
    assert lines[0] == ("iteration,systemTime-ms,numObservedEntities,logLikelihood,popSize,aggDist-by,aggDist-fname_c1,"
                        "recDistortion-0,recDistortion-1,recDistortion-2")  # DiagnosticsWriter.scala:39-45
    f = lines[1].split(",")
    assert f[0] == "7" and f[2] == "8" and f[3] == "-1.234560000e+02" and f[4:] == ["10", "3", "7", "5", "1", "0"]
    w.save_cluster_size_distribution(an.cluster_size_distribution(chain), str(tmp_path))
    assert open(os.path.join(tmp_path, "cluster-size-distribution.csv")).read().splitlines()[0] == "iteration,0,1,2"
    w.save_partition_sizes(an.partition_sizes(chain), str(tmp_path))
    assert open(os.path.join(tmp_path, "partition-sizes.csv")).read().splitlines() == ["iteration,0,1", "10,3,1", "20,3,1"]


def test_sampler_argument_checks():
    from dblink_b200 import sampler

    for kw in (dict(sample_size=0), dict(sample_size=1, burnin_interval=-1), dict(sample_size=1, thinning_interval=0),
               dict(sample_size=1, sampler="Metropolis")):
        args = dict(sample_size=1, burnin_interval=0, thinning_interval=1, sampler="PCG-I")
        args.update(kw)
        with pytest.raises(ValueError):
            sampler.sample(None, [], [], args["sample_size"], "/tmp/x", args["burnin_interval"], args["thinning_interval"],
                           sampler=args["sampler"])


def test_bench_reference_arm_runs():
    """`bench.py --impl reference` (the CPU arm beside the GPU arm) prints one JSON line and writes nothing into the
    tree (its -march=native oracle build goes to a temporary directory)"""
    import json
    import subprocess
    import sys

    from helpers import tree_files

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for sampler in ("PCG-II", "PCG-I"):
        before = tree_files(root)
        res = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--records", "20000",
                              "--steps", "1", "--warmup", "0", "--cpu-sample", "500", "--sampler", sampler],
                             capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, res.stderr[-2000:]
        assert tree_files(root) == before
        line = json.loads(res.stdout.strip().splitlines()[-1])
        assert line["impl"] == "reference" and line["value"] > 0 and line["unit"] == "iterations/s"
        assert line["cpu_baseline"]["kind"] == "port" and line["e2e"]["h2d_bytes_per_step"] == 0


def test_bench_dump_outputs_sample_and_size(tmp_path):
    """bench.py --dump-outputs on a state the size of the benchmark's: float32 / float64 files under 64 MB in all, the
    same fixed rows on every call, values taken from those rows"""
    import importlib.util

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    R, A, F = 1_000_000, 10, 2
    rng = np.random.default_rng(3)
    state = {"link": rng.integers(0, R, R, dtype=np.int32), "z": rng.integers(0, 2, (R, A), dtype=np.uint8),
             "y": rng.integers(0, 50_000, (R, A), dtype=np.int32), "block": rng.integers(0, 64, R, dtype=np.int32),
             "theta": rng.uniform(0, 1, (A, F))}
    summary = {"agg_dist": rng.integers(0, R, (A, F)), "rec_dist": rng.integers(0, R, A + 1), "log_likelihood": -1.5e7,
               "num_isolates": 12345, "iteration": 11}
    dirs = [tmp_path / "a", tmp_path / "b"]
    for d in dirs:
        bench.dump_outputs(str(d), state, summary)
    files = sorted(p.name for p in dirs[0].iterdir())
    assert {"link.npy", "y.npy", "z.npy", "block.npy", "theta.npy", "record_ids.npy", "entity_ids.npy"} <= set(files)
    assert sum((dirs[0] / f).stat().st_size for f in files) <= 64 << 20
    for f in files:
        a, b = np.load(dirs[0] / f), np.load(dirs[1] / f)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b), f
    out = {f[:-4]: np.load(dirs[0] / f) for f in files}
    rec, ent = out["record_ids"].astype(np.int64), out["entity_ids"].astype(np.int64)
    assert 100_000 < len(rec) < R and np.all(np.diff(rec) > 0) and np.all(np.diff(ent) > 0)
    np.testing.assert_array_equal(out["link"], state["link"][rec])
    np.testing.assert_array_equal(out["z"], state["z"][rec])
    np.testing.assert_array_equal(out["y"], state["y"][ent])
    np.testing.assert_array_equal(out["block"], state["block"][ent])
    np.testing.assert_array_equal(out["theta"], state["theta"])
    assert out["log_likelihood"][0] == -1.5e7 and out["iteration"][0] == 11


def test_arrow_linkage_structure_equals_list_form(tmp_path):
    """linkage_structure_arrow (no Python loop over clusters) == linkage_structure, in memory and through the
    hive-partitioned Parquet chain; mixed buffers (Arrow + list rows) are written too."""
    import time

    from dblink_b200 import writers as w

    rng = np.random.default_rng(3)
    for R, E, P in ((1, 1, 1), (50, 50, 4), (3000, 2500, 8)):
        link = rng.integers(0, E, R).astype(np.int32)
        blk = rng.integers(0, P, E).astype(np.int32)
        ids = ["rec-%d" % i for i in range(R)]
        lists = w.linkage_structure(link, blk, ids)
        arrow = w.linkage_structure_arrow(link, blk, ids)
        assert {p: a.to_pylist() for p, a in arrow.items()} == lists
        path = os.path.join(tmp_path, "chain-%d.parquet" % R)
        lw = w.LinkageChainWriter(path, write_buffer_size=3)
        lw.append(0, arrow)
        lw.append(5, lists)   # one buffer holding both forms
        lw.append(10, arrow)
        lw.append(15, arrow)
        lw.close()
        chain = w.read_linkage_chain(path)
        assert [c[0] for c in chain] == [0, 5, 10, 15]
        assert all(c[1] == lists for c in chain)
    # the point of the Arrow form: no per-cluster Python work
    R = 200_000
    link = rng.integers(0, R, R).astype(np.int32)
    blk = rng.integers(0, 16, R).astype(np.int32)
    import pyarrow as pa

    ids = pa.array(["r%d" % i for i in range(R)], pa.string())
    t0 = time.perf_counter()
    arrow = w.linkage_structure_arrow(link, blk, ids)
    dt = time.perf_counter() - t0
    assert sum(len(a) for a in arrow.values()) == len(np.unique(link))
    assert dt < 2.0


def test_array_summaries_equal_the_set_based_ones(tmp_path):
    """analysis_arrays (vectorised: signatures, run-length mode, contingency tables) == analysis (sets and loops) on
    random chains read back from linkage-chain.parquet, including ties between equally frequent clusters."""
    from dblink_b200 import analysis as an, analysis_arrays as aa, writers as w

    rng = np.random.default_rng(11)
    for trial, (R, E, P, S) in enumerate(((6, 4, 2, 4), (40, 25, 3, 7), (300, 220, 5, 9))):
        ids = ["id%03d" % i for i in range(R)]
        blk = rng.integers(0, P, E).astype(np.int32)
        path = os.path.join(tmp_path, "chain%d.parquet" % trial)
        lw = w.LinkageChainWriter(path, write_buffer_size=4)
        base = rng.integers(0, E, R).astype(np.int32)
        for s in range(S):
            link = base.copy()
            move = rng.random(R) < 0.3                      # samples share most clusters: repeated and tied modes
            link[move] = rng.integers(0, E, int(move.sum()))
            if s % 3 == 0:
                base = link
            lw.append(10 * s, w.linkage_structure_arrow(link, blk, ids))
        lw.close()
        for cutoff in (0, 20):
            ch = w.read_linkage_chain(path, cutoff)
            ca = aa.read_chain_arrays(path, cutoff)
            assert list(ca.iterations) == [c[0] for c in ch]
            assert aa.cluster_size_distribution(ca) == an.cluster_size_distribution(ch)
            assert aa.partition_sizes(ca) == an.partition_sizes(ch)
            labels = aa.shared_most_probable_clusters(ca)
            got = {frozenset(c) for c in aa.labels_to_clusters(labels, ca.record_ids)}
            assert got == set(an.shared_most_probable_clusters(ch))
            truth_of = rng.integers(0, max(2, R // 2), R)
            id_list = ca.record_ids.to_pylist()
            truth_sets = an.membership_to_clusters(id_list, truth_of)
            pm_a, pm_s = aa.pairwise_metrics(labels, truth_of), an.pairwise_metrics(list(got), truth_sets)
            assert (pm_a["TP"], pm_a["FP"], pm_a["FN"]) == (pm_s["TP"], pm_s["FP"], pm_s["FN"])
            assert pm_a["f1score"] == pytest.approx(pm_s["f1score"], nan_ok=True)
            assert aa.adjusted_rand_index(labels, truth_of) == pytest.approx(an.adjusted_rand_index(list(got), truth_sets))
    # a sample straight from link arrays
    link = np.array([3, 0, 3, 2, 0, 4], np.int32)
    mem, off, part = aa.sample_from_links(link, np.array([0, 1, 1, 0, 0], np.int32))
    assert [list(mem[off[i]:off[i + 1]]) for i in range(len(off) - 1)] == [[1, 4], [3], [0, 2], [5]]
    assert list(part) == [0, 1, 0, 0]


def test_columnar_records_path_equals_the_list_path(tmp_path):
    """read_csv_columns + build_cache_from_columns (pyarrow, no loop over records) give the same value ids, file
    ids, index sizes and missing counts as read_csv + RecordsCache.build + transform_records."""
    from dblink_b200 import records as R

    rng = np.random.default_rng(5)
    path = os.path.join(tmp_path, "d.csv")
    names = ["c0", "s0", "s1"]
    vocab = [["a", "b", "c"], ["SMITH", "SMYTH", "JONES", "JONAS", "BROWN"], ["ANN", "ANNE", "BOB", ""]]
    with open(path, "w") as fh:
        fh.write("id,src," + ",".join(names) + ",truth\n")
        for r in range(400):
            vals = [("NA" if rng.random() < 0.1 else vocab[a][rng.integers(len(vocab[a]))]) for a in range(3)]
            fh.write("r%d,%s,%s,e%d\n" % (r, "fileB" if rng.random() < 0.4 else "fileA", ",".join(vals), r // 2))
    attrs = [R.Attribute("c0"), R.Attribute("s0", R.SimilarityFn("LevenshteinSimilarityFn", 7, 10)),
             R.Attribute("s1", R.SimilarityFn("LevenshteinSimilarityFn", 7, 10))]
    for file_col in ("src", None):
        ri, f, v, e = R.read_csv(path, "id", names, file_col, "truth", "NA")
        c1 = R.RecordsCache.build(v, f, attrs, 5)
        x1, f1 = c1.transform_records(v, f)
        ri2, f2, cols, e2 = R.read_csv_columns(path, "id", names, file_col, "truth", "NA")
        c2, x2, ff2 = R.build_cache_from_columns(cols, f2, attrs, 5)
        assert ri2.to_pylist() == ri and e2.to_pylist() == e
        np.testing.assert_array_equal(x1, x2)
        np.testing.assert_array_equal(f1, ff2)
        assert (c1.file_ids, c1.file_sizes, c1.missing_counts) == (c2.file_ids, c2.file_sizes, c2.missing_counts)
        for a in range(3):
            assert c1.indexes[a].num_values == c2.indexes[a].num_values
            for v_ in set(vocab[a]) - {""}:
                assert c1.indexes[a].value_idx_of(v_) == c2.indexes[a].value_idx_of(v_)
    with pytest.raises(ValueError):
        R.build_cache_from_columns(cols[:2], f2, attrs, 5)


def test_array_summaries_edge_cases(tmp_path):
    from dblink_b200 import analysis_arrays as aa, writers as w

    # one sample, one record
    path = os.path.join(tmp_path, "one.parquet")
    lw = w.LinkageChainWriter(path)
    lw.append(0, w.linkage_structure_arrow(np.array([0], np.int32), np.array([0], np.int32), ["only"]))
    lw.close()
    ca = aa.read_chain_arrays(path)
    assert list(ca.iterations) == [0] and ca.num_records == 1
    assert aa.cluster_size_distribution(ca) == {0: {1: 1}} and aa.partition_sizes(ca) == {0: {0: 1}}
    labels = aa.shared_most_probable_clusters(ca)
    assert list(labels) == [0]
    assert aa.labels_to_clusters(labels, ca.record_ids) == [["only"]]
    m = aa.pairwise_metrics(labels, np.array([7]))
    assert (m["TP"], m["FP"], m["FN"]) == (0, 0, 0) and m["f1score"] != m["f1score"]  # NaN, as PairwiseMetrics does
    # cutoff beyond the chain: empty
    empty = aa.read_chain_arrays(path, lower_iteration_cutoff=5)
    assert len(empty.samples) == 0 and empty.num_records == 0
    # a record whose two candidate clusters are equally frequent keeps the one seen first
    ids = ["a", "b", "c"]
    blk = np.zeros(3, np.int32)
    path2 = os.path.join(tmp_path, "tie.parquet")
    lw = w.LinkageChainWriter(path2)
    lw.append(0, w.linkage_structure_arrow(np.array([0, 0, 2], np.int32), blk, ids))   # {a,b} {c}
    lw.append(1, w.linkage_structure_arrow(np.array([0, 1, 1], np.int32), blk, ids))   # {a} {b,c}
    lw.close()
    ca = aa.read_chain_arrays(path2)
    got = {frozenset(c) for c in aa.labels_to_clusters(aa.shared_most_probable_clusters(ca), ca.record_ids)}
    assert got == {frozenset("ab"), frozenset("c")}


def test_run_txt_describes_the_project_and_its_steps(tmp_path):
    """Run.main writes Project.mkString and ProjectSteps.mkString to run.txt before executing (Run.scala:38-43)"""
    from dblink_b200 import config
    from dblink_b200.project import Project

    data = os.path.join(GOLDEN, "RLdata500.csv.gz")
    out = str(tmp_path) + "/"
    p = Project(config.parse_string(make_conf(data, out, 1, '["fname_c1"]')), base_dir="")
    p.write_run_txt()
    txt = open(os.path.join(out, "run.txt")).read()
    for needle in ("Data settings", "  * The record identifier attribute is 'rec_id'", "  * There is no file identifier",
                   "  * The matching attributes are 'by', 'bm', 'bd', 'fname_c1', 'lname_c1'",
                   "  * 'fname_c1' (id=3) with LevenshteinSimilarityFn(threshold=7.0, maxSimilarity=10.0) and "
                   "BetaShapeParameters(alpha=0.5, beta=50.0)",
                   "  * KDTreePartitioner(numLevels=1, attributeIds=[3])", "  * Using randomSeed=319158",
                   "Scheduled steps",
                   "  * SampleStep: Evolving the chain from new initial state with sampleSize=100, burninInterval=0, "
                   "thinningInterval=10 and sampler=PCG-I",
                   "  * SummarizeStep: Calculating summary quantities", "  * EvaluateStep: Evaluating sMPC clusters"):
        assert needle in txt, needle


def test_saved_state_fingerprint_covers_seed_and_partitioner(tmp_path):
    """a state saved under another randomSeed / populationSize / partitioner must not be continued (it would run on
    another Philox key or another partition function)"""
    from dblink_b200 import config
    from dblink_b200.project import Project

    data = os.path.join(GOLDEN, "RLdata500.csv.gz")
    base = make_conf(data, str(tmp_path) + "/", 1, '["fname_c1"]')
    fp = Project(config.parse_string(base), base_dir="").fingerprint()
    assert Project(config.parse_string(base), base_dir="").fingerprint() == fp
    for changed in (base.replace("randomSeed : 319158", "randomSeed : 7"),
                    base.replace("numLevels : 1", "numLevels : 0").replace('["fname_c1"]', "[]"),
                    base.replace('matchingAttributes : ["fname_c1"]', 'matchingAttributes : ["lname_c1"]')):
        assert changed != base
        assert Project(config.parse_string(changed), base_dir="").fingerprint() != fp
