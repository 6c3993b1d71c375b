"""Shared builders for tests: the same synthetic problem through the product host code and the oracle."""
import collections

import numpy as np


def synth_problem(seed=1, R=600, attrs=None, dup=0.3, distortion=0.1, missing=0.03, n_files=1):
    from dblink_b200 import synth

    if attrs is None:
        attrs = [synth.SynthAttr("c0", "constant", 8, 0.5), synth.SynthAttr("c1", "constant", 20, 0.5),
                 synth.SynthAttr("s0", "levenshtein", 120, 1.0), synth.SynthAttr("s1", "levenshtein", 160, 1.0)]
    return synth.generate(seed, R, attrs, dup=dup, distortion=distortion, missing=missing, n_files=n_files)


def oracle_indexes(O, g, kmax=10):
    """Oracle attribute indexes built independently from the strings (value counts as RecordsCache.scala:90-96)."""
    out = []
    for a, attr in enumerate(g["attributes"]):
        cnt = collections.Counter(v[a] for v in g["values"] if v[a] is not None)
        sf = attr.similarity_fn
        out.append(O.Index.build({k: float(v) for k, v in cnt.items()}, attr.is_constant, sf.threshold,
                                 sf.max_similarity, kmax))
    return out


def encode(O_indexes, g):
    A = len(O_indexes)
    R = len(g["values"])
    x = np.full((R, A), -1, np.int32)
    for a, ix in enumerate(O_indexes):
        cache = {}
        for r in range(R):
            v = g["values"][r][a]
            if v is not None:
                if v not in cache:
                    cache[v] = ix.value_id(v)
                x[r, a] = cache[v]
    fids = sorted(set(g["files"]))
    fmap = {f: i for i, f in enumerate(fids)}
    file = np.array([fmap[f] for f in g["files"]], np.int32)
    return x, file, len(fids)


def oracle_setup(O, g, seed, levels=0, attr_ids=(), pop=0, kmax=10):
    """-> (model_with_tree, state at iteration 0, tree, x, file)"""
    idx = oracle_indexes(O, g, kmax)
    x, file, F = encode(idx, g)
    alpha = [a.alpha for a in g["attributes"]]
    beta = [a.beta for a in g["attributes"]]
    m0 = O.Model(idx, alpha, beta, None, seed, F)
    s0 = O.State.init(m0, x, file, pop)
    tree = O.KDTree.fit(s0.y, levels, list(attr_ids))
    m = O.Model(idx, alpha, beta, tree, seed, F)
    s = O.State.from_arrays(m, x, file, s0.z, s0.link, s0.y, s0.theta, 0)
    s._keep = (m0, s0)
    return m, s, tree, x, file


def product_setup(g, seed, levels=0, attr_ids=(), pop=0, kmax=10):
    """-> (engine at iteration 0, records cache, x, file) through the public host API."""
    import dblink_b200 as D

    rc = D.RecordsCache.build(g["values"], g["files"], g["attributes"], kmax)
    x, file = rc.transform_records(g["values"], g["files"])
    eng = D.GibbsEngine(rc.indexes, [a.alpha for a in g["attributes"]], [a.beta for a in g["attributes"]], None, seed,
                        len(rc.file_ids))
    eng.init_state(x, file, pop)
    part = D.KDTreePartitioner(levels, list(attr_ids))
    part.fit(eng.download_state()["y"])
    eng.set_partitioner(part)
    return eng, rc, x, file


def random_state(rng, x, E, Vs, theta_scale=0.05):
    """A random but *valid* state (z=0 & x>=0 => x == y[link]) for single-sweep parity tests."""
    R, A = x.shape
    y = np.stack([rng.integers(0, Vs[a], E) for a in range(A)], axis=1).astype(np.int32)
    link = rng.integers(0, E, R).astype(np.int32)
    # make many records agree with their entity so that non-distorted paths are exercised
    for r in range(R):
        if rng.random() < 0.7:
            e = link[r]
            for a in range(A):
                if x[r, a] >= 0 and rng.random() < 0.8:
                    y[e, a] = x[r, a]
    z = np.zeros((R, A), np.uint8)
    for r in range(R):
        for a in range(A):
            if x[r, a] < 0:
                z[r, a] = rng.random() < 0.1
            elif x[r, a] != y[link[r], a]:
                z[r, a] = 1
            else:
                z[r, a] = rng.random() < 0.2
    return y, link, z


def _mix64(z):
    z = np.asarray(z, np.uint64)
    with np.errstate(over="ignore"):
        z = z + np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def state_hash_numpy(y, link, z):
    """(entities, records): the row fingerprints dbl_state_hash computes on the device, restated with numpy from host
    arrays (e.g. the ORACLE's state): sum over rows of a mixed hash of (row id, row contents), mod 2^64."""
    y = np.asarray(y)
    E, A = y.shape
    h = _mix64(np.uint64(0xE000000000000000) ^ np.arange(E, dtype=np.uint64))
    for a in range(A):
        h = _mix64(h ^ y[:, a].astype(np.uint32).astype(np.uint64))
    with np.errstate(over="ignore"):
        he = int(np.add.reduce(h, dtype=np.uint64))
    R = len(link)
    zm = np.zeros(R, np.uint64)
    for a in range(A):
        zm |= np.asarray(z)[:, a].astype(np.uint64) << np.uint64(a)
    g = _mix64(np.uint64(0xA000000000000000) ^ np.arange(R, dtype=np.uint64))
    g = _mix64(g ^ np.asarray(link).astype(np.uint32).astype(np.uint64))
    g = _mix64(g ^ zm)
    with np.errstate(over="ignore"):
        hr = int(np.add.reduce(g, dtype=np.uint64))
    return he, hr


def host_threads(cap=256):
    """CPU threads this process may really use: the scheduler affinity mask, cut by a cgroup CPU quota when there is
    one (a container that shows 128 CPUs may be allowed 8)."""
    import math
    import os

    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]  # cgroup v2
        if q != "max":
            n = min(n, max(1, math.ceil(int(q) / int(p))))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, math.ceil(q / p)))
        except Exception:
            pass
    return max(1, min(cap, n))


def tree_files(root):
    """Every file under the repository tree (but .git), with its size and mtime: taken before and after a run of
    bench.py, which must write nothing into the tree (it may be read-only where the bench runs)."""
    import os

    out = {}
    for dp, dirs, files in os.walk(root):
        dirs[:] = [d for d in dirs if d != ".git"]
        for f in files:
            st = os.stat(os.path.join(dp, f))
            out[os.path.relpath(os.path.join(dp, f), root)] = (st.st_size, st.st_mtime_ns)
    return out


def agreeing_cluster(rng, x, y, link, z, K, distorted=(), flag_rate=0.0):
    """A valid state in which records 0..K-1 all copy record 0 and link to entity 0, whose values are theirs: a
    cluster of K agreeing records, built on the state (y, link, z) of the records x.  The cluster's flags are 1 on
    the attributes in `distorted` and 0 elsewhere; every other flag is set to 1 with probability flag_rate (a valid
    change at any rate) so that the next theta draw lands near flag_rate.  -> x, y, link, z"""
    x, y, link, z = (np.array(t, copy=True) for t in (x, y, link, z))
    x[:K] = x[0]
    link[:K] = 0
    y[0] = np.where(x[0] >= 0, x[0], y[0])
    z[:K] = 0
    for a in distorted:
        z[:K, a] = 1
    z[K:] |= (rng.random(z[K:].shape) < flag_rate).astype(z.dtype)
    obs = x >= 0
    z |= (obs & (x != y[link])).astype(z.dtype)  # records of entity 0 outside the cluster
    z[:K][~obs[:K]] = 1
    return x, y, link, z
