"""An independent check of the link draws of a sweep: an extended-precision inverse CDF of the literal conditional.

Every link kernel, whatever its internals, draws the new link of record r by inverse CDF:
  * the candidates are the entities of the record's block (the block of its current link) in ascending id; the
    cumulative sums run over them in the draw order of DESIGN.md 4.2: chunk (a chunk is ceil(tiles/32) tiles of 128
    candidates), then lane (position mod 32), then step (position div 32).  That order is a fixed permutation of the
    candidates, independent of the weights and of the uniform, so any such order draws from the same categorical;
    it is the one piece of the kernels' protocol this check takes over, because it decides WHICH entity a uniform
    picks;
  * the weights are updateEntityIdCollapsed GU:363-395 (PCG-II) or updateEntityIdSeq GU:434-466 (PCG-I, Gibbs,
    Gibbs-Sequential), up to a constant factor per record;
  * the uniform is u0 of uniform2(seed, PH_LINK, iteration + 1, r, 0).
So the state before a sweep and theta after it (k_theta runs first in a sweep, before the link update) determine the
drawn entity, except where u0 * total lies within rounding distance of a boundary of the cumulative sums.

This module restates the weights from the attribute tables (phi, norm, CSR similarity rows) in np.longdouble and
shares nothing with the kernels or with the oracle's sweep but the Philox stream (oracle.uniform2, pinned by the
known-answer vectors).  It does not call the oracle's link weights.
"""
import numpy as np

PH_LINK = 2
SAMPLERS = {"PCG-I": 0, "PCG-II": 1, "Gibbs": 2, "Gibbs-Sequential": 3}
LD = np.longdouble
_MAX_PAIRS = 1 << 21  # (record, candidate) pairs scored at once


def tables_of(indexes):
    """Per attribute {phi, norm, rowptr, col, expsim, is_const} from product AttributeIndex objects (their tables()) or
    from oracle.Index objects; the two are bit-identical (tests/test_oracle_golden.py, test_abi_and_host.py)."""
    out = []
    for ix in indexes:
        if hasattr(ix, "tables"):
            t = dict(ix.tables())
            t["is_const"] = bool(ix.is_constant)
        else:
            t = {"phi": ix.phi, "norm": ix.norm, "rowptr": ix.rowptr, "col": ix.col, "expsim": ix.expsim,
                 "is_const": bool(ix.is_const)}
        out.append(t)
    return out


def snapshot(obj):
    """{link, y, z, block, theta, iteration} of a GibbsEngine or of an oracle State."""
    if hasattr(obj, "download_state"):
        d = obj.download_state()
        d["iteration"] = obj.iteration
        return d
    return {"link": obj.link, "y": obj.y, "z": obj.z, "block": obj.block, "theta": obj.theta,
            "iteration": obj.iteration}


class _Attr:
    def __init__(self, t):
        self.is_const = bool(t["is_const"])
        self.phi = np.asarray(t["phi"], np.float64).astype(LD)
        self.norm = np.asarray(t["norm"], np.float64).astype(LD)
        self.V = len(self.phi)
        if not self.is_const:
            rowptr = np.asarray(t["rowptr"], np.int64)
            col = np.asarray(t["col"], np.int64)
            row = np.repeat(np.arange(self.V, dtype=np.int64), np.diff(rowptr))
            keys = row * self.V + col
            order = np.argsort(keys, kind="stable")
            self.keys = keys[order]
            self.vals = np.asarray(t["expsim"], np.float64)[order].astype(LD)

    def exp_sim(self, xv, yv):
        """E(x, y) of AttributeIndex.expSimOf: the CSR entry of (x, y), 1 when y is not in x's row.  xv[n, 1], yv[1, m]."""
        keys = np.maximum(xv, 0).astype(np.int64) * self.V + yv.astype(np.int64)
        if len(self.keys) == 0:
            return np.ones(keys.shape, LD)
        i = np.minimum(np.searchsorted(self.keys, keys), len(self.keys) - 1)
        return np.where(self.keys[i] == keys, self.vals[i], LD(1))


def literal_weights(attrs, sampler, xr, fr, zr, ycand, theta, missing_norm=True):
    """Weights [n, m] of n records (x rows xr, files fr, flags zr) for m candidates (value rows ycand), np.longdouble.

    PCG-II (GU:363-395): prod over observed attributes of [x==y](1-theta) + theta*phi(x) (constant) or
    + theta*phi(x)*n(y)*E(x,y) (non-constant).
    PCG-I / Gibbs / Gibbs-Sequential (GU:434-466): 0 unless every observed attribute with z = 0 agrees; otherwise the
    product over observed distorted attributes of phi(x) (constant) or phi(x)*n(y)*E(x,y) (non-constant).
    missing_norm=False multiplies the PCG-II weight by n(y) of every missing non-constant attribute: what a kernel
    that skipped the 1/n(y) factor of its protocol form would draw from (a negative control of the tests)."""
    n, m = xr.shape[0], ycand.shape[0]
    s = SAMPLERS[sampler] if isinstance(sampler, str) else int(sampler)
    w = np.ones((n, m), LD)
    for a, at in enumerate(attrs):
        xa = xr[:, a][:, None]
        ya = ycand[:, a][None, :]
        obs = xa >= 0
        phi = np.where(obs, at.phi[np.maximum(xa, 0)], LD(0))
        if at.is_const:
            sim = phi
        else:
            sim = phi * at.norm[ya] * at.exp_sim(xa, ya)
        eq = xa == ya
        if s == SAMPLERS["PCG-II"]:
            th = np.asarray(theta[a], np.float64)[fr].astype(LD)[:, None]
            f = np.where(eq, LD(1) - th, LD(0)) + th * sim
            w *= np.where(obs, f, LD(1))
            if not missing_norm and not at.is_const:
                w *= np.where(obs, LD(1), at.norm[ya])
        else:
            must = obs & (zr[:, a][:, None] == 0)
            w *= np.where(must, eq.astype(LD), np.where(obs, sim, LD(1)))
    return w


def draw_order(m):
    """Positions 0..m-1 of a block's candidates in the order their weights are accumulated (DESIGN.md 4.2)."""
    j = np.arange(m)
    ntiles = (m + 127) // 128
    tpc = max(1, (ntiles + 31) // 32)
    return np.lexsort((j // 32, j % 32, j // (128 * tpc)))


def _groups(before, recs):
    """(block, candidates in ascending id, records of recs whose current link is in that block), block by block."""
    block = np.asarray(before["block"])
    rblk = block[np.asarray(before["link"])[recs]]
    ent_order = np.argsort(block, kind="stable")
    bptr = np.searchsorted(block[ent_order], np.arange(block.max() + 2))
    for b in np.unique(rblk):
        yield int(b), ent_order[bptr[b]:bptr[b + 1]], recs[rblk == b]


def exact_draws(before, theta, tables, x, file, seed, sampler, records=None, missing_norm=True):
    """The links the inverse CDF of literal_weights picks, in extended precision -> {record id: entity id}.  With
    missing_norm=False: the draws of a kernel that drops the 1/n(y) factor of missing non-constant attributes."""
    from oracle import oracle as O

    attrs = [_Attr(t) for t in tables]
    theta = np.asarray(theta, np.float64).reshape(len(attrs), -1)
    it = (int(before["iteration"]) + 1) & 0xFFFFFFFF
    recs = np.arange(len(x)) if records is None else np.unique(np.asarray(records, np.int64))
    out = {}
    for b, cand, rs in _groups(before, recs):
        w = literal_weights(attrs, sampler, np.asarray(x)[rs], np.asarray(file)[rs], np.asarray(before["z"])[rs],
                            np.asarray(before["y"])[cand], theta, missing_norm)
        order = draw_order(len(cand))
        C = np.cumsum(w[:, order], axis=1)
        u0 = np.array([O.uniform2(seed, PH_LINK, it, int(r), 0)[0] for r in rs], np.float64).astype(LD)
        j = np.minimum((C <= (u0 * C[:, -1])[:, None]).sum(axis=1), len(cand) - 1)
        out.update(zip(rs.tolist(), cand[order[j]].tolist()))
    return out


def check_link_draws(before, after, tables, x, file, seed, sampler, records=None, verbose=5):
    """Check the links of `after` against the inverse CDF of the literal link conditional of `before`.

    before: {link, y, z, block, iteration} of the state the sweep started from (links, values, flags, block ids);
    after: {link, theta} of the state it produced (theta is drawn first in a sweep, the link update uses it);
    tables: tables_of(indexes); x[R, A], file[R]: the records; records: the record ids to check (default all).

    The drawn position j must satisfy C[j-1] <= t < C[j] with C the cumulative weights over the candidates in draw
    order (draw_order) and t = u0 * C[-1], both in extended precision; only within delta = 4 (m + A) 2^-53 C[-1] of a
    boundary may the pick be the other side of it (the rounding of a kernel's binary64 weights and sums).  The drawn
    entity must always have a weight > 0.
    -> {checked, band, mismatches, bad: [record ids], band_records: [record ids]}"""
    from oracle import oracle as O

    assert np.finfo(LD).nmant >= 63, "np.longdouble is not an extended-precision type on this platform"
    attrs = [_Attr(t) for t in tables]
    A = len(attrs)
    x = np.asarray(x)
    file = np.asarray(file)
    y = np.asarray(before["y"])
    z = np.asarray(before["z"])
    it = (int(before["iteration"]) + 1) & 0xFFFFFFFF
    link1 = np.asarray(after["link"])
    theta = np.asarray(after["theta"], np.float64).reshape(A, -1)
    recs = np.arange(x.shape[0]) if records is None else np.unique(np.asarray(records, np.int64))
    res = {"checked": 0, "band": 0, "mismatches": 0, "bad": [], "band_records": []}
    eps = LD(2.0) ** -53
    for b, cand, rb in _groups(before, recs):
        m = len(cand)
        order = draw_order(m)
        rank = np.empty(m, np.int64)
        rank[order] = np.arange(m)  # place of a candidate position in the draw order
        yc = y[cand[order]]
        step = max(1, _MAX_PAIRS // max(m, 1))
        for i0 in range(0, len(rb), step):
            rs = rb[i0:i0 + step]
            w = literal_weights(attrs, sampler, x[rs], file[rs], z[rs], yc, theta)
            C = np.cumsum(w, axis=1)
            T = C[:, -1]
            u0 = np.array([O.uniform2(seed, PH_LINK, it, int(r), 0)[0] for r in rs], np.float64).astype(LD)
            t = u0 * T
            delta = LD(4 * (m + A)) * eps * T
            expect = (C <= t[:, None]).sum(axis=1)  # first position whose cumulative weight exceeds t
            j = np.minimum(np.searchsorted(cand, link1[rs]), m - 1)
            is_cand = cand[j] == link1[rs]
            pos = rank[j]  # place of the drawn entity in the draw order
            rows = np.arange(len(rs))
            lo = np.where(pos > 0, C[rows, np.maximum(pos - 1, 0)], LD(0))
            hi = C[rows, pos]
            wpos = w[rows, pos]
            ok = is_cand & (wpos > 0) & (T > 0) & np.isfinite(T)
            ok &= (pos == expect) | ((lo - delta <= t) & (t <= hi + delta))
            ec = np.minimum(expect, m - 1)
            near = (np.abs(C[rows, ec] - t) <= delta) | ((ec > 0) & (np.abs(t - C[rows, np.maximum(ec - 1, 0)]) <= delta))
            res["checked"] += len(rs)
            res["band"] += int(near.sum())
            res["band_records"] += rs[near].tolist()
            for k in np.flatnonzero(~ok):
                res["mismatches"] += 1
                res["bad"].append(int(rs[k]))
                if res["mismatches"] <= verbose:
                    print(f"link draw mismatch ({sampler}): record {int(rs[k])} block {int(b)} drew entity "
                          f"{int(link1[rs[k]])} (draw-order place {int(pos[k]) if is_cand[k] else 'none'} of {m}, "
                          f"weight {float(wpos[k]):.6g}); the inverse CDF gives place {int(expect[k])}, "
                          f"t/T = {float(u0[k]):.17g}, T = {float(T[k]):.6g}")
    return res
