"""An independent check of everything a sweep draws or computes besides the links: theta, the entity values, the
distortion flags, the block ids and the summary, each against the literal conditional of the reference restated in
np.longdouble.  The sibling of link_exact.py, which checks the links.

A sweep (update_owned in dblink_b200/csrc/dbl_engine.cu) runs
  1. theta ~ Beta(aggDist + alpha, fileSize - aggDist + beta) from the flags of the state it starts from (GU:305-320);
  2. the links (link_exact.py);
  3. the entity values from the NEW links and the OLD flags (GU:534-599, 605-646);
  4. the flags from the new values (GU:324-359);
  5. block ids (GU:206) and the summary of the new state (GU:219-301).
The check takes the state before and after the sweep (link_exact.snapshot) and shares with the kernels only
  * the Philox stream (uniform2 below, a numpy restatement checked against oracle.uniform2): phase THETA = 1 (through
    dbl_draw_theta), VALUE = 3 with (id, sub) = (entity, attribute), DIST = 4 with (record, attribute);
  * the orders that decide which value a uniform picks (DESIGN.md 4.3): the base distribution is inverted in
    ascending value id, the perturbation part in first-appearance order of the linked records' similarity rows.
It does not call the oracle's value or distortion routines or its sweep.

Values.  p~(v) = phi(v) prod_r [(1-theta_r)[x_r=v] + theta_r phi(x_r) n(v) E(x_r,v)] (PCG-I, PCG-II) or
phi(v) prod_r phi(x_r) n(v) E(x_r,v) over the (all distorted) records (Gibbs, Gibbs-Sequential; a record with z = 0
forces its value; a constant attribute with every record distorted draws from the prior).  The draw protocol is the
mixture p~ / D = b + W with D = prod_r theta_r phi(x_r) (or prod_r phi(x_r)), b(v) = phi(v) n(v)^k:
u0 < B / (B + sum W) picks the base b (inverse CDF at u1), otherwise W (inverse CDF at u1 sum W).  Each comparison
may fall the other way only within a rounding band around its boundary; the drawn value must have p~ > 0."""
import numpy as np

from link_exact import LD, SAMPLERS, _Attr

PH_THETA, PH_VALUE, PH_DIST = 1, 3, 4
EPS = LD(2.0) ** -53
_M32 = np.uint64(0xFFFFFFFF)


def uniform2(seed, phase, it, ids, subs):
    """(u0, u1) of the protocol's Philox4x32-10 stream (dbl_internal.h uniform2) for arrays of (id, sub), float64."""
    ids, subs = np.broadcast_arrays(np.asarray(ids, np.uint64), np.asarray(subs, np.uint64))
    c0, c1 = ids & _M32, subs & _M32
    c2 = np.full(c0.shape, np.uint64(it) & _M32)
    c3 = np.full(c0.shape, np.uint64(phase))
    k0, k1 = int(seed) & 0xFFFFFFFF, (int(seed) >> 32) & 0xFFFFFFFF
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c0
        p1 = np.uint64(0xCD9E8D57) * c2
        n0 = (p1 >> np.uint64(32)) ^ c1 ^ np.uint64(k0)
        n2 = (p0 >> np.uint64(32)) ^ c3 ^ np.uint64(k1)
        c1, c3, c0, c2 = p1 & _M32, p0 & _M32, n0, n2
        k0, k1 = (k0 + 0x9E3779B9) & 0xFFFFFFFF, (k1 + 0xBB67AE85) & 0xFFFFFFFF
    unit = lambda lo, hi: (((hi << np.uint64(32)) | lo) >> np.uint64(12)).astype(np.float64) * 2.0 ** -52 + 2.0 ** -53
    return unit(c0, c1), unit(c2, c3)


class _VAttr(_Attr):
    """_Attr plus the similarity rows in stored order and the base distributions b_k, built once per k."""

    def __init__(self, t):
        super().__init__(t)
        if not self.is_const:
            self.rowptr = np.asarray(t["rowptr"], np.int64)
            self.col = np.asarray(t["col"], np.int64)
        self._base = {}

    def support(self, xo):
        """values of the observed x's rows (a constant attribute: the x's themselves) in first-appearance order"""
        if self.is_const:
            cat = xo
        else:
            cat = np.concatenate([self.col[self.rowptr[v]:self.rowptr[v + 1]] for v in xo])
        _, first = np.unique(cat, return_index=True)
        return cat[np.sort(first)]

    def base(self, k):
        """(b, cumulative b in ascending id) of b_k(v) = phi(v) n(v)^k (k = 0 for a constant attribute)"""
        k = 0 if self.is_const else int(k)
        if k not in self._base:
            b = self.phi * self.norm ** k
            self._base[k] = (b, np.cumsum(b))
        return self._base[k]


def _inv(C, t, j, delta):
    """inverse-CDF check of position j at target t over cumulative sums C -> (ok, near, expected position)"""
    m = len(C)
    expect = min(int((C <= t).sum()), m - 1)
    ok = 0 <= j < m and (j == expect or ((C[j - 1] if j > 0 else LD(0)) - delta <= t <= C[j] + delta))
    near = abs(C[expect] - t) <= delta or (expect > 0 and abs(t - C[expect - 1]) <= delta)
    return ok, near, expect


def value_conditional(at, sampler, xo, fo, zo, theta_a, variant=None):
    """The protocol mixture of one (entity, attribute) with observed linked records xo (ascending record id), files
    fo and old flags zo -> ("forced", value) | ("base", k) | ("mix", k, support, W).
    variant (negative controls of the tests): "drop_theta_term" omits (1-theta)[x=v] (GU:557/560); "ignore_forced"
    treats every record as distorted."""
    s = SAMPLERS[sampler] if isinstance(sampler, str) else int(sampler)
    collapsed = s in (SAMPLERS["PCG-I"], SAMPLERS["PCG-II"])
    k = len(xo)
    if k == 0:
        return ("base", 0)
    if not collapsed:
        keep = np.flatnonzero(zo == 0)
        if len(keep) and variant != "ignore_forced":
            return ("forced", int(xo[keep[0]]))
        if at.is_const:
            return ("base", 0)
    sup = at.support(xo)
    phix = at.phi[xo][:, None]
    if at.is_const:
        sim = phix * np.ones((1, len(sup)), LD)
    else:
        sim = phix * at.norm[sup][None, :] * at.exp_sim(xo[:, None], sup[None, :])
    if collapsed:
        th = np.asarray(theta_a, np.float64)[fo].astype(LD)[:, None]
        eq = LD(0) if variant == "drop_theta_term" else np.where(xo[:, None] == sup[None, :], LD(1) - th, LD(0))
        ratio = np.prod((eq + th * sim) / (th * phix), axis=0)  # prod_r factor_r(v) / (theta_r phi(x_r))
    else:
        ratio = np.prod(sim / phix, axis=0)
    b, _ = at.base(k)
    W = at.phi[sup] * ratio - b[sup]  # p~(v) / D - b(v)
    return ("mix", k, sup, W)


def _pick(at, cond, u0, u1):
    """the value the extended-precision inverse CDF of a conditional picks (no rounding band)"""
    if cond[0] == "forced":
        return cond[1]
    b, Cb = at.base(cond[1])
    if cond[0] == "mix":
        sup, W = cond[2], cond[3]
        T = W.sum()
        if not u0 < Cb[-1] / (Cb[-1] + T):
            C = np.cumsum(W)
            return int(sup[min(int((C <= LD(u1) * T).sum()), len(sup) - 1)])
    return min(int((Cb <= LD(u1) * Cb[-1]).sum()), at.V - 1)


def _groups_by_entity(link, E):
    order = np.argsort(link, kind="stable")
    ptr = np.searchsorted(link[order], np.arange(E + 1))
    return order, ptr


def exact_values(before, after, tables, x, file, seed, sampler, entities=None, variant=None):
    """the values the inverse CDF of value_conditional picks -> y[E, A] (rows outside `entities` copied from after)"""
    attrs = [_VAttr(t) for t in tables]
    x, file = np.asarray(x), np.asarray(file)
    z0, link1, y1 = np.asarray(before["z"]), np.asarray(after["link"]), np.asarray(after["y"])
    theta = np.asarray(after["theta"], np.float64).reshape(len(attrs), -1)
    it = (int(before["iteration"]) + 1) & 0xFFFFFFFF
    order, ptr = _groups_by_entity(link1, len(y1))
    ents = np.arange(len(y1)) if entities is None else np.asarray(entities, np.int64)
    out = y1.copy()
    for e in ents:
        rs = order[ptr[e]:ptr[e + 1]]
        for a, at in enumerate(attrs):
            obs = rs[x[rs, a] >= 0]
            u0, u1 = uniform2(seed, PH_VALUE, it, [e], [a])
            cond = value_conditional(at, sampler, x[obs, a], file[obs], z0[obs, a], theta[a], variant)
            out[e, a] = _pick(at, cond, u0[0], u1[0])
    return out


def check_values(before, after, tables, x, file, seed, sampler, entities=None, verbose=5):
    """every y[e, a] of `after` against the protocol mixture of the literal conditional
    -> {checked, band, mismatches, overflow, bad: [(e, a)], band_cells: [(e, a)]}; overflow counts the draws whose
    binary64 sums are not finite (a product of similarity factors or sum W / B past DBL_MAX, or b_k(v) below the
    smallest double for every v)"""
    attrs = [_VAttr(t) for t in tables]
    A = len(attrs)
    x, file = np.asarray(x), np.asarray(file)
    z0, link1, y1 = np.asarray(before["z"]), np.asarray(after["link"]), np.asarray(after["y"])
    theta = np.asarray(after["theta"], np.float64).reshape(A, -1)
    it = (int(before["iteration"]) + 1) & 0xFFFFFFFF
    order, ptr = _groups_by_entity(link1, len(y1))
    ents = np.arange(len(y1)) if entities is None else np.asarray(entities, np.int64)
    U0, U1 = uniform2(seed, PH_VALUE, it, np.repeat(ents, A), np.tile(np.arange(A), len(ents)))
    res = {"checked": 0, "band": 0, "mismatches": 0, "overflow": 0, "bad": [], "band_cells": []}
    tiny, huge = LD(np.finfo(np.float64).tiny) * LD(2.0) ** -52, LD(np.finfo(np.float64).max)
    for i, e in enumerate(ents):
        rs = order[ptr[e]:ptr[e + 1]]
        for a, at in enumerate(attrs):
            u0, u1 = LD(U0[i * A + a]), LD(U1[i * A + a])
            v = int(y1[e, a])
            obs = rs[x[rs, a] >= 0]
            cond = value_conditional(at, sampler, x[obs, a], file[obs], z0[obs, a], theta[a])
            near = False
            if cond[0] == "forced":
                ok = v == cond[1]
            else:
                b, Cb = at.base(cond[1])
                B = Cb[-1]
                if cond[0] == "base":
                    rel = LD(8 * (at.V + 4)) * EPS
                    ok, near, _ = _inv(Cb, u1 * B, v, rel * B)
                else:
                    k, sup, W = cond[1], cond[2], cond[3]
                    T = W.sum()
                    if (W / b[sup]).max() + 1 > huge or T / B > huge or b.max() < tiny:
                        res["overflow"] += 1
                    lsc = float(np.max(np.abs(np.log(np.maximum(W + b[sup], LD(1e-4000))))))
                    rel = LD(8 * (at.V + len(sup) + k + 4) * (1.0 + lsc)) * EPS
                    pb = B / (B + T)
                    ok_b, near_b, _ = _inv(Cb, u1 * B, v, rel * B)
                    j = np.flatnonzero(sup == v)
                    ok_w, near_w = False, False
                    if len(j):
                        ok_w, near_w, _ = _inv(np.cumsum(W), u1 * T, int(j[0]), rel * T)
                        ok_w = ok_w and W[j[0]] > 0
                    if u0 < pb * (1 - rel):
                        ok, near = ok_b, near_b
                    elif u0 >= pb * (1 + rel):
                        ok, near = ok_w, near_w
                    else:
                        ok, near = ok_b or ok_w, True
                ok = ok and 0 <= v < at.V and at.phi[v] > 0  # p~(v) > 0: phi(v) > 0 and every factor positive
            res["checked"] += 1
            if near:
                res["band"] += 1
                res["band_cells"].append((int(e), a))
            if not ok:
                res["mismatches"] += 1
                res["bad"].append((int(e), a))
                if res["mismatches"] <= verbose:
                    print(f"value draw mismatch ({sampler}): entity {int(e)} attribute {a} drew {v}; "
                          f"{cond[0]} conditional, inverse CDF picks {_pick(at, cond, u0, u1)}, u = ({float(u0):.17g}, "
                          f"{float(u1):.17g}), {len(obs)} observed linked records")
    return res


def dist_probability(tables, x, yl, th, with_diag=True):
    """P(z = 1 | x, y) of GU:324-359 per (record, attribute), long double: theta for a missing x, 1 for x != y,
    theta phi(x) n(x) E(x,x) / (theta phi(x) n(x) E(x,x) + 1 - theta) for x = y, E(x,x) from the CSR row.
    with_diag=False omits E(x,x) (a negative control of the tests)."""
    attrs = [_VAttr(t) for t in tables]
    p = np.empty(x.shape, LD)
    for a, at in enumerate(attrs):
        xa, ya, t = x[:, a], yl[:, a], th[:, a].astype(LD)
        xs = np.maximum(xa, 0)
        pr1 = t * at.phi[xs]
        if not at.is_const:
            pr1 = pr1 * at.norm[xs] * (at.exp_sim(xs[:, None], xs[:, None])[:, 0] if with_diag else LD(1))
        pe = pr1 / (pr1 + (LD(1) - t))
        p[:, a] = np.where(xa < 0, t, np.where(xa != ya, LD(1), pe))
    return p


def exact_dist(before, after, tables, x, file, seed, with_diag=True):
    """the flags the uniforms give under dist_probability -> z[R, A] (uint8)"""
    x, file = np.asarray(x), np.asarray(file)
    R, A = x.shape
    th = np.asarray(after["theta"], np.float64).reshape(A, -1)[:, file].T
    p = dist_probability(tables, x, np.asarray(after["y"])[np.asarray(after["link"])], th, with_diag)
    it = (int(before["iteration"]) + 1) & 0xFFFFFFFF
    u0, _ = uniform2(seed, PH_DIST, it, np.repeat(np.arange(R), A), np.tile(np.arange(A), R))
    return (u0.reshape(R, A).astype(LD) < p).astype(np.uint8)


def check_dist(before, after, tables, x, file, seed, verbose=5):
    """every flag of `after` against u0 < P(z = 1) (dist_probability with the new links, values and theta); within
    16 ulp of p either flag is accepted -> {checked, band, mismatches, bad: [(r, a)]}"""
    x, file = np.asarray(x), np.asarray(file)
    R, A = x.shape
    th = np.asarray(after["theta"], np.float64).reshape(A, -1)[:, file].T
    p = dist_probability(tables, x, np.asarray(after["y"])[np.asarray(after["link"])], th)
    it = (int(before["iteration"]) + 1) & 0xFFFFFFFF
    u0, _ = uniform2(seed, PH_DIST, it, np.repeat(np.arange(R), A), np.tile(np.arange(A), R))
    u0 = u0.reshape(R, A).astype(LD)
    near = np.abs(u0 - p) <= 16 * EPS * p
    bad = ((np.asarray(after["z"]) != 0) != (u0 < p)) & ~near
    idx = np.argwhere(bad)
    for r, a in idx[:verbose]:
        print(f"distortion mismatch: record {r} attribute {a} z = {int(after['z'][r, a])}, p = {float(p[r, a]):.17g}, "
              f"u0 = {float(u0[r, a]):.17g}")
    return {"checked": R * A, "band": int(near.sum()), "mismatches": len(idx), "bad": [tuple(map(int, t)) for t in idx]}


def literal_counts(z, file, F):
    """aggDist[A, F] (flags per attribute and file, missing values included, GU:244-246) and the file sizes"""
    z, file = np.asarray(z), np.asarray(file)
    agg = np.stack([np.bincount(file, weights=z[:, a], minlength=F) for a in range(z.shape[1])]).astype(np.int64)
    return agg, np.bincount(file, minlength=F).astype(np.int64)


def draw_theta(alpha, beta, seed, agg, fs, iteration):
    """theta of the protocol (dbl_draw_theta, the host build of the device's draw_theta_one) for literal counts"""
    import ctypes as C

    from dblink_b200 import _lib

    A, F = agg.shape
    alpha, beta = np.ascontiguousarray(alpha, np.float64), np.ascontiguousarray(beta, np.float64)
    agg, fs = np.ascontiguousarray(agg, np.int64), np.ascontiguousarray(fs, np.int64)
    out = np.zeros((A, F))
    p = lambda a, t: a.ctypes.data_as(t)
    rc = _lib.load().dbl_draw_theta(A, F, p(alpha, _lib.f64p), p(beta, _lib.f64p), C.c_uint64(int(seed)),
                                    p(agg, _lib.i64p), p(fs, _lib.i64p), int(iteration), p(out, _lib.f64p))
    assert rc == 0
    return out


def check_theta(before, after, file, seed, alpha, beta):
    """theta of `after` must be the protocol's Beta draw on the literal counts of the flags of `before`
    -> (ok, expected theta)"""
    A = len(alpha)
    theta = np.asarray(after["theta"], np.float64).reshape(A, -1)
    agg, fs = literal_counts(before["z"], file, theta.shape[1])
    expect = draw_theta(alpha, beta, seed, agg, fs, int(before["iteration"]) + 1)
    return bool(np.array_equal(theta, expect)), expect


def leaf_ids(tree, y):
    """the block id of each entity row: the k-d tree walk (MutableBST.getLeafNumber) over an exported tree
    {attr, kind, split, set_ptr, set_val, leaf_no}; None = one block"""
    y = np.asarray(y)
    if tree is None:
        return np.zeros(len(y), np.int64)
    t = {k: np.asarray(tree[k] if isinstance(tree, dict) else getattr(tree, k)) for k in
         ("attr", "kind", "split", "set_ptr", "set_val", "leaf_no")}
    node = np.zeros(len(y), np.int64)
    while True:
        act = np.flatnonzero((node < len(t["attr"])) & (t["attr"][np.minimum(node, len(t["attr"]) - 1)] >= 0))
        if len(act) == 0:
            break
        nd = node[act]
        v = y[act, t["attr"][nd]]
        right = np.where(t["kind"][nd] != 0, False, v > t["split"][nd])
        for n in np.unique(nd[t["kind"][nd] != 0]):
            sel = nd == n
            right[sel] = np.isin(v[sel], t["set_val"][t["set_ptr"][n]:t["set_ptr"][n + 1]])
        node[act] = np.where(right, 2 * nd + 2, 2 * nd + 1)
    return t["leaf_no"][node].astype(np.int64)


def literal_summary(after, tables, x, file, alpha, beta):
    """updateSummaryVariables GU:219-301 of a state, long double -> {num_isolates, agg_dist, rec_dist,
    log_likelihood, abs_terms (sum of the absolute values of the terms of the log-likelihood)}"""
    attrs = [_VAttr(t) for t in tables]
    x, file = np.asarray(x), np.asarray(file)
    y, link, z = np.asarray(after["y"]), np.asarray(after["link"]), np.asarray(after["z"]) != 0
    A = len(attrs)
    theta = np.asarray(after["theta"], np.float64).reshape(A, -1)
    F = theta.shape[1]
    agg, fs = literal_counts(z.astype(np.int64), file, F)
    terms = []
    yl = y[link]
    for a, at in enumerate(attrs):
        terms.append(np.log(at.phi[y[:, a]]))  # GU:234-237, 271-274
        d = np.flatnonzero(z[:, a] & (x[:, a] >= 0))
        xa, ya = x[d, a], yl[d, a]
        pr = at.phi[xa] if at.is_const else at.phi[xa] * at.norm[ya] * at.exp_sim(xa[:, None], ya[:, None])[:, 0]
        terms.append(np.log(pr))  # GU:248-258
    th = theta.astype(LD)
    nd = agg.astype(LD)
    al = np.asarray(alpha, np.float64).astype(LD)[:, None]
    be = np.asarray(beta, np.float64).astype(LD)[:, None]
    terms.append(((al + nd - 1) * np.log(th)).ravel())  # GU:282-289
    terms.append(((be + fs.astype(LD)[None, :] - nd - 1) * np.log(LD(1) - th)).ravel())
    t = np.concatenate(terms)
    return {"num_isolates": int(len(y) - len(np.unique(link))), "agg_dist": agg,
            "rec_dist": np.bincount(z.sum(axis=1), minlength=A + 1).astype(np.int64), "log_likelihood": t.sum(),
            "abs_terms": np.abs(t).sum()}


def check_summary(summary, after, tables, x, file, alpha, beta):
    """the summary of a sweep against literal_summary of the state it left -> list of the fields that differ"""
    ref = literal_summary(after, tables, x, file, alpha, beta)
    E, R, A = len(after["y"]), len(x), len(tables)
    bad = [k for k in ("num_isolates", "agg_dist", "rec_dist") if not np.array_equal(np.asarray(summary[k]), ref[k])]
    tol = 4 * (E + R) * A * EPS * ref["abs_terms"]
    if not abs(LD(summary["log_likelihood"]) - ref["log_likelihood"]) <= tol:
        bad.append("log_likelihood")
        print(f"log-likelihood {summary['log_likelihood']!r}, literal {float(ref['log_likelihood'])!r}, "
              f"tolerance {float(tol):.3g}")
    return bad


def check_sweep(before, after, summary, tables, x, file, seed, sampler, alpha, beta, tree=None, entities=None,
                verbose=5):
    """all five checks of one sweep -> {values, dist: result dicts; theta, blocks: bool; summary: list of bad fields}
    (summary None: not checked)"""
    out = {"values": check_values(before, after, tables, x, file, seed, sampler, entities, verbose),
           "dist": check_dist(before, after, tables, x, file, seed, verbose),
           "theta": check_theta(before, after, file, seed, alpha, beta)[0],
           "blocks": bool(np.array_equal(np.asarray(after["block"]), leaf_ids(tree, after["y"])))}
    out["summary"] = [] if summary is None else check_summary(summary, after, tables, x, file, alpha, beta)
    return out


def assert_sweep_ok(out, label=""):
    v, d = out["values"], out["dist"]
    print(f"sweep_exact {label}: values {v['checked']} checked, {v['band']} in the band, {v['mismatches']} mismatches, "
          f"{v['overflow']} past binary64; flags {d['checked']} checked, {d['band']} in the band, "
          f"{d['mismatches']} mismatches; theta {'ok' if out['theta'] else 'WRONG'}, blocks "
          f"{'ok' if out['blocks'] else 'WRONG'}, summary {out['summary'] or 'ok'}")
    assert v["mismatches"] == 0, v["bad"][:10]
    assert d["mismatches"] == 0, d["bad"][:10]
    assert out["theta"] and out["blocks"] and out["summary"] == []
    assert v["band"] <= max(1, 0.005 * v["checked"]) and d["band"] <= max(1, 0.005 * d["checked"])
