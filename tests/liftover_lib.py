"""Reference implementations of sccg_archive_liftover (include/sccg.h) for the tests, on the whole-archive records of
variants_lib.variants_whole.  Two independent ones: `Brute` builds the owner of every target base and reads the answer off
it (small cases), `lift` is the closed form with numpy searchsorted (any size); `check_small` cross-checks them.
`check_splice` is the splice identity of the header.  A row is [start, end, same, subst, records, flags]; a query
[archive, start, end, from]."""
import numpy as np

import variants_lib as vl

START_INSIDE, END_INSIDE, LENGTH_CHANGE = 1, 2, 4


def side(recs: np.ndarray, rlen: int, dlen: int, frm: int):
    """(records as (k, ke, o, oe): source span, target span; len(source), len(target)) for direction frm"""
    recs = np.asarray(recs, dtype=np.int64).reshape(-1, 4)
    return (recs[:, [2, 3, 0, 1]], dlen, rlen) if frm else (recs, rlen, dlen)


class Brute:
    """queries of one archive and direction by ownership: owner[i] is the source base aligned with target base i, or the
    key of the record that owns it; inside / sub mark the source bases inside records / substitution records"""

    def __init__(self, recs: np.ndarray, rlen: int, dlen: int, frm: int):
        self.R, self.ls, lt = side(recs, rlen, dlen, frm)
        owner, pe = [], 0
        for k, ke, o, oe in self.R.tolist():
            owner += list(range(pe, k)) + [k] * (oe - o)
            pe = ke
        owner += list(range(pe, self.ls))
        assert len(owner) == lt
        self.owner = np.array(owner, dtype=np.int64)
        self.inside = np.zeros(self.ls, dtype=bool)
        self.sub = np.zeros(self.ls, dtype=bool)
        for k, ke, o, oe in self.R.tolist():
            self.inside[k:ke] = True
            self.sub[k:ke] = ke - k == oe - o

    def __call__(self, s: int, e: int) -> list:
        hi = e + 1 if e == self.ls else e                                 # the len rule, at the end only
        idx = np.flatnonzero((self.owner >= s) & (self.owner < hi))
        start, end = (int(idx[0]), int(idx[-1]) + 1) if len(idx) else (int((self.owner < s).sum()),) * 2
        same = int((~self.inside[s:e]).sum())
        subst = int(self.sub[s:e].sum())
        R = self.R
        owned = R[(R[:, 0] >= s) & (R[:, 0] < hi)] if len(R) else R
        flags = 0
        if len(R) and ((R[:, 0] < s) & (R[:, 1] > s)).any():
            flags |= START_INSIDE
        if len(owned) and (owned[:, 1] > e).any():
            flags |= END_INSIDE
        if len(owned) and (owned[:, 1] - owned[:, 0] != owned[:, 3] - owned[:, 2]).any():
            flags |= LENGTH_CHANGE
        return [start, end, same, subst, len(owned), flags]


def lift(recs: np.ndarray, rlen: int, dlen: int, s, e, frm: int) -> np.ndarray:
    """queries [s, e) of one archive in one direction by the closed form -> (n, 6) rows"""
    R, ls, lt = side(recs, rlen, dlen, frm)
    s, e = np.asarray(s, dtype=np.int64), np.asarray(e, dtype=np.int64)
    k, ke, o, oe = R[:, 0], R[:, 1], R[:, 2], R[:, 3]
    is_sub = ke - k == oe - o
    pk = np.concatenate([[0], np.cumsum(ke - k)])
    ps = np.concatenate([[0], np.cumsum(np.where(is_sub, ke - k, 0))])
    pn = np.concatenate([[0], np.cumsum(~is_sub)])
    js = np.searchsorted(k, s, "left") - 1                                # last record with key < s
    je = np.searchsorted(k, np.where(e == ls, e + 1, e), "left") - 1
    jsc, jec = np.maximum(js, 0), np.maximum(je, 0)

    def at(a, j):
        return a[j] if len(a) else np.zeros_like(j)

    def F(j, jc, b):
        return np.where(j < 0, b, at(oe, jc) + np.maximum(0, b - at(ke, jc)))

    def inside(j, jc, b, pref, sub_only):
        part = np.minimum(b, at(ke, jc)) - at(k, jc)
        if sub_only:
            part = np.where(at(is_sub, jc), part, 0)
        return np.where(j < 0, 0, pref[jc] + part)
    start = F(js, jsc, s)
    end = np.where(e == ls, lt, F(je, jec, e))
    same = (e - s) - (inside(je, jec, e, pk, False) - inside(js, jsc, s, pk, False))
    subst = inside(je, jec, e, ps, True) - inside(js, jsc, s, ps, True)
    flags = np.where((js >= 0) & (at(ke, jsc) > s), START_INSIDE, 0)
    flags |= np.where((je > js) & (at(ke, jec) > e), END_INSIDE, 0)
    flags |= np.where(pn[je + 1] != pn[js + 1], LENGTH_CHANGE, 0)
    return np.stack([start, end, same, subst, je - js, flags], axis=1).astype(np.int64).reshape(-1, 6)


def lift_queries(wholes: list, rlen: int, dlens: list, queries) -> np.ndarray:
    """rows of any queries [archive, start, end, from] over archives with whole-archive records wholes[a]"""
    q = np.asarray(queries, dtype=np.int64).reshape(-1, 4)
    out = np.zeros((len(q), 6), dtype=np.int64)
    for a in np.unique(q[:, 0]) if len(q) else []:
        for frm in (0, 1):
            m = (q[:, 0] == a) & (q[:, 3] == frm)
            if m.any():
                out[m] = lift(wholes[a], rlen, dlens[a], q[m, 1], q[m, 2], frm)
    return out


def check_splice(R: bytes, D: bytes, recs: np.ndarray, s: int, e: int, frm: int, row) -> None:
    """the splice identity: the target piece up(T[start:end]) equals up(S[s:e]) with every owned record's source span
    replaced by its target span (taken whole past e) and the source bases inside a record that begins before s dropped"""
    Rr, ls, _ = side(recs, len(R), len(D), frm)
    S, T = (D, R) if frm else (R, D)
    hi = e + 1 if e == ls else e
    lo_r = max(int(np.searchsorted(Rr[:, 0], s, "left")) - 1, 0)         # the last record before s, then the owned ones
    hi_r = int(np.searchsorted(Rr[:, 0], hi, "left"))
    parts, cur = [], s
    for k, ke, o, oe in Rr[lo_r:hi_r].tolist():
        if k < s < ke:
            cur = ke
        if s <= k < hi:
            parts.append(S[cur:k] if cur < k else b"")
            parts.append(T[o:oe])
            cur = max(cur, ke)
    if cur < e:
        parts.append(S[cur:e])
    assert vl.up(T[row[0]:row[1]]) == vl.up(b"".join(parts)), (frm, s, e, list(row))


def boundary_queries(ls: int, rng, n_random: int = 200) -> list:
    """every [b, b) and [b, b + 1), plus random intervals, of a source of length ls"""
    q = [(b, b) for b in range(ls + 1)] + [(b, b + 1) for b in range(ls)]
    for _ in range(n_random):
        s = int(rng.integers(0, ls + 1))
        q.append((s, int(rng.integers(s, ls + 1))))
    return q


def check_small(recs: np.ndarray, R: bytes, D: bytes, rows, queries) -> None:
    """device rows of queries [s, e, from] (one archive) against both references and the splice identity"""
    q = np.asarray(queries, dtype=np.int64).reshape(-1, 3)
    rows = np.asarray(rows).reshape(-1, 6)
    for frm in (0, 1):
        m = q[:, 2] == frm
        if not m.any():
            continue
        exp = lift(recs, len(R), len(D), q[m, 0], q[m, 1], frm)
        assert np.array_equal(rows[m], exp), first_difference(rows[m], exp, q[m])
    brute = [Brute(recs, len(R), len(D), frm) for frm in (0, 1)]
    for (s, e, frm), row in zip(q.tolist(), rows.tolist()):
        assert brute[frm](s, e) == row, (s, e, frm, row, brute[frm](s, e))
        check_splice(R, D, recs, s, e, frm, row)


def first_difference(got, exp, q) -> str:
    for i in range(min(len(got), len(exp))):
        if not np.array_equal(got[i], exp[i]):
            return f"query {q[i].tolist()}: got {got[i].tolist()}, expected {exp[i].tolist()}"
    return f"{len(got)} rows, expected {len(exp)}"
