"""Both archive search engines over the whole of their contract on the B200 through the product library: the battery of
test_emu_search_space.py, and 1,024 A/C/G/T 23-mers over the whole chr1-sized synthetic archive at k = 0 and 1 with both
engines: the automatic launch cut (a launch's hits must fit 32 bits), strand symmetry, case invariance and monotone k on
the whole archive, and every hit in a 5 Mbp window against a pigeonhole reference over 2-bit k-mer codes."""
import numpy as np
import pytest

import sccg_b200
from test_emu_archive import revcomp
from test_emu_search import MISS
from test_emu_search_edits import expect, probe  # noqa: F401
from test_emu_search_space import (check_counter_widths, check_every_byte, check_many_patterns, check_properties,
                                   check_window_shapes)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = sccg_b200.Context(0)
    yield c
    c.close()


def test_every_byte(ctx, probe):  # noqa: F811
    check_every_byte(ctx, probe)


def test_counter_widths(ctx, probe):  # noqa: F811
    check_counter_widths(ctx, probe)


def test_many_patterns(ctx, probe):  # noqa: F811
    check_many_patterns(ctx, probe)


def test_window_shapes(ctx, probe):  # noqa: F811
    check_window_shapes(ctx, probe)


CODE = np.full(256, 4, dtype=np.uint64)
for _i, _c in enumerate(b"ACGT"):
    CODE[_c] = CODE[_c | 0x20] = _i


def kmer_codes(D: np.ndarray, L: int) -> np.ndarray:
    """2-bit code of the L-mer at every start of D (upper-cased A/C/G/T), all ones where it holds another byte"""
    c = CODE[D]
    n = len(D) - L + 1
    k = np.zeros(n, dtype=np.uint64)
    bad = np.zeros(n, dtype=bool)
    for j in range(L):
        k = (k << np.uint64(2)) | (c[j:j + n] & np.uint64(3))
        bad |= c[j:j + n] == 4
    k[bad] = ~np.uint64(0)
    return k


def pigeonhole(D: np.ndarray, pats, k: int):
    """candidate starts of A/C/G/T patterns (both strands: pattern j of pats + their reverse complements) with at most k
    mismatches or edits: one of k + 1 disjoint parts occurs exactly, at offset a from the start c, so c = t - a for an
    occurrence at t -> (pattern j, c) arrays, unique; c may lie before 0 or end past len(D)"""
    m = len(pats[0])
    cut = [m * j // (k + 1) for j in range(k + 2)]
    pj, ps = [], []
    for a, b in zip(cut, cut[1:]):
        codes = kmer_codes(D, b - a)
        order = np.argsort(codes, kind="stable")
        srt = codes[order]
        q = np.array([sum(int(x) << (2 * (b - a - 1 - t)) for t, x in enumerate(CODE[np.frombuffer(p[a:b], dtype=np.uint8)]))
                      for p in pats], dtype=np.uint64)
        lo = np.searchsorted(srt, q, "left")
        hi = np.searchsorted(srt, q, "right")
        cnt = hi - lo
        j = np.repeat(np.arange(len(pats)), cnt)
        at = order[np.concatenate([np.arange(x, y) for x, y in zip(lo, hi)]) if cnt.sum() else np.zeros(0, np.int64)]
        pj.append(j)
        ps.append(at.astype(np.int64) - a)
    key = np.unique(np.concatenate(pj).astype(np.int64) * (1 << 40) + np.concatenate(ps) + m)
    return key >> 40, (key & ((1 << 40) - 1)) - m


def hamming_ref(D: np.ndarray, pats, k: int, base: int) -> np.ndarray:
    """every hit [0, pos, pattern, strand, mismatches] of the A/C/G/T patterns in D (positions offset by base)"""
    both = list(pats) + [revcomp(p) for p in pats]
    j, c = pigeonhole(D, both, k)
    keep = (c >= 0) & (c + len(pats[0]) <= len(D))
    j, c = j[keep], c[keep]
    P = np.frombuffer(b"".join(both), dtype=np.uint8).reshape(len(both), -1)
    mm = np.zeros(len(c), dtype=np.int64)
    for t in range(P.shape[1]):
        mm += MISS[P[j, t], D[c + t]]
    h = np.stack([np.zeros(len(c), np.int64), c + base, j % len(pats), j // len(pats), mm], axis=1)[mm <= k]
    return h[np.lexsort((h[:, 3], h[:, 2], h[:, 1], h[:, 0]))]


def edits_ref(probe, D: np.ndarray, pats, k: int, base: int) -> np.ndarray:  # noqa: F811
    """every edit hit of the A/C/G/T patterns in D (offset by base): an alignment with at most k edits leaves one of k + 1
    disjoint parts of the pattern unedited, within k bytes of its offset, so every alignment lies in [c - k, c + m + 2k) of
    a candidate start c of the pigeonhole filter; regions of one pattern (both strands) are merged and scored by the probe"""
    m = len(pats[0])
    both = list(pats) + [revcomp(p) for p in pats]
    j, c = pigeonhole(D, both, k)
    Db = D.tobytes()
    rows = []
    for i, p in enumerate(pats):
        st = np.sort(c[(j == i) | (j == i + len(pats))])
        merged = []
        for s in st.tolist():
            s0, e0 = max(0, s - k), min(len(Db), s + m + 2 * k)
            if merged and s0 <= merged[-1][1]:
                merged[-1][1] = max(merged[-1][1], e0)
            else:
                merged.append([s0, e0])
        if not merged:
            continue
        pieces = [Db[s:e] for s, e in merged]
        h = expect(probe, pieces, [(x, 0, len(y)) for x, y in enumerate(pieces)], [p], k, 3)
        off = np.array([s for s, _ in merged], dtype=np.int64)[h[:, 0]] + base
        h[:, 1] += off
        h[:, 2] += off
        h[:, 0] = 0
        h[:, 3] = i
        rows.append(h)
    h = np.concatenate(rows)
    return h[np.lexsort((h[:, 4], h[:, 3], h[:, 2], h[:, 0]))]


def test_full_size_1024(ctx, probe):  # noqa: F811
    """1,024 patterns x 2 strands: a launch takes at most 0xffffffff / 2,048 = 2,097,151 candidate positions, so the
    chr1-sized archive takes 119 launches, each a count pass and a scan, and an emit pass where it found hits"""
    from sccg_genome_compression_b200 import synth
    ref_np, tgt_np = synth.local_pair(synth.CHR1_LEN, synth.seed_for(2, 0))
    ctx.set_reference(ref_np.tobytes())
    inter, mode = ctx.compress_resident(tgt_np.tobytes())
    D = tgt_np.tobytes()
    r = np.random.default_rng(31)
    W0, W1 = 100_000_000, 105_000_000
    pats = []
    while len(pats) < 1024:
        s = int(r.integers(W0, W1 - 23)) if len(pats) % 4 else int(r.integers(0, len(D) - 23))
        p = D[s:s + 23]
        if set(p.upper()) <= set(b"ACGT"):
            pats.append(p.upper())
    n_launch = -(-len(D) // (0xffffffff // 2048))
    assert n_launch == 119
    Dw = tgt_np[W0:W1]
    with ctx.open_archive(inter) as a:
        for edits in (False, True):
            for k in (0, 1):
                got = (ctx.search_edits([a], pats, max_edits=k) if edits else ctx.search([a], pats, max_mismatches=k))
                launches = ctx.profile()["launches"]
                assert 2 * n_launch <= launches <= 3 * n_launch, (edits, k, launches)
                assert len(np.unique(got[:, 3 if edits else 2])) == 1024
                win = (ctx.search_edits([a], pats, [(0, W0, W1)], max_edits=k) if edits
                       else ctx.search([a], pats, [(0, W0, W1)], max_mismatches=k))
                exp = edits_ref(probe, Dw, pats, k, W0) if edits else hamming_ref(Dw, pats, k, W0)
                assert len(exp) >= 256 and np.array_equal(win, exp), (edits, k, len(win), len(exp))
                if edits:                                                   # ends whose alignments all start in the window
                    got, win = (h[(h[:, 2] >= W0 + 23 + k) & (h[:, 2] <= W1)] for h in (got, win))
                else:
                    got = got[(got[:, 1] >= W0) & (got[:, 1] + 23 <= W1)]
                assert np.array_equal(got, win), (edits, k)
        check_properties(ctx, [a], pats, [(0, 0, len(D))], 1)
    ctx.clear_reference()
