"""Pattern search in open archives (sccg_archive_search) on the B200 through the product library: the battery of
test_emu_search.py, and the chr1-sized synthetic archive searched whole for four 23-mers of its D with up to 2 mismatches on
both strands, against a NumPy brute force."""
import numpy as np
import pytest

import sccg_b200
from test_emu_search import MISS, check_archive_set, check_contract, check_golden_search, revcomp

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = sccg_b200.Context(0)
    yield c
    c.close()


def test_archive_set(ctx):
    check_archive_set(ctx)


def test_golden_cases(ctx, golden):
    check_golden_search(ctx, golden)


def test_contract(ctx):
    ctx2 = sccg_b200.Context(0)
    try:
        check_contract(ctx, ctx2)
    finally:
        ctx2.close()


def brute_acgt(D: bytes, patterns, k: int) -> np.ndarray:
    """every hit of A/C/G/T patterns on both strands over the whole of D: a pattern with at most k mismatches matches one of
    k + 1 disjoint parts exactly (A/C/G/T match only themselves, in either case), so every exact occurrence of a part in
    upper(D) is a candidate, and each candidate is scored with the match table"""
    U = D.upper()
    Dn = np.frombuffer(D, dtype=np.uint8)
    rows = []
    for i, p in enumerate(patterns):
        L = len(p)
        cut = [L * j // (k + 1) for j in range(k + 2)]
        for st in (0, 1):
            pp = revcomp(p) if st else p
            cand = []
            for a, b in zip(cut, cut[1:]):
                part = pp[a:b].upper()
                at = U.find(part)
                while at >= 0:
                    cand.append(at - a)
                    at = U.find(part, at + 1)
            c = np.unique(np.array(cand, dtype=np.int64))
            c = c[(c >= 0) & (c + L <= len(D))]
            mm = np.zeros(len(c), dtype=np.int16)
            for j in range(L):
                mm += MISS[pp[j]][Dn[c + j]]
            keep = mm <= k
            rows.append(np.stack([np.zeros(keep.sum(), np.int64), c[keep], np.full(keep.sum(), i), np.full(keep.sum(), st), mm[keep]], axis=1))
    h = np.concatenate(rows).astype(np.int64)
    return h[np.lexsort((h[:, 3], h[:, 2], h[:, 1], h[:, 0]))]


def test_full_size(ctx):
    from sccg_genome_compression_b200 import synth
    ref_np, tgt_np = synth.local_pair(synth.CHR1_LEN, synth.seed_for(2, 0))
    ctx.set_reference(ref_np.tobytes())
    inter, mode = ctx.compress_resident(tgt_np.tobytes())
    D = tgt_np.tobytes()
    r = np.random.default_rng(23)
    pats = []
    while len(pats) < 4:
        s = int(r.integers(0, len(D) - 23))
        p = D[s:s + 23]
        if set(p.upper()) <= set(b"ACGT"):
            pats.append(p)
    with ctx.open_archive(inter) as a:
        assert a.seq_len == len(D)
        got = ctx.search([a], pats, max_mismatches=2)
        assert ctx.profile()["launches"] >= 3
    exp = brute_acgt(D, pats, 2)
    assert len(exp) >= 4
    assert np.array_equal(got, exp)
    ctx.clear_reference()
