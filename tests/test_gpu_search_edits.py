"""Edit-distance pattern search in open archives (sccg_archive_search_edits) on the B200 through the product library: the
battery of test_emu_search_edits.py, and the chr1-sized synthetic archive searched whole for four 23-nt guides that each carry
a planted 1-bp indel, with up to 2 edits on both strands, against tests/edit_probe.cpp run on candidate regions."""
import numpy as np
import pytest

import sccg_b200
from test_emu_search_edits import check_archive_set, check_contract, check_golden_search, expect_acgt, probe  # noqa: F401

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = sccg_b200.Context(0)
    yield c
    c.close()


def test_archive_set(ctx, probe):  # noqa: F811
    check_archive_set(ctx, probe)


def test_golden_cases(ctx, probe, golden):  # noqa: F811
    check_golden_search(ctx, probe, golden)


def test_contract(ctx, probe):  # noqa: F811
    ctx2 = sccg_b200.Context(0)
    try:
        check_contract(ctx, ctx2, probe)
    finally:
        ctx2.close()


def test_full_size(ctx, probe):  # noqa: F811
    from sccg_genome_compression_b200 import synth
    ref_np, tgt_np = synth.local_pair(synth.CHR1_LEN, synth.seed_for(2, 0))
    ctx.set_reference(ref_np.tobytes())
    inter, mode = ctx.compress_resident(tgt_np.tobytes())
    D = tgt_np.tobytes()
    r = np.random.default_rng(29)
    pats = []
    while len(pats) < 4:
        s = int(r.integers(0, len(D) - 30))
        w = D[s:s + 24]
        if not set(w.upper()) <= set(b"ACGT"):
            continue
        c = int(r.integers(6, 17))
        if len(pats) % 2:
            pats.append(w[:c] + w[c + 1:])                                       # one base of D deleted from the guide
        else:
            pats.append(w[:c] + bytes([b"ACGT"[int(r.integers(0, 4))]]) + w[c:22])  # one base inserted into it
    with ctx.open_archive(inter) as a:
        assert a.seq_len == len(D)
        got = ctx.search_edits([a], pats, max_edits=2)
        assert ctx.profile()["launches"] >= 3
        ham = ctx.search([a], pats, max_mismatches=2)
    exp = expect_acgt(probe, D, pats, 2)
    assert len(exp) >= 4 and all(p in set(exp[:, 3].tolist()) for p in range(4))
    assert np.array_equal(got, exp)
    # the planted occurrences: an edit hit with one edit; the Hamming search misses at least one of them
    ends = {(int(e), int(i)) for _, _, e, i, _, d in got.tolist() if d <= 1}
    ham_ends = {(int(p) + 23, int(i)) for _, p, i, _, _ in ham.tolist()}
    assert len(ends - ham_ends) >= 1
    ctx.clear_reference()
