"""Archives (sccg_archive_open / sccg_archive_extract) on the B200 through the product library: the battery of
test_emu_archive.py, full-size archives answering W2-style queries on both strands, and a set of 20 archives with random
queries."""
import numpy as np
import pytest

import sccg_b200
from test_emu_archive import (COMP, check_argument_errors, check_complement_table, check_golden_archives, check_lifetime,
                              check_many_archives, check_no_body_line, check_reference_generation, expect)

pytestmark = pytest.mark.gpu

COMP_NP = np.frombuffer(COMP, dtype=np.uint8)


@pytest.fixture(scope="module")
def ctx():
    c = sccg_b200.Context(0)
    yield c
    c.close()


def test_golden_cases(ctx, golden):
    check_golden_archives(ctx, golden)


def test_many_archives(ctx):
    check_many_archives(ctx)


def test_lifetime(ctx):
    check_lifetime(ctx)


def test_reference_generation(ctx):
    check_reference_generation(ctx)


def test_argument_errors(ctx):
    ctx2 = sccg_b200.Context(0)
    try:
        check_argument_errors(ctx, ctx2)
    finally:
        ctx2.close()


def test_complement_table(ctx):
    check_complement_table(ctx)


def test_no_body_line(ctx):
    check_no_body_line(ctx)


def expect_np(Ds, q):
    parts = [COMP_NP[Ds[a][s:e][::-1]] if st else Ds[a][s:e] for a, s, e, st in q.tolist()]
    return np.concatenate(parts)


def w2_queries(lens, n, seed, grouped):
    r = np.random.default_rng(seed)
    ks = r.integers(0, len(lens), n)
    if grouped:
        ks.sort()
    st = (r.random(n) * (np.asarray(lens)[ks] - 150)).astype(np.int64)
    return np.ascontiguousarray(np.stack([ks, st, st + 150, r.integers(0, 2, n)], axis=1).astype(np.int64))


def test_full_size(ctx):
    """the chr1-sized local-mode archive and a global-mode archive against the same reference open together, and the
    chr19-shaped gap archive (BASELINE cfg 1) on a second context: 200,000 x 150 bp queries on both strands"""
    from sccg_genome_compression_b200 import synth
    ref_np, tgt_np = synth.local_pair(synth.CHR1_LEN, synth.seed_for(2, 0))
    g = ref_np.copy()
    synth.substitute(np.random.default_rng(3), g, 0.001)
    g = np.concatenate([g[:10_000], g[15_000:]])
    ctx.set_reference(ref_np.tobytes())
    archives, Ds = [], []
    for t, mode in ((tgt_np, 0), (g, 1)):
        inter, m = ctx.compress_resident(t.tobytes())
        assert m == mode
        a = ctx.open_archive(inter)
        assert a.mode == mode and a.seq_len == t.size
        archives.append(a); Ds.append(t)
    gref, gtgt = synth.global_gap_pair(63_811_651, 59_128_983, synth.seed_for(1, 0))
    ctx2 = sccg_b200.Context(0)
    try:
        ctx2.set_reference(gref.tobytes())
        inter, m = ctx2.compress_resident(gtgt.tobytes())
        G = ctx2.open_archive(inter)
        assert G.mode == 1 and m == 1
        for grouped in (True, False):
            q = w2_queries([D.size for D in Ds], 200_000, 11, grouped)
            got = np.frombuffer(ctx.query(archives, q), dtype=np.uint8)
            assert np.array_equal(got, expect_np(Ds, q))
            q = w2_queries([gtgt.size], 200_000, 12, grouped)
            got = np.frombuffer(ctx2.query([G], q), dtype=np.uint8)
            assert np.array_equal(got, expect_np([gtgt], q))
        whole = np.array([[0, 0, Ds[0].size, 1], [1, 0, Ds[1].size, 0]], dtype=np.int64)
        assert np.array_equal(np.frombuffer(ctx.query(archives, whole), dtype=np.uint8), expect_np(Ds, whole))
        G.close()
    finally:
        ctx2.close()
    for a in archives:
        a.close()
    ctx.clear_reference()


def test_twenty_archives(ctx):
    from sccg_genome_compression_b200 import synth
    ref_np, _ = synth.local_pair(2_000_000, synth.seed_for(4, 9))
    ctx.set_reference(ref_np.tobytes())
    archives, Ds = [], []
    for i in range(20):
        rng = np.random.default_rng(100 + i)
        t = ref_np.copy()
        synth.substitute(rng, t, 0.002)
        t = synth.compensated_indels(rng, t, 40)
        synth.lowercase_runs(rng, t, 0.3)
        if i % 5 == 4:
            t = np.concatenate([t[:2000], t[7000:]])                       # global mode
        inter, _ = ctx.compress_resident(t.tobytes())
        archives.append(ctx.open_archive(inter)); Ds.append(t)
    assert {a.mode for a in archives} == {0, 1}
    r = np.random.default_rng(5)
    for n, maxlen in ((50_000, 3), (20_000, 400), (300, 30_000)):
        ks = r.integers(0, 20, n)
        lens = np.array([D.size for D in Ds])[ks]
        st = (r.random(n) * lens).astype(np.int64)
        en = np.minimum(lens, st + r.integers(0, maxlen, n))
        q = np.ascontiguousarray(np.stack([ks, st, en, r.integers(0, 2, n)], axis=1).astype(np.int64))
        got = np.frombuffer(ctx.query(archives, q), dtype=np.uint8)
        assert np.array_equal(got, expect_np(Ds, q))
    assert ctx.query(archives, q[:50]) == expect([D.tobytes() for D in Ds], q[:50].tolist())
    for a in archives:
        a.close()
    ctx.clear_reference()
