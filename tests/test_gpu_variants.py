"""Variant records of open archives (sccg_archive_variants) on the B200 through the product library: the battery of
test_emu_variants.py, the chr1-sized synthetic archive whole (splice check against the target itself, equality with the
reference implementation, record counts by kind), a full-size global-mode gap pair shaped like BASELINE config 1, and a
65-archive call against per-archive calls."""
import numpy as np
import pytest

import sccg_b200
import variants_lib as vl
from test_emu_variants import (check_argument_errors, check_caps, check_global, check_golden, check_hand_files, check_repeats,
                               check_substitutions_only, check_uncompensated, check_windows, first_difference)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = sccg_b200.Context(0)
    yield c
    c.close()


def test_battery(ctx, golden):
    check_golden(ctx, golden)
    check_substitutions_only(ctx, 400_000)
    check_uncompensated(ctx, 300_000)
    check_repeats(ctx)
    check_hand_files(ctx)
    check_global(ctx)
    check_windows(ctx, 400_000, rounds=5)
    check_caps(ctx)
    ctx2 = sccg_b200.Context(0)
    try:
        check_argument_errors(ctx, ctx2)
    finally:
        ctx2.close()


def whole_against_reference(ctx, ref: bytes, tgt: bytes, want_mode: int) -> np.ndarray:
    ctx.set_reference(ref)
    inter, mode = ctx.compress_resident(tgt)
    assert mode == want_mode
    D = vl.decoded(ref, inter)
    assert D == tgt
    with ctx.open_archive(inter) as a:
        rec, alt = ctx.variants([a])
        assert ctx.variants([a], count_only=True) == (len(rec), len(alt))
    vl.check_invariants(ref, tgt, rec, alt)                               # splices into up(R) to give the target itself
    exp = vl.variants_whole(ref, inter, D)
    assert np.array_equal(rec[:, 1:5], exp), first_difference(rec[:, 1:5], exp)
    ctx.clear_reference()
    return rec


def test_chr1_whole(ctx):
    from sccg_genome_compression_b200 import synth
    ref_np, tgt_np = synth.local_pair(synth.CHR1_LEN, synth.seed_for(2, 0))
    rec = whole_against_reference(ctx, ref_np.tobytes(), tgt_np.tobytes(), 0)
    k = vl.kinds(rec)
    print("chr1-sized archive:", len(rec), "records", k)
    assert k["substitution"] > 200_000 and k["insertion"] > 0 and k["deletion"] > 0


def test_global_gap_full_size(ctx):
    from sccg_genome_compression_b200 import synth
    ref_np, tgt_np = synth.global_gap_pair(63_811_651, 59_128_983, synth.seed_for(1, 0))
    rec = whole_against_reference(ctx, ref_np.tobytes(), tgt_np.tobytes(), 1)
    k = vl.kinds(rec)
    print("cfg-1-shaped global gap pair:", len(rec), "records", k)
    assert k["deletion"] >= 4                                              # the resized N gaps


def cohort(n_ref: int = 4_000_000, k: int = 64):
    """64 local-mode individuals and one global-mode one (an uncompensated 5 kb deletion near the start) of one reference"""
    from sccg_genome_compression_b200 import synth
    ref_np, _ = synth.local_pair(n_ref, synth.seed_for(4, 0))
    out = []
    for i in range(k):
        rng = np.random.default_rng(synth.seed_for(4, i))
        t = ref_np.copy()
        synth.substitute(rng, t, 0.001)
        t = synth.compensated_indels(rng, t, int(t.size * 20e-6))
        synth.lowercase_runs(rng, t)
        out.append(t)
    rng = np.random.default_rng(synth.seed_for(4, 255))
    g = ref_np.copy()
    synth.substitute(rng, g, 0.001)
    out.append(np.concatenate([g[:10_000], g[15_000:]]))
    return ref_np, out


def test_cohort_one_call(ctx):
    ref_np, tgts = cohort()
    ref = ref_np.tobytes()
    ctx.set_reference(ref)
    arch = []
    for t in tgts:
        inter, _ = ctx.compress_resident(t.tobytes())
        arch.append(ctx.open_archive(inter))
    assert arch[-1].mode == 1 and all(a.mode == 0 for a in arch[:-1])
    rec, alt = ctx.variants(arch)
    n = 0
    for k, a in enumerate(arch):
        r1, a1 = ctx.variants([a])
        mine = rec[rec[:, 0] == k]
        assert np.array_equal(mine[:, 1:5], r1[:, 1:5]), k
        assert b"".join(alt[o:o + e - s] for o, s, e in mine[:, [5, 3, 4]].tolist()) == a1
        vl.check_invariants(ref, tgts[k].tobytes(), r1, a1)
        n += len(r1)
    assert n == len(rec)
    g0 = 2_000_000                                                          # one 10 kb window across the 65 archives
    w = [(k, g0, g0 + 10_000) for k in range(len(arch))]
    rw, aw = ctx.variants(arch, w)
    exp, exp_alt = vl.filter_windows([rec[rec[:, 0] == k][:, 1:5] for k in range(len(arch))], [t.tobytes() for t in tgts], w, len(ref))
    assert np.array_equal(rw, exp) and aw == exp_alt
    for a in arch:
        a.close()
    ctx.clear_reference()
