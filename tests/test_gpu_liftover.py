"""Coordinates lifted between the reference and open archives (sccg_archive_liftover) on the B200 through the product
library: the battery of test_emu_liftover.py, the chr1-sized synthetic archive with 200,000 random intervals in each
direction against the closed form of tests/liftover_lib.py (plus record counts against sccg_archive_variants and the splice
identity on a sample), and the 65-archive cohort of tools/archive_bench.py in one call."""
import sys
from pathlib import Path

import numpy as np
import pytest

import liftover_lib as ll
import sccg_b200
import variants_lib as vl
from test_emu_liftover import (check_argument_errors, check_global, check_golden, check_hand_files, check_lifecycle,
                               check_synthetic)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = sccg_b200.Context(0)
    yield c
    c.close()


def test_battery(ctx, golden):
    check_golden(ctx, golden)
    check_synthetic(ctx)
    check_hand_files(ctx)
    check_global(ctx)
    check_lifecycle(ctx, lambda: sccg_b200.Context(0))
    ctx2 = sccg_b200.Context(0)
    try:
        check_argument_errors(ctx, ctx2)
    finally:
        ctx2.close()


def random_intervals(rng, ls: int, n: int) -> tuple:
    s = rng.integers(0, ls + 1, size=n)
    e = np.minimum(ls, s + rng.choice([0, 1, 150, 5_000, 100_000], size=n))
    s[:4], e[:4] = [0, 0, ls, ls - 1], [0, ls, ls, ls]
    return s, e


def test_chr1(ctx):
    from sccg_genome_compression_b200 import synth
    ref_np, tgt_np = synth.local_pair(synth.CHR1_LEN, synth.seed_for(2, 0))
    ref, tgt = ref_np.tobytes(), tgt_np.tobytes()
    ctx.set_reference(ref)
    inter, mode = ctx.compress_resident(tgt)
    assert mode == 0
    D = vl.decoded(ref, inter)
    assert D == tgt
    recs = vl.variants_whole(ref, inter, D)
    rng = np.random.default_rng(5)
    with ctx.open_archive(inter) as a:
        before = a.device_bytes
        q = []
        for frm, ls in ((0, len(ref)), (1, len(D))):
            s, e = random_intervals(rng, ls, 200_000)
            q.append(np.stack([np.zeros_like(s), s, e, np.full_like(s, frm)], axis=1))
        q = np.concatenate(q)
        rows = ctx.liftover([a], q)
        build = ctx.profile()
        assert a.device_bytes == before + 4 * (8 * len(recs) + 4)
        exp = ll.lift_queries([recs], len(ref), [len(D)], q)
        assert np.array_equal(rows, exp), ll.first_difference(rows, exp, q)
        again = ctx.liftover([a], q)
        p = ctx.profile()
        assert np.array_equal(again, rows) and p["launches"] == 1
        print("chr1-sized archive:", len(recs), "records; first call kernels_ms", build["kernels_ms"], "gather_ms", build["gather_ms"],
              "launches", build["launches"], "; second call gather_ms", p["gather_ms"])
        w = q[q[:, 3] == 0][:3000, :3]
        rec, _ = ctx.variants([a], w)
        assert np.array_equal(np.bincount(rec[:, 0], minlength=len(w)), rows[:3000, 4])
        for i in rng.choice(len(q), 300, replace=False).tolist():
            ll.check_splice(ref, D, recs, int(q[i, 1]), int(q[i, 2]), int(q[i, 3]), rows[i])
    ctx.clear_reference()


def test_cohort_one_call(ctx):
    sys.path.insert(0, str(Path(__file__).resolve().parent.parent / "tools"))
    from archive_bench import individuals
    from sccg_genome_compression_b200 import synth
    ref_np, _ = synth.local_pair(50_000_000, synth.seed_for(4, 0))
    ref = ref_np.tobytes()
    tgts = individuals(ref_np, 64)
    ctx.set_reference(ref)
    arch = []
    for t in tgts:
        inter, _ = ctx.compress_resident(t.tobytes())
        arch.append(ctx.open_archive(inter))
    assert arch[-1].mode == 1 and all(a.mode == 0 for a in arch[:-1])
    rec, alt = ctx.variants(arch)
    wholes = [rec[rec[:, 0] == k][:, 1:5] for k in range(len(arch))]
    dlens = [len(t) for t in tgts]
    rng = np.random.default_rng(9)
    n = 20_000
    k = rng.integers(0, len(arch), size=n)
    frm = rng.integers(0, 2, size=n)
    ls = np.where(frm == 1, np.array(dlens)[k], len(ref))
    s = (rng.random(n) * ls).astype(np.int64)
    e = np.minimum(ls, s + rng.integers(1_000, 100_000, size=n))
    q = np.stack([k, s, e, frm], axis=1)
    rows = ctx.liftover(arch, q)
    exp = ll.lift_queries(wholes, len(ref), dlens, q)
    assert np.array_equal(rows, exp), ll.first_difference(rows, exp, q)
    assert np.array_equal(ctx.liftover(arch, q), rows) and ctx.profile()["launches"] == 1
    # the same region lifted into every archive and extracted equals the per-archive slices of D
    g = [(j, 20_000_000, 20_010_000, 0) for j in range(len(arch))]
    lifted = ctx.liftover(arch, g)
    got = ctx.query(arch, [(j, x, y, 0) for j, (x, y) in enumerate(lifted[:, :2].tolist())])
    assert got == b"".join(tgts[j].tobytes()[x:y] for j, (x, y) in enumerate(lifted[:, :2].tolist()))
    for a in arch:
        a.close()
    ctx.clear_reference()
