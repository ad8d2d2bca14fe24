"""Coordinates lifted between the reference and open archives (sccg_archive_liftover, include/sccg.h) on the CPU (SIMT
emulator build): every row must equal the closed form of tests/liftover_lib.py and, on small cases, the owner-of-every-base
reference and the splice identity (D read through Context.query); the record counts must equal what sccg_archive_variants
reports for the same windows; tables are built once per archive and live as long as it.  The check_* functions are shared
with test_gpu_liftover.py."""
import ctypes as C

import numpy as np
import pytest

import liftover_lib as ll
import sccg_b200
import variants_lib as vl
from emu_lib import emu_context
from test_emu_archive import archive_set
from test_emu_extract import CASES, seq_of, unpack
from test_emu_variants import compressed, hand_file, tokens

ARG = sccg_b200.SCCG_E_ARG


@pytest.fixture(scope="module")
def ctx():
    c = emu_context()
    yield c
    c.close()


def edge_points(recs: np.ndarray, ls: int, frm: int) -> list:
    """source positions worth probing: both ends, and every record edge +- 1 (on the source side of direction frm)"""
    cols = recs[:, 2:4] if frm else recs[:, 0:2]
    pts = {0, ls}
    for b in cols.reshape(-1).tolist():
        pts.update((b - 1, b, b + 1))
    return sorted(p for p in pts if 0 <= p <= ls)


def small_queries(recs: np.ndarray, R: bytes, D: bytes, rng, n_random: int = 200, full: int = 8000) -> list:
    """[s, e, from]: every [b, b) and [b, b + 1) (every b when the source is at most `full` long, else the record edges),
    plus random intervals and intervals between record edges, both directions"""
    q = []
    for frm, ls in ((0, len(R)), (1, len(D))):
        pts = range(ls + 1) if ls <= full else edge_points(recs, ls, frm)
        q += [(b, b, frm) for b in pts] + [(b, b + 1, frm) for b in pts if b < ls]
        for _ in range(n_random):
            s = int(rng.integers(0, ls + 1))
            q.append((s, int(rng.integers(s, ls + 1)), frm))
        ep = edge_points(recs, ls, frm)
        for _ in range(n_random):
            a, b = sorted(int(x) for x in rng.choice(ep, 2))
            q.append((a, b, frm))
    return q


def check_one(ctx, ref: bytes, inter: bytes, D: bytes, seed: int = 0, n_random: int = 200, full: int = 8000) -> np.ndarray:
    """one archive: boundary and random queries in both directions against both references and the splice identity, the
    records of from = 0 queries against sccg_archive_variants, a second call equal to the first -> the records"""
    recs = vl.variants_whole(ref, inter, D)
    rng = np.random.default_rng(seed)
    q = small_queries(recs, ref, D, rng, n_random, full)
    ctx.set_reference(ref)
    with ctx.open_archive(inter) as a:
        assert ctx.query([a], [(0, 0, len(D), 0)]) == D
        qa = [(0, s, e, f) for s, e, f in q]
        rows = ctx.liftover([a], qa)
        ll.check_small(recs, ref, D, rows, q)
        assert np.array_equal(ctx.liftover([a], qa), rows)
        assert ctx.profile()["launches"] == 1                              # the table is built: one launch, the lift
        w = [(0, s, e) for s, e, f in q if f == 0]
        rec, _ = ctx.variants([a], w)
        per_window = np.bincount(rec[:, 0], minlength=len(w)) if len(rec) else np.zeros(len(w), np.int64)
        assert np.array_equal(per_window, rows[np.array([f == 0 for _, _, f in q]), 4])
    ctx.clear_reference()
    return recs


def check_golden(ctx, golden):
    n = 0
    for case in CASES:
        g = golden["cases"][case.name]
        inter = unpack(g["intermediate_z"])
        ctx.set_reference(case.ref)
        try:
            D = seq_of(ctx.decompress_resident(inter))
        except sccg_b200.SccgError:
            continue
        check_one(ctx, case.ref, inter, D, n, n_random=40)
        n += 1
    ctx.clear_reference()
    assert n > 10


def check_synthetic(ctx, n=30_000, seed=3):
    """SNPs only; compensated indels with a target N run; an uncompensated insertion and deletion"""
    from sccg_genome_compression_b200 import synth
    rng = np.random.default_rng(seed)
    r = synth.random_bases(rng, n)
    t = r.copy()
    synth.substitute(rng, t, 0.004)
    synth.lowercase_runs(rng, t, 0.3, 10, 2000)
    ref = r.tobytes()
    inter, D, mode = compressed(ref, t.tobytes())
    recs = check_one(ctx, ref, inter, D, 1)
    assert len(recs) > 50 and (recs[:, 1] - recs[:, 0] == recs[:, 3] - recs[:, 2]).all()
    r2, t2 = synth.local_pair(n, 21, snp=0.002, indels_per_mbp=300)
    t2[5000:5080] = ord("N")
    inter, D, _ = compressed(r2.tobytes(), t2.tobytes())
    recs = check_one(ctx, r2.tobytes(), inter, D, 2)
    assert (recs[:, 1] - recs[:, 0] != recs[:, 3] - recs[:, 2]).any()
    a, b = n // 3, 2 * n // 3
    t3 = r.copy()
    tgt = t3[:a].tobytes() + b"GATTACA" + t3[a:b].tobytes() + t3[b + 3:].tobytes()
    inter, D, _ = compressed(ref, tgt)
    recs = check_one(ctx, ref, inter, D, 3)
    assert len(recs) == 2


def repeat_ref(rng) -> bytes:
    from sccg_genome_compression_b200 import synth
    r = bytearray(synth.random_bases(rng, 2000).tobytes())
    r[999] = ord("G"); r[1000:1020] = b"CA" * 10; r[1020] = ord("G")
    return bytes(r)


def check_hand_files(ctx, seed=8):
    """edits at both ends, insertions at pos 0 and len(R), a deletion at the end of D, adjacent records after left-alignment
    in a repeat, identical, empty and literal-only targets, complex records, lowercase in R; and the end-only len rules"""
    from sccg_genome_compression_b200 import synth
    rng = np.random.default_rng(seed)
    R = bytearray(synth.random_bases(rng, 3000).tobytes())
    R[100:400] = bytes(R[100:400]).lower()
    R[2989], R[2999] = ord("C"), ord("A")                                  # the end records cannot left-align away
    R = bytes(R)
    other = lambda c: b"T" if vl.up(bytes([c])) != b"T" else b"G"           # noqa: E731
    bodies = {
        "identical": tokens((0, 3000)),
        "empty": b"",
        "sub_at_0": other(R[0]) + tokens((1, 2999)),
        "sub_at_end": tokens((0, 2999)) + other(R[-1]),
        "ins_at_0": b"GG" + tokens((0, 3000)),
        "ins_at_end": tokens((0, 3000)) + b"GG",
        "del_at_0": tokens((5, 2995)),
        "del_at_end": tokens((0, 2990)),
        "literal_only": R[:1500].lower() + b"ACGTNN" + R[1500:],
        "duplication": tokens((0, 1000), (500, 800), (1300, 1700)),
        "permuted": tokens((2000, 1000), (0, 1000), (1000, 1000)),
        "complex": tokens((0, 1200)) + b"ACGTACGTTT" + tokens((1205, 1795)),
        "mixed_ends": b"TT" + tokens((3, 1000), (1004, 1990)),
    }
    for i, (name, body) in enumerate(bodies.items()):
        inter = hand_file(body)
        D = vl.decoded(R, inter)
        recs = check_one(ctx, R, inter, D, 10 + i, n_random=60)
        if name == "identical":
            assert len(recs) == 0
        ctx.set_reference(R)
        with ctx.open_archive(inter) as a:
            L, LD = len(R), len(D)
            end_r, end_d = ctx.liftover([a], [(0, L, L, 0), (0, LD, LD, 1)])
            if name == "ins_at_end":                                       # [len(R), len(R)) owns the trailing insertion
                assert end_r.tolist()[:2] == [LD - 2, LD] and end_r[4] == 1 and end_r[5] == ll.LENGTH_CHANGE
                assert ctx.variants([a], [(0, L, L)], count_only=True)[0] == 1
            if name == "del_at_end":                                       # [len(D), len(D)) owns the trailing deletion
                assert end_d.tolist()[:2] == [L - 10, L] and end_d[4] == 1 and end_d[5] == ll.LENGTH_CHANGE
                assert end_r[4] == 0 and end_r[0] == end_r[1] == LD
            if name == "ins_at_0":                                         # [0, 0) owns nothing, [0, 1) the insertion at 0
                assert ctx.liftover([a], [(0, 0, 0, 0), (0, 0, 1, 0)]).tolist() == [[0, 0, 0, 0, 0, 0], [0, 3, 1, 0, 1, ll.LENGTH_CHANGE]]
            if name == "empty":
                assert ctx.liftover([a], [(0, 0, L, 0)])[0].tolist() == [0, 0, 0, 0, 1, ll.LENGTH_CHANGE]
        ctx.clear_reference()
    # adjacent records after left-alignment: two deletions, two insertions, a deletion then an insertion, in one repeat
    R2 = repeat_ref(rng)
    rep = 1000
    for j, body in enumerate((tokens((0, rep + 2), (rep + 4, 12), (rep + 18, 2000 - rep - 18)),
                              tokens((0, rep + 2), b"CA", (rep + 2, 12), b"AC", (rep + 14, 2000 - rep - 14)),
                              tokens((0, rep + 2), (rep + 4, 12), b"CACA", (rep + 16, 2000 - rep - 16)),
                              tokens((0, rep + 2), (rep + 4, 2000 - rep - 4)) + b"",
                              tokens((0, rep)) + b"TTT" + tokens((rep + 2, 2000 - rep - 2)))):
        inter = hand_file(body)
        D = vl.decoded(R2, inter)
        recs = check_one(ctx, R2, inter, D, 40 + j, n_random=100)
        assert len(recs) >= 1


def check_global(ctx):
    """global-mode gap and divergent pairs: N runs in R and D"""
    from sccg_genome_compression_b200 import synth
    for i, (r, t) in enumerate((synth.global_gap_pair(41_000, 40_000, 7), synth.divergent_pair(30_000, 9, blocks=6))):
        inter, D, mode = compressed(r.tobytes(), t.tobytes())
        assert mode == 1
        recs = check_one(ctx, r.tobytes(), inter, D, 50 + i, n_random=100, full=0)
        assert len(recs) > 0


def lift_tables_bytes(n: int) -> int:
    return 4 * (8 * n + 4)


def check_lifecycle(ctx, make_ctx, n=30_000, seed=74):
    """several archives: tables built lazily and once, calls that mix archives with and without a table, repeated archives,
    device_bytes, zero queries, close and destroy with tables built"""
    ref, files = archive_set(n, seed)
    ctx.set_reference(ref)
    arch = [ctx.open_archive(inter) for inter, _, _ in files]
    Ds = [D for _, D, _ in files]
    whole = [vl.variants_whole(ref, inter, D) for inter, D, _ in files]
    L = len(ref)
    bytes0 = [a.device_bytes for a in arch]
    rng = np.random.default_rng(seed)

    def queries(ks, m=60):
        q = []
        for k in ks:
            for _ in range(m):
                frm = int(rng.integers(0, 2))
                ls = len(Ds[k]) if frm else L
                s = int(rng.integers(0, ls + 1))
                q.append((k, s, min(ls, s + int(rng.choice([0, 1, 150, 5000, ls]))), frm))
            q += [(k, 0, L, 0), (k, 0, len(Ds[k]), 1), (k, L, L, 0), (k, len(Ds[k]), len(Ds[k]), 1)]
        rng.shuffle(q)
        return q
    # zero queries: nothing built, nothing launched
    assert ctx.liftover(arch, []).shape == (0, 6)
    assert ctx.profile()["launches"] == 0 and [a.device_bytes for a in arch] == bytes0
    # archive 0 alone: its table is built, the others stay as they were
    q = queries([0])
    rows = ctx.liftover(arch, q)
    assert np.array_equal(rows, ll.lift_queries(whole, L, [len(D) for D in Ds], q))
    build1 = ctx.profile()["launches"]
    assert build1 > 1
    assert arch[0].device_bytes == bytes0[0] + lift_tables_bytes(len(whole[0]))
    assert [a.device_bytes for a in arch[1:]] == bytes0[1:]
    # a call mixing built and unbuilt tables, archives listed twice (the same handle at two indices)
    listed = arch + [arch[1], arch[0]]
    n_a = len(arch)
    q = queries(range(n_a)) + [(n_a, 0, 100, 0), (n_a + 1, 7, 9, 1)]
    rows = ctx.liftover(listed, q)
    exp = ll.lift_queries(whole + [whole[1], whole[0]], L, [len(D) for D in Ds] + [len(Ds[1]), len(Ds[0])], q)
    assert np.array_equal(rows, exp)
    assert ctx.profile()["launches"] > 1
    for k, a in enumerate(arch):
        assert a.device_bytes == bytes0[k] + lift_tables_bytes(len(whole[k]))
    # every table built: one launch, the same rows; kernels_ms - gather_ms is the build, here none
    again = ctx.liftover(listed, q)
    p = ctx.profile()
    assert np.array_equal(again, rows) and p["launches"] == 1 and p["kernels_ms"] == p["gather_ms"]
    # per-archive calls equal the multi-archive call
    qa = np.array(q)
    for k in range(n_a):
        m = qa[:, 0] == k
        one = qa[m].copy(); one[:, 0] = 0
        assert np.array_equal(ctx.liftover([arch[k]], one), rows[m])
    # close one archive with its table; the others keep working
    arch[0].close()
    q = queries(range(1, n_a))
    assert np.array_equal(ctx.liftover(arch[1:], [(k - 1, s, e, f) for k, s, e, f in q]),
                          ll.lift_queries(whole, L, [len(D) for D in Ds], q))
    for a in arch[1:]:
        a.close()
    ctx.clear_reference()
    # destroy a context with tables built and archives still open
    c2 = make_ctx()
    c2.set_reference(ref)
    b = [c2.open_archive(inter) for inter, _, _ in files[:2]]
    c2.liftover(b, [(0, 0, L, 0), (1, 0, 10, 1)])
    c2.close()


def check_argument_errors(ctx, ctx2):
    """the error list of include/sccg.h, in its order, whichever queries commit the errors; nothing is launched"""
    ref, files = archive_set(30_000, 74)
    ctx.set_reference(ref)
    A = ctx.open_archive(files[0][0])
    D = files[0][1]
    L, LD = len(ref), len(D)
    assert L != LD
    good = [(0, 3, 4000, 0), (0, 5, 100, 1)]
    exp = ctx.liftover([A], good)

    def fails(msg, archives, queries):
        with pytest.raises(sccg_b200.SccgError) as e:
            ctx.liftover(archives, queries)
        assert e.value.code == ARG and msg in str(e.value), str(e.value)
        assert ctx.profile()["launches"] == 0
        assert np.array_equal(ctx.liftover([A], good), exp)               # the context survived
    lib = ctx.lib
    arr = (C.c_void_p * 1)(A.handle)
    qa = np.zeros(1, dtype=ctx._LIFT_QUERY)
    qa[0] = (0, 0, 1, 0, 0)
    out = np.zeros(1, dtype=ctx._LIFT)
    call = lambda *t: lib.sccg_archive_liftover(ctx.handle, *t)           # noqa: E731
    assert call(None, 1, qa.ctypes.data, 1, out.ctypes.data) == ARG        # NULL with a count
    assert call(arr, 1, None, 1, out.ctypes.data) == ARG
    assert call(arr, 1, qa.ctypes.data, 1, None) == ARG
    assert call(arr, -1, qa.ctypes.data, 1, out.ctypes.data) == ARG
    assert call(arr, 1, qa.ctypes.data, -1, out.ctypes.data) == ARG
    assert call(arr, 1 << 31, qa.ctypes.data, 1, out.ctypes.data) == ARG
    assert call(arr, 1, qa.ctypes.data, 1 << 31, out.ctypes.data) == ARG
    assert lib.sccg_archive_liftover(None, arr, 1, qa.ctypes.data, 1, out.ctypes.data) == ARG
    assert call(None, 0, None, 0, None) == 0
    assert call(arr, 1, qa.ctypes.data, 1, out.ctypes.data) == 0 and out["end"][0] >= out["start"][0]
    fails("out of range", [A], [(1, 0, 1, 0)])
    fails("out of range", [A], [(-1, 0, 1, 0)])
    fails("null argument", [A, type("Closed", (), {"handle": None})()], [(1, 0, 1, 0)])
    ctx2.set_reference(ref)
    X = ctx2.open_archive(files[0][0])
    fails("another context", [A, X], [(1, 0, 1, 0)])
    fails("from must be 0", [A], [(0, 0, 1, 2)])
    fails("from must be 0", [A], [(0, 0, 1, -1)])
    fails("from must be 0", [A], [(0, 0, 1, 1 << 32)])
    fails("start <= end", [A], [(0, -1, 3, 0)])
    fails("start <= end", [A], [(0, 5, 4, 1)])
    fails("past the end of its source", [A], [(0, 0, L + 1, 0)])
    fails("past the end of its source", [A], [(0, 0, LD + 1, 1)])
    fails("past the end of its source", [A], [(0, 0, max(L, LD), 0 if LD > L else 1)])   # legal the other way only
    ctx.liftover([A], [(0, 0, L, 0), (0, 0, LD, 1)])
    # the order of the list, whichever queries commit the errors
    fails("out of range", [A, X], [(0, 9, 1, 0), (1, 0, 1, 0), (0, 0, 1, 5), (2, 0, 1, 0)])
    fails("another context", [A, X], [(0, 9, 1, 0), (0, 0, 1, 7), (1, 0, 1, 0)])
    fails("from must be 0", [A], [(0, 0, L + 1, 0), (0, 9, 1, 0), (0, 0, 1, 3)])
    fails("start <= end", [A], [(0, 0, L + 1, 0), (0, 9, 1, 1)])
    X.close()
    # a stale archive: replaced and cleared references
    ctx.set_reference(ref)
    with pytest.raises(sccg_b200.SccgError) as e:
        ctx.liftover([A], [(0, 0, 10, 0)])
    assert e.value.code == ARG and "replaced or cleared" in str(e.value)
    B = ctx.open_archive(files[0][0])
    assert np.array_equal(ctx.liftover([B], good), exp)
    ctx.clear_reference()
    with pytest.raises(sccg_b200.SccgError) as e:
        ctx.liftover([B], [(0, 0, 0, 0)])
    assert e.value.code == ARG and "replaced or cleared" in str(e.value)
    A.close(); B.close()
    ctx2.clear_reference()


def test_golden_cases(ctx, golden):
    check_golden(ctx, golden)


def test_synthetic(ctx):
    check_synthetic(ctx)


def test_hand_files(ctx):
    check_hand_files(ctx)


def test_global_pairs(ctx):
    check_global(ctx)


def test_lifecycle(ctx):
    check_lifecycle(ctx, emu_context)


def test_argument_errors(ctx):
    ctx2 = emu_context()
    try:
        check_argument_errors(ctx, ctx2)
    finally:
        ctx2.close()
