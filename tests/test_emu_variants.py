"""Variant records of open archives (sccg_archive_variants, include/sccg.h) on the CPU (SIMT emulator build): every record
list must equal the reference implementation of tests/variants_lib.py (steps 1-5 in Python from the oracle's token loop) and
pass the invariant and splice check of the header; windows must be a filter of the whole-archive records; counts, caps,
errors and archive lifetime follow the contract.  The check_* functions are shared with test_gpu_variants.py."""
import ctypes as C
import random

import numpy as np
import pytest

import oracle_lib as ol
import sccg_b200
import variants_lib as vl
from emu_lib import emu_context
from test_emu_archive import archive_set
from test_emu_extract import CASES, seq_of, unpack

ARG = sccg_b200.SCCG_E_ARG


@pytest.fixture(scope="module")
def ctx():
    c = emu_context()
    yield c
    c.close()


def compressed(ref: bytes, tgt: bytes):
    rc, inter, mode = ol.orc_compress(ref, tgt, b">t")
    assert rc == 0
    return inter, vl.decoded(ref, inter), mode


def check_archive(ctx, ref: bytes, inter: bytes, D: bytes) -> np.ndarray:
    """one archive, whole: the records must equal the reference implementation's and pass the invariants -> the records"""
    exp = vl.variants_whole(ref, inter, D)
    vl.check_invariants(ref, D, exp)
    ctx.set_reference(ref)
    with ctx.open_archive(inter) as a:
        assert a.seq_len == len(D)
        rec, alt = ctx.variants([a])
        assert ctx.variants([a], count_only=True) == (len(rec), len(alt))
    vl.check_invariants(ref, D, rec, alt)
    assert rec.shape == (len(exp), 6) and np.array_equal(rec[:, 1:5], exp), first_difference(rec[:, 1:5], exp)
    assert (rec[:, 0] == 0).all()
    return rec


def first_difference(got, exp) -> str:
    for i in range(min(len(got), len(exp))):
        if not np.array_equal(got[i], exp[i]):
            return f"record {i}: got {got[i].tolist()}, expected {exp[i].tolist()} ({len(got)} vs {len(exp)} records)"
    return f"{len(got)} records, expected {len(exp)}"


def hand_file(body: bytes, low: bytes = b"") -> bytes:
    """a local-mode record file written by hand"""
    return b">hand\n" + low + b"\n,\n" + body + b"\n"


def tokens(*copies) -> bytes:
    """(absolute start, length) copies and literal bytes -> a record body with delta-encoded starts"""
    out, prev = [], 0
    for c in copies:
        if isinstance(c, bytes):
            out.append(c)
        else:
            out.append(b"(%d,%d)" % (c[0] - prev, c[1]))
            prev = c[0]
    return b"".join(out)


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
        check_archive(ctx, case.ref, inter, D)
        n += 1
    ctx.clear_reference()
    assert n > 10


def check_substitutions_only(ctx, n=40_000, seed=3):
    """local mode, substitutions only, lowercase in R and D: the records are the maximal runs of up(R) != up(D)"""
    from sccg_genome_compression_b200 import synth
    rng = np.random.default_rng(seed)
    r = synth.random_bases(rng, n)
    t = r.copy()
    synth.substitute(rng, t, 0.004)
    t[1000:1003] = [ord(c) for c in "ACG"] if bytes(r[1000:1003]) != b"ACG" else [ord(c) for c in "TTT"]   # (an MNP, maybe)
    synth.lowercase_runs(rng, t, 0.3, 10, 2000)
    synth.lowercase_runs(rng, r, 0.3, 10, 2000)
    ref, tgt = r.tobytes(), t.tobytes()
    inter, D, mode = compressed(ref, tgt)
    assert mode == 0 and D == tgt
    rec = check_archive(ctx, ref, inter, D)
    d = np.frombuffer(vl.up(ref), np.uint8) != np.frombuffer(vl.up(tgt), np.uint8)
    e = np.diff(np.concatenate([[0], d.astype(np.int8), [0]]))
    runs = np.stack([np.flatnonzero(e == 1), np.flatnonzero(e == -1)], axis=1)
    assert np.array_equal(rec[:, 1:3], runs) and np.array_equal(rec[:, 3:5], runs)


def left_aligned_deletion(R: bytes, pos: int, n: int) -> int:
    U = vl.up(R)
    end = pos + n
    while pos > 0 and U[pos - 1] == U[end - 1]:
        pos -= 1; end -= 1
    return pos


def left_aligned_insertion(R: bytes, pos: int, ins: bytes) -> int:
    U = vl.up(R)
    while pos > 0 and U[pos - 1] == ins[-1]:
        ins = bytes([U[pos - 1]]) + ins[:-1]
        pos -= 1
    return pos


def check_uncompensated(ctx, n=30_000, seed=11):
    """one +7 insertion and one -3 deletion, not compensated, plus SNPs: among the non-substitution records exactly one
    insertion and one deletion, at the planted sites after left-alignment"""
    from sccg_genome_compression_b200 import synth
    rng = np.random.default_rng(seed)
    r = synth.random_bases(rng, n)
    t = r.copy()
    synth.substitute(rng, t, 0.001)
    a, b = n // 3, 2 * n // 3
    t[a - 20:a + 20] = r[a - 20:a + 20]
    t[b - 20:b + 20] = r[b - 20:b + 20]
    ins = b"GATTACA"
    tgt = t[:a].tobytes() + ins + t[a:b].tobytes() + t[b + 3:].tobytes()
    ref = r.tobytes()
    inter, D, mode = compressed(ref, tgt)
    rec = check_archive(ctx, ref, inter, D)
    lr, ld = rec[:, 2] - rec[:, 1], rec[:, 4] - rec[:, 3]
    other = rec[lr != ld]
    assert len(other) == 2, other
    i_row = other[other[:, 2] == other[:, 1]]
    d_row = other[other[:, 4] == other[:, 3]]
    assert len(i_row) == 1 and len(d_row) == 1
    assert i_row[0, 1] == left_aligned_insertion(ref, a, ins) and i_row[0, 4] - i_row[0, 3] == 7
    assert d_row[0, 1] == left_aligned_deletion(ref, b, 3) and d_row[0, 2] - d_row[0, 1] == 3


def check_repeats(ctx, n=20_000, seed=5):
    """homopolymer and tandem-repeat expansions and contractions: compressed pairs, and hand-written files with two indels in
    one repeat, where the previous record bounds the left shift"""
    from sccg_genome_compression_b200 import synth
    rng = np.random.default_rng(seed)
    r = bytearray(synth.random_bases(rng, n).tobytes())
    sites = [(2000, b"A", 14, 1), (5000, b"CA", 12, -1), (8000, b"AGT", 8, 1), (11_000, b"T", 25, -2), (14_000, b"GATC", 9, 2)]
    for s, unit, k, _ in sites:
        rep = unit * k
        r[s - 1] = ord("G") if unit[-1] != ord("G") else ord("C")
        r[s:s + len(rep)] = rep
        r[s + len(rep)] = ord("G") if unit[0] != ord("G") else ord("C")
    ref = bytes(r)
    t = bytearray(ref)
    for s, unit, k, d in reversed(sites):                                  # expansions and contractions inside the repeats
        at = s + len(unit) * (k // 2)
        if d > 0:
            t[at:at] = unit * d
        else:
            del t[at:at + len(unit) * -d]
    tgt = bytes(t)
    inter, D, _ = compressed(ref, tgt)
    check_archive(ctx, ref, inter, D)
    # hand-written: two CA deletions in one (CA)x10 repeat; the second is bounded by the first's end
    rep = 1000
    r2 = bytearray(ref[:2000])
    r2[rep - 1] = ord("G"); r2[rep:rep + 20] = b"CA" * 10; r2[rep + 20] = ord("G")
    R2 = bytes(r2)
    for body in (tokens((0, rep + 2), (rep + 4, 12), (rep + 18, 2000 - rep - 18)),       # two deletions of CA
                 tokens((0, rep + 2), b"CA", (rep + 2, 12), b"AC", (rep + 14, 2000 - rep - 14)),   # two insertions
                 tokens((0, rep + 2), (rep + 4, 12), b"CACA", (rep + 16, 2000 - rep - 16))):       # a deletion, then an insertion
        inter = hand_file(body)
        D = vl.decoded(R2, inter)
        rec = check_archive(ctx, R2, inter, D)
        assert len(rec) >= 2
        assert rec[1, 1] >= rec[0, 2]


def check_hand_files(ctx, seed=8):
    """edits at D position 0 and at its end, identical and empty targets, a literal-only file, overlapping and contained
    copies (the clipping of step 2), lowercase in R"""
    from sccg_genome_compression_b200 import synth
    rng = np.random.default_rng(seed)
    R = bytearray(synth.random_bases(rng, 3000).tobytes())
    R[100:400] = bytes(R[100:400]).lower()
    R = bytes(R)
    other = lambda c: b"T" if vl.up(bytes([c])) != b"T" else b"G"           # noqa: E731
    bodies = {
        "identical": tokens((0, 3000)),
        "empty": b"",
        "sub_at_0": other(R[0]) + tokens((1, 2999)),
        "sub_at_end": tokens((0, 2999)) + other(R[-1]),
        "ins_at_0": b"GG" + tokens((0, 3000)),
        "ins_at_end": tokens((0, 3000)) + b"CC",
        "del_at_0": tokens((5, 2995)),
        "del_at_end": tokens((0, 2990)),
        "literal_only": R[:1500].lower() + b"ACGTNN" + R[1500:],
        "literal_same_length": R[:700] + other(R[700]) + R[701:],
        "duplication": tokens((0, 1000), (500, 800), (1300, 1700)),
        "contained": tokens((0, 1000), (100, 50), (1000, 2000)),
        "permuted": tokens((2000, 1000), (0, 1000), (1000, 1000)),
        "lower_copy": tokens((0, 3000)),
    }
    for name, body in bodies.items():
        low = b"(0,50)" if name == "lower_copy" else b""
        inter = hand_file(body, low)
        D = vl.decoded(R, inter)
        rec = check_archive(ctx, R, inter, D)
        if name in ("identical", "lower_copy"):
            assert len(rec) == 0, name
        if name == "empty":
            assert rec[:, 1:5].tolist() == [[0, 3000, 0, 0]]
        if name == "sub_at_0":
            assert rec[0, 1:5].tolist() == [0, 1, 0, 1]
        if name == "ins_at_0":
            assert rec[0, 1:5].tolist() == [0, 0, 0, 2]


def check_global(ctx):
    from sccg_genome_compression_b200 import synth
    for r, t in (synth.global_gap_pair(41_000, 40_000, 7), synth.divergent_pair(30_000, 9, blocks=6)):
        inter, D, mode = compressed(r.tobytes(), t.tobytes())
        assert mode == 1
        rec = check_archive(ctx, r.tobytes(), inter, D)
        assert len(rec) > 0


def random_windows(rng: random.Random, n_arch: int, L: int, n: int = 40):
    w = [(0, 0, 0), (0, L, L), (n_arch - 1, 0, L), (0, 0, L)]
    for _ in range(n):
        k = rng.randrange(n_arch)
        s = rng.randrange(L + 1)
        e = min(L, s + rng.choice([0, 1, 10, 500, 5000, L]))
        w.append((k, s, e))
    w += w[4:10]                                                           # repeated
    rng.shuffle(w)
    return w


def check_windows(ctx, n=60_000, seed=74, rounds=3):
    """several archives in one call, random windows: the records of each window are the filter of the whole-archive records"""
    ref, files = archive_set(n, seed)
    ctx.set_reference(ref)
    arch = [ctx.open_archive(inter) for inter, _, _ in files]
    Ds = [D for _, D, _ in files]
    whole = [vl.variants_whole(ref, inter, D) for inter, D, _ in files]
    for k, (inter, D, _) in enumerate(files):
        rec, alt = ctx.variants([arch[k]])
        assert np.array_equal(rec[:, 1:5], whole[k]), (k, first_difference(rec[:, 1:5], whole[k]))
    rng = random.Random(seed)
    for _ in range(rounds):
        w = random_windows(rng, len(arch), len(ref))
        rec, alt = ctx.variants(arch, w)
        exp, exp_alt = vl.filter_windows(whole, Ds, w, len(ref))
        assert np.array_equal(rec, exp), first_difference(rec, exp)
        assert alt == exp_alt
        assert ctx.variants(arch, w, count_only=True) == (len(exp), len(exp_alt))
    # windows=None: the whole reference of each archive, in order; one call equals per-archive calls
    rec, alt = ctx.variants(arch)
    exp, exp_alt = vl.filter_windows(whole, Ds, [(k, 0, len(ref)) for k in range(len(arch))], len(ref))
    assert np.array_equal(rec, exp) and alt == exp_alt
    for a in arch:
        a.close()
    ctx.clear_reference()


def raw_call(ctx, archives, windows, vars_cap, alt_cap, null_vars=False, null_alt=False):
    arr = (C.c_void_p * max(len(archives), 1))(*[a.handle for a in archives])
    w = np.ascontiguousarray(np.asarray(windows, dtype=np.int64).reshape(-1, 3))
    out = np.zeros(max(vars_cap, 1), dtype=ctx._VARIANT)
    alt = C.create_string_buffer(max(alt_cap, 1))
    n, na = C.c_int64(-1), C.c_int64(-1)
    rc = ctx.lib.sccg_archive_variants(ctx.handle, arr, len(archives), w.ctypes.data if len(w) else None, len(w),
                                       None if null_vars else out.ctypes.data, vars_cap, C.byref(n), None if null_alt else alt, alt_cap, C.byref(na))
    return rc, n.value, na.value, out, alt


def check_caps(ctx, n=30_000, seed=75):
    ref, files = archive_set(n, seed)
    ctx.set_reference(ref)
    A = ctx.open_archive(files[0][0])
    w = [(0, 0, len(ref)), (0, 100, 9000)]
    rec, alt = ctx.variants([A], w)
    nv, na = len(rec), len(alt)
    assert nv > 2 and na > 2
    assert raw_call(ctx, [A], w, 0, 0, null_vars=True, null_alt=True)[:3] == (0, nv, na)          # counting only
    rc, n1, n2, out, buf = raw_call(ctx, [A], w, nv, na)                                              # exact caps
    assert (rc, n1, n2) == (0, nv, na)
    assert np.array_equal(np.stack([out[f][:nv] for f, _ in ctx._VARIANT], axis=1), rec) and buf.raw[:na] == alt
    assert raw_call(ctx, [A], w, nv - 1, na)[:3] == (ARG, nv, na)
    assert raw_call(ctx, [A], w, nv, na - 1)[:3] == (ARG, nv, na)
    assert raw_call(ctx, [A], w, nv - 1, na - 1)[:3] == (ARG, nv, na)
    assert raw_call(ctx, [A], w, nv, na, null_alt=True)[0] == ARG
    assert raw_call(ctx, [A], [], 0, 0)[:3] == (0, 0, 0)
    assert ctx.variants([A], []) [0].shape == (0, 6)
    A.close()
    ctx.clear_reference()


def check_argument_errors(ctx, ctx2):
    """the error list of include/sccg.h, in its order, whichever windows commit the errors (as check_argument_errors of
    test_emu_archive.py does for sccg_archive_extract)"""
    ref, files = archive_set(30_000, 74)
    ctx.set_reference(ref)
    A = ctx.open_archive(files[0][0])
    L = len(ref)
    good = [(0, 3, 4000)]
    exp = ctx.variants([A], good)

    def fails(msg, archives, windows):
        with pytest.raises(sccg_b200.SccgError) as e:
            ctx.variants(archives, windows)
        assert e.value.code == ARG and msg in str(e.value), str(e.value)
        got = ctx.variants([A], good)                                     # the context survived
        assert np.array_equal(got[0], exp[0]) and got[1] == exp[1]
    lib = ctx.lib
    n, na = C.c_int64(), C.c_int64()
    arr = (C.c_void_p * 1)(A.handle)
    wa = np.array([[0, 0, 1]], dtype=np.int64)
    call = lambda *t: lib.sccg_archive_variants(ctx.handle, *t)           # noqa: E731
    assert call(None, 1, wa.ctypes.data, 1, None, 0, C.byref(n), None, 0, C.byref(na)) == ARG          # NULL with a count
    assert call(arr, 1, None, 1, None, 0, C.byref(n), None, 0, C.byref(na)) == ARG
    assert call(arr, -1, wa.ctypes.data, 1, None, 0, C.byref(n), None, 0, C.byref(na)) == ARG
    assert call(arr, 1, wa.ctypes.data, -1, None, 0, C.byref(n), None, 0, C.byref(na)) == ARG
    assert call(arr, 1, wa.ctypes.data, 1, None, -1, C.byref(n), None, 0, C.byref(na)) == ARG
    assert call(arr, 1, wa.ctypes.data, 1, None, 0, C.byref(n), None, -1, C.byref(na)) == ARG
    assert call(arr, 1, wa.ctypes.data, 1, None, 0, None, None, 0, C.byref(na)) == ARG
    assert call(arr, 1, wa.ctypes.data, 1, None, 0, C.byref(n), None, 0, None) == ARG
    assert call(arr, 1, wa.ctypes.data, 1 << 31, None, 0, C.byref(n), None, 0, C.byref(na)) == ARG
    assert lib.sccg_archive_variants(None, arr, 1, wa.ctypes.data, 1, None, 0, C.byref(n), None, 0, C.byref(na)) == ARG
    assert call(None, 0, None, 0, None, 0, C.byref(n), None, 0, C.byref(na)) == 0 and n.value == 0 and na.value == 0
    fails("out of range", [A], [(1, 0, 1)])
    fails("out of range", [A], [(-1, 0, 1)])
    fails("null argument", [A, type("Closed", (), {"handle": None})()], [(1, 0, 1)])
    ctx2.set_reference(ref)
    X = ctx2.open_archive(files[0][0])
    fails("another context", [A, X], [(1, 0, 1)])
    fails("start <= end", [A], [(0, -1, 3)])
    fails("start <= end", [A], [(0, 5, 4)])
    fails("past the end of the resident reference", [A], [(0, 0, L + 1)])
    fails("past the end of the resident reference", [A], [(0, L + 5, L + 5)])
    # windows end past len(D) but inside len(R): not an error (reference coordinates)
    D = files[0][1]
    if len(D) < L:
        ctx.variants([A], [(0, len(D), L)])
    # the order of the list, whichever windows commit the errors
    fails("out of range", [A, X], [(0, 9, 1), (1, 0, 1), (0, 0, L + 1), (2, 0, 1)])
    fails("another context", [A, X], [(0, 9, 1), (0, 0, L + 1), (1, 0, 1)])
    fails("start <= end", [A], [(0, 0, L + 1), (0, 9, 1)])
    X.close()
    # a stale archive: replaced and cleared references
    ctx.set_reference(ref)
    with pytest.raises(sccg_b200.SccgError) as e:
        ctx.variants([A], [(0, 0, 10)])
    assert e.value.code == ARG and "replaced or cleared" in str(e.value)
    B = ctx.open_archive(files[0][0])
    got = ctx.variants([B], good)
    assert np.array_equal(got[0], exp[0]) and got[1] == exp[1]
    ctx.clear_reference()
    with pytest.raises(sccg_b200.SccgError) as e:
        ctx.variants([B], [(0, 0, 0)])
    assert e.value.code == ARG and "replaced or cleared" in str(e.value)
    A.close(); B.close()
    ctx2.clear_reference()


def test_golden_cases(ctx, golden):
    check_golden(ctx, golden)


def test_substitutions_only(ctx):
    check_substitutions_only(ctx)


def test_compensated_indels_n_lowercase(ctx):
    from sccg_genome_compression_b200 import synth
    r, t = synth.local_pair(60_000, 21, snp=0.002, indels_per_mbp=300)
    t[5000:5080] = ord("N")                                                # target-only N run
    synth.lowercase_runs(np.random.default_rng(2), r, 0.3, 10, 3000)
    inter, D, mode = compressed(r.tobytes(), t.tobytes())
    assert mode == 0
    check_archive(ctx, r.tobytes(), inter, D)


def test_uncompensated_indels(ctx):
    check_uncompensated(ctx)


def test_repeats(ctx):
    check_repeats(ctx)


def test_hand_files(ctx):
    check_hand_files(ctx)


def test_global_pairs(ctx):
    check_global(ctx)


def test_windows(ctx):
    check_windows(ctx)


def test_caps(ctx):
    check_caps(ctx)


def test_argument_errors(ctx):
    ctx2 = emu_context()
    try:
        check_argument_errors(ctx, ctx2)
    finally:
        ctx2.close()
