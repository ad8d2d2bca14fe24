"""Variant records of open archives (sccg_archive_variants, include/sccg.h) over the whole of their contract on the CPU (SIMT
emulator build): inputs built to land where the pipeline of csrc/sccg_variants.cuh can go wrong -- runs of differences at
the 16-byte thread and 4,096-byte tile edges of the gap-byte space, long gaps whose trims combine across CTAs, scans at
their tile and chunk sizes, global-mode N runs at every split point, the reference N-run table across reference changes,
many archives in one call, odd bytes and token forms, and the output paths of empty windows and empty ALTs.  Every record
list and ALT string is compared with tests/variants_lib.py (whole-archive records through filter_windows), every
whole-archive list passes check_invariants (splice check included), and every count-only total equals the full result.
Each edge test asserts through variants_lib.gap_layout that its input really puts a record start, a run end or an archive
seam on the gap byte it claims.  The check_* functions are shared with test_gpu_variants_space.py."""
import functools
import random

import numpy as np
import pytest

import oracle_lib as ol
import token_grammar_cases as tg
import variants_lib as vl
from emu_lib import emu_context
from test_emu_archive import every_byte_archive
from test_emu_extract import tolerance_cases
from test_emu_search_space import odd_target_archive
from test_emu_variants import first_difference, hand_file, raw_call, tokens

# csrc/sccg_variants.cuh: gap bytes per thread (VR_BPT), gap bytes per CTA (VR_TILE), scan elements per CTA (VR_STILE) and
# per pass of the one-CTA top scan (VR_T * VR_STILE)
THREAD, TILE, STILE, CHUNK = 16, 4096, 1024, 262_144
EMU_GRID = 8 * 8                                                              # sm_count x 8 CTAs: the emulator reports 8 SMs


@pytest.fixture(scope="module")
def ctx():
    c = emu_context()
    yield c
    c.close()


def bases(n: int, seed) -> bytes:
    from sccg_genome_compression_b200 import synth
    return synth.random_bases(np.random.default_rng(seed), n).tobytes()


def other(c: int) -> bytes:
    """a base that differs from byte c, case folded"""
    return b"T" if vl.up(bytes([c])) != b"T" else b"G"


def flipped(s: bytes, runs=None) -> bytes:
    """s with every byte of the [a, b) runs (all of s when None) replaced by a different base"""
    out = bytearray(s)
    for a, b in runs if runs is not None else [(0, len(s))]:
        for i in range(a, b):
            out[i] = other(s[i])[0]
    return bytes(out)


def run_list(runs) -> bytes:
    """(start, length) runs in raw D coordinates -> an N or lowercase line as the oracle writes it (start deltas;
    a one-byte run as 'delta,')"""
    out, prev = [], 0
    for s, n in runs:
        out.append(b"%d," % (s - prev) if n == 1 else b"(%d,%d)" % (s - prev, n))
        prev = s
    return b"".join(out)


def global_file(body: bytes, nline: bytes = b"", low: bytes = b"") -> bytes:
    """a global-mode record file written by hand: body copies in N-stripped reference coordinates, N runs in raw D"""
    assert nline != b","
    return b">glob\n" + low + b"\n" + nline + b"\n" + body + b"\n"


class Call:
    """one sccg_archive_variants call over record files against R, checked against variants_lib"""

    def __init__(self, ctx, R: bytes, inters, windows=None, set_ref=True, modes=None):
        if set_ref:
            ctx.set_reference(R)
        self.R, self.Ds = R, [vl.decoded(R, i) for i in inters]
        self.pieces = [vl.copy_pieces(R, i, D) for i, D in zip(inters, self.Ds)]
        self.whole = [vl.variants_from_pieces(R, D, P) for D, P in zip(self.Ds, self.pieces)]
        for D, W in zip(self.Ds, self.whole):
            vl.check_invariants(R, D, W)
        arch = [ctx.open_archive(i) for i in inters]
        try:
            if modes is not None:
                assert [a.mode for a in arch] == list(modes)
            self.windows = windows if windows is not None else [(k, 0, len(R)) for k in range(len(arch))]
            self.rec, self.alt = ctx.variants(arch, self.windows)
            exp, exp_alt = vl.filter_windows(self.whole, self.Ds, self.windows, len(R))
            assert np.array_equal(self.rec, exp), first_difference(self.rec, exp)
            assert self.alt == exp_alt
            assert ctx.variants(arch, self.windows, count_only=True) == (len(self.rec), len(self.alt))
            if windows is None:
                for k, D in enumerate(self.Ds):
                    vl.check_invariants(R, D, self.rec[self.rec[:, 0] == k], self.alt)
        finally:
            for a in arch:
                a.close()
        self.layout = vl.gap_layout(R, self.Ds, self.pieces)

    @functools.cached_property
    def gap_bytes(self):
        return vl.record_gap_bytes(self.layout, self.R, self.Ds, self.pieces, self.whole)

    @property
    def first(self) -> np.ndarray:
        return self.gap_bytes[0]

    @property
    def last(self) -> np.ndarray:
        return self.gap_bytes[1]

    @property
    def width(self) -> int:
        return int(self.layout[:, 1].sum())

    def tiles(self) -> int:
        return -(-self.width // TILE)


def around(*edges):
    return {e + d for e in edges for d in (-1, 0, 1)}


# ------------------------------------------------------------------------------------------------ 1. thread and tile edges
def check_thread_tile_edges(ctx):
    """equal-length literal runs whose runs of differences start, end and span thread and tile edges (the look-back of
    vr_starts into another thread's byte), a run that ends at its gap's end, a gap that starts mid-thread, short and
    zero-width gaps inside one thread, and two archives whose seam falls mid-thread and on a tile edge"""
    R = bases(5 * TILE + 3000, 101)
    L = 4 * TILE + 50
    starts, lasts = set(), set()
    for d in (-1, 0, 1):
        runs = [(160 + d, 163 + d), (478 + d, 481 + d), (797, 803), (TILE + d, TILE + 3 + d), (2 * TILE - 2 + d, 2 * TILE + 1 + d),
                (3 * TILE - 40, 3 * TILE + 40), (3 * TILE + 60, 3 * TILE + 99), (L - 3, L)]
        c = Call(ctx, R, [hand_file(flipped(R[:L], runs) + tokens((L, len(R) - L)))])
        assert c.layout[0].tolist() == [0, L, L, L]                           # gap byte = D position
        starts |= set(c.first.tolist()); lasts |= set(c.last.tolist())
        assert L - 1 in c.last                                                 # a run ends at its gap's end
        for e in (800, 3 * TILE, 3 * TILE + 16, 3 * TILE + 32, 3 * TILE + 64, 3 * TILE + 96):                # spanned edges: one record across each
            assert ((c.first < e) & (c.last >= e)).sum() == 1, e
    assert around(160, TILE) <= starts and around(480, 2 * TILE) <= lasts
    # a gap that starts mid-thread (goff 3): record starts on thread and tile edges of the gap-byte space
    g0 = 3
    edges = (16 * 20, 16 * 40, TILE)
    lit = flipped(R[103:103 + TILE + 200], [(e - g0 - 1, e - g0 + 2) for e in edges])      # gap bytes [e - 1, e + 2)
    c = Call(ctx, R, [hand_file(tokens(flipped(R[:3]), (3, 100), lit, (303 + TILE, len(R) - 303 - TILE)))])
    assert c.layout[1, 0] == g0 and c.layout[1, 0] % THREAD != 0
    assert {e - 1 for e in edges} <= set(c.first.tolist()) and {e + 1 for e in edges} <= set(c.last.tolist())
    # short gaps, some of zero width, inside one thread's 16 bytes (and across the edge at 16)
    for pre in (0, 13):
        body = tokens(flipped(R[:pre]), (pre, 10), other(R[pre + 10]), (pre + 11, 2), (pre + 13, 3), other(R[pre + 16]), (pre + 17, 1),
                      flipped(R[pre + 18:pre + 20]), (pre + 20, len(R) - pre - 20))
        c = Call(ctx, R, [hand_file(body)])
        w = c.layout[:, 1]
        assert (w == 0).sum() >= 2 and c.width == pre + 4 and len(c.whole[0]) == (1 if pre else 0) + 3
    # two archives in one call: the first ends on a copy to len(R) (its max-scan key must not clip the second's copies)
    for LA in (TILE, 16 * 100 + 7):
        A = hand_file(flipped(R[:LA], [(LA - 2, LA)]) + tokens((LA, len(R) - LA)))
        B = hand_file(tokens(flipped(R[:500], [(0, 2), (THREAD - 1, THREAD + 1)]), (500, 1000), (1600, len(R) - 1600)))
        c = Call(ctx, R, [A, B])
        seam = int(vl.gap_layout(R, c.Ds[:1], c.pieces[:1])[:, 1].sum())
        assert seam == LA and {LA - 2, LA} <= set(c.first.tolist()) and LA - 1 in c.last
        assert (c.rec[:, 0] == 1).sum() == 3                                  # two substitutions, then a 100-byte deletion


# ------------------------------------------------------------------------------------------------ 2. long gaps
def first_diffs(GR: bytes, GD: bytes):
    """(first difference from the start, first difference from the end) of an unequal-length gap, capped at min length"""
    m = min(len(GR), len(GD))
    p = next((i for i in range(m) if GR[i] != GD[i]), m)
    s = next((i for i in range(m) if GR[len(GR) - 1 - i] != GD[len(GD) - 1 - i]), m)
    return p, s


def check_long_gaps(ctx, big: int = 10 * 1024, grid: int = 64):
    """unequal gaps of 4 KiB and `big` bytes whose first differences from the start and from the end lie in different CTAs,
    trims that overlap (min(p0, m - s) binds), insertions and deletions longer than a tile, an equal-length gap of more
    than two tiles that differs everywhere, and a call with more gap tiles than the grid of `grid` CTAs"""
    n = max(3 * big, 60_000)
    R = bytearray(bases(n + 2 * big, 202))
    a2 = n // 2
    R[a2:a2 + 6000] = b"A" * 6000                                              # a poly-A stretch for the overlapping trims
    R = bytes(R)
    for nr, g0 in ((TILE, TILE - 1000), (big, 0)):
        a = 2 * TILE
        off = nr // 8
        GR = R[a:a + nr]
        GD = GR[:off] + GR[off + 50:]
        lead = flipped(R[:g0])
        c = Call(ctx, R, [hand_file(tokens(lead, (g0, a - g0), GD, (a + nr, len(R) - a - nr)))])
        p, s = first_diffs(GR, GD)
        row = c.layout[1]
        assert row[2:].tolist() == [nr - 50, nr] and (row[0] + p) // TILE != (row[0] + s) // TILE, (row.tolist(), p, s)
    # overlapping trims: 5,000 A's for 6,000 A's, so p0 = s = m
    c = Call(ctx, R, [hand_file(tokens((0, a2), b"A" * 5000, (a2 + 6000, len(R) - a2 - 6000)))])
    p, s = first_diffs(R[a2:a2 + 6000], b"A" * 5000)
    assert p == s == 5000 and len(c.whole[0]) == 1
    # a pure deletion and a pure insertion longer than a tile, an equal-length gap differing everywhere over > 2 tiles
    a = 3 * TILE + 5
    c = Call(ctx, R, [hand_file(tokens((0, a), (a + TILE + 700, len(R) - a - TILE - 700))),
                      hand_file(tokens((0, a), bases(TILE + 900, 7), (a, len(R) - a))),
                      hand_file(tokens((0, a), flipped(R[a:a + 2 * TILE + 300]), (a + 2 * TILE + 300, len(R) - a - 2 * TILE - 300)))])
    assert [len(W) for W in c.whole] == [1, 1, 1] and c.whole[2][0, 1] - c.whole[2][0, 0] == 2 * TILE + 300
    # more gap tiles than CTAs: a long deletion, then substitutions in tiles past the grid
    R2 = bases(grid * TILE + 40_000, 203)
    cut = grid * TILE + 10_000
    body = tokens((0, 1000), (1000 + cut, 5000), other(R2[6000 + cut]), (6001 + cut, 3000), other(R2[9001 + cut]),
                  (9002 + cut, len(R2) - 9002 - cut))
    c = Call(ctx, R2, [hand_file(body)])
    assert c.tiles() > grid and c.first.min() // TILE >= grid and len(c.whole[0]) == 3


# ------------------------------------------------------------------------------------------------ 3. scan sizes
def segments(c: "Call") -> int:
    """the segments of a single local-mode archive of one-byte copies and one-byte literals: its copies and literal bytes"""
    return len(c.pieces[0]) + sum(1 for d, r in zip(c.Ds[0], c.R) if d != r)


def scan_body(R: bytes, nseg: int, every: int = 0, snps: int | None = None) -> bytes:
    """nseg segments over R[:nseg]: one-byte copies, with a substituted literal byte at every `every`-th position among
    the first `snps` segments -> nseg + 1 elements"""
    out, prev = [], 0
    snps = nseg if snps is None else snps
    for i in range(nseg):
        if every and i < snps and i % every == every - 1:
            out.append(other(R[i]))
        else:
            out.append(b"(%d,1)" % (i - prev)); prev = i
    return b"".join(out)


def far_right_body(R: bytes, J: int, after: int) -> bytes:
    """one-byte copies (a substitution every 4th), then at segment J a copy of the last 100 bytes of R, then `after`
    one-byte copies that it clips entirely"""
    body = scan_body(R, J, 4)
    prev = max((i for i in range(J) if i % 4 != 3), default=0)
    far = len(R) - 100
    out = [body, b"(%d,100)" % (far - prev)]
    prev = far
    for i in range(J, J + after):
        out.append(b"(%d,1)" % (i - prev)); prev = i
    return b"".join(out)


def check_scan_sizes(ctx, big: bool = True):
    """element counts (segments + 1), record counts and window counts on both sides of the scan tile (1,024) and, with
    big, of the top-scan chunk (262,144); a far-right copy first, just before a scan-tile edge and just before a chunk
    edge, followed by copies it clips (the max-scan carry)"""
    sizes = [STILE - 1, STILE, STILE + 1] + ([CHUNK - 1, CHUNK, CHUNK + 1, CHUNK + STILE + 3] if big else [])
    R = bases(2 * CHUNK + 60_000 if big else 8000, 303)
    for ne in sizes:                                                          # elements: ne - 1 segments
        c = Call(ctx, R, [hand_file(scan_body(R, ne - 1, 2, snps=min(ne - 1, 2000)))])
        assert segments(c) == ne - 1
    for nrec in sizes:                                                        # records: nrec - 1 substitutions + the deletion at the end
        c = Call(ctx, R, [hand_file(scan_body(R, 2 * nrec - 1, 2))])
        assert len(c.rec) == nrec
    A = hand_file(scan_body(R, 6000, 5))
    rng = random.Random(5)
    for nw in sizes:
        w = [(0, s, s + rng.choice([0, 1, 7, 40])) for s in (rng.randrange(6000) for _ in range(nw))]
        c = Call(ctx, R, [A], w)
        assert len(c.windows) == nw and len(c.rec) > 0
    for J in [0, STILE - 1] + ([CHUNK - 1] if big else []):
        after = 2 * CHUNK + 1000 - J if big else 2 * STILE + 100
        c = Call(ctx, R, [hand_file(far_right_body(R, J, after))])
        P = c.pieces[0]
        assert P[J - J // 4, 1] == len(R) - 100 and len(P) == J - J // 4 + 1 + after
        assert len(vl.anchors(R, c.Ds[0], P)) == len(P) - after + 1          # every copy after the far one is clipped away


# ------------------------------------------------------------------------------------------------ 4. global-mode N runs
def n_reference():
    """R starting and ending with N, runs of 30 and 1, lowercase n (a base, not a run) -> (R, its N-stripped form)"""
    A, B, C, E = (bases(1000, s) for s in (41, 42, 43, 44))
    R = b"N" * 5 + A + b"N" * 30 + B + b"N" + C + b"nnnn" + E + b"N" * 7
    return R, R.replace(b"N", b"")


def check_global_n_runs(ctx):
    """hand-written global files: copies spanning one and many reference N runs, starting and ending on N-run edges of
    either sequence, a target and a reference N run at one split point, clip points on N-run edges, a file whose anchors
    fill the host bound nseg + 1 + n_k + rn_k exactly, a reference with no N, lowercase n in R and D"""
    R, S = n_reference()                                                      # stripped: A [0,1000) B [1000,2000) C [2000,3000) nnnn E [3004,4004)
    files = [
        global_file(tokens((0, len(S)))),                                     # every reference N run inside one copy
        global_file(tokens((500, 1000))),                                     # one run
        global_file(tokens((1000, 500), (2000, 1000), (1500, 500), (3000, 1004))),   # starts and ends on reference run edges
        global_file(tokens((0, 2000)), run_list([(1000, 20)])),               # a target run at the reference run's split point
        global_file(tokens((0, 700), (700, 300)), run_list([(0, 5), (705, 10)])),     # D starts with N; a copy starts on a target run edge
        global_file(tokens((0, 1000), b"ACGTn", (1000, 3004)), run_list([(995, 1), (1010, 12), (4022, 3)]), run_list([(990, 40)])),
        global_file(tokens((0, 1000), (500, 1200), (1500, 500), (1800, 700))),       # clip points M = 1000 and 2000: run edges
        global_file(tokens((2000, 3), b"GG", (10, 2990)), b""),
    ]
    c = Call(ctx, R, files, modes=[1] * len(files))
    assert all(len(W) for W in c.whole)
    # a target run and a reference run cut the copy at the same point: one cut, not two
    P3 = c.pieces[3]
    assert P3[:, 2].tolist() == [1000, 1000]
    # the anchors fill the host bound exactly (no leading or trailing reference run, target runs away from its runs)
    R2 = S[:1000] + b"N" * 30 + S[1000:2000] + b"N" * 2 + S[2000:3000]
    f = global_file(tokens((0, 3000)), run_list([(500, 3), (2503, 4)]))
    c = Call(ctx, R2, [f], modes=[1])
    nseg, n_k, rn_k = 1, 2, 2
    assert len(vl.anchors(R2, c.Ds[0], c.pieces[0])) == nseg + 1 + n_k + rn_k
    # a global archive against a reference with no N
    R3 = S[:3000]
    Call(ctx, R3, [global_file(tokens((0, 1500), b"TT", (1502, 1498)), run_list([(700, 9)])), global_file(tokens((0, 3000)))], modes=[1, 1])
    ctx.clear_reference()


def check_nrun_cache(ctx):
    """the reference N-run table over one context's life: a local call before the first global one; reference A, then B
    of the same length with an N run moved; A, clear, A"""
    R, S = n_reference()
    i = R.index(b"N" * 30)
    RB = R[:i] + R[i + 30:i + 45] + b"N" * 30 + R[i + 45:]                  # the 30-N run 15 bytes to the right
    assert len(RB) == len(R) and RB.count(b"N") == R.count(b"N")
    g = [global_file(tokens((0, len(S)))), global_file(tokens((900, 200), (1990, 30)), run_list([(100, 2)]))]
    loc = hand_file(tokens((0, 3000), b"ACG", (3003, len(R) - 3003)))
    ctx.set_reference(R)
    Call(ctx, R, [loc], set_ref=False, modes=[0])
    a = Call(ctx, R, g, set_ref=False, modes=[1, 1])
    b = Call(ctx, RB, g, modes=[1, 1])
    assert not np.array_equal(a.rec, b.rec)
    Call(ctx, R, g + [loc], modes=[1, 1, 0])
    ctx.clear_reference()
    a2 = Call(ctx, R, g, modes=[1, 1])
    assert np.array_equal(a.rec, a2.rec) and a.alt == a2.alt
    ctx.clear_reference()


# ------------------------------------------------------------------------------------------------ 6. many archives
def random_file(r: random.Random, R: bytes, glob: bool) -> bytes:
    """a small file of copies, substitutions, insertions and deletions (global: with target N runs)"""
    body, at = [], 0
    while at < len(R) - 50:
        n = r.randint(20, 400)
        body.append((at, min(n, len(R) - at)))
        at += n
        kind = r.randrange(4)
        if kind == 0 and at < len(R):
            body.append(other(R[at])); at += 1
        elif kind == 1:
            body.append(bases(r.randint(1, 5), r.randrange(1 << 30)))
        elif kind == 2:
            at += r.randint(1, 6)
    body = tokens(*[b if isinstance(b, bytes) else (b[0], b[1]) for b in body if isinstance(b, bytes) or b[1] > 0 and b[0] < len(R)])
    if glob:
        return global_file(body, run_list([(r.randrange(10, 200), r.randint(1, 5)), (r.randrange(600, 900), 3)]))
    return hand_file(body)


def check_many_archives(ctx, n: int = 300):
    """left-alignment bounded within an archive only (archive k ends with a record near len(R), archive k + 1 starts with
    indels in a repeat at the start of R); n small local and global archives named out of order and as a subset; one call
    equals per-archive calls"""
    R = b"A" * 12 + bases(3000, 606)
    L = len(R)
    tail = hand_file(tokens((0, L - 40), other(R[L - 40]), (L - 39, 39)))
    cross = [tail, hand_file(tokens((0, 5), (6, L - 6))), tail, hand_file(tokens((0, 6), b"A", (6, L - 6))),
             tail, global_file(tokens((0, 7), (9, L - 9)))]
    c = Call(ctx, R, cross, modes=[0, 0, 0, 0, 0, 1])
    assert [c.rec[c.rec[:, 0] == k][0, 1] for k in (1, 3, 5)] == [0, 0, 0]
    r = random.Random(66)
    files = [random_file(r, R, k % 7 == 3) for k in range(n)]
    subset = r.sample(range(n), n * 2 // 3)
    w = [(k, r.randrange(L // 2), L) for k in subset] + [(k, 0, r.randrange(L)) for k in subset[::5]] + [(subset[0], 0, L)]
    Call(ctx, R, files, w)
    every = Call(ctx, R, files)
    for k in r.sample(range(n), 12):
        one = Call(ctx, R, [files[k]], set_ref=False)
        mine = every.rec[every.rec[:, 0] == k]
        assert np.array_equal(mine[:, 1:5], one.rec[:, 1:5])
        assert b"".join(every.alt[o:o + e - s] for o, s, e in mine[:, [5, 3, 4]].tolist()) == one.alt
    ctx.clear_reference()


# ------------------------------------------------------------------------------------------------ 7. bytes and token forms
def check_odd_bytes(ctx):
    """D holding every byte value but '\\n', the odd-byte target of the search tests, an R with lowercase and IUPAC bytes"""
    ref, inter, D = every_byte_archive()
    c = Call(ctx, ref, [inter])
    assert len(c.rec) and max(c.alt) >= 0x80
    ref2, inter2, mode2, _, D2 = odd_target_archive()
    c = Call(ctx, ref2, [inter2], modes=[mode2])
    assert max(c.alt) >= 0x80 and min(c.alt) < 0x20
    from sccg_genome_compression_b200 import synth
    R = bytearray(bases(20_000, 707))
    rr = random.Random(7)
    for i in range(0, len(R), 37):
        R[i] = rr.choice(b"RYSWKMBDHVryswkmbdhv")
    for a in range(500, len(R), 3000):
        R[a:a + 700] = bytes(R[a:a + 700]).lower()
    R = bytes(R)
    t = np.frombuffer(R, np.uint8).copy()
    synth.substitute(np.random.default_rng(7), t, 0.003)
    tgt = t.tobytes()[:9000] + b"GATTACA" + t.tobytes()[9000:15000] + t.tobytes()[15010:]
    rc, inter3, mode3 = ol.orc_compress(R, tgt, b">iupac")
    assert rc == 0
    Call(ctx, R, [inter3], modes=[mode3])
    ctx.clear_reference()


def token_form_files(slice_sweep: int = 1):
    """(R, record file) of every body of the token table and the sweep (every slice_sweep-th) that the oracle decodes and
    the library must accept, of a fuzz corpus slice, and of the tolerance cases"""
    out = []
    sweep = tg.sweep_bodies()[::slice_sweep]
    for body in tg.token_table() + sweep:
        rc, _ = ol.orc_reconstruct(tg.TABLE_REF, body, b"", b"")
        if rc == 0 and tg.pinned_class(body) is None and b"\n" not in body:
            out.append((tg.TABLE_REF, hand_file(body)))
    for ref, body, nlist, low in tg.fuzz_corpus([1, 2]):
        rc, _ = ol.orc_reconstruct(ref, body, nlist, low)
        if rc == 0 and tg.pinned_class(body) is None:
            out.append((ref, b">f\n" + low + b"\n" + (nlist or b",") + b"\n" + body + b"\n"))
    tref = bases(9000, 808)
    for body, nlist, low in tolerance_cases():
        inter = b">tol\n" + low + b"\n" + nlist + b"\n" + body + b"\n"
        if ol.orc_decompress(tref, inter)[0] == 0:
            out.append((tref, inter))
    return out


def check_token_forms(ctx, slice_sweep: int = 1, per_call: int = 250):
    """every decodable body of token_grammar_cases (table, sweep, fuzz slice) and the tolerance cases, many archives a call"""
    by_ref = {}
    for R, inter in token_form_files(slice_sweep):
        by_ref.setdefault(R, []).append(inter)
    n = 0
    for R, files in by_ref.items():
        for b in range(0, len(files), per_call):
            Call(ctx, R, files[b:b + per_call])
            n += len(files[b:b + per_call])
    assert n > 400
    ctx.clear_reference()


# ------------------------------------------------------------------------------------------------ 8. output paths
def check_output_paths(ctx):
    """windows with no records at the start, middle and end of the list; [len(R), len(R)) with and without insertions at
    len(R); a call whose records are all deletions (alt_len 0, alt NULL); count-only calls with records but no ALT bytes"""
    R = bases(5000, 909)
    L = len(R)
    A = hand_file(tokens((0, 1000), other(R[1000]), (1001, 2000), other(R[3001]), (3002, L - 3002), b"GG"))
    B = hand_file(tokens((0, 1000), other(R[1000]), (1001, L - 1001)))
    w = [(0, 0, 500), (1, 0, 10), (0, 900, 1100), (0, 1500, 2500), (1, 1200, 1300), (0, 2900, 3100), (0, L, L), (1, L, L),
         (0, 4000, 4500), (1, 2000, L - 1), (0, 10, 10)]
    c = Call(ctx, R, [A, B], w)
    per = np.bincount(c.rec[:, 0], minlength=len(w)).tolist()
    assert per == [0, 0, 1, 0, 0, 1, 1, 0, 0, 0, 0], per
    # all deletions: no ALT bytes, so alt may be NULL
    Dl = hand_file(tokens((0, 100), (110, 2000), (2150, L - 2150)))
    c = Call(ctx, R, [Dl])
    assert len(c.rec) == 2 and c.alt == b""
    arch = ctx.open_archive(Dl)
    try:
        rc, n, na, out, _ = raw_call(ctx, [arch], [(0, 0, L)], 4, 0, null_alt=True)
        assert (rc, n, na) == (0, 2, 0)
        got = np.stack([out[f][:n] for f, _ in ctx._VARIANT], axis=1)
        assert np.array_equal(got, c.rec)
        assert raw_call(ctx, [arch], [(0, 0, L)], 0, 0, null_vars=True, null_alt=True)[:3] == (0, 2, 0)
        assert raw_call(ctx, [arch], [(0, 0, 50), (0, 200, 300)], 0, 0, null_alt=True)[:3] == (0, 0, 0)
    finally:
        arch.close()
    ctx.clear_reference()


def test_thread_tile_edges(ctx):
    check_thread_tile_edges(ctx)


def test_long_gaps(ctx):
    check_long_gaps(ctx, grid=EMU_GRID)


def test_scan_sizes(ctx):
    check_scan_sizes(ctx)


def test_global_n_runs(ctx):
    check_global_n_runs(ctx)


def test_nrun_cache(ctx):
    check_nrun_cache(ctx)


def test_many_archives(ctx):
    check_many_archives(ctx)


def test_odd_bytes(ctx):
    check_odd_bytes(ctx)


def test_token_forms(ctx):
    check_token_forms(ctx)


def test_output_paths(ctx):
    check_output_paths(ctx)
