"""The diagonal-hypothesis path of the local segment matcher (`lm_diag_parse`) on the CPU emulator, judged by the oracle.

A near-identical segment pair is parsed in closed form from its mismatch positions, once a proof shows that no k-mer the parse
looks up occurs in r off the diagonal.  The proof hashes the 8-byte chunks t[u..u+8), u = j..j+3, of every looked-up window j
and probes the 4-aligned chunks of r.  The cases below plant exactly the occurrences it has to find (at every phase of p
against the 4- and 8-byte grids, at both ends of the segment), sit on the limits of the path (30 / 31 mismatching symbols, 16 / 17
mismatching words, 32 looked-up windows), force equal chunks at different positions, and run the shapes that reach the path
in other ways (short last pairs, lowercase and N in the target, k other than 14, two-phase launches, the path switched off).
Shared with tests/test_gpu_diag_proof.py."""
import random

import pytest

import oracle_lib as ol
from emu_lib import emu_context

L = 1000
K = 14
# p of the planted occurrence: every phase against the 8-byte grid at the start, in the middle and at the end of the segment
# (p = 0; p = 986 = L - k)
PLANT_P = list(range(0, 8)) + list(range(203, 211)) + list(range(979, 987))


def _other(c: int) -> int:
    return {65: 67, 67: 71, 71: 84, 84: 65}.get(c, 65)


def _random_seg(r: random.Random, n: int = L, alphabet: bytes = b"ACGT") -> bytearray:
    return bytearray(r.choice(alphabet) for _ in range(n))


def planted_pair(p: int, kind: str, seed=0, n: int = L) -> tuple[bytes, bytes]:
    return planted_case(p, kind, seed, n)[:2]


def planted_case(p: int, kind: str, seed=0, n: int = L) -> tuple[bytes, bytes, int]:
    """(r, t, j): one segment pair whose looked-up window t[j..j+k) also occurs in r at p, off the diagonal.
    kind "clean": j starts a mismatch-free interval of 20 symbols; the planted copy runs 6 symbols past its end, so the
    reference's parse takes p (longer than the diagonal match).  kind "mutated": j is a mismatch; the planted copy turns the
    literal of the diagonal parse into a match.  The copy goes into r and t alike, so the diagonal stays clean there."""
    r = random.Random(repr(("dvp", p, kind, seed, n)))
    ref = _random_seg(r, n)
    tgt = bytearray(ref)
    m1 = (n * 6 // 10 if p < n // 2 else min(100, n // 10)) + r.randrange(8)
    tgt[m1] = _other(ref[m1])
    if kind == "clean":
        tgt[m1 + 21] = _other(ref[m1 + 21])
        j, ln = m1 + 1, 26
    else:
        j, ln = m1, 20
    ln = min(ln, n - p)
    piece = bytes(tgt[j:j + ln])
    ref[p:p + ln] = piece
    tgt[p:p + ln] = piece
    return bytes(ref), bytes(tgt), j


def snp_pair(positions, seed=0, n: int = L, alphabet: bytes = b"ACGT", plant: bool = False) -> tuple[bytes, bytes]:
    """r random, t = r with a substitution at every listed position; plant: a mutated window's k-mer copied to a free place"""
    r = random.Random(repr(("snp", tuple(positions), seed, n, alphabet)))
    ref = _random_seg(r, n, alphabet)
    tgt = bytearray(ref)
    for q in positions:
        tgt[q] = _other(ref[q]) if alphabet == b"ACGT" else r.choice([c for c in alphabet if c != ref[q]] or [67])
    if plant and positions:
        m = r.choice(list(positions))
        if m + K <= n:
            free = [q for q in range(0, n - K + 1) if all(abs(q - x) > K + 1 for x in positions)]
            if free:
                at = r.choice(free)
                piece = bytes(tgt[m:m + K])
                ref[at:at + K] = piece
                tgt[at:at + K] = piece
    return bytes(ref), bytes(tgt)


def edge_snps(r: random.Random, n: int = L) -> list[int]:
    """substitutions next to the segment borders, closer together than k, and windows that start at L - k"""
    pool = [0, 1, 2, 7, 8, 13, 14, 15, n - K - 1, n - K, n - K + 1, n - 8, n - 2, n - 1]
    pos = set(q for q in r.sample(pool, r.randint(1, 5)) if 0 <= q < n)
    for _ in range(r.randint(0, 3)):                                    # a cluster: gaps < k
        c = r.randrange(n)
        pos.update(q for q in range(c, c + r.randint(2, 40), r.randint(1, 13)) if q < n)
    if r.random() < 0.3:
        pos.update(q for q in range(r.randrange(n // 2), n, r.randint(15, 60)))   # evenly spaced, many windows
    return sorted(pos)


def run_snps(start: int, count: int) -> list[int]:
    return list(range(start, start + count))


def word_pairs(words: int, first: int = 40) -> list[int]:
    """`words` mismatching 8-byte words with as few looked-up windows as possible: adjacent symbols across a word border"""
    pos = []
    w = first // 8
    while len(set(q // 8 for q in pos)) + 2 <= words:
        pos += [8 * w + 7, 8 * w + 8]
        w += 6
    if len(set(q // 8 for q in pos)) < words:
        pos.append(8 * w + 3)
    return pos


def low_complexity_pair(kind: int, seed=0) -> tuple[bytes, bytes]:
    """equal 8-byte chunks at different positions of t (the table cannot hold both) and crowded slots"""
    r = random.Random(repr(("lowc", kind, seed)))
    if kind == 0:
        ref = bytearray(b"A" * L)
    elif kind == 1:
        unit = bytes(r.choice(b"ACGT") for _ in range(r.choice([2, 3, 4, 6, 8])))
        ref = bytearray((unit * L)[:L])
    elif kind == 2:
        ref = _random_seg(r, L, b"AC")
    else:                                                               # random, with a periodic stretch around the looked-up windows
        ref = _random_seg(r, L)
        unit = bytes(r.choice(b"ACGT") for _ in range(r.choice([1, 2, 7, 8])))
        at = r.randrange(0, 600)
        ref[at:at + 300] = (unit * 300)[:300]
    tgt = bytearray(ref)
    for q in r.sample(range(L), r.randint(1, 6)):
        tgt[q] = r.choice([c for c in b"ACGT" if c != ref[q]])
    return bytes(ref), bytes(tgt)


def looked_up_windows(ref: bytes, tgt: bytes, k: int = K) -> list[int]:
    """the windows the diagonal path looks up (its closed form of the greedy parse, for a pair with few mismatches)"""
    n = len(tgt)
    mis = [q for q in range(n) if ref[q] != tgt[q]]
    wins, a = [], 0
    for i, b in enumerate(mis + [n]):
        if b - a >= k:
            wins.append(a)
        else:
            wins += range(a, min(b, n - k + 1))
        if i < len(mis) and b <= n - k:
            wins.append(b)
        a = b + 1
    return wins


def proof_slot(tgt: bytes, u: int) -> tuple[int, int]:
    """(table slot under the first slot function, entry) of the proof's chunk t[u..u+8) (dv_hash, dv_slot)"""
    c = tgt[u:u + 8]
    h = (((int.from_bytes(c[:4], "little") * 0x9E3779B1) + int.from_bytes(c[4:], "little")) * 0x85EBCA6B) & 0xffffffff
    return h >> 22, (h & ~1023 & 0xffffffff) | 1024 | u


def colliding_planted_pair(p: int, kind: str) -> tuple[bytes, bytes]:
    """planted_pair whose chunk that reveals the planted occurrence shares its table slot with another looked-up chunk: the
    table is rebuilt under the second slot function (or the generic path runs), and the occurrence is still found"""
    for seed in range(20000):
        ref, tgt, j = planted_case(p, kind, ("slot", seed))
        us = set(w + o for w in looked_up_windows(ref, tgt) for o in range(4))
        u_star = j + (-p) % 4                                          # u = j + (ceil4(p) - p)
        slot, ent = proof_slot(tgt, u_star)
        if any(proof_slot(tgt, u)[0] == slot and proof_slot(tgt, u)[1] != ent for u in us if u != u_star):
            return ref, tgt
    raise AssertionError("no colliding case found")


def check_match(ctx, ref: bytes, tgt: bytes, k: int = K):
    exp = [(x.p, x.l, x.lit) for x in ol.orc_match_sequences(ref, tgt, k, 0, False, 0)]
    got = [(x.p, x.l, x.lit) for x in ctx.match_sequences(ref, tgt, k, 0, False, 0)]
    assert got == exp, (k, ref, tgt)


def check_file(ctx, ref: bytes, tgt: bytes, header: bytes = b">diag proof", compress=None):
    """compress: (ctx, ref, tgt, header) -> (file, mode); default the host-pointer entry point"""
    rc, exp, mode = ol.orc_compress(ref, tgt, header)
    assert rc == 0
    got, gmode = (compress or (lambda c, a, b, h: c.compress(a, b, h)))(ctx, ref, tgt, header)
    assert (gmode, got) == (mode, exp)


def compress_device_emu(ctx, ref: bytes, tgt: bytes, header: bytes):
    """the device-resident entry point under the emulator (device memory is host memory there)"""
    import numpy as np
    r = np.frombuffer(ref + bytes(64), dtype=np.uint8).copy(); t = np.frombuffer(tgt + bytes(64), dtype=np.uint8).copy()
    ptr, n, mode = ctx.compress_device(r.ctypes.data, len(ref), t.ctypes.data, len(tgt), header)
    return ctx.download(ptr, n), mode


def planted_file(seed) -> tuple[bytes, bytes]:
    """a file of segments that reach the diagonal path: planted occurrences of both kinds, edge and clustered SNPs, the
    limits, low-complexity segments, identical segments, and a short last pair"""
    r = random.Random(repr(("dvfile", seed)))
    refs, tgts = [], []
    for i in range(40):
        x = r.randrange(7)
        if x == 0:
            a, b = planted_pair(r.choice(PLANT_P), r.choice(["clean", "mutated"]), (seed, i))
        elif x == 1:
            a, b = snp_pair(edge_snps(r), (seed, i), plant=r.random() < 0.5)
        elif x == 2:
            a, b = snp_pair(run_snps(r.randrange(0, L - 31), r.choice([30, 31])), (seed, i), plant=r.random() < 0.5)
        elif x == 3:
            a, b = snp_pair(word_pairs(r.choice([16, 17])), (seed, i), plant=r.random() < 0.5)
        elif x == 4:
            a, b = low_complexity_pair(r.randrange(4), (seed, i))
        elif x == 5:
            a = bytes(_random_seg(r)); b = a
        else:
            a, b = snp_pair(sorted(r.sample(range(L), r.randint(1, 4))), (seed, i))
        refs.append(a); tgts.append(b)
    n = r.choice([14, 15, 100, 517, 999])
    a, b = snp_pair(edge_snps(r, n), (seed, "last"), n=n, plant=True)
    refs.append(a); tgts.append(b)
    return b"".join(refs), b"".join(tgts)


def lower_n_target(tgt: bytes, seed) -> bytes:
    """lowercase runs and N symbols in the target (the matcher upper-cases, N is just another symbol on the diagonal)"""
    r = random.Random(repr(("lowN", seed)))
    t = bytearray(tgt)
    for _ in range(r.randint(2, 8)):
        a = r.randrange(len(t)); b = min(len(t), a + r.randint(1, 900))
        t[a:b] = t[a:b].lower()
    for _ in range(r.randint(1, 6)):
        a = r.randrange(len(t)); b = min(len(t), a + r.randint(1, 3))
        t[a:b] = b"N" * (b - a)
    return bytes(t)


@pytest.fixture(params=[0, 1, 2], ids=["asc", "desc", "mixed"])
def sweep_order(request, monkeypatch):
    monkeypatch.setenv("SCCG_EMU_ORDER", str(request.param))
    return request.param


@pytest.fixture(scope="module")
def ctx():
    c = emu_context()
    yield c
    c.close()


@pytest.mark.parametrize("kind", ["clean", "mutated"])
@pytest.mark.parametrize("p", PLANT_P)
def test_planted_occurrence(ctx, p, kind):
    ref, tgt = planted_pair(p, kind)
    check_match(ctx, ref, tgt)


@pytest.mark.parametrize("kind", ["clean", "mutated"])
@pytest.mark.parametrize("p", PLANT_P[::2])
def test_planted_occurrence_behind_a_slot_collision(ctx, p, kind, sweep_order):
    """the chunk that reveals the occurrence shares a table slot (the emulator runs the lanes in three orders)"""
    check_match(ctx, *colliding_planted_pair(p, kind))


@pytest.mark.parametrize("seed", range(40))
def test_edge_and_clustered_snps(ctx, seed):
    r = random.Random(repr(("edge", seed)))
    ref, tgt = snp_pair(edge_snps(r), seed, plant=seed % 2 == 1)
    check_match(ctx, ref, tgt)


@pytest.mark.parametrize("plant", [False, True])
@pytest.mark.parametrize("count", [29, 30, 31])
def test_mismatch_symbol_limit(ctx, count, plant):
    for start in (0, 100, 501, L - count):
        ref, tgt = snp_pair(run_snps(start, count), start, plant=plant)
        check_match(ctx, ref, tgt)


@pytest.mark.parametrize("plant", [False, True])
@pytest.mark.parametrize("words", [15, 16, 17])
def test_mismatch_word_limit(ctx, words, plant):
    pos = word_pairs(words)
    assert len(set(q // 8 for q in pos)) == words
    ref, tgt = snp_pair(pos, words, plant=plant)
    check_match(ctx, ref, tgt)


@pytest.mark.parametrize("seed", range(3))
@pytest.mark.parametrize("kind", range(4))
def test_low_complexity_segments(ctx, kind, seed):
    ref, tgt = low_complexity_pair(kind, seed)
    check_match(ctx, ref, tgt)


@pytest.mark.parametrize("n", [14, 15, 21, 100, 517, 993, 999])
def test_short_last_pair(ctx, n):
    for seed in range(4):
        r = random.Random(repr(("short", n, seed)))
        ref, tgt = snp_pair(edge_snps(r, n), seed, n=n, plant=seed % 2 == 1)
        check_match(ctx, ref, tgt)
        if n > 40:
            ref, tgt = planted_pair(r.choice([0, n - K, n // 2]), ["clean", "mutated"][seed % 2], seed, n=n)
            check_match(ctx, ref, tgt)


@pytest.mark.parametrize("k", range(10, 17))
def test_other_k(ctx, k):
    r = random.Random(repr(("k", k)))
    for p in PLANT_P[::3]:
        check_match(ctx, *planted_pair(p, ["clean", "mutated"][p % 2], k), k=k)
    for seed in range(6):
        check_match(ctx, *snp_pair(edge_snps(r), (k, seed), plant=True), k=k)


@pytest.mark.parametrize("seed", range(3))
def test_files_lowercase_and_n(ctx, seed):
    ref, tgt = planted_file(seed)
    check_file(ctx, ref, tgt)
    check_file(ctx, ref, lower_n_target(tgt, seed))


@pytest.mark.parametrize("two_phase", [1, 0])
@pytest.mark.parametrize("seed", range(2))
def test_files_two_phase(ctx, seed, two_phase, monkeypatch):
    monkeypatch.setenv("SCCG_LM_TWO_PHASE_MIN", "0" if two_phase else "2000000000")
    ref, tgt = planted_file(("2ph", seed))
    check_file(ctx, ref, lower_n_target(tgt, seed), compress=compress_device_emu)


def test_no_diag_parity(ctx, monkeypatch):
    """the generic path alone (SCCG_NO_DIAG=1) writes the same files"""
    monkeypatch.setenv("SCCG_NO_DIAG", "1")
    plain = emu_context()
    try:
        for seed in range(2):
            ref, tgt = planted_file(("nodiag", seed))
            tgt = lower_n_target(tgt, seed)
            assert plain.compress(ref, tgt, b">x") == ctx.compress(ref, tgt, b">x")
            check_file(plain, ref, tgt, b">x")
    finally:
        plain.close()
