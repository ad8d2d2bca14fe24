"""TEST INFRASTRUCTURE ONLY: a reference implementation of sccg_archive_variants (include/sccg.h, steps 1-5) in Python and
numpy, from the record file and R alone: the pieces come from the oracle's own token loop (tests/pieces_probe.c), never from
the library.  Also the invariant and splice check of the header, the window filter and a VCF renderer for the CLI tests."""
from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

import numpy as np

from oracle_lib import orc_decompress, prepare_reference, split_intermediate

HERE = Path(__file__).resolve().parent
_lib = None
_UP = bytes(c - 32 if 97 <= c <= 122 else c for c in range(256))


def up(b: bytes) -> bytes:
    return b.translate(_UP)


def pieces_lib(directory: Path | None = None):
    """the oracle's token loop reporting its copies (built once per process into a temporary directory)"""
    global _lib
    if _lib is None:
        import tempfile
        d = Path(directory or tempfile.mkdtemp(prefix="pieces_probe"))
        so = d / "libpieces_probe.so"
        subprocess.check_call(["gcc", "-O2", "-shared", "-fPIC", "-w", str(HERE / "pieces_probe.c"), "-o", str(so)])
        lib = C.CDLL(str(so))
        lp = C.POINTER(C.c_long)
        lib.orc_reconstruct_pieces.argtypes = [C.c_char_p, C.c_long, C.c_char_p, C.c_long, C.c_char_p, C.c_long,
                                               C.POINTER(lp), lp, lp, C.POINTER(lp), lp]
        lib.orc_free.argtypes = [C.c_void_p]
        _lib = lib
    return _lib


def decoded(ref_raw: bytes, intermediate: bytes) -> bytes:
    """D: the oracle's decoded sequence (no header line, no newlines)"""
    rc, text = orc_decompress(ref_raw, intermediate)
    assert rc == 0, rc
    return text.split(b"\n", 1)[1].replace(b"\n", b"")


def copy_pieces(ref_raw: bytes, intermediate: bytes, D: bytes) -> np.ndarray:
    """step 1: the copy pieces (x, p, l) in raw D / R coordinates, in D order, as an (n, 3) int64 array"""
    _, _, nline, body = split_intermediate(intermediate)
    local = nline == b","
    prep = prepare_reference(ref_raw, nline)
    lib = pieces_lib()
    pc, ins = C.POINTER(C.c_long)(), C.POINTER(C.c_long)()
    npc, rec_len, nins = C.c_long(), C.c_long(), C.c_long()
    rc = lib.orc_reconstruct_pieces(prep, len(prep), body, len(body), b"" if local else nline, 0 if local else len(nline),
                                    C.byref(pc), C.byref(npc), C.byref(rec_len), C.byref(ins), C.byref(nins))
    assert rc == 0, rc
    P = np.ctypeslib.as_array(pc, shape=(npc.value * 3,)).reshape(-1, 3).astype(np.int64).copy() if npc.value else np.zeros((0, 3), np.int64)
    I = np.ctypeslib.as_array(ins, shape=(nins.value,)).astype(np.int64).copy() if nins.value else np.zeros(0, np.int64)
    lib.orc_free(C.cast(pc, C.c_void_p)); lib.orc_free(C.cast(ins, C.c_void_p))
    if local:
        return P
    # global mode: record-stream position s is D position dmap[s]; stripped reference position q is raw position rmap[q]
    keep = np.ones(len(D), dtype=bool)
    keep[I[I < len(D)]] = False
    dmap = np.flatnonzero(keep)
    rmap = np.flatnonzero(np.frombuffer(ref_raw, dtype=np.uint8) != ord("N"))
    out = []
    for s, q, l in P.tolist():
        dp, rp = dmap[s:s + l], rmap[q:q + l]
        cuts = np.flatnonzero((np.diff(dp) != 1) | (np.diff(rp) != 1)) + 1
        b = 0
        for c in list(cuts) + [l]:
            out.append((int(dp[b]), int(rp[b]), int(c - b)))
            b = c
    return np.array(out, dtype=np.int64).reshape(-1, 3)


def variants_whole(ref_raw: bytes, intermediate: bytes, D: bytes | None = None) -> np.ndarray:
    """steps 1-4: the records of the whole archive, an (n, 4) int64 array [pos, end, d_start, d_end]"""
    if D is None:
        D = decoded(ref_raw, intermediate)
    return variants_from_pieces(ref_raw, D, copy_pieces(ref_raw, intermediate, D))


def anchors(R: bytes, D: bytes, P: np.ndarray) -> list:
    """step 2: the anchors [x, p, l] of the copy pieces P, then the sentinel [len(D), len(R), 0]"""
    if len(P):
        x, p, l = P[:, 0], P[:, 1], P[:, 2]
        M = np.concatenate([[0], np.maximum.accumulate(p + l)[:-1]])
        s = np.maximum(0, M - p)
        a = s < l
        anc = np.stack([x[a] + s[a], p[a] + s[a], l[a] - s[a]], axis=1)
    else:
        anc = np.zeros((0, 3), np.int64)
    return np.concatenate([anc, [[len(D), len(R), 0]]]).astype(np.int64).tolist()


def gap_layout(R: bytes, Ds: list[bytes], pieces: list[np.ndarray]) -> np.ndarray:
    """the gap-byte space of one call over the archives with D = Ds[k] and copy pieces pieces[k], in that order: per gap
    (goff, width, nd, nr), goff the exclusive prefix sum of width = max(nd, nr) over every gap of every archive (zero-width
    gaps included) -> an (n, 4) int64 array"""
    rows = []
    for D, P in zip(Ds, pieces):
        lx = lp = 0
        for ax, ap, al in anchors(R, D, P):
            rows.append((ax - lx, ap - lp))
            lx, lp = ax + al, ap + al
    nd = np.array([r[0] for r in rows], np.int64)
    nr = np.array([r[1] for r in rows], np.int64)
    w = np.maximum(nd, nr)
    goff = np.concatenate([[0], np.cumsum(w)[:-1]]).astype(np.int64)
    return np.stack([goff, w, nd, nr], axis=1).reshape(-1, 4)


def record_gap_bytes(layout: np.ndarray, R: bytes, Ds: list[bytes], pieces: list[np.ndarray], whole: list[np.ndarray]):
    """where the substitution records of whole[k] (variants_whole) fall in the gap-byte space of gap_layout, for the gaps of
    equal length: -> (first byte, last byte) of each record's run of differences"""
    first, last = [], []
    g = 0
    for D, P, W in zip(Ds, pieces, whole):
        lx = lp = 0
        for ax, ap, al in anchors(R, D, P):
            if ax - lx == ap - lp:
                for pos, end, ds, de in W[(W[:, 0] >= lp) & (W[:, 1] <= ap) & (W[:, 2] >= lx) & (W[:, 3] <= ax)].tolist():
                    if pos - lp == ds - lx and end - pos == de - ds:
                        first.append(int(layout[g, 0]) + pos - lp); last.append(int(layout[g, 0]) + end - lp - 1)
            g += 1
            lx, lp = ax + al, ap + al
    return np.array(first, np.int64), np.array(last, np.int64)


def variants_from_pieces(R: bytes, D: bytes, P: np.ndarray) -> np.ndarray:
    UR, UD = up(R), up(D)
    anc = anchors(R, D, P)                                                  # step 2
    # step 3: gaps
    recs = []
    lx = lp = 0
    for ax, ap, al in anc:
        GR, GD = UR[lp:ap], UD[lx:ax]
        if GR != GD:
            if len(GR) == len(GD):
                d = np.frombuffer(GR, np.uint8) != np.frombuffer(GD, np.uint8)
                e = np.diff(np.concatenate([[0], d.astype(np.int8), [0]]))
                for b, f in zip(np.flatnonzero(e == 1), np.flatnonzero(e == -1)):
                    recs.append([lp + b, lp + f, lx + b, lx + f])
            else:
                m = min(len(GR), len(GD))
                suf = 0
                while suf < m and GR[len(GR) - 1 - suf] == GD[len(GD) - 1 - suf]:
                    suf += 1
                pre = 0
                while pre < m - suf and GR[pre] == GD[pre]:
                    pre += 1
                recs.append([lp + pre, ap - suf, lx + pre, ax - suf])
        lx, lp = ax + al, ap + al
    # step 4: left-alignment, bounded by the previous record's step-3 end
    out = []
    prev_end = 0
    for pos, end, ds, de in recs:
        bound = prev_end
        prev_end = end
        dele, ins = de == ds, end == pos
        if dele != ins:
            while pos > bound:
                last = UR[end - 1] if dele else UD[de - 1]
                if UR[pos - 1] != last:
                    break
                pos -= 1; end -= 1; ds -= 1; de -= 1
        out.append([pos, end, ds, de])
    return np.array(out, dtype=np.int64).reshape(-1, 4)


def filter_windows(whole: list[np.ndarray], Ds: list[bytes], windows, rlen: int) -> tuple[np.ndarray, bytes]:
    """step 5 over whole-archive records (whole[k] for archive k): -> ((n, 6) records, ALT bytes) as the library lays them out"""
    rows, alt = [], bytearray()
    for w, (k, s, e) in enumerate(windows):
        W = whole[k]
        e = e + 1 if e == rlen else e                                      # (insertions at len(R) belong to a window ending there)
        for pos, end, ds, de in W[(W[:, 0] >= s) & (W[:, 0] < e)].tolist():
            rows.append([w, pos, end, ds, de, len(alt)])
            alt += up(Ds[k][ds:de])
    return np.array(rows, dtype=np.int64).reshape(-1, 6), bytes(alt)


def check_invariants(R: bytes, D: bytes, recs: np.ndarray, alt: bytes | None = None) -> None:
    """the invariants of include/sccg.h for the records of one archive ([.., pos, end, d_start, d_end, alt_off] in the last
    five columns or [pos, end, d_start, d_end]); splicing their ALTs into up(R) must give up(D)"""
    UR, UD = up(R), up(D)
    r4 = recs[:, -5:-1] if recs.shape[1] >= 5 else recs
    out = bytearray()
    pe = de_prev = 0
    for j, (pos, end, ds, de) in enumerate(r4.tolist()):
        assert pos >= pe and ds >= de_prev, (j, pos, pe, ds, de_prev)
        assert 0 <= pos <= end <= len(R) and 0 <= ds <= de <= len(D)
        assert UR[pe:pos] == UD[de_prev:ds], j
        assert (end - pos) + (de - ds) > 0
        a = UD[ds:de]
        if alt is not None:
            off = int(recs[j, -1])
            assert alt[off:off + de - ds] == a
        ref = UR[pos:end]
        if len(ref) == len(a):
            assert all(x != y for x, y in zip(ref, a)), j
        elif ref and a:
            assert ref[0] != a[0] and ref[-1] != a[-1], j
        out += UR[pe:pos] + a
        pe, de_prev = end, de
    out += UR[pe:]
    assert bytes(out) == UD


def kinds(recs: np.ndarray) -> dict:
    """record counts by kind: substitution, insertion, deletion, complex"""
    r4 = recs[:, -5:-1] if recs.shape[1] >= 5 else recs
    lr, ld = r4[:, 1] - r4[:, 0], r4[:, 3] - r4[:, 2]
    return {"substitution": int(((lr == ld)).sum()), "insertion": int(((lr == 0) & (ld > 0)).sum()),
            "deletion": int(((ld == 0) & (lr > 0)).sum()), "complex": int(((lr != ld) & (lr > 0) & (ld > 0)).sum())}
