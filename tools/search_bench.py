"""Pattern search in open archives (sccg_archive_search) on one GPU, against extracting the same windows (sccg_archive_extract)
and against extracting them to the host followed by a host scan.

    S1  one 23-mer, k = 0, both strands, the whole chr1-sized archive
    S2  the same with k = 3
    S3  100 guides of 23 nt, k = 3, both strands, the whole chr1-sized archive
    S4  100 guides of 23 nt taken from the gene, k = 3, in one 10 kb gene window across the 65 archives of tools/archive_bench.py
    S5  one 23-mer of the first archive, k = 0, in the whole sequence of all 65 archives in one call (several launches)
Per workload: the search's gather_ms (its kernels), wall time and hit count; ext_gather_k's gather_ms for the same windows
(Context.query); and the baseline, Context.query to the host followed by a host scan.  The host scan is exact for A/C/G/T
patterns: a hit with at most k mismatches matches one of k + 1 disjoint parts exactly, so the exact occurrences of the parts
(bytes.find on the upper-cased bytes; a 5-mer index for S3) give the candidates, which NumPy scores with the 256 x 256 match
table of the rule.  Every hit list is compared with the host scan before a number is written; each shape is warmed up and
the median of many calls is kept.

    python tools/search_bench.py [--calls 10] [--out profiles/r4_search_bench.json]
"""
from __future__ import annotations

import argparse
import json
import statistics
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
import sccg_b200  # noqa: E402
from archive_bench import individuals  # noqa: E402
from extract_bench import gpu_info  # noqa: E402
from sccg_genome_compression_b200 import synth  # noqa: E402

COMP = bytearray(range(256))
for _a, _b in (b"AT", b"CG", b"RY", b"KM", b"BV", b"DH"):
    for _x, _y in ((_a, _b), (_a | 0x20, _b | 0x20)):
        COMP[_x], COMP[_y] = _y, _x
UP = bytes(b - 32 if 97 <= b <= 122 else b for b in range(256))
MISS = np.ones((256, 256), dtype=np.int16)                 # A/C/G/T pattern bytes only: p matches d when up(d) == up(p)
for _p in b"ACGTacgt":
    for _d in range(256):
        MISS[_p, _d] = UP[_d] != UP[_p]
CODE = np.full(256, 255, dtype=np.uint8)
for _i, _c in enumerate(b"ACGT"):
    CODE[_c] = CODE[_c | 0x20] = _i


def revcomp(p: bytes) -> bytes:
    return p.translate(bytes(COMP))[::-1]


class Index5:
    """positions of every 5-mer of upper(D) made of A/C/G/T, grouped by 5-mer"""

    def __init__(self, D: np.ndarray):
        c = CODE[D]
        n = len(D) - 4
        key = np.zeros(n, dtype=np.uint16)
        bad = np.zeros(n, dtype=bool)
        for j in range(5):
            key = (key << 2) | (c[j:j + n] & 3)
            bad |= c[j:j + n] == 255
        key[bad] = 1024
        self.order = np.argsort(key, kind="stable").astype(np.int64)
        self.start = np.searchsorted(key[self.order], np.arange(1026))

    def find(self, part: bytes) -> np.ndarray:
        k = 0
        for b in part.upper()[:5]:
            k = (k << 2) | int(CODE[b])
        return self.order[self.start[k]:self.start[k + 1]]


def host_scan(D: bytes, patterns, k: int, index: Index5 | None = None) -> np.ndarray:
    """hits [0, pos, pattern, strand, mismatches] over the whole of D, in (pos, pattern, strand) order"""
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
                if index is not None:
                    cand.append(index.find(pp[a:b]) - a)
                    continue
                part, at, got = pp[a:b].upper(), U.find(pp[a:b].upper()), []
                while at >= 0:
                    got.append(at - a)
                    at = U.find(part, at + 1)
                cand.append(np.array(got, dtype=np.int64))
            c = np.unique(np.concatenate(cand))
            c = c[(c >= 0) & (c + L <= len(D))]
            mm = np.zeros(len(c), dtype=np.int16)
            for j in range(L):
                mm += MISS[pp[j]][Dn[c + j]]
            keep = mm <= k
            rows.append(np.stack([np.zeros(keep.sum(), np.int64), c[keep], np.full(keep.sum(), i), np.full(keep.sum(), st), mm[keep]], axis=1))
    h = np.concatenate(rows).astype(np.int64)
    return h[np.lexsort((h[:, 3], h[:, 2], h[:, 1]))]


def expected(Ds, windows, patterns, k, index=None) -> np.ndarray:
    """the host scan of each window's bytes, shifted to D coordinates"""
    out = []
    for w, (a, s, e) in enumerate(windows):
        piece = Ds[a][s:e]
        h = host_scan(piece, patterns, k, index if (s, e) == (0, len(Ds[a])) else None)
        h[:, 0] = w
        h[:, 1] += s
        out.append(h)
    return np.concatenate(out)


def median_call(ctx, fn, calls):
    fn()
    walls, profs = [], []
    for _ in range(calls):
        t0 = time.perf_counter()
        fn()
        walls.append((time.perf_counter() - t0) * 1e3)
        profs.append(ctx.profile())
    prof = {k: statistics.median(p[k] for p in profs) for k in ("h2d_ms", "gather_ms", "kernels_ms", "d2h_ms")}
    prof["launches"] = profs[-1]["launches"]
    return {"wall_ms": statistics.median(walls), **prof}


def workload(ctx, archives, Ds, windows, patterns, k, calls, index=None):
    w = np.array(windows, dtype=np.int64)
    got = ctx.search(archives, patterns, w, max_mismatches=k)
    t0 = time.perf_counter()
    exp = expected(Ds, windows, patterns, k, index)
    scan_ms = (time.perf_counter() - t0) * 1e3
    assert np.array_equal(got, exp), (got.shape, exp.shape)
    res = {"patterns": len(patterns), "k": k, "windows": len(windows), "bases": int(sum(e - s for _, s, e in windows)), "hits": int(len(got))}
    res["search"] = median_call(ctx, lambda: ctx.search(archives, patterns, w, max_mismatches=k), calls)
    q = np.array([(a, s, e, 0) for a, s, e in windows], dtype=np.int64)
    if res["bases"] < 1 << 31:
        res["archive_extract_same_windows"] = median_call(ctx, lambda: ctx.query(archives, q), calls)
    else:                                                  # past sccg_archive_extract's 2^31-byte limit: one call per window
        per = [median_call(ctx, lambda i=i: ctx.query(archives, q[i:i + 1]), max(1, calls // 3)) for i in range(len(q))]
        res["archive_extract_same_windows"] = {key: sum(x[key] for x in per) for key in per[0]}
        res["archive_extract_same_windows"]["note"] = "sum over one call per window"
    t0 = time.perf_counter()
    for a, s, e in windows:
        ctx.query(archives, [(a, s, e, 0)])
    query_ms = (time.perf_counter() - t0) * 1e3
    res["baseline_query_then_host_scan"] = {"query_ms": query_ms, "host_scan_ms": scan_ms, "total_ms": query_ms + scan_ms,
                                            "note": "one call each; the host scan is the one that checked the hit list"}
    return res


def guides(D: bytes, n: int, seed: int):
    r = np.random.default_rng(seed)
    out = []
    while len(out) < n:
        s = int(r.integers(0, len(D) - 23))
        p = D[s:s + 23]
        if set(p.upper()) <= set(b"ACGT"):
            out.append(p.upper())
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r4_search_bench.json"))
    args = ap.parse_args()
    res = {"gpu": gpu_info(), "calls": args.calls, "statistic": "median"}
    ctx = sccg_b200.Context(0)
    ref_np, tgt_np = synth.local_pair(synth.CHR1_LEN, synth.seed_for(2, 0))
    ctx.set_reference(ref_np.tobytes())
    inter, mode = ctx.compress_resident(tgt_np.tobytes())
    A = ctx.open_archive(inter)
    D = tgt_np.tobytes()
    one = guides(D, 1, 1)
    hundred = guides(D, 100, 2)
    whole = [(0, 0, len(D))]
    for name, pats, k, idx in (("S1", one, 0, None), ("S2", one, 3, None), ("S3", hundred, 3, "index")):
        index = Index5(tgt_np) if idx else None
        res[name] = workload(ctx, [A], [D], whole, pats, k, args.calls, index)
        print(name, json.dumps(res[name]), flush=True)
    A.close()
    ref_np, _ = synth.local_pair(50_000_000, synth.seed_for(4, 0))
    tgts = individuals(ref_np, 64)
    ctx.set_reference(ref_np.tobytes())
    archives = []
    for t in tgts:
        it, _ = ctx.compress_resident(t.tobytes())
        archives.append(ctx.open_archive(it))
    Ds = [t.tobytes() for t in tgts]
    g0 = 20_000_000
    gene = guides(Ds[0][g0:g0 + 10_000], 100, 3)          # guides of the gene itself, so that the individuals hold hits
    res["S4"] = workload(ctx, archives, Ds, [(a, g0, g0 + 10_000) for a in range(len(Ds))], gene, 3, args.calls)
    print("S4", json.dumps(res["S4"]), flush=True)
    res["S5"] = workload(ctx, archives, Ds, [(a, 0, len(x)) for a, x in enumerate(Ds)], guides(Ds[0], 1, 4), 0, max(3, args.calls // 3))
    print("S5", json.dumps(res["S5"]), flush=True)
    for a in archives:
        a.close()
    ctx.close()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res, indent=1) + "\n")
    print("wrote", args.out)


if __name__ == "__main__":
    main()
