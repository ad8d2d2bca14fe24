"""Archives (sccg_archive_open / sccg_archive_extract) against per-call region extraction (sccg_extract_resident), on one GPU.

    A1  one 1 kb region of the open chr1-sized archive, one query per call (>= 200 calls), against sccg_extract_resident
    A2  one 10 kb region from 65 archives in one call: 64 individuals derived from the reference of synth.local_pair(50 Mbp)
        (substitutions, compensated indels, lowercase runs under 64 seeds) and one target with an uncompensated 5 kb
        deletion near its start plus 0.1 % SNPs (global mode); against 65 sccg_extract_resident calls
    A3  200,000 x 150 bp spread over those 65 archives in one call (the bytes of extract_bench's W2, which reads one archive)
    A4  sccg_archive_open of the chr1-sized archive: wall time, front-end time, device bytes
With --parent-tree, tools/extract_bench.py (W1-W4) also runs from that tree (the parent build) and from this one, alternating,
so the gather times of the two builds come from the same GPU session.  Every output is compared with slices (or reverse
complements) of the targets before a number is written; each shape is warmed up and the median of many calls is kept.

    python tools/archive_bench.py [--calls 50] [--parent-tree DIR] [--rounds 2] [--out profiles/r4_archive_bench.json]
"""
from __future__ import annotations

import argparse
import json
import statistics
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
import sccg_b200  # noqa: E402
from extract_bench import gpu_info, slices  # noqa: E402
from sccg_genome_compression_b200 import synth  # noqa: E402

COMP = bytearray(range(256))
for _a, _b in (b"AT", b"CG", b"RY", b"KM", b"BV", b"DH"):
    for _x, _y in ((_a, _b), (_a | 0x20, _b | 0x20)):
        COMP[_x], COMP[_y] = _y, _x
COMP_NP = np.frombuffer(bytes(COMP), dtype=np.uint8)


def expect(Ds, q: np.ndarray) -> np.ndarray:
    parts = []
    for a, s, e, st in q.tolist():
        p = Ds[a][s:e]
        parts.append(COMP_NP[p[::-1]] if st else p)
    return np.concatenate(parts) if parts else np.zeros(0, np.uint8)


def timed(ctx, fn, calls: int):
    fn()
    walls, profs = [], []
    for _ in range(calls):
        t0 = time.perf_counter()
        fn()
        walls.append((time.perf_counter() - t0) * 1e3)
        profs.append(ctx.profile())
    prof = {k: statistics.median(p[k] for p in profs) for k in ("h2d_ms", "serialize_ms", "gather_ms", "kernels_ms", "d2h_ms")}
    prof["launches"] = profs[-1]["launches"]
    return statistics.median(walls), prof


def pinned(lib, n):
    import ctypes as C
    p = lib.sccg_pinned_alloc(max(n, 1))
    return p, np.ctypeslib.as_array((C.c_uint8 * max(n, 1)).from_address(p))


def individuals(ref_np: np.ndarray, k: int):
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
    out.append(np.concatenate([g[:10_000], g[15_000:]]))                  # 5 kb deleted near the start, not compensated
    return out


def archive_part(calls: int) -> dict:
    ctx = sccg_b200.Context(0)
    lib = ctx.lib
    res = {}
    # ---- A1, A4: the chr1-sized pair
    ref_np, tgt_np = synth.local_pair(synth.CHR1_LEN, synth.seed_for(2, 0))
    ref, tgt = ref_np.tobytes(), tgt_np.tobytes()
    inter, mode = ctx.compress(ref, tgt, b">bench")
    ctx.set_reference(ref)
    opens = []
    for _ in range(5):
        t0 = time.perf_counter()
        a = ctx.open_archive(inter)
        opens.append(((time.perf_counter() - t0) * 1e3, ctx.profile()["serialize_ms"]))
        a.close()
    A = ctx.open_archive(inter)
    assert A.seq_len == len(tgt) and A.mode == mode == 0
    res["A4_open"] = {"symbols": len(tgt), "record_file_bytes": len(inter), "wall_ms": statistics.median(o[0] for o in opens),
                      "serialize_ms": statistics.median(o[1] for o in opens), "device_bytes": A.device_bytes, "opens": len(opens)}
    s = int(np.random.default_rng(7).integers(0, len(tgt) - 1000))
    buf, out = pinned(lib, 1000)
    for strand in (0, 1):
        q = np.array([[0, s, s + 1000, strand]], dtype=np.int64)
        assert ctx.query([A], q, buf, 1000) == 1000 and np.array_equal(out[:1000], expect([tgt_np], q))
    q = np.array([[0, s, s + 1000, 0]], dtype=np.int64)
    wall, prof = timed(ctx, lambda: ctx.query([A], q, buf, 1000), max(calls, 200))
    regs = np.array([[s, s + 1000]], dtype=np.int64)
    assert ctx.extract_resident(inter, regs, buf, 1000) == 1000 and np.array_equal(out[:1000], tgt_np[s:s + 1000])
    wall_x, prof_x = timed(ctx, lambda: ctx.extract_resident(inter, regs, buf, 1000), max(calls, 200))
    res["A1_point_query"] = {"calls": max(calls, 200), "region_bytes": 1000, "archive_extract": {"wall_ms": wall, **prof},
                             "extract_resident": {"wall_ms": wall_x, **prof_x}, "speedup": wall_x / wall}
    print("A1", json.dumps(res["A1_point_query"]), flush=True)
    print("A4", json.dumps(res["A4_open"]), flush=True)
    lib.sccg_pinned_free(buf)
    A.close()
    # ---- A2, A3: 65 archives against one 50 Mbp reference
    ref_np, _ = synth.local_pair(50_000_000, synth.seed_for(4, 0))
    ref = ref_np.tobytes()
    tgts = individuals(ref_np, 64)
    ctx.set_reference(ref)
    inters, archives = [], []
    for t in tgts:
        it, m = ctx.compress_resident(t.tobytes())
        inters.append(it)
        archives.append(ctx.open_archive(it))
    modes = [a.mode for a in archives]
    assert modes[-1] == 1 and all(m == 0 for m in modes[:-1]), modes
    n = len(archives)
    g0 = 20_000_000
    q = np.array([[k, g0, g0 + 10_000, 0] for k in range(n)], dtype=np.int64)
    total = 10_000 * n
    buf, out = pinned(lib, total)
    assert ctx.query(archives, q, buf, total) == total and np.array_equal(out[:total], expect(tgts, q))
    wall, prof = timed(ctx, lambda: ctx.query(archives, q, buf, total), calls)
    regs = np.array([[g0, g0 + 10_000]], dtype=np.int64)

    def separate():
        for k in range(n):
            ctx.extract_resident(inters[k], regs, buf + 10_000 * k, 10_000)
    separate()
    assert np.array_equal(out[:total], expect(tgts, q))
    wall_x, _ = timed(ctx, separate, max(5, calls // 5))
    res["A2_gene_across_individuals"] = {"archives": n, "modes": {"local": modes.count(0), "global": modes.count(1)}, "region_bytes": 10_000,
                                         "reference_symbols": len(ref), "archive_extract_one_call": {"wall_ms": wall, **prof},
                                         "extract_resident_65_calls_wall_ms": wall_x, "speedup": wall_x / wall,
                                         "device_bytes_per_archive_median": statistics.median(a.device_bytes for a in archives)}
    print("A2", json.dumps(res["A2_gene_across_individuals"]), flush=True)
    lib.sccg_pinned_free(buf)
    rng = np.random.default_rng(20261020)
    ks = rng.integers(0, n, 200_000)
    lens = np.array([t.size for t in tgts])
    st = (rng.random(200_000) * (lens[ks] - 150)).astype(np.int64)
    grouped = np.argsort(ks, kind="stable")
    for order, label in ((grouped, "grouped_by_archive"), (np.arange(200_000), "interleaved")):
        q = np.ascontiguousarray(np.stack([ks, st, st + 150, np.zeros_like(ks)], axis=1)[order].astype(np.int64))
        total = 150 * len(q)
        buf, out = pinned(lib, total)
        assert ctx.query(archives, q, buf, total) == total and np.array_equal(out[:total], expect(tgts, q))
        wall, prof = timed(ctx, lambda: ctx.query(archives, q, buf, total), calls)
        res.setdefault("A3_gather_across_archives", {})[label] = {"queries": len(q), "output_bytes": total, "wall_ms": wall, **prof}
        print("A3", label, json.dumps(res["A3_gather_across_archives"][label]), flush=True)
        lib.sccg_pinned_free(buf)
    for a in archives:
        a.close()
    ctx.close()
    return res


def extract_rounds(parent: Path, rounds: int, calls: int) -> dict:
    """tools/extract_bench.py from the parent tree and from this tree, alternating: W1-W4 gather_ms and wall_ms of each run"""
    runs = {"parent": [], "this": []}
    with tempfile.TemporaryDirectory() as td:
        for r in range(rounds):
            for label, tree in (("parent", parent), ("this", ROOT)):
                out = Path(td) / f"{label}{r}.json"
                subprocess.check_call([sys.executable, str(tree / "tools" / "extract_bench.py"), "--calls", str(calls), "--out", str(out)])
                d = json.loads(out.read_text())
                runs[label].append({f"{p}/{w}": {"gather_ms": e["gather_ms"], "wall_ms": e["wall_ms"]}
                                    for p, pr in d["pairs"].items() for w, e in pr["workloads"].items()})
    summary = {}
    for key in runs["this"][0]:
        g_p = statistics.median(x[key]["gather_ms"] for x in runs["parent"])
        g_t = statistics.median(x[key]["gather_ms"] for x in runs["this"])
        summary[key] = {"parent_gather_ms": g_p, "this_gather_ms": g_t, "ratio": g_t / g_p if g_p else None}
    return {"rounds": rounds, "order": "parent, this, parent, this, ...", "runs": runs, "median_of_rounds": summary}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--parent-tree", default=None)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--extract-calls", type=int, default=20)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r4_archive_bench.json"))
    args = ap.parse_args()
    result = {"gpu": gpu_info(), "calls": args.calls, "statistic": "median"}
    result.update(archive_part(args.calls))
    if args.parent_tree:
        result["extract_bench_parent_vs_this"] = extract_rounds(Path(args.parent_tree).resolve(), args.rounds, args.extract_calls)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(result, indent=1) + "\n")
    print("wrote", args.out)


if __name__ == "__main__":
    main()
