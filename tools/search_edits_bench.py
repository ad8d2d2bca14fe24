"""Edit-distance pattern search in open archives (sccg_archive_search_edits) on one GPU, against the Hamming search
(sccg_archive_search) on the same windows and patterns, and against extracting the windows to the host followed by a host scan.

    S1  one 23-mer, the whole chr1-sized archive, k = 1 and k = 3
    S3  100 guides of 23 nt, the whole chr1-sized archive, k = 1
    S4  100 guides of 23 nt taken from the gene, in one 10 kb gene window across the 64 archives of tools/archive_bench.py,
        k = 1 and k = 3
All on both strands.  S3 runs at k = 1 only: at k = 3 its host check would score tens of millions of candidate regions.
Per workload and k: both engines' gather_ms (their kernels) and wall time, the median of --calls calls made alternately
(edit, Hamming, edit, ...) after a warm-up of each; hit counts; and the baseline, Context.query to the host followed by the host
scan, which is tests/edit_probe.cpp: over the windows for S4, and over the candidate regions of the exact occurrences of k + 1
pattern parts (tests/test_emu_search_edits.expect_acgt) for the whole archive.  Every hit list is compared with the host scan
before a number is written.

    python tools/search_edits_bench.py [--calls 10] [--out profiles/r6_search_edits_bench.json]
"""
from __future__ import annotations

import argparse
import json
import statistics
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
sys.path.insert(0, str(ROOT / "tests"))
import sccg_b200  # noqa: E402
from archive_bench import individuals  # noqa: E402
from extract_bench import gpu_info  # noqa: E402
from search_bench import guides  # noqa: E402
from sccg_genome_compression_b200 import synth  # noqa: E402
from test_emu_search_edits import build_probe, expect, expect_acgt  # noqa: E402


def timed(ctx, fn):
    t0 = time.perf_counter()
    fn()
    wall = (time.perf_counter() - t0) * 1e3
    p = ctx.profile()
    return {"wall_ms": wall, "gather_ms": p["gather_ms"], "kernels_ms": p["kernels_ms"], "h2d_ms": p["h2d_ms"], "d2h_ms": p["d2h_ms"],
            "launches": p["launches"]}


def alternate(ctx, fns: dict, calls: int) -> dict:
    for f in fns.values():
        f()
    runs = {k: [] for k in fns}
    for _ in range(calls):
        for k, f in fns.items():
            runs[k].append(timed(ctx, f))
    out = {}
    for k, rs in runs.items():
        out[k] = {key: statistics.median(r[key] for r in rs) for key in ("wall_ms", "gather_ms", "kernels_ms", "h2d_ms", "d2h_ms")}
        out[k]["launches"] = rs[-1]["launches"]
    return out


def workload(ctx, probe, archives, Ds, windows, patterns, k, calls):
    w = np.array(windows, dtype=np.int64)
    got = ctx.search_edits(archives, patterns, w, max_edits=k)
    t0 = time.perf_counter()
    if len(windows) == 1 and windows[0][1:] == (0, len(Ds[windows[0][0]])):
        exp = expect_acgt(probe, Ds[windows[0][0]], patterns, k)
    else:
        exp = expect(probe, Ds, windows, patterns, k)
    scan_ms = (time.perf_counter() - t0) * 1e3
    assert np.array_equal(got, exp), (got.shape, exp.shape)
    ham = ctx.search(archives, patterns, w, max_mismatches=k)
    res = {"patterns": len(patterns), "k": k, "windows": len(windows), "bases": int(sum(e - s for _, s, e in windows)),
           "edit_hits": int(len(got)), "hamming_hits": int(len(ham))}
    res.update(alternate(ctx, {"edits": lambda: ctx.search_edits(archives, patterns, w, max_edits=k),
                               "hamming": lambda: ctx.search(archives, patterns, w, max_mismatches=k)}, calls))
    res["edits_over_hamming_gather"] = res["edits"]["gather_ms"] / res["hamming"]["gather_ms"]
    t0 = time.perf_counter()
    for a, s, e in windows:
        ctx.query(archives, [(a, s, e, 0)])
    query_ms = (time.perf_counter() - t0) * 1e3
    res["baseline_query_then_host_scan"] = {"query_ms": query_ms, "host_scan_ms": scan_ms, "total_ms": query_ms + scan_ms,
                                            "note": "one call each; the host scan is the one that checked the hit list"}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r6_search_edits_bench.json"))
    args = ap.parse_args()
    res = {"gpu": gpu_info(), "calls": args.calls, "statistic": "median"}
    tmp = tempfile.TemporaryDirectory()
    probe = build_probe(Path(tmp.name))
    ctx = sccg_b200.Context(0)
    ref_np, tgt_np = synth.local_pair(synth.CHR1_LEN, synth.seed_for(2, 0))
    ctx.set_reference(ref_np.tobytes())
    inter, mode = ctx.compress_resident(tgt_np.tobytes())
    A = ctx.open_archive(inter)
    D = tgt_np.tobytes()
    one = guides(D, 1, 1)
    hundred = guides(D, 100, 2)
    whole = [(0, 0, len(D))]
    for name, pats, k in (("S1_k1", one, 1), ("S1_k3", one, 3), ("S3_k1", hundred, 1)):
        res[name] = workload(ctx, probe, [A], [D], whole, pats, k, args.calls)
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
    for k in (1, 3):
        res[f"S4_k{k}"] = workload(ctx, probe, archives, Ds, [(a, g0, g0 + 10_000) for a in range(len(Ds))], gene, k, args.calls)
        print(f"S4_k{k}", json.dumps(res[f"S4_k{k}"]), flush=True)
    for a in archives:
        a.close()
    ctx.close()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res, indent=1) + "\n")
    print("wrote", args.out)


if __name__ == "__main__":
    main()
