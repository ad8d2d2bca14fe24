"""Coordinates lifted between the reference and open archives (sccg_archive_liftover), on one GPU.

    L1  lift-table build of the chr1-sized local-mode archive (synth.local_pair(CHR1_LEN, seed_for(2, 0))): the first
        liftover call after an open (kernels_ms - gather_ms; the archive is reopened before each call), next to one
        whole-archive sccg_archive_variants call in the same run
    L2  200,000 exome-like 150 bp intervals on the cached chr1 table, reference -> archive and archive -> reference
    L3  20,000 gene-sized intervals (1 to 30 kb, reference coordinates) across the 65-archive cohort of tools/archive_bench.py
        in one call, and the `--reference-coords` extraction of them (that liftover call, then one sccg_archive_extract call)
Per workload: kernel time (gather_ms: CUDA events around the lift kernel), wall time per call, h2d_ms (query table) and
d2h_ms (results), each the median over repeated calls after a warm-up.  For comparison, labelled as such: numpy searchsorted
over the same records on the host (tests/liftover_lib.py lift).  Every device result is checked against tests/liftover_lib.py
before a number is written.

    python tools/liftover_bench.py [--calls 20] [--out profiles/r8_liftover_bench.json]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import statistics
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
sys.path.insert(0, str(ROOT / "tests"))
import liftover_lib as ll  # noqa: E402
import sccg_b200  # noqa: E402
import variants_lib as vl  # noqa: E402
from archive_bench import individuals  # noqa: E402
from extract_bench import gpu_info  # noqa: E402
from sccg_genome_compression_b200 import synth  # noqa: E402


def raw_lift(ctx, arch, q: np.ndarray):
    """one sccg_archive_liftover call on prebuilt query and result tables (what a caller that times it would do) -> (run, out)"""
    t = np.zeros(len(q), dtype=ctx._LIFT_QUERY)
    t["archive"], t["start"], t["end"], t["from"] = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
    out = np.zeros(len(q), dtype=ctx._LIFT)
    handles = (C.c_void_p * len(arch))(*[a.handle for a in arch])

    def run():
        ctx._check(ctx.lib.sccg_archive_liftover(ctx.handle, handles, len(arch), t.ctypes.data, len(t), out.ctypes.data))
    return run, out


def rows_of(out) -> np.ndarray:
    return np.stack([out[f].astype(np.int64) for f, _ in sccg_b200.Context._LIFT[:6]], axis=1)


def timed(ctx, fn, calls: int) -> dict:
    fn()
    walls, profs = [], []
    for _ in range(calls):
        t0 = time.perf_counter()
        fn()
        walls.append((time.perf_counter() - t0) * 1e3)
        profs.append(ctx.profile())
    r = {k: statistics.median(p[k] for p in profs) for k in ("gather_ms", "kernels_ms", "h2d_ms", "d2h_ms")}
    r.update({"wall_ms": statistics.median(walls), "launches": profs[-1]["launches"], "calls": calls})
    return r


def host_searchsorted(wholes, rlen, dlens, q: np.ndarray, calls: int) -> dict:
    walls = []
    for _ in range(max(3, calls // 4)):
        t0 = time.perf_counter()
        ll.lift_queries(wholes, rlen, dlens, q)
        walls.append((time.perf_counter() - t0) * 1e3)
    return {"what": "host numpy searchsorted over the same records (tests/liftover_lib.py), one thread", "wall_ms": statistics.median(walls)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r8_liftover_bench.json"))
    args = ap.parse_args()
    res = {"gpu": gpu_info(), "statistic": "median",
           "timing": "gather_ms: CUDA events around the lift kernel; kernels_ms - gather_ms: the lift-table build; wall: host clock per call"}
    ctx = sccg_b200.Context(0)
    # ---- L1
    ref_np, tgt_np = synth.local_pair(synth.CHR1_LEN, synth.seed_for(2, 0))
    ref, tgt = ref_np.tobytes(), tgt_np.tobytes()
    ctx.set_reference(ref)
    inter, mode = ctx.compress_resident(tgt)
    assert mode == 0
    A = ctx.open_archive(inter)
    rec, alt = ctx.variants([A])
    vl.check_invariants(ref, tgt, rec, alt)
    recs = rec[:, 1:5]
    builds = []
    for i in range(max(5, args.calls // 4) + 1):
        A.close()
        A = ctx.open_archive(inter)
        b0 = A.device_bytes
        t0 = time.perf_counter()
        ctx.liftover([A], [(0, 0, 1, 0)])
        wall = (time.perf_counter() - t0) * 1e3
        p = ctx.profile()
        if i:                                                               # (the first is the warm-up)
            builds.append((p["kernels_ms"] - p["gather_ms"], wall, p["launches"]))
    v = {}
    for _ in range(args.calls):
        ctx.variants([A])
        v.setdefault("gather_ms", []).append(ctx.profile()["gather_ms"])
    l1 = {"symbols": len(tgt), "records": int(len(recs)), "table_bytes": A.device_bytes - b0,
          "build": {"kernel_ms": statistics.median(b[0] for b in builds), "first_call_wall_ms": statistics.median(b[1] for b in builds),
                    "launches": builds[-1][2], "builds": len(builds)},
          "sccg_archive_variants_whole": {"gather_ms": statistics.median(v["gather_ms"]), "calls": args.calls}}
    res["L1_chr1_table_build"] = l1
    print("L1", json.dumps(l1), flush=True)
    # ---- L2
    rng = np.random.default_rng(11)
    l2 = {"intervals": 200_000, "length": 150, "bytes_in_per_query": 32, "bytes_out_per_query": 48}
    for frm, ls in ((0, len(ref)), (1, len(tgt))):
        s = rng.integers(0, ls - 150, size=200_000)
        q = np.stack([np.zeros_like(s), s, s + 150, np.full_like(s, frm)], axis=1)
        run, out = raw_lift(ctx, [A], q)
        run()
        exp = ll.lift_queries([recs], len(ref), [len(tgt)], q)
        assert np.array_equal(rows_of(out), exp)
        l2["reference_to_archive" if frm == 0 else "archive_to_reference"] = {
            "sccg_archive_liftover": timed(ctx, run, args.calls), "host_searchsorted": host_searchsorted([recs], len(ref), [len(tgt)], q, args.calls)}
    res["L2_chr1_exome_intervals"] = l2
    print("L2", json.dumps(l2), flush=True)
    A.close()
    # ---- L3
    ref_np, _ = synth.local_pair(50_000_000, synth.seed_for(4, 0))
    ref = ref_np.tobytes()
    tgts = individuals(ref_np, 64)
    ctx.set_reference(ref)
    arch = []
    for t in tgts:
        it, _ = ctx.compress_resident(t.tobytes())
        arch.append(ctx.open_archive(it))
    rec, _ = ctx.variants(arch)
    wholes = [rec[rec[:, 0] == k][:, 1:5] for k in range(len(arch))]
    print("L3: 65 archives open", flush=True)
    dlens = [len(t) for t in tgts]
    n = 20_000
    k = rng.integers(0, len(arch), size=n)
    s = rng.integers(0, len(ref) - 30_000, size=n)
    q = np.stack([k, s, s + rng.integers(1_000, 30_001, size=n), np.zeros(n, np.int64)], axis=1)
    run, out = raw_lift(ctx, arch, q)
    t0 = time.perf_counter()
    run()
    first = ctx.profile()
    first_wall = (time.perf_counter() - t0) * 1e3
    rows = rows_of(out)
    assert np.array_equal(rows, ll.lift_queries(wholes, len(ref), dlens, q))
    eq = np.ascontiguousarray(np.stack([q[:, 0], rows[:, 0], rows[:, 1], np.zeros(n, np.int64)], axis=1))
    total = int((rows[:, 1] - rows[:, 0]).sum())
    buf = ctx.lib.sccg_pinned_alloc(total + 64)
    ctx.query(arch, eq, buf, total + 64)
    got = C.string_at(buf, total)
    tb = [t.tobytes() for t in tgts]
    assert got == b"".join(tb[a][x:y] for a, x, y in eq[:, :3].tolist())
    del tb
    del got

    def extract_ref_coords():
        run()
        lifted = rows_of(out)
        eq[:, 1], eq[:, 2] = lifted[:, 0], lifted[:, 1]
        ctx.query(arch, eq, buf, total + 64)
    walls, ext = [], []
    extract_ref_coords()
    for _ in range(args.calls):
        t0 = time.perf_counter()
        extract_ref_coords()
        walls.append((time.perf_counter() - t0) * 1e3)
        ext.append(ctx.profile())
    ctx.lib.sccg_pinned_free(buf)
    l3 = {"archives": len(arch), "intervals": n, "interval_bytes": "1 to 30 kb (reference)", "lifted_bytes": total,
          "first_call": {"kernels_ms": first["kernels_ms"], "build_kernel_ms": first["kernels_ms"] - first["gather_ms"], "wall_ms": first_wall,
                         "launches": first["launches"]},
          "sccg_archive_liftover": timed(ctx, run, args.calls),
          "host_searchsorted": host_searchsorted(wholes, len(ref), dlens, q, args.calls),
          "reference_coords_extraction": {"what": "the liftover call, then one sccg_archive_extract call of the lifted pieces into page-locked memory",
                                          "wall_ms": statistics.median(walls),
                                          "extract_gather_ms": statistics.median(p["gather_ms"] for p in ext),
                                          "extract_d2h_ms": statistics.median(p["d2h_ms"] for p in ext), "calls": args.calls}}
    res["L3_cohort_gene_intervals"] = l3
    print("L3", json.dumps(l3), flush=True)
    for a in arch:
        a.close()
    ctx.close()
    res["gpu_after"] = gpu_info()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res, indent=1) + "\n")
    print("wrote", args.out)


if __name__ == "__main__":
    main()
