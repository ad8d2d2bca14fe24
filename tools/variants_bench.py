"""Variant records of open archives (sccg_archive_variants), on one GPU.

    V1  the chr1-sized local-mode archive (synth.local_pair(CHR1_LEN, seed_for(2, 0))), whole
    V2  the 65-archive cohort of tools/archive_bench.py (50 Mbp reference, 64 local-mode individuals and one global-mode one),
        whole, in one call
    V3  one 10 kb reference window across those 65 archives, in one call
Per workload: kernel time (gather_ms, the CUDA-event time of the variant kernels; median over repeated calls after a warm-up),
wall time per call, record counts (by kind) and ALT bytes.  In the same run, for comparison and labelled as such:
sccg_decompress_resident_into of the same archives (kernels_ms and wall), and the host Python reference implementation of
tests/variants_lib.py on the same record files (wall; V2: the first 8 archives only).  Every device result is checked against
the reference implementation (V1, and the archives it runs on in V2) and the splice invariant before a number is written.

    python tools/variants_bench.py [--calls 20] [--out profiles/r7_variants_bench.json]
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
sys.path.insert(0, str(ROOT / "tests"))
import sccg_b200  # noqa: E402
import variants_lib as vl  # noqa: E402
from archive_bench import individuals  # noqa: E402
from extract_bench import gpu_info  # noqa: E402
from sccg_genome_compression_b200 import synth  # noqa: E402


def timed(ctx, fn, calls: int, key: str):
    fn()
    walls, ks = [], []
    for _ in range(calls):
        t0 = time.perf_counter()
        fn()
        walls.append((time.perf_counter() - t0) * 1e3)
        ks.append(ctx.profile()[key])
    p = ctx.profile()
    return {"wall_ms": statistics.median(walls), f"{key}_median": statistics.median(ks), f"{key}_min": min(ks), "launches": p["launches"],
            "h2d_ms": p["h2d_ms"], "d2h_ms": p["d2h_ms"], "calls": calls}


def decompress_time(ctx, inters, calls: int):
    """sccg_decompress_resident_into of each record file (summed over the files per round)"""
    cap = 0
    for it in inters:
        cap = max(cap, len(ctx.decompress_resident(it)))
    p = ctx.lib.sccg_pinned_alloc(cap + 64)

    def once():
        k = 0.0
        for it in inters:
            ctx.decompress_resident(it, p, cap + 64)
            k += ctx.profile()["kernels_ms"]
        return k
    once()
    walls, ks = [], []
    for _ in range(calls):
        t0 = time.perf_counter()
        ks.append(once())
        walls.append((time.perf_counter() - t0) * 1e3)
    ctx.lib.sccg_pinned_free(p)
    return {"what": "sccg_decompress_resident_into of the same record files", "files": len(inters), "wall_ms": statistics.median(walls),
            "kernels_ms_median": statistics.median(ks), "calls": calls}


def python_reference(ref: bytes, inters, Ds, got_by_archive):
    t0 = time.perf_counter()
    outs = [vl.variants_whole(ref, it, D) for it, D in zip(inters, Ds)]
    wall = (time.perf_counter() - t0) * 1e3
    for k, exp in enumerate(outs):
        assert np.array_equal(got_by_archive[k], exp), k
    return {"what": "host Python reference implementation (tests/variants_lib.py)", "files": len(inters), "wall_ms": wall}


def exact_call(ctx, arch, windows=None):
    """one sccg_archive_variants call into buffers of the exact sizes (counted once beforehand), as a caller that times it would"""
    import ctypes as C
    w = np.ascontiguousarray(np.asarray(windows if windows is not None else [(k, 0, ctx.ref_len) for k in range(len(arch))], dtype=np.int64))
    nv, na = ctx.variants(arch, w, count_only=True)
    out = np.zeros(max(nv, 1), dtype=ctx._VARIANT)
    alt = C.create_string_buffer(max(na, 1))
    handles = (C.c_void_p * len(arch))(*[a.handle for a in arch])
    n, m = C.c_int64(), C.c_int64()

    def run():
        ctx._check(ctx.lib.sccg_archive_variants(ctx.handle, handles, len(arch), w.ctypes.data, len(w), out.ctypes.data, nv, C.byref(n), alt, na, C.byref(m)))
    return run


def summary(rec: np.ndarray, alt: bytes) -> dict:
    return {"records": int(len(rec)), "alt_bytes": len(alt), "kinds": vl.kinds(rec)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r7_variants_bench.json"))
    args = ap.parse_args()
    res = {"gpu": gpu_info(), "statistic": "median", "timing": "gather_ms: CUDA events around the variant kernels of one call"}
    ctx = sccg_b200.Context(0)
    # ---- V1
    ref_np, tgt_np = synth.local_pair(synth.CHR1_LEN, synth.seed_for(2, 0))
    ref, tgt = ref_np.tobytes(), tgt_np.tobytes()
    ctx.set_reference(ref)
    inter, mode = ctx.compress_resident(tgt)
    assert mode == 0
    A = ctx.open_archive(inter)
    rec, alt = ctx.variants([A])
    vl.check_invariants(ref, tgt, rec, alt)
    v1 = {"symbols": len(tgt), "record_file_bytes": len(inter), **summary(rec, alt),
          "sccg_archive_variants": timed(ctx, exact_call(ctx, [A]), args.calls, "gather_ms")}
    v1["sccg_decompress_resident_into"] = decompress_time(ctx, [inter], args.calls)
    v1["python_reference"] = python_reference(ref, [inter], [tgt], [rec[:, 1:5]])
    res["V1_chr1_whole"] = v1
    print("V1", json.dumps(v1), flush=True)
    A.close()
    # ---- V2, V3
    ref_np, _ = synth.local_pair(50_000_000, synth.seed_for(4, 0))
    ref = ref_np.tobytes()
    tgts = individuals(ref_np, 64)
    ctx.set_reference(ref)
    inters, arch = [], []
    for t in tgts:
        it, _ = ctx.compress_resident(t.tobytes())
        inters.append(it)
        arch.append(ctx.open_archive(it))
    modes = [a.mode for a in arch]
    assert modes[-1] == 1 and all(m == 0 for m in modes[:-1]), modes
    rec, alt = ctx.variants(arch)
    by = [rec[rec[:, 0] == k] for k in range(len(arch))]
    for k in range(len(arch)):
        vl.check_invariants(ref, tgts[k].tobytes(), by[k], alt)
    v2 = {"archives": len(arch), "modes": {"local": modes.count(0), "global": modes.count(1)}, "reference_symbols": len(ref), **summary(rec, alt),
          "sccg_archive_variants": timed(ctx, exact_call(ctx, arch), args.calls, "gather_ms")}
    v2["sccg_decompress_resident_into"] = decompress_time(ctx, inters, max(3, args.calls // 5))
    sub = list(range(8))
    v2["python_reference"] = python_reference(ref, [inters[k] for k in sub], [tgts[k].tobytes() for k in sub], [by[k][:, 1:5] for k in sub])
    v2["python_reference"]["archives"] = "the first 8 of the 65"
    res["V2_cohort_whole"] = v2
    print("V2", json.dumps(v2), flush=True)
    g0 = 20_000_000
    w = [(k, g0, g0 + 10_000) for k in range(len(arch))]
    rw, aw = ctx.variants(arch, w)
    exp, exp_alt = vl.filter_windows([b[:, 1:5] for b in by], [t.tobytes() for t in tgts], w, len(ref))
    assert np.array_equal(rw, exp) and aw == exp_alt
    v3 = {"archives": len(arch), "window": [g0, g0 + 10_000], **summary(rw, aw),
          "sccg_archive_variants": timed(ctx, exact_call(ctx, arch, w), args.calls, "gather_ms")}
    res["V3_window_across_cohort"] = v3
    print("V3", json.dumps(v3), flush=True)
    for a in arch:
        a.close()
    ctx.close()
    res["gpu_after"] = gpu_info()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res, indent=1) + "\n")
    print("wrote", args.out)


if __name__ == "__main__":
    main()
