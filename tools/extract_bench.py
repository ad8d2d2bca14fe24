"""Region extraction (sccg_extract*) against the full-decompress alternative, on one GPU.

Pairs: the chr1-sized local-mode pair and the chr19-shaped gap pair (global mode), made by synth with the seeds bench.py uses.
Workloads (regions in the decoded sequence D; for these lossless synthetic pairs D is the target):
    W1  the whole sequence as one region
    W2  200,000 regions of 150 bp at seeded uniform positions (exome-like)
    W3  1,000,000 single-base queries
    W4  1,000 regions of 1 kb inside one 2 Mbp window
W1-W3 run through extract_resident, W4 through sccg_extract with the reference in host memory.  The alternative is
decompress_resident_into (decompress_into for W4) of the whole image followed by slicing on the host.  Every output is
compared with slices of the target before a number is written; every shape is warmed up and the median of --calls calls is kept.
W2 and W3 are also timed with the gather forced onto either tile path (SCCG_EXT_LANE_MIN), which is what the default threshold
rests on.  Gather bandwidth counts one byte read and one byte written per output byte.

    python tools/extract_bench.py [--calls 20] [--out profiles/r3_extract_bench.json]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import sccg_b200  # noqa: E402
from sccg_genome_compression_b200 import synth  # noqa: E402

DATASHEET_GBS = 7700.0


def hbm_peak() -> tuple[float, str]:
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return DATASHEET_GBS, "data sheet (HGX B200, 7.7 TB/s per GPU), not measured"


def gpu_info() -> dict:
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        name, power = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:
        return {"name": "unknown", "power_limit": f"unknown ({type(e).__name__})"}


def workloads(Lm: int, seed: int) -> dict:
    r = np.random.default_rng(seed)
    w2 = r.integers(0, Lm - 150, 200_000)
    w3 = r.integers(0, Lm, 1_000_000)
    w0 = int(r.integers(0, Lm - 2_000_000))
    w4 = w0 + r.integers(0, 2_000_000 - 1000, 1000)
    pairs = lambda s, n: np.ascontiguousarray(np.stack([s, s + n], axis=1).astype(np.int64))
    return {"W1": np.array([[0, Lm]], dtype=np.int64), "W2": pairs(w2, 150), "W3": pairs(w3, 1), "W4": pairs(w4, 1000)}


def slices(seq: np.ndarray, regs: np.ndarray) -> np.ndarray:
    """concatenated seq[start:end] (seq: uint8 array of D)"""
    if len(regs) == 1:
        return seq[regs[0, 0]:regs[0, 1]]
    lens = regs[:, 1] - regs[:, 0]
    off = np.concatenate([[0], np.cumsum(lens)[:-1]])
    pos = np.repeat(regs[:, 0] - off, lens) + np.arange(int(lens.sum()))
    return seq[pos]


def image_slices(img: np.ndarray, hl: int, regs: np.ndarray) -> np.ndarray:
    """the alternative's host step: the same pieces cut out of the wrapped image (50 symbols + '\\n' per line after the header)"""
    if len(regs) == 1:                                              # the whole sequence: drop every newline
        body = img[hl:]
        n = int(regs[0, 1])
        full = n // 50
        out = body[:full * 51].reshape(full, 51)[:, :50].ravel()
        return np.concatenate([out, body[full * 51:full * 51 + n - full * 50]])
    lens = regs[:, 1] - regs[:, 0]
    off = np.concatenate([[0], np.cumsum(lens)[:-1]])
    b = np.repeat(regs[:, 0] - off, lens) + np.arange(int(lens.sum()))
    return img[hl + b + b // 50]


def timed(fn, calls: int):
    fn()                                                            # warm-up of this shape
    walls, profs = [], []
    for _ in range(calls):
        t0 = time.perf_counter()
        fn()
        walls.append((time.perf_counter() - t0) * 1e3)
        profs.append(ctx.profile())
    keys = ("h2d_ms", "serialize_ms", "gather_ms", "kernels_ms", "d2h_ms")
    prof = {k: statistics.median(p[k] for p in profs) for k in keys}
    prof["launches"] = profs[-1]["launches"]
    return statistics.median(walls), prof


def main():
    global ctx
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r3_extract_bench.json"))
    args = ap.parse_args()
    peak, peak_src = hbm_peak()
    ctx = sccg_b200.Context(0)
    result = {"gpu": gpu_info(), "hbm_peak_gbs": peak, "hbm_peak_source": peak_src, "calls": args.calls, "statistic": "median", "pairs": {}}
    for name, make in (("chr1_local", lambda: synth.local_pair(synth.CHR1_LEN, synth.seed_for(2, 0))),
                       ("chr19_gap_global", lambda: synth.global_gap_pair(63_811_651, 59_128_983, synth.seed_for(1, 0)))):
        ref_np, tgt_np = make()
        ref, tgt = ref_np.tobytes(), tgt_np.tobytes()
        inter, mode = ctx.compress(ref, tgt, b">bench")
        Lm = len(tgt)
        ctx.set_reference(ref)
        img_cap = Lm + Lm // 50 + 4096
        img_buf = sccg_b200.load_library().sccg_pinned_alloc(img_cap)
        img = np.ctypeslib.as_array((C.c_uint8 * img_cap).from_address(img_buf))
        n_img = ctx.decompress_resident(inter, img_buf, img_cap)
        hl = bytes(img[:4096]).index(b"\n") + 1
        assert n_img == hl + Lm + (Lm + 49) // 50
        pr = {"mode": "local" if mode == 0 else "global", "symbols": Lm, "record_file_bytes": len(inter), "workloads": {}}
        for wname, regs in workloads(Lm, 20261020).items():
            exp = slices(tgt_np, regs)
            total = len(exp)
            out_buf = sccg_b200.load_library().sccg_pinned_alloc(max(total, 1))
            out = np.ctypeslib.as_array((C.c_uint8 * max(total, 1)).from_address(out_buf))
            host_ref = wname == "W4"
            call = (lambda: ctx.extract(ref, inter, regs, out_buf, total)) if host_ref else (lambda: ctx.extract_resident(inter, regs, out_buf, total))
            assert call() == total and np.array_equal(out[:total], exp), (name, wname)
            wall, prof = timed(call, args.calls)
            entry = {"regions": int(len(regs)), "output_bytes": total, "entry_point": "sccg_extract" if host_ref else "sccg_extract_resident",
                     "wall_ms": wall, **prof}
            g = prof["gather_ms"]
            entry["gather_gbs"] = 2 * total / (g * 1e6) if g > 0 else None
            entry["gather_share_of_hbm_peak"] = entry["gather_gbs"] / peak if entry["gather_gbs"] else None
            if wname in ("W2", "W3"):
                for path, v in (("lane_path", "0"), ("warp_path", str(1 << 30))):
                    os.environ["SCCG_EXT_LANE_MIN"] = v
                    assert call() == total and np.array_equal(out[:total], exp)
                    entry[f"{path}_gather_ms"] = timed(call, args.calls)[1]["gather_ms"]
                    del os.environ["SCCG_EXT_LANE_MIN"]
            # the alternative: the whole image, then the host cuts the pieces out
            def alt():
                if host_ref:
                    ctx.decompress_into(ref, inter, img_buf, img_cap)
                else:
                    ctx.decompress_resident(inter, img_buf, img_cap)
                return image_slices(img, hl, regs)
            assert np.array_equal(alt(), exp), (name, wname, "alternative")
            t_alt, p_alt = timed(alt, args.calls)
            entry["full_decompress_alternative"] = {"entry_point": "sccg_decompress_into" if host_ref else "sccg_decompress_resident_into",
                                                    "wall_ms_with_host_slicing": t_alt, **p_alt, "image_bytes": int(n_img)}
            entry["speedup_vs_alternative"] = t_alt / wall
            pr["workloads"][wname] = entry
            sccg_b200.load_library().sccg_pinned_free(out_buf)
            print(name, wname, json.dumps({k: v for k, v in entry.items() if k != "full_decompress_alternative"}), flush=True)
        sccg_b200.load_library().sccg_pinned_free(img_buf)
        ctx.clear_reference()
        result["pairs"][name] = pr
    ctx.close()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(result, indent=1) + "\n")
    print("wrote", args.out)


if __name__ == "__main__":
    main()
