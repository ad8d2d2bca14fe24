#!/usr/bin/env python
"""bench.py -- SCCG hot path on B200.

Headline (BASELINE.json configs[3] / [4]): whole-genome compression and decompression of the 24-pair synthetic
hg19-vs-hg18-shaped set (3,095,677,412 target bp), STRONG scaling over N GPUs: the pairs are LPT-packed onto the ranks by
the C++ multi-GPU layer (sccg_mgpu_assign), every rank works through its own pairs, and the encoded record streams are
gathered to rank 0 over NCCL (sccg_mgpu_gather) inside the timed region.  A "step" is one pass over the whole genome.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One JSON line on stdout (rank 0):
    value / ms_per_step   compression, inputs resident in HBM: per rank the device time of its calls (CUDA events on the
                          library stream) + the gather, max over ranks
    e2e                   the same job through the host-pointer C ABI: pinned host buffers in, H2D + kernels + NCCL gather + D2H
                          inside the timed region (wall clock between barriers, max over ranks)
    decompress            the same two numbers for decompression (Gbp/s)
    roofline              seg_match_k on the chr1-sized pair (BASELINE configs[1]) against the measured HBM peak
    chr1_local            configs[1] on one GPU: device-resident and end-to-end, both directions, with both kernels' rooflines
    global_gap_chr19 / global_divergent_chr21   configs[0]-shaped / configs[2] pairs through the global fallback
    chr1_sharded (N > 1)  one chromosome over all ranks by segment range (sccg_mgpu_compress_sharded)
    cpu_baseline          the reference's CPU implementation on a bounded sample, same box (N = 1 only)
    verified_against_oracle / parity_vs_reference   untimed byte comparisons of the outputs that were timed

--dump-outputs DIR (rank 0) writes what the timed legs returned in their last step as DIR/<name>.npy, one float32 value per
output byte (float64 for lengths), so that two builds can be compared output for output on the same seeded inputs:
    genome_compressed          the 24 encoded streams of the headline leg, back to back in pair order (sampled)
    genome_compressed_lengths  their lengths
    genome_decompressed_pair<i>  the FASTA image of rank 0's last pair from the end-to-end decompression leg (sampled)
    <global pair>_compressed / _decompressed   the end-to-end outputs of the two global-mode pairs (sampled)
An output longer than its share of the 64 MB budget is sampled: 4 KiB blocks at positions drawn with a fixed seed.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
if __name__ == "__main__":
    sys.dont_write_bytecode = True      # run as the benchmark, it leaves the tree as it found it (it may be read-only)

METRIC = "compress Mbp/s (decompress Gbp/s in `decompress`), whole-genome 24-pair synthetic hg19-vs-hg18 shape"
CHR1_HEADER = b">chr1 synthetic hg19-vs-hg18 shape"

import sccg_b200  # noqa: E402  (registers the hyphenated package dir as sccg_genome_compression_b200)


def header_of(i: int) -> bytes:
    return CHR1_HEADER if i == 0 else b">chr%d synthetic hg19-vs-hg18 shape" % (i + 1)


def ncu_traffic(kernel: str):
    """DRAM bytes (read + write) per launch of `kernel` from the committed `ncu --set full` capture of the chr1-sized workload
    (profiles/traffic.json, written by tools/ncu_traffic.py from the .ncu-rep); None if no capture is committed"""
    p = ROOT / "profiles" / "traffic.json"
    try:
        return json.loads(p.read_text())["kernels"][kernel]["dram_bytes_per_launch"]
    except Exception:
        return None


def bind_to_gpu_numa_node(index: int) -> str:
    """Pins this process to the CPUs closest to its GPU (NVML's ideal affinity) so that the page-locked host buffers of the
    end-to-end legs live on that NUMA node; with 8 ranks the PCIe copies otherwise cross the socket interconnect."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        pynvml.nvmlDeviceSetCpuAffinity(h)
        return f"{len(os.sched_getaffinity(0))} cpus"
    except Exception as e:                               # no NVML / not permitted: run unbound
        return f"unbound ({type(e).__name__})"


def peaks() -> tuple[float, str]:
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """streams `nvidia-smi -lms 100` (clocks, throttle reasons) while the timed regions run"""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.samples, self.proc, self.thread = index, [], None, None

    def _run(self):
        for line in self.proc.stdout:
            parts = [x.strip() for x in line.split(",")]
            if len(parts) >= 6:
                self.samples.append(parts)

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._run, daemon=True)
            self.thread.start()
            time.sleep(0.35)                      # let the first sample land before the timed region starts
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
            self.thread.join(timeout=5)

    def summary(self) -> dict:
        sm = [int(s[0]) for s in self.samples if s[0].isdigit()]
        mx = [int(s[1]) for s in self.samples if s[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for s in self.samples for i in range(4) if s[2 + i].lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.samples)}


# ----------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the reference's own CPU implementation (oracle/_ref where build() could
# compile it from the reference's sources, else the C oracle port), timed on this box's host cores.
# ----------------------------------------------------------------------------------------------
def _ref_compress_worker(args):
    """one process: reference `compress` + `decompress` executables on one FASTA slice; keeps the two output files"""
    import oracle_lib as ol
    ref_fa, tgt_fa, out_dir, n_bp = args
    t0 = time.perf_counter()
    r = subprocess.run([str(ol.REF_DIR / "compress"), ref_fa, tgt_fa, out_dir], env=ol.shim_env(), stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    t1 = time.perf_counter()
    d = subprocess.run([str(ol.REF_DIR / "decompress"), out_dir + "/compressed_genome.txt.7z", ref_fa, out_dir + "/dec"], env=ol.shim_env(),
                       stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    t2 = time.perf_counter()
    return r.returncode, d.returncode, t1 - t0, t2 - t1, n_bp


def _port_compress_worker(args):
    import oracle_lib as ol
    ref, tgt, header = args
    t0 = time.perf_counter()
    rc, text, _ = ol.orc_compress(ref, tgt, header)
    t1 = time.perf_counter()
    rc2, _ = ol.orc_decompress(ref, text)
    t2 = time.perf_counter()
    return rc, rc2, t1 - t0, t2 - t1, len(tgt)


def cpu_reference_pass(jobs_sym: list[tuple[bytes, bytes, bytes]], tmp: Path, keep: bool = False) -> dict:
    """one process per job, all at once; each runs the reference on its own (reference, target, header) symbols.
    keep: return the first job's compressed_genome.txt / reconstructed_genome.fa (reference kind only)"""
    import concurrent.futures as cf
    import oracle_lib as ol
    kind = "reference" if ol.have_reference() else "port"
    jobs = []
    for c, (r, t, h) in enumerate(jobs_sym):
        if kind == "reference":
            d = tmp / f"job{c}"
            d.mkdir(parents=True, exist_ok=True)
            ol.write_fasta(d / "ref.fa", r, b">ref")
            ol.write_fasta(d / "tgt.fa", t, h)
            jobs.append((str(d / "ref.fa"), str(d / "tgt.fa"), str(d / "out"), len(t)))
        else:
            jobs.append((r, t, h))
    t0 = time.perf_counter()
    with cf.ProcessPoolExecutor(max_workers=len(jobs)) as ex:
        res = list(ex.map(_ref_compress_worker if kind == "reference" else _port_compress_worker, jobs))
    wall = time.perf_counter() - t0
    assert all(r[0] == 0 and r[1] == 0 for r in res), "reference run failed"
    bp = sum(r[4] for r in res)
    comp_wall = max(r[2] for r in res)
    dec_wall = max(r[3] for r in res)
    out = {"kind": kind, "cores": len(jobs), "bp": bp, "compress_s": comp_wall, "decompress_s": dec_wall, "wall_s": wall,
           "compress_mbp_s": bp / comp_wall / 1e6, "decompress_gbp_s": bp / dec_wall / 1e9}
    if keep and kind == "reference":
        out["intermediate"] = (tmp / "job0" / "out" / "compressed_genome.txt").read_bytes()
        out["reconstructed"] = (tmp / "job0" / "out" / "dec" / "reconstructed_genome.fa").read_bytes()
    return out


def genome_lengths(scale: float) -> list[int]:
    from sccg_genome_compression_b200 import synth
    if scale == 1.0:
        return list(synth.HG19_LENGTHS)
    return [max(20_000, int(n * scale)) for n in synth.HG19_LENGTHS]


def workload_name(scale: float) -> str:
    base = ("whole-genome synthetic hg19-vs-hg18 shape: 24 pairs with the hg19 chromosome lengths (249,250,621 ... 48,129,895; "
            "3,095,677,412 target bp), every target = its reference with 0.1% SNPs + compensated small indels, 50% lowercase runs, "
            "co-located and target-only N runs; local segment-matching path")
    return base if scale == 1.0 else base + f" -- REDUCED by x{scale} (debug run, not the named config)"


def run_reference_arm(args, rank: int) -> None:
    if rank != 0:
        return
    from sccg_genome_compression_b200 import synth
    import oracle_lib as ol
    cores = os.cpu_count() or 1
    slice_bp = 4_000_000
    n = min(synth.CHR1_LEN, cores * slice_bp + slice_bp)
    if args.size > 0:
        n = max(2 * slice_bp, min(n, args.size))
    ref, tgt = synth.local_pair(n, synth.seed_for(2, 0))
    ref, tgt = ref.tobytes(), tgt.tobytes()
    jobs = []
    for c in range(cores):
        a = (c * slice_bp) % max(1, n - slice_bp)
        a -= a % 1000
        jobs.append((ref[a:a + slice_bp], tgt[a:a + slice_bp], CHR1_HEADER))
    times_c, times_d, bp = [], [], 0
    with tempfile.TemporaryDirectory() as d:
        for step in range(args.warmup + args.steps):
            r = cpu_reference_pass(jobs, Path(d))
            if step >= args.warmup:
                times_c.append(r["compress_s"]); times_d.append(r["decompress_s"]); bp = r["bp"]
    ms = 1e3 * sum(times_c) / len(times_c)
    value = bp / (ms / 1e3) / 1e6
    dec = bp / (sum(times_d) / len(times_d)) / 1e9
    sample = (f"{cores} processes x {slice_bp} bp slices of the genome's chr1-sized pair per step (local-mode segments are independent, the "
              "reference is single-threaded: slices on all cores are the most favourable way to run it); whole `compress` program (FASTA read + "
              "match + write + delta_encode; 7z replaced by a copy shim), wall time of the slowest process")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "Mbp/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": workload_name(1.0), "bp_per_step": bp},
            "decompress": {"value": dec, "unit": "Gbp/s"},
            "cpu_baseline": {"value": value, "unit": "Mbp/s", "cores": cores, "kind": r["kind"], "sample": sample},
            "e2e": {"value": value, "unit": "Mbp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    # like-for-like companion: ONE reference process on the full chr1-sized pair (its per-bp cost grows with the size:
    # delta_encode is quadratic in the number of tokens).  Once, --gpus 1 only (a few minutes).
    if args.gpus == 1 and not args.no_ref_full and ol.have_reference():
        ref, tgt = synth.local_pair(synth.CHR1_LEN, synth.seed_for(2, 0))
        with tempfile.TemporaryDirectory() as d:
            r = cpu_reference_pass([(ref.tobytes(), tgt.tobytes(), CHR1_HEADER)], Path(d))
        line["reference_full_config"] = {"workload": "chr1-sized pair (249,250,621 bp), one reference process, one core", "compress_s": r["compress_s"],
                                         "decompress_s": r["decompress_s"], "compress_mbp_s": r["compress_mbp_s"], "decompress_gbp_s": r["decompress_gbp_s"]}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------
def _cbuf(t, n=None):
    """zero-copy view of the first n bytes of a pinned CPU uint8 tensor as a ctypes char buffer"""
    return (ctypes.c_char * (t.numel() if n is None else n)).from_address(t.data_ptr())


def fasta_image(header: bytes, tgt) -> bytes:
    """the FASTA text `decompress` must give back for a target on the lossless envelope (decompression.cpp:266-274, :322)"""
    import numpy as np
    n = tgt.size
    full = n // 50 * 50
    body = np.empty((full // 50, 51), dtype=np.uint8)
    body[:, :50] = tgt[:full].reshape(-1, 50)
    body[:, 50] = 10
    tail = tgt[full:].tobytes()
    return header + b"\n" + body.tobytes() + (tail + b"\n" if tail else b"")


DUMP_BLOCK = 4096


def dump_sample(data, cap: int):
    """bytes / uint8 array -> float32 array of every byte, or of `cap` bytes in DUMP_BLOCK-sized blocks whose positions are
    drawn with a fixed seed (in ascending order) when the output is longer than that"""
    import numpy as np
    a = np.frombuffer(data, dtype=np.uint8) if isinstance(data, (bytes, bytearray)) else np.asarray(data, dtype=np.uint8)
    if a.size > cap:
        blocks = a[:a.size // DUMP_BLOCK * DUMP_BLOCK].reshape(-1, DUMP_BLOCK)
        pick = np.sort(np.random.default_rng(0).choice(blocks.shape[0], cap // DUMP_BLOCK, replace=False))
        a = blocks[pick].ravel()
    return a.astype(np.float32)


def oracle_compress_many(items: list) -> list[bytes]:
    """the C oracle (test infrastructure: the checker) on several pairs at once: ctypes releases the GIL, one thread per pair"""
    import concurrent.futures as cf
    import oracle_lib as ol
    lib = ol.oracle()

    def one(it):
        ref, tgt, header = it
        out = ctypes.c_void_p(); n = ctypes.c_long(); mode = ctypes.c_int()
        rc = lib.orc_compress(ctypes.cast(ref.ctypes.data, ctypes.c_char_p), ref.size, ctypes.cast(tgt.ctypes.data, ctypes.c_char_p), tgt.size,
                              header, len(header), ctypes.byref(out), ctypes.byref(n), ctypes.byref(mode))
        data = ctypes.string_at(out, n.value) if out.value else b""
        if out.value:
            lib.orc_free(out)
        return (rc, mode.value, data)
    with cf.ThreadPoolExecutor(max_workers=max(1, min(len(items), os.cpu_count() or 1))) as ex:
        return list(ex.map(one, items))


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scale", type=float, default=1.0, help="shrink every chromosome (debug runs only; 1.0 = the named config)")
    ap.add_argument("--no-verify", action="store_true", help="skip the untimed oracle / reference comparisons")
    ap.add_argument("--no-global", action="store_true", help="skip the global-mode sub-benchmarks")
    ap.add_argument("--no-ref-full", action="store_true", help="reference arm: skip the one-off full chr1-sized run")
    ap.add_argument("--size", type=int, default=0, help="reference arm: bp of the chr1-sized pair generated for the slices (default: as many as the cores need)")
    ap.add_argument("--cpu-sample", type=int, default=20_000_000, help="bp of the chr1-sized pair timed on 1 host core as cpu_baseline")
    ap.add_argument("--dump-outputs", metavar="DIR", type=Path, help="write the outputs of the last timed step as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    import oracle_lib as ol
    from sccg_genome_compression_b200 import synth

    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_numa_node(local_rank)             # before any page-locked allocation: first touch puts the buffers next to the GPU
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce(x: float, op="max") -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op={"max": dist.ReduceOp.MAX, "min": dist.ReduceOp.MIN, "sum": dist.ReduceOp.SUM}[op])
        return float(t.item())

    # ---- communicator of the C++ multi-GPU layer: rank 0 creates the NCCL id, torch.distributed only carries its 128 bytes
    ctx = sccg_b200.Context(local_rank)
    uid = torch.zeros(sccg_b200.MGPU_ID_BYTES, dtype=torch.uint8)
    if rank == 0:
        uid = torch.frombuffer(bytearray(sccg_b200.mgpu_unique_id()), dtype=torch.uint8)
    if world > 1:
        uid = uid.cuda(); dist.broadcast(uid, 0); uid = uid.cpu()
    mg = sccg_b200.Mgpu(ctx, bytes(uid.numpy().tobytes()), rank, world)

    # ---- workload: 24 pairs, LPT over the ranks; this rank's pairs in pinned host memory AND in HBM, before any clock starts
    lengths = genome_lengths(args.scale)
    total_bp = sum(lengths)
    owner = sccg_b200.mgpu_assign(lengths, world)
    mine = [i for i in range(len(lengths)) if owner[i] == rank]
    pad = torch.zeros(64, dtype=torch.uint8)                    # *_device entry points may read a few bytes past the end
    pairs = {}
    for i in mine:
        ref_np, tgt_np = synth.local_pair(lengths[i], synth.seed_for(2, i))
        assert not bool((ref_np >= 97).any())                    # upper-case reference: it is its own prepared form (decompression.cpp:110)
        h_ref = torch.cat([torch.from_numpy(ref_np), pad]).pin_memory()
        h_tgt = torch.cat([torch.from_numpy(tgt_np), pad]).pin_memory()
        pairs[i] = {"n": int(tgt_np.size), "nr": int(ref_np.size), "h_ref": h_ref, "h_tgt": h_tgt, "d_ref": h_ref.cuda(), "d_tgt": h_tgt.cuda(),
                    "ref_np": h_ref.numpy()[:ref_np.size], "tgt_np": h_tgt.numpy()[:tgt_np.size], "header": header_of(i)}
        del ref_np, tgt_np
    my_bp = sum(p["n"] for p in pairs.values())
    max_tgt = max([p["n"] for p in pairs.values()], default=0)

    # untimed: one device-resident pass; the encoded images feed the decompress halves and the verification
    for i, p in pairs.items():
        ptr, n, mode = ctx.compress_device(p["d_ref"].data_ptr(), p["nr"], p["d_tgt"].data_ptr(), p["n"], p["header"])
        assert mode == 0, "workload left the local path"
        enc = ctx.download(ptr, n)
        header, low, nline, body = ol.split_intermediate(enc)
        p["enc"] = enc
        p["h_inter"] = torch.frombuffer(bytearray(enc), dtype=torch.uint8).pin_memory()
        p["d_body"] = torch.cat([torch.frombuffer(bytearray(body), dtype=torch.uint8), pad]).cuda(); p["n_body"] = len(body)
        p["d_low"] = torch.cat([torch.frombuffer(bytearray(low), dtype=torch.uint8), pad]).cuda(); p["n_low"] = len(low)
    d_n = torch.zeros(64, dtype=torch.uint8, device="cuda")
    enc_total = int(reduce(float(sum(len(p["enc"]) for p in pairs.values())), "sum"))
    h_gather = torch.empty(enc_total + 4096 if rank == 0 else 16, dtype=torch.uint8).pin_memory()
    h_out = torch.empty(max_tgt + max_tgt // 50 + 4096, dtype=torch.uint8).pin_memory()

    launches = 0

    def genome_compress(device_resident: bool):
        """one pass over this rank's pairs + the NCCL gather of the encoded streams to rank 0 -> (device ms, launches, items)"""
        dev_ms, nl = 0.0, 0
        for i, p in pairs.items():
            if device_resident:
                mg.compress_item_device(i, p["d_ref"].data_ptr(), p["nr"], p["d_tgt"].data_ptr(), p["n"], p["header"])
            else:
                mg.compress_item(i, _cbuf(p["h_ref"], p["nr"]), _cbuf(p["h_tgt"], p["n"]), p["header"])
            pr = ctx.profile(); dev_ms += pr["kernels_ms"]; nl += pr["launches"]
        # inputs resident in HBM: the gathered streams stay in rank 0's HBM as well (like sccg_compress_device's image); from host
        # buffers: they go on to rank 0's page-locked buffer
        items = mg.gather_device() if device_resident else mg.gather(h_gather.data_ptr(), h_gather.numel())
        dev_ms += ctx.profile()["exchange_ms"]
        return dev_ms, nl, items

    def genome_decompress(device_resident: bool):
        """one pass over this rank's pairs -> (device ms, launches, output length of the last pair)"""
        dev_ms, nl, n_out = 0.0, 0, 0
        for i, p in pairs.items():
            if device_resident:
                _, n_out = ctx.reconstruct_device(p["d_ref"].data_ptr(), p["nr"], p["d_body"].data_ptr(), p["n_body"], d_n.data_ptr(), 0, p["d_low"].data_ptr(), p["n_low"])
            else:
                n_out = ctx.decompress_into(_cbuf(p["h_ref"], p["nr"]), _cbuf(p["h_inter"]), h_out.data_ptr(), h_out.numel())
            pr = ctx.profile(); dev_ms += pr["kernels_ms"]; nl += pr["launches"]
        return dev_ms, nl, n_out

    for _ in range(args.warmup):
        genome_compress(True); genome_decompress(True); genome_compress(False); genome_decompress(False)

    def timed(fn, steps):
        """K steps between barriers -> (device ms per step summed over this rank's calls, wall ms per step), both max over ranks"""
        nonlocal launches
        barrier()
        t0 = time.perf_counter()
        dev = 0.0
        last = None
        for _ in range(steps):
            r = fn()
            dev += r[0]; launches += r[1]; last = r
        barrier()
        wall = (time.perf_counter() - t0) * 1e3 / steps
        return reduce(dev / steps), reduce(wall), last

    K = args.steps
    res = {}
    dump = {} if args.dump_outputs and rank == 0 else None
    with ClockSampler(local_rank) as clocks:
        res["c_dev"] = timed(lambda: genome_compress(True), K)
        if dump is not None:                                      # the gathered streams live until the next gather
            d_streams, spans = res["c_dev"][2][2]
            streams = b"".join(ctx.download(d_streams + spans[i][0], spans[i][1]) for i in sorted(spans))
            dump["genome_compressed"] = dump_sample(streams, 5 << 20)
            dump["genome_compressed_lengths"] = np.array([spans[i][1] for i in sorted(spans)], dtype=np.float64)
            del streams
        res["d_dev"] = timed(lambda: genome_decompress(True), K)
        res["c_e2e"] = timed(lambda: genome_compress(False), K)
        gathered = res["c_e2e"][2][2]
        res["d_e2e"] = timed(lambda: genome_decompress(False), K)
        if dump is not None:                                      # h_out holds the last pair's image until the chr1 leg below
            dump[f"genome_decompressed_pair{list(pairs)[-1]}"] = dump_sample(h_out[:res["d_e2e"][2][2]].numpy(), 3 << 20)

        # ---- chr1-sized pair on ONE GPU (BASELINE configs[1]): rank 0 owns pair 0; the other ranks wait at the barrier
        chr1 = None
        if rank == 0:
            p = pairs[0]
            cm = mm = dm = gm = 0.0
            for _ in range(K):
                ctx.compress_device(p["d_ref"].data_ptr(), p["nr"], p["d_tgt"].data_ptr(), p["n"], p["header"])
                pr = ctx.profile(); cm += pr["kernels_ms"]; mm += pr["match_ms"]; launches += pr["launches"]
            for _ in range(K):
                ctx.reconstruct_device(p["d_ref"].data_ptr(), p["nr"], p["d_body"].data_ptr(), p["n_body"], d_n.data_ptr(), 0, p["d_low"].data_ptr(), p["n_low"])
                pr = ctx.profile(); dm += pr["kernels_ms"]; gm += pr["gather_ms"]; launches += pr["launches"]
            h_enc = torch.empty(len(p["enc"]) + 4096, dtype=torch.uint8).pin_memory()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(K):
                e_len, e_mode = ctx.compress_into(_cbuf(p["h_ref"], p["nr"]), _cbuf(p["h_tgt"], p["n"]), p["header"], h_enc.data_ptr(), h_enc.numel())
                e2e_prof = ctx.profile(); launches += e2e_prof["launches"]
            c_e2e_ms = (time.perf_counter() - t0) * 1e3 / K
            t0 = time.perf_counter()
            for _ in range(K):
                d_len = ctx.decompress_into(_cbuf(p["h_ref"], p["nr"]), _cbuf(p["h_inter"]), h_out.data_ptr(), h_out.numel())
                e2e_dprof = ctx.profile(); launches += e2e_dprof["launches"]
            d_e2e_ms = (time.perf_counter() - t0) * 1e3 / K
            assert bytes(h_enc[:e_len].numpy()) == p["enc"], "end-to-end output differs from the device-resident output"
            chr1 = {"comp_ms": cm / K, "match_ms": mm / K, "dec_ms": dm / K, "gather_ms": gm / K, "c_e2e_ms": c_e2e_ms, "d_e2e_ms": d_e2e_ms,
                    "e2e_prof": e2e_prof, "e2e_dprof": e2e_dprof, "d_len": d_len}
        barrier()

        # ---- one chromosome over all ranks by segment range (N > 1): every rank holds the chr1-sized pair in pinned memory
        sharded = None
        if world > 1:
            if rank == 0:
                s_ref, s_tgt = pairs[0]["h_ref"], pairs[0]["h_tgt"]
            else:
                r_np, t_np = synth.local_pair(lengths[0], synth.seed_for(2, 0))
                s_ref = torch.cat([torch.from_numpy(r_np), pad]).pin_memory(); s_tgt = torch.cat([torch.from_numpy(t_np), pad]).pin_memory()
            n0 = lengths[0]
            h_sh = torch.empty(max(len(pairs[0]["enc"]) + 4096 if rank == 0 else 16, 16), dtype=torch.uint8).pin_memory()

            def shard_step():
                got = mg.compress_sharded(_cbuf(s_ref, n0), _cbuf(s_tgt, n0), CHR1_HEADER, h_sh.data_ptr() if rank == 0 else 0, h_sh.numel() if rank == 0 else 0)
                return 0.0, ctx.profile()["launches"], got
            for _ in range(args.warmup):
                shard_step()
            _, sh_wall, sh_last = timed(shard_step, K)
            ok = True
            if rank == 0:
                n_img, _, was_sharded = sh_last[2]
                ok = bool(was_sharded) and bytes(h_sh[:n_img].numpy()) == pairs[0]["enc"]
            sharded = {"ms_per_step": sh_wall, "value": n0 / (sh_wall / 1e3) / 1e6, "unit": "Mbp/s", "byte_identical_to_unsharded": ok,
                       "api": "sccg_mgpu_compress_sharded: pinned host buffers on every rank, slices uploaded per rank, image on rank 0"}
            assert ok, "sharded output differs from the unsharded file"

        # ---- global-mode pairs (BASELINE configs[0] shape and configs[2]) on one GPU
        glob = {}
        if rank == 0 and not args.no_global:
            for name, cfg, gen in (("global_gap_chr19", 1, lambda s: synth.global_gap_pair(int(63_811_651 * s), int(59_128_983 * s), synth.seed_for(1, 0))),
                                   ("global_divergent_chr21", 3, lambda s: synth.divergent_pair(int(48_129_895 * s), synth.seed_for(3, 0)))):
                glob[name] = global_bench(ctx, ol, gen, args, name, cfg, dump)
                launches += glob[name].pop("_launches")
        barrier()
    launches = int(reduce(float(launches), "sum"))
    if dump is not None:
        assert sum(a.nbytes for a in dump.values()) <= 64_000_000
        args.dump_outputs.mkdir(parents=True, exist_ok=True)
        for name, a in dump.items():
            np.save(args.dump_outputs / f"{name}.npy", a)

    # ---- the host's PCIe ceiling with all ranks copying at once (plain cudaMemcpyAsync from / to page-locked memory, no kernels):
    #      what the end-to-end numbers above can reach at most on this box
    pcie = {}
    nbytes = 256 << 20
    h_probe = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    d_probe = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    for name, fn in (("h2d", lambda: d_probe.copy_(h_probe, non_blocking=True)), ("d2h", lambda: h_probe.copy_(d_probe, non_blocking=True))):
        fn(); barrier()
        t0 = time.perf_counter()
        for _ in range(8):
            fn()
        barrier()
        dt = reduce(time.perf_counter() - t0)
        pcie[name + "_gbs_aggregate"] = world * 8 * nbytes / dt / 1e9
    pcie["note"] = f"{world} rank(s) copying simultaneously, 8 x 256 MiB each; e2e compress moves {2 * total_bp / 1e9:.2f} GB host->device per step"
    del h_probe, d_probe

    # ---- untimed verification of what was timed
    verified = parity_ref = None
    if not args.no_verify:
        ok = True
        # (a) every pair of this rank: GPU image == C oracle image (the oracle is the checker), all ranks in parallel
        exp = oracle_compress_many([(p["ref_np"], p["tgt_np"], p["header"]) for p in pairs.values()])
        for (i, p), (rc, mode, data) in zip(pairs.items(), exp):
            ok = ok and rc == 0 and mode == 0 and data == p["enc"]
        # (b) the gathered streams on rank 0 are those images
        if rank == 0:
            ok = ok and sorted(gathered) == list(range(len(lengths)))
            for i, p in pairs.items():
                off, n = gathered[i]
                ok = ok and bytes(h_gather[off:off + n].numpy()) == p["enc"]
        # (c) decompression gives back every target's FASTA text (round trip; targets are on the lossless envelope)
        for i, p in pairs.items():
            d_len = ctx.decompress_into(_cbuf(p["h_ref"], p["nr"]), _cbuf(p["h_inter"]), h_out.data_ptr(), h_out.numel())
            want = fasta_image(p["header"], p["tgt_np"])
            ok = ok and d_len == len(want) and bytes(h_out[:d_len].numpy()) == want
        if rank == 0:                                             # ... and equals the oracle's decoder on the chr1-sized pair
            p = pairs[0]
            rc, oback = ol.orc_decompress(p["ref_np"].tobytes(), p["enc"])
            d_len = ctx.decompress_into(_cbuf(p["h_ref"], p["nr"]), _cbuf(p["h_inter"]), h_out.data_ptr(), h_out.numel())
            ok = ok and rc == 0 and bytes(h_out[:d_len].numpy()) == oback
        verified = reduce(1.0 if ok else 0.0, "min") == 1.0
        assert verified, "output differs from the oracle"

    # ---- CPU baseline beside it (rank 0, N = 1 only): the reference on one host core, bounded sample of the chr1-sized pair;
    #      its two output files are compared with the GPU's output on the same sample
    cpu = None
    if rank == 0 and world == 1 and args.cpu_sample > 0:
        p = pairs[0]
        sample = min(args.cpu_sample, p["n"])
        r_s, t_s = p["ref_np"][:sample].tobytes(), p["tgt_np"][:sample].tobytes()
        with tempfile.TemporaryDirectory() as d:
            r = cpu_reference_pass([(r_s, t_s, CHR1_HEADER)], Path(d), keep=True)
        cpu = {"value": r["compress_mbp_s"], "unit": "Mbp/s", "cores": 1, "kind": r["kind"],
               "decompress_gbp_s": r["decompress_gbp_s"],
               "sample": f"first {sample} bp of the chr1-sized pair; whole reference `compress` program on 1 core (FASTA read + match + write + "
                         f"delta_encode, 7z = copy shim): {r['compress_s']:.2f} s; `decompress`: {r['decompress_s']:.2f} s"}
        if "intermediate" in r and not args.no_verify:
            g_enc, g_mode = ctx.compress(r_s, t_s, CHR1_HEADER)
            g_back = ctx.decompress(r_s, g_enc)
            parity_ref = bool(g_enc == r["intermediate"] and g_back == r["reconstructed"])
            assert parity_ref, "GPU output differs from the reference executable's files on the sample"

    if rank == 0:
        hbm, which = peaks()
        c_dev_ms, c_wall_ms, _ = res["c_dev"]; d_dev_ms, d_wall_ms, _ = res["d_dev"]
        _, c_e2e_ms, _ = res["c_e2e"]; _, d_e2e_ms, _ = res["d_e2e"]
        p = pairs[0]
        algo = p["nr"] + p["n"]                     # segment-match kernel: both genomes read once (SURVEY 8d, 2.0 B/bp)
        ach = algo / (chr1["match_ms"] / 1e3) / 1e9
        out_len = p["n"] + (p["n"] + 49) // 50
        dec_bytes = p["n_body"] + p["n"] + out_len    # gather kernel: record stream + copied reference symbols + wrapped text (2.02 B/bp)
        dach = dec_bytes / (chr1["gather_ms"] / 1e3) / 1e9
        full = args.scale == 1.0
        roof_c = {"bound": "hbm", "kernel": "seg_match_k (two launches for a device-resident pair: seg_match_defer_k + seg_match_queue_k)", "achieved": ach, "peak": hbm, "unit": "GB/s", "frac": ach / hbm,
                  "traffic": ncu_traffic("seg_match_k") if full else None, "algorithmic_bytes_per_launch": algo, "kernel_ms": chr1["match_ms"],
                  "peak_source": which, "measured_on": "chr1-sized pair (pair 0 of the genome), CUDA events around the matcher launches inside sccg_compress_device"}
        roof_d = {"bound": "hbm", "kernel": "dec_gather_k", "achieved": dach, "peak": hbm, "unit": "GB/s", "frac": dach / hbm,
                  "traffic": ncu_traffic("dec_gather_k") if full else None, "algorithmic_bytes_per_launch": dec_bytes, "kernel_ms": chr1["gather_ms"],
                  "peak_source": which}
        h2d_genome = sum(lengths) * 2                 # references have the targets' lengths in this set
        d2h_dec = sum(n + (n + 49) // 50 + len(header_of(i)) + 1 for i, n in enumerate(lengths))
        line = {
            "metric": METRIC, "value": total_bp / (c_dev_ms / 1e3) / 1e6, "unit": "Mbp/s", "n_gpus": world, "steps": K, "warmup": args.warmup,
            "ms_per_step": c_dev_ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": workload_name(args.scale), "bp_per_step": total_bp, "pairs": len(lengths),
                       "sharding": "pairs LPT-packed onto the ranks (sccg_mgpu_assign), encoded streams gathered to rank 0 over NCCL inside the timed region "
                                   "(value: sccg_mgpu_gather_device, into rank 0's HBM; e2e: sccg_mgpu_gather, on to rank 0's page-locked host buffer)",
                       "pairs_per_rank": [owner.count(r) for r in range(world)], "bp_on_busiest_rank": max(sum(lengths[i] for i in range(len(lengths)) if owner[i] == r) for r in range(world)),
                       "l2": "every pair (2 x 48..249 MB) is larger than the 126 MB L2 and 24 pairs (6.2 GB) are cycled through, no flush needed",
                       "timing": "value: per rank, CUDA events on the library stream around every call (first launch to last completion) + the gather, summed, max over ranks; "
                                 "e2e: wall clock between barriers, max over ranks",
                       "cpu_affinity": numa, "encoded_bytes": enc_total, "mode": "local"},
            "wall_ms_per_step": c_wall_ms,
            "decompress": {"value": total_bp / (d_dev_ms / 1e3) / 1e9, "unit": "Gbp/s", "ms_per_step": d_dev_ms, "wall_ms_per_step": d_wall_ms,
                           "roofline": roof_d,
                           "e2e": {"value": total_bp / (d_e2e_ms / 1e3) / 1e9, "unit": "Gbp/s", "ms_per_step": d_e2e_ms,
                                   "h2d_bytes_per_step": sum(lengths) + enc_total, "d2h_bytes_per_step": d2h_dec,
                                   "api": "sccg_decompress_into per pair: pinned reference + record file in, pinned FASTA image out (every rank keeps its own pairs' text)"}},
            "roofline": roof_c,
            "cpu_baseline": cpu,
            "e2e": {"value": total_bp / (c_e2e_ms / 1e3) / 1e6, "unit": "Mbp/s", "h2d_bytes_per_step": h2d_genome, "d2h_bytes_per_step": enc_total,
                    "ms_per_step": c_e2e_ms, "frac_of_pcie_ceiling": (h2d_genome / (c_e2e_ms / 1e3) / 1e9) / pcie["h2d_gbs_aggregate"],
                    "api": "sccg_mgpu_compress_item per pair (pinned host buffers in, pipelined upload) + sccg_mgpu_gather (NCCL) -> pinned buffer on rank 0"},
            "chr1_local": {
                "workload": "chr1-sized pair (249,250,621 bp), BASELINE configs[1], one GPU" if full else "pair 0 (reduced)",
                "compress": {"value": p["n"] / (chr1["comp_ms"] / 1e3) / 1e6, "unit": "Mbp/s", "ms_per_step": chr1["comp_ms"], "roofline": roof_c,
                             "e2e": {"value": p["n"] / (chr1["c_e2e_ms"] / 1e3) / 1e6, "unit": "Mbp/s", "ms_per_step": chr1["c_e2e_ms"],
                                     "h2d_bytes_per_step": p["nr"] + p["n"], "d2h_bytes_per_step": len(p["enc"]), "h2d_ms": chr1["e2e_prof"]["h2d_ms"],
                                     "d2h_ms": chr1["e2e_prof"]["d2h_ms"], "api": "sccg_compress_into"}},
                "decompress": {"value": p["n"] / (chr1["dec_ms"] / 1e3) / 1e9, "unit": "Gbp/s", "ms_per_step": chr1["dec_ms"], "roofline": roof_d,
                               "e2e": {"value": p["n"] / (chr1["d_e2e_ms"] / 1e3) / 1e9, "unit": "Gbp/s", "ms_per_step": chr1["d_e2e_ms"],
                                       "h2d_bytes_per_step": p["nr"] + len(p["enc"]), "d2h_bytes_per_step": chr1["d_len"], "h2d_ms": chr1["e2e_dprof"]["h2d_ms"],
                                       "d2h_ms": chr1["e2e_dprof"]["d2h_ms"], "api": "sccg_decompress_into"}}},
            "gpu_launches": launches,
            "pcie_ceiling": pcie,
            "clocks": clocks.summary(),
        }
        line.update(glob)
        if sharded is not None:
            line["chr1_sharded"] = sharded
        if verified is not None:
            line["verified_against_oracle"] = verified
            line["verified_what"] = ("all 24 encoded images (every rank its own, C oracle on the host cores), the NCCL-gathered streams on rank 0, every decompressed "
                                     "image against its target's FASTA text, the chr1-sized image against the oracle's decoder")
        if parity_ref is not None:
            line["parity_vs_reference"] = parity_ref
        print(json.dumps(line), flush=True)
    mg.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def global_bench(ctx, ol, gen, args, name: str, cfg: int, dump: dict | None) -> dict:
    """one global-mode pair at full size on one GPU: device-resident + end to end, rooflines of the index build and of the
    parse, the reference beside it on a bounded sample, output verified against the oracle (untimed); the end-to-end
    outputs of the last step go to `dump` when it is given"""
    import torch
    full = args.scale == 1.0
    ref_np, tgt_np = gen(1.0 if full else args.scale)
    nr, nt = int(ref_np.size), int(tgt_np.size)
    header = b">" + name.encode()
    pad = torch.zeros(64, dtype=torch.uint8)
    h_ref = torch.cat([torch.from_numpy(ref_np), pad]).pin_memory(); h_tgt = torch.cat([torch.from_numpy(tgt_np), pad]).pin_memory()
    d_ref, d_tgt = h_ref.cuda(), h_tgt.cuda()
    K = args.steps
    for _ in range(2):
        ptr, n, mode = ctx.compress_device(d_ref.data_ptr(), nr, d_tgt.data_ptr(), nt, header)
    assert mode == 1, "pair did not take the global path"
    enc = ctx.download(ptr, n)
    km = im = pm = mm = 0.0
    nl = 0
    for _ in range(K):
        ctx.compress_device(d_ref.data_ptr(), nr, d_tgt.data_ptr(), nt, header)
        pr = ctx.profile(); km += pr["kernels_ms"]; im += pr["index_ms"]; pm += pr["parse_ms"]; mm += pr["match_ms"]; nl += pr["launches"]
    rounds, steps_front, stride = pr["spec_rounds"], pr["front_steps"], pr["index_stride"]
    h_enc = torch.empty(len(enc) + 4096, dtype=torch.uint8).pin_memory()
    ctx.compress_into(_cbuf(h_ref, nr), _cbuf(h_tgt, nt), header, h_enc.data_ptr(), h_enc.numel())
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(K):
        e_len, _ = ctx.compress_into(_cbuf(h_ref, nr), _cbuf(h_tgt, nt), header, h_enc.data_ptr(), h_enc.numel())
        nl += ctx.profile()["launches"]
    e2e_ms = (time.perf_counter() - t0) * 1e3 / K
    assert bytes(h_enc[:e_len].numpy()) == enc
    if dump is not None:
        dump[name + "_compressed"] = dump_sample(h_enc[:e_len].numpy(), 2 << 20)
    # decompression of the same record stream
    h_inter = torch.frombuffer(bytearray(enc), dtype=torch.uint8).pin_memory()
    h_out = torch.empty(nt + nt // 50 + 4096, dtype=torch.uint8).pin_memory()
    ctx.decompress_into(_cbuf(h_ref, nr), _cbuf(h_inter), h_out.data_ptr(), h_out.numel())
    t0 = time.perf_counter()
    for _ in range(K):
        d_len = ctx.decompress_into(_cbuf(h_ref, nr), _cbuf(h_inter), h_out.data_ptr(), h_out.numel())
        dpr = ctx.profile(); nl += dpr["launches"]
    d_e2e_ms = (time.perf_counter() - t0) * 1e3 / K
    if dump is not None:
        dump[name + "_decompressed"] = dump_sample(h_out[:d_len].numpy(), 1 << 20)
    hbm, which = peaks()
    n_strip_r = nr - int((ref_np == ord("N")).sum()); n_strip_t = nt - int((tgt_np == ord("N")).sum())
    idx_bytes = 5 * n_strip_r + 4 * ((1 << 20) + 1)       # SURVEY 8d: R' read once + one 4-byte position per k-mer written + the bucket table
    parse_bytes = n_strip_r + n_strip_t + len(enc)        # both stripped sequences read once + the records written (2 B/bp)
    out = {"workload": f"{name}: reference {nr} / target {nt} symbols" + ("" if full else " (REDUCED)"), "mode": "global",
           "value": nt / (km / K / 1e3) / 1e6, "unit": "Mbp/s", "ms_per_step": km / K, "index_ms": im / K, "parse_ms": pm / K, "spec_rounds": rounds,
           "front_steps": steps_front, "encoded_bytes": len(enc), "index_stride": stride,
           "roofline": {"index_build": {"bound": "hbm", "kernels": "rs_hist_k + rs_scatter_k x3 + kmer_buckets_k" + (" over every %dth position + gp_first_k / gp_first_scan_k / gp_first_collect_k (one or three passes over R')" % stride if stride > 1 else ""),
                                        "note": "algorithmic bytes = SURVEY 8d's formula for an index of EVERY reference k-mer (what the reference builds); with index_stride > 1 the parse gets by with a sampled index, so less than that is moved", "achieved": idx_bytes / (im / K / 1e3) / 1e9, "peak": hbm,
                                        "unit": "GB/s", "frac": idx_bytes / (im / K / 1e3) / 1e9 / hbm, "algorithmic_bytes": idx_bytes, "ms": im / K},
                        "parse": {"bound": "hbm", "kernels": "gp_spec_k + gp_front_k + gp_concat_k", "achieved": parse_bytes / (pm / K / 1e3) / 1e9, "peak": hbm, "unit": "GB/s",
                                  "frac": parse_bytes / (pm / K / 1e3) / 1e9 / hbm, "algorithmic_bytes": parse_bytes, "ms": pm / K}, "peak_source": which},
           "e2e": {"value": nt / (e2e_ms / 1e3) / 1e6, "unit": "Mbp/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": nr + nt, "d2h_bytes_per_step": len(enc), "api": "sccg_compress_into"},
           "decompress_e2e": {"value": nt / (d_e2e_ms / 1e3) / 1e9, "unit": "Gbp/s", "ms_per_step": d_e2e_ms, "kernels_ms": dpr["kernels_ms"], "api": "sccg_decompress_into"},
           "_launches": nl}
    if not args.no_verify:
        rc, exp, emode = ol.orc_compress(ref_np.tobytes(), tgt_np.tobytes(), header)
        want = fasta_image(header, tgt_np)
        out["verified_against_oracle"] = bool(rc == 0 and emode == 1 and exp == enc and bytes(h_out[:d_len].numpy()) == want)
        assert out["verified_against_oracle"], name + ": output differs from the oracle"
    if args.cpu_sample > 0 and not args.no_verify:
        # the reference itself on a 1/20 scale model of the same pair (its global mode needs ~100 B of RAM per base and minutes at full size)
        s_ref, s_tgt = gen(0.05 if full else min(0.05, args.scale))
        with tempfile.TemporaryDirectory() as d:
            r = cpu_reference_pass([(s_ref.tobytes(), s_tgt.tobytes(), header)], Path(d), keep=True)
        g_enc, g_mode = ctx.compress(s_ref.tobytes(), s_tgt.tobytes(), header)
        out["cpu_baseline"] = {"value": r["compress_mbp_s"], "unit": "Mbp/s", "cores": 1, "kind": r["kind"], "decompress_gbp_s": r["decompress_gbp_s"],
                               "sample": f"1/20 scale model of the pair ({s_tgt.size} target symbols), whole reference `compress` / `decompress` programs: "
                                         f"{r['compress_s']:.2f} s / {r['decompress_s']:.2f} s"}
        if "intermediate" in r:
            out["parity_vs_reference"] = bool(g_mode == 1 and g_enc == r["intermediate"])
            assert out["parity_vs_reference"], name + ": GPU output differs from the reference executable on the sample"
    return out


if __name__ == "__main__":
    main()
