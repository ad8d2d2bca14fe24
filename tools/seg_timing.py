#!/usr/bin/env python
"""Development aid: per-segment clock64() cost of seg_match_k on the bench workload (needs the
-DSCCG_SEG_TIMING build written to /tmp by this script).  usage: seg_timing.py [chrom]"""
import ctypes, subprocess, sys
from pathlib import Path
ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import numpy as np, torch
import sccg_b200
from sccg_genome_compression_b200 import synth
so = "/tmp/libsccg_timing.so"
prebuilt = [a for a in sys.argv[1:] if a.endswith(".so")]
sys.argv = [a for a in sys.argv if not a.endswith(".so")]
if prebuilt: so = prebuilt[0]
else: subprocess.check_call(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xcompiler", "-fPIC", "-shared", "--cudart", "static",
                       "-ccbin", "/usr/bin/g++", "-DSCCG_SEG_TIMING", "-o", so, str(ROOT / "sccg-genome-compression_b200/csrc/sccg_b200.cu")])
chrom = int(sys.argv[1]) if len(sys.argv) > 1 else 1
ref, tgt = synth.local_pair(synth.CHR1_LEN, synth.seed_for(2, chrom))
ctx = sccg_b200.Context(0, lib_path=so)
pad = torch.zeros(64, dtype=torch.uint8)
d_ref = torch.cat([torch.from_numpy(ref), pad]).cuda(); d_tgt = torch.cat([torch.from_numpy(tgt), pad]).cuda()
nseg = (ref.size + 999) // 1000
cyc = torch.zeros(7 * nseg, dtype=torch.int64, device="cuda")      # totals + 6 phase arrays (generic segments)
ctx.lib.sccg_debug_seg_timing.argtypes = [ctypes.c_void_p]
for _ in range(2):
    ctx.compress_device(d_ref.data_ptr(), ref.size, d_tgt.data_ptr(), tgt.size, b">x")
assert ctx.lib.sccg_debug_seg_timing(cyc.data_ptr()) == 0
ctx.compress_device(d_ref.data_ptr(), ref.size, d_tgt.data_ptr(), tgt.size, b">x")
print(ctx.profile())
call = cyc.cpu().numpy().reshape(7, nseg)
c = call[0]
ph = call[1:]
gen = ph[1] > 0
print("generic segments", int(gen.sum()), "mean cycles: staged %.0f diagonal attempt %.0f runs %.0f index %.0f parse %.0f epilogue %.0f" % tuple(ph[i][gen].mean() for i in range(6)), " total mean", c[gen].mean())
print("segments", nseg, "sum cycles", c.sum(), "mean", c.mean(), "median", np.median(c), "p99", np.percentile(c, 99), "max", c.max())
tu = np.where((tgt >= 97) & (tgt <= 122), tgt - 32, tgt).astype(np.uint8)
ru = np.where((ref >= 97) & (ref <= 122), ref - 32, ref).astype(np.uint8)
# path of each segment: identical pairs are decided in registers, generic segments record their phases, the rest took the
# diagonal-hypothesis path (the same split for any build of the library, so two builds can be compared)
m = min(ru.size, tu.size) // 1000 * 1000
ident = np.zeros(nseg, dtype=bool)
ident[:m // 1000] = (ru[:m] == tu[:m]).reshape(-1, 1000).all(axis=1)
diag = ~ident & ~gen
for name, sel in (("identical", ident), ("diagonal", diag), ("generic", gen)):
    print(f"path {name}: {int(sel.sum())} segments, mean cycles {c[sel].mean() if sel.any() else 0.0:.0f}, sum {int(c[sel].sum())}")
top = np.argsort(-c)[:15]
for i in top:
    r = ref[i * 1000:(i + 1) * 1000]; t = tu[i * 1000:(i + 1) * 1000]
    m = min(r.size, t.size)
    print("   phases", [int(ph[q][i]) for q in range(6)])
    print(f"seg {i}: cycles {c[i]}  mismatches {(r[:m] != t[:m]).sum()}  rN {(r == 78).sum()} tN {(t == 78).sum()}  r[:40]={r[:40].tobytes()}")
reg = 10_000                                     # segments per region (10 Mbp)
for a in range(0, nseg, reg):
    x = c[a:a + reg]
    print(f"segments {a:>7d}..: mean cycles {x.mean():9.0f}  max {x.max():9d}  > 100k cycles: {(x > 100000).sum()}")
hist = np.bincount(np.minimum(c // 20000, 50).astype(np.int64))
print("histogram (20k-cycle bins):", hist.tolist())
