"""bench.py contract.  On the CPU: the reference arm (`--impl reference`) runs the compiled reference (oracle/_ref; the C oracle
port where it is not built) on host cores and prints one JSON line with the agreed keys; the sample behind --dump-outputs is
fixed.  On the GPU: --dump-outputs writes the outputs the timed legs computed."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import oracle_lib as ol

ROOT = Path(__file__).resolve().parent.parent


def test_reference_arm_json_line():
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--size", "9000000", "--steps", "1", "--warmup", "0", "--no-ref-full"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-500:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
                "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["unit"] == "Mbp/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == ("reference" if ol.have_reference() else "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"]
    assert "workload" in line["config"]


def test_reference_arm_other_ranks_stay_silent(monkeypatch):
    import os
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "2", "--size", "9000000", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_dump_sample_is_fixed():
    import bench
    B = bench.DUMP_BLOCK
    data = np.random.default_rng(5).integers(0, 256, 100 * B + 17, dtype=np.uint8)
    whole = bench.dump_sample(data[:5000], 2 * B)
    assert whole.dtype == np.float32 and np.array_equal(whole, data[:5000])
    a = bench.dump_sample(data, 40 * B)
    assert a.dtype == np.float32 and a.size == 40 * B
    assert np.array_equal(a, bench.dump_sample(data.tobytes(), 40 * B))        # same sample from run to run
    where = {data[k * B:(k + 1) * B].tobytes(): k for k in range(100)}
    picked = [where[blk.astype(np.uint8).tobytes()] for blk in a.reshape(40, B)]
    assert picked == sorted(set(picked))                                          # whole aligned blocks, ascending, no repeats


@pytest.mark.gpu
def test_dump_outputs_are_the_timed_outputs(tmp_path):
    """--dump-outputs on a reduced genome (small enough that nothing is sampled): every array is the C oracle's output for
    its pair, so two builds that dump the same arrays computed the same files.  (At this scale every target still decodes
    to its own FASTA text, which the bench checks; at 0.004 the first pair does not.)"""
    import bench
    from sccg_genome_compression_b200 import synth
    scale = 0.01
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--scale", str(scale), "--steps", "2", "--warmup", "1", "--cpu-sample", "0",
                        "--dump-outputs", str(tmp_path / "out")], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-800:]
    got = {p.stem: np.load(p) for p in (tmp_path / "out").glob("*.npy")}
    assert sum(a.nbytes for a in got.values()) <= 64_000_000
    lengths = bench.genome_lengths(scale)
    last = len(lengths) - 1
    images, tgts = [], {}
    for i, n in enumerate(lengths):
        ref, tgt = synth.local_pair(n, synth.seed_for(2, i))
        rc, img, mode = ol.orc_compress(ref.tobytes(), tgt.tobytes(), bench.header_of(i))
        assert rc == 0 and mode == 0
        images.append(img)
        tgts[i] = tgt
    assert got["genome_compressed_lengths"].dtype == np.float64 and got["genome_compressed_lengths"].tolist() == [len(x) for x in images]
    assert got["genome_compressed"].dtype == np.float32
    assert np.array_equal(got["genome_compressed"], np.frombuffer(b"".join(images), dtype=np.uint8))
    assert np.array_equal(got[f"genome_decompressed_pair{last}"], np.frombuffer(bench.fasta_image(bench.header_of(last), tgts[last]), dtype=np.uint8))
    for name, (ref, tgt) in (("global_gap_chr19", synth.global_gap_pair(int(63_811_651 * scale), int(59_128_983 * scale), synth.seed_for(1, 0))),
                             ("global_divergent_chr21", synth.divergent_pair(int(48_129_895 * scale), synth.seed_for(3, 0)))):
        header = b">" + name.encode()
        rc, img, mode = ol.orc_compress(ref.tobytes(), tgt.tobytes(), header)
        assert rc == 0 and mode == 1
        assert np.array_equal(got[name + "_compressed"], np.frombuffer(img, dtype=np.uint8))
        assert np.array_equal(got[name + "_decompressed"], np.frombuffer(bench.fasta_image(header, tgt), dtype=np.uint8))
    assert len(got) == 7
