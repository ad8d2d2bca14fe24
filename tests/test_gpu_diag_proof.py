"""The diagonal-hypothesis path of the local segment matcher on the GPU (`-m gpu`), judged by the oracle: the cases of
tests/test_emu_diag_proof.py through match_sequences, compress and compress_device."""
import random

import pytest

from test_emu_diag_proof import (K, PLANT_P, check_file, check_match, edge_snps, low_complexity_pair, lower_n_target, planted_file,
                                 planted_pair, run_snps, snp_pair, word_pairs)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    import sccg_b200
    c = sccg_b200.Context(0)
    yield c
    c.close()


def compress_device_gpu(ctx, ref: bytes, tgt: bytes, header: bytes):
    import torch
    pad = torch.zeros(64, dtype=torch.uint8)
    d_ref = torch.cat([torch.frombuffer(bytearray(ref), dtype=torch.uint8), pad]).cuda()
    d_tgt = torch.cat([torch.frombuffer(bytearray(tgt), dtype=torch.uint8), pad]).cuda()
    ptr, n, mode = ctx.compress_device(d_ref.data_ptr(), len(ref), d_tgt.data_ptr(), len(tgt), header)
    return ctx.download(ptr, n), mode


def test_segments(ctx):
    """every single-segment case of the emulator tests, at k = 14 and at k = 10 .. 16"""
    for kind in ("clean", "mutated"):
        for p in PLANT_P:
            check_match(ctx, *planted_pair(p, kind))
    for seed in range(40):
        check_match(ctx, *snp_pair(edge_snps(random.Random(repr(("edge", seed)))), seed, plant=seed % 2 == 1))
    for plant in (False, True):
        for count in (29, 30, 31):
            for start in (0, 100, 501, 1000 - count):
                check_match(ctx, *snp_pair(run_snps(start, count), start, plant=plant))
        for words in (15, 16, 17):
            check_match(ctx, *snp_pair(word_pairs(words), words, plant=plant))
    for kind in range(4):
        for seed in range(3):
            check_match(ctx, *low_complexity_pair(kind, seed))
    for n in (14, 15, 21, 100, 517, 993, 999):
        for seed in range(4):
            r = random.Random(repr(("short", n, seed)))
            check_match(ctx, *snp_pair(edge_snps(r, n), seed, n=n, plant=seed % 2 == 1))
            if n > 40:
                check_match(ctx, *planted_pair(r.choice([0, n - K, n // 2]), ["clean", "mutated"][seed % 2], seed, n=n))
    for k in range(10, 17):
        r = random.Random(repr(("k", k)))
        for p in PLANT_P[::3]:
            check_match(ctx, *planted_pair(p, ["clean", "mutated"][p % 2], k), k=k)
        for seed in range(6):
            check_match(ctx, *snp_pair(edge_snps(r), (k, seed), plant=True), k=k)


@pytest.mark.parametrize("seed", range(4))
def test_files(ctx, seed):
    ref, tgt = planted_file(("gpu", seed))
    check_file(ctx, ref, tgt)
    check_file(ctx, ref, lower_n_target(tgt, seed))


@pytest.mark.parametrize("two_phase", [1, 0])
def test_files_two_phase(ctx, two_phase, monkeypatch):
    monkeypatch.setenv("SCCG_LM_TWO_PHASE_MIN", "0" if two_phase else "2000000000")
    refs, tgts = zip(*(planted_file(("gpu-2ph", s)) for s in range(8)))
    ref, tgt = b"".join(refs), lower_n_target(b"".join(tgts), two_phase)
    for _ in range(2):
        check_file(ctx, ref, tgt, compress=compress_device_gpu)


def test_no_diag_parity(ctx, monkeypatch):
    import sccg_b200
    monkeypatch.setenv("SCCG_NO_DIAG", "1")
    plain = sccg_b200.Context(0)
    try:
        for seed in range(3):
            ref, tgt = planted_file(("gpu-nodiag", seed))
            tgt = lower_n_target(tgt, seed)
            assert plain.compress(ref, tgt, b">x") == ctx.compress(ref, tgt, b">x")
            check_file(plain, ref, tgt, b">x")
    finally:
        plain.close()
