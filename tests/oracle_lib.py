"""ctypes bindings for the CPU oracle (oracle/libsccg_oracle.so) and, when it has been built,
the compiled UNMODIFIED reference (oracle/_ref/libsccg_ref.so + executables).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  The product package never imports this module.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile
from dataclasses import dataclass
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
ORACLE_DIR = ROOT / "oracle"
REF_DIR = ORACLE_DIR / "_ref"


def build_oracle(force: bool = False) -> Path:
    so = ORACLE_DIR / "libsccg_oracle.so"
    src = ORACLE_DIR / "sccg_oracle.c"
    if force or not so.exists() or so.stat().st_mtime < src.stat().st_mtime:
        subprocess.check_call(["make", "-C", str(ORACLE_DIR), "oracle"], stdout=subprocess.DEVNULL)
    return so


def build_reference() -> bool:
    """Compile the reference into oracle/_ref where its sources are readable (__graft_entry__.oracle_make says where they
    are looked for); True if oracle/_ref is usable."""
    import __graft_entry__ as g
    subprocess.check_call(g.oracle_make("ref"), stdout=subprocess.DEVNULL)
    return have_reference()


def have_reference() -> bool:
    return (REF_DIR / "libsccg_ref.so").exists() and (REF_DIR / "compress").exists()


class _OrcRecord(C.Structure):
    _fields_ = [("p", C.c_int), ("l", C.c_int), ("lit_off", C.c_long), ("lit_len", C.c_long)]


class _OrcRecords(C.Structure):
    _fields_ = [("rec", C.POINTER(_OrcRecord)), ("n", C.c_long), ("lits", C.c_void_p), ("lits_len", C.c_long)]


@dataclass
class Record:
    p: int
    l: int
    lit: bytes  # b"" for a match record

    def __repr__(self):
        return f"({self.p},{self.l})" if not self.lit else f"lit[{len(self.lit)}]{self.lit[:24]!r}"


_oracle = None


def oracle():
    global _oracle
    if _oracle is None:
        lib = C.CDLL(str(build_oracle()))
        lib.orc_match_sequences.argtypes = [C.c_char_p, C.c_long, C.c_char_p, C.c_long, C.c_int, C.c_int, C.c_int,
                                            C.c_int, C.POINTER(_OrcRecords)]
        lib.orc_records_free.argtypes = [C.POINTER(_OrcRecords)]
        lib.orc_compress.argtypes = [C.c_char_p, C.c_long, C.c_char_p, C.c_long, C.c_char_p, C.c_long,
                                     C.POINTER(C.c_void_p), C.POINTER(C.c_long), C.POINTER(C.c_int)]
        lib.orc_delta_encode.argtypes = [C.c_char_p, C.c_long, C.POINTER(C.c_void_p), C.POINTER(C.c_long)]
        lib.orc_reconstruct.argtypes = [C.c_char_p, C.c_long, C.c_char_p, C.c_long, C.c_char_p, C.c_long, C.c_char_p,
                                        C.c_long, C.POINTER(C.c_void_p), C.POINTER(C.c_long)]
        lib.orc_parse_reference_fasta.argtypes = [C.c_char_p, C.c_long, C.POINTER(C.c_void_p), C.POINTER(C.c_long)]
        lib.orc_parse_target_fasta.argtypes = [C.c_char_p, C.c_long, C.POINTER(C.c_void_p), C.POINTER(C.c_long),
                                               C.POINTER(C.c_void_p), C.POINTER(C.c_long)]
        lib.orc_free.argtypes = [C.c_void_p]
        _oracle = lib
    return _oracle


def _take(lib_free, ptr: C.c_void_p, n: int) -> bytes:
    data = C.string_at(ptr, n) if ptr.value else b""
    if ptr.value:
        lib_free(ptr)
    return data


# ----------------------------------------------------------------------------- oracle wrappers
def orc_match_sequences(Sr: bytes, St: bytes, k: int, m: int, is_global: bool, offset: int = 0) -> list[Record]:
    lib = oracle()
    out = _OrcRecords()
    rc = lib.orc_match_sequences(Sr, len(Sr), St, len(St), k, m, int(is_global), offset, C.byref(out))
    assert rc == 0
    lits = C.string_at(out.lits, out.lits_len) if out.lits else b""
    recs = []
    for i in range(out.n):
        r = out.rec[i]
        recs.append(Record(r.p, r.l, lits[r.lit_off:r.lit_off + r.lit_len]))
    lib.orc_records_free(C.byref(out))
    return recs


def orc_compress(ref: bytes, tgt: bytes, header: bytes) -> tuple[int, bytes, int]:
    """-> (rc, compressed_genome.txt bytes, mode 0 local / 1 global)"""
    lib = oracle()
    out = C.c_void_p(); n = C.c_long(); mode = C.c_int()
    rc = lib.orc_compress(ref, len(ref), tgt, len(tgt), header, len(header), C.byref(out), C.byref(n), C.byref(mode))
    return rc, _take(lib.orc_free, out, n.value), mode.value


def orc_delta_encode(text: bytes) -> tuple[int, bytes]:
    lib = oracle()
    out = C.c_void_p(); n = C.c_long()
    rc = lib.orc_delta_encode(text, len(text), C.byref(out), C.byref(n))
    return rc, _take(lib.orc_free, out, n.value)


def orc_reconstruct(ref: bytes, enc: bytes, n_idx: bytes, low_idx: bytes) -> tuple[int, bytes]:
    lib = oracle()
    out = C.c_void_p(); n = C.c_long()
    rc = lib.orc_reconstruct(ref, len(ref), enc, len(enc), n_idx, len(n_idx), low_idx, len(low_idx),
                             C.byref(out), C.byref(n))
    return rc, _take(lib.orc_free, out, n.value)


def orc_parse_reference_fasta(data: bytes) -> bytes:
    lib = oracle()
    out = C.c_void_p(); n = C.c_long()
    lib.orc_parse_reference_fasta(data, len(data), C.byref(out), C.byref(n))
    return _take(lib.orc_free, out, n.value)


def orc_parse_target_fasta(data: bytes) -> tuple[bytes, bytes]:
    lib = oracle()
    out = C.c_void_p(); n = C.c_long(); h = C.c_void_p(); nh = C.c_long()
    lib.orc_parse_target_fasta(data, len(data), C.byref(out), C.byref(n), C.byref(h), C.byref(nh))
    return _take(lib.orc_free, out, n.value), _take(lib.orc_free, h, nh.value)


def split_intermediate(data: bytes) -> tuple[bytes, bytes, bytes, bytes]:
    """decompress_genome's line split (decompression.cpp:66-101): -> (header, lowercase, nline, body)."""
    lines = data.split(b"\n")
    if data.startswith(b">"):
        return lines[0], lines[1], lines[2], lines[3]
    return b"", lines[0], lines[1], lines[2]


def prepare_reference(ref_raw: bytes, nline: bytes) -> bytes:
    """decompression.cpp:105-110: strip 'N' (before upper-casing!) unless the N line is ','."""
    if nline != b",":
        ref_raw = ref_raw.replace(b"N", b"")
    return ref_raw.upper() if ref_raw.isascii() else bytes(c - 32 if 97 <= c <= 122 else c for c in ref_raw)


def orc_decompress(ref_raw: bytes, intermediate: bytes) -> tuple[int, bytes]:
    """reference `decompress` minus 7z and file I/O: -> (rc, reconstructed_genome.fa bytes)."""
    header, low, nline, body = split_intermediate(intermediate)
    rc, text = orc_reconstruct(prepare_reference(ref_raw, nline), body, b"" if nline == b"," else nline, low)
    return rc, header + b"\n" + text


# ------------------------------------------------------------------- compiled-reference wrappers
_ref = None


def ref():
    global _ref
    if _ref is None:
        lib = C.CDLL(str(REF_DIR / "libsccg_ref.so"))
        lib.sccg_ref_match_sequences.argtypes = [C.c_char_p, C.c_long, C.c_char_p, C.c_long, C.c_int, C.c_int, C.c_int,
                                                 C.c_int, C.POINTER(C.c_long), C.POINTER(C.POINTER(C.c_int)),
                                                 C.POINTER(C.POINTER(C.c_int)), C.POINTER(C.POINTER(C.c_long)),
                                                 C.POINTER(C.c_void_p)]
        lib.sccg_ref_compress_genome.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, C.POINTER(C.c_double)]
        lib.sccg_ref_delta_encode.argtypes = [C.c_char_p]
        lib.sccg_ref_reconstruct_genome.argtypes = [C.c_char_p, C.c_long, C.c_char_p, C.c_long, C.c_char_p, C.c_long,
                                                    C.c_char_p, C.c_long, C.POINTER(C.c_void_p), C.POINTER(C.c_long),
                                                    C.POINTER(C.c_double)]
        lib.sccg_ref_free.argtypes = [C.c_void_p]
        _ref = lib
    return _ref


def shim_env() -> dict:
    env = dict(os.environ)
    env["PATH"] = str(REF_DIR / "bin") + os.pathsep + env.get("PATH", "")
    return env


def ref_match_sequences(Sr: bytes, St: bytes, k: int, m: int, is_global: bool, offset: int = 0) -> list[Record]:
    lib = ref()
    n = C.c_long(); p = C.POINTER(C.c_int)(); l = C.POINTER(C.c_int)(); off = C.POINTER(C.c_long)(); lits = C.c_void_p()
    rc = lib.sccg_ref_match_sequences(Sr, len(Sr), St, len(St), k, m, int(is_global), offset, C.byref(n), C.byref(p),
                                      C.byref(l), C.byref(off), C.byref(lits))
    assert rc == 0
    total = off[n.value]
    lb = C.string_at(lits, total) if total else b""
    recs = [Record(p[i], l[i], lb[off[i]:off[i + 1]]) for i in range(n.value)]
    for q in (p, l, off):
        lib.sccg_ref_free(C.cast(q, C.c_void_p))
    lib.sccg_ref_free(lits)
    return recs


def ref_reconstruct(ref_prepared: bytes, enc: bytes, n_idx: bytes, low_idx: bytes) -> tuple[int, bytes, float]:
    lib = ref()
    out = C.c_void_p(); n = C.c_long(); secs = C.c_double()
    rc = lib.sccg_ref_reconstruct_genome(ref_prepared, len(ref_prepared), enc, len(enc), n_idx, len(n_idx), low_idx,
                                         len(low_idx), C.byref(out), C.byref(n), C.byref(secs))
    return rc, _take(lib.sccg_ref_free, out, n.value), secs.value


def ref_compress_cli(ref_fa: Path, tgt_fa: Path, out_dir: Path) -> tuple[int, bytes]:
    """Run the reference `compress` executable (7z shim on PATH); -> (exit code, compressed_genome.txt)."""
    r = subprocess.run([str(REF_DIR / "compress"), str(ref_fa), str(tgt_fa), str(out_dir)], env=shim_env(),
                       stdout=subprocess.DEVNULL, stderr=subprocess.PIPE)
    f = Path(out_dir) / "compressed_genome.txt"
    return r.returncode, (f.read_bytes() if f.exists() else b"")


def ref_decompress_cli(archive: Path, ref_fa: Path, out_dir: Path) -> tuple[int, bytes, bytes]:
    r = subprocess.run([str(REF_DIR / "decompress"), str(archive), str(ref_fa), str(out_dir)], env=shim_env(),
                       stdout=subprocess.DEVNULL, stderr=subprocess.PIPE)
    f = Path(out_dir) / "reconstructed_genome.fa"
    return r.returncode, (f.read_bytes() if f.exists() else b""), r.stderr


def write_fasta(path: Path, seq: bytes, header: bytes | None = b">seq", width: int = 50, newline: bytes = b"\n",
                trailing_newline: bool = True) -> None:
    parts = []
    if header is not None:
        parts.append(header)
    parts += [seq[i:i + width] for i in range(0, len(seq), width)]
    data = newline.join(parts) + (newline if trailing_newline else b"")
    Path(path).write_bytes(data)


def ref_roundtrip(ref_seq: bytes, tgt_seq: bytes, header: bytes | None = b">tgt") -> dict:
    """compress -> decompress through the reference executables on FASTA files made from the symbols."""
    with tempfile.TemporaryDirectory() as d:
        d = Path(d)
        write_fasta(d / "ref.fa", ref_seq, b">ref")
        write_fasta(d / "tgt.fa", tgt_seq, header)
        rc_c, inter = ref_compress_cli(d / "ref.fa", d / "tgt.fa", d / "out")
        rc_d, recon, err = ref_decompress_cli(d / "out" / "compressed_genome.txt.7z", d / "ref.fa", d / "dec")
        return {"rc_compress": rc_c, "intermediate": inter, "rc_decompress": rc_d, "reconstructed": recon,
                "target_file": (d / "tgt.fa").read_bytes(), "stderr": err}
