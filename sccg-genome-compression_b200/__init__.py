"""sccg-genome-compression_b200 -- host-side Python mirror of the reference's hot-path functions
(match_sequences / compress_genome / reconstruct_genome of Jan-Celin/SCCG-genome-compression) over
the C ABI of libsccg_b200.so (include/sccg.h).  The library is hand-written CUDA for sm_100a; there
is no CPU fallback: importing works anywhere, but creating a context without the built library or
without a CUDA device raises.

The directory name contains a hyphen, so import it through the shim module at the repo root:

    import sccg_b200
    ctx = sccg_b200.Context(device=0)
    text, mode = ctx.compress(ref_symbols, tgt_symbols, header)
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
DEFAULT_LIB = PKG_DIR / "libsccg_b200.so"

SCCG_OK, SCCG_E_CUDA, SCCG_E_ARG, SCCG_E_FORMAT, SCCG_E_BOUNDS, SCCG_E_NOMEM, SCCG_E_STOI = 0, -1, -2, -3, -4, -5, -6


class SccgError(RuntimeError):
    def __init__(self, code: int, message: str, partial: bytes | None = None):
        super().__init__(f"sccg error {code}: {message}")
        self.code = code
        self.partial = partial      # SCCG_E_STOI: the un-rewritten image the reference leaves on disk before it exits 1


class _Records(C.Structure):
    _fields_ = [("n", C.c_int64), ("p", C.POINTER(C.c_int32)), ("l", C.POINTER(C.c_int32)),
                ("lit_off", C.POINTER(C.c_int64)), ("lits", C.c_void_p)]


class Profile(C.Structure):
    _fields_ = [("h2d_ms", C.c_float), ("kernels_ms", C.c_float), ("d2h_ms", C.c_float), ("match_ms", C.c_float),
                ("serialize_ms", C.c_float), ("gather_ms", C.c_float), ("launches", C.c_int32), ("mode", C.c_int32),
                ("front_steps", C.c_int32), ("spec_rounds", C.c_int32), ("index_ms", C.c_float), ("parse_ms", C.c_float), ("exchange_ms", C.c_float), ("index_stride", C.c_int32)]

    def as_dict(self) -> dict:
        return {k: getattr(self, k) for k, _ in self._fields_}


class ShardInfo(C.Structure):
    """sccg_shard_info (include/sccg.h): what one shard reports across its borders"""
    _fields_ = [("n_segments", C.c_int64), ("abort_inside", C.c_int32), ("has_paren", C.c_int32), ("head_status", C.c_int32 * 4),
                ("tail_status", C.c_int32 * 4), ("has_match", C.c_int32), ("last_p", C.c_int32), ("n_runs", C.c_int64),
                ("first_run_start", C.c_int64), ("first_run_len", C.c_int64), ("last_run_start", C.c_int64), ("last_run_len", C.c_int64)]

    def as_dict(self) -> dict:
        d = {k: getattr(self, k) for k, _ in self._fields_}
        d["head_status"] = list(self.head_status); d["tail_status"] = list(self.tail_status)
        return d


class ShardCarry(C.Structure):
    """sccg_shard_carry (include/sccg.h)"""
    _fields_ = [("prev_p", C.c_int32), ("skip_first_run", C.c_int32), ("extra_last_len", C.c_int64), ("prev_run_start", C.c_int64),
                ("last_run_reaches_end", C.c_int32), ("reserved", C.c_int32)]


@dataclass
class Record:
    """One element of match_sequences' vector<Position> (compression.cpp:20-24)."""
    p: int
    l: int
    lit: bytes

    def __repr__(self):
        return f"({self.p},{self.l})" if not self.lit else f"lit[{len(self.lit)}]{self.lit[:24]!r}"


def _as_char_p(buf):
    """bytes and ctypes char arrays stay as they are; numpy uint8 arrays are passed by address (no copy)"""
    if isinstance(buf, (bytes, bytearray)):
        return bytes(buf) if isinstance(buf, bytearray) else buf
    if isinstance(buf, C.Array):
        return buf
    return C.cast(buf.ctypes.data, C.c_char_p) if len(buf) else b""


SINK_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64)       # sccg_sink_fn (include/sccg.h)

_libs: dict[str, C.CDLL] = {}


def load_library(path: str | os.PathLike | None = None) -> C.CDLL:
    p = Path(path) if path else DEFAULT_LIB
    key = str(p)
    if key in _libs:
        return _libs[key]
    if not p.exists():
        raise OSError(f"{p} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                      "(nvcc, sm_100a). There is no CPU fallback.")
    lib = C.CDLL(key)
    vp, i64, cp = C.c_void_p, C.c_int64, C.c_char_p
    lib.sccg_create.restype = vp
    lib.sccg_create.argtypes = [C.c_int]
    lib.sccg_destroy.argtypes = [vp]
    lib.sccg_last_error.restype = cp
    lib.sccg_version.restype = cp
    lib.sccg_free.argtypes = [vp]
    lib.sccg_records_free.argtypes = [C.POINTER(_Records)]
    lib.sccg_get_profile.argtypes = [vp, C.POINTER(Profile)]
    lib.sccg_download.argtypes = [vp, vp, i64, vp]
    lib.sccg_compress.argtypes = [vp, cp, i64, cp, i64, cp, i64, C.POINTER(vp), C.POINTER(i64), C.POINTER(C.c_int)]
    lib.sccg_compress_device.argtypes = [vp, vp, i64, vp, i64, cp, i64, C.POINTER(vp), C.POINTER(i64), C.POINTER(C.c_int)]
    lib.sccg_match_sequences.argtypes = [vp, cp, i64, cp, i64, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(_Records)]
    lib.sccg_reconstruct.argtypes = [vp, cp, i64, cp, i64, cp, i64, cp, i64, C.POINTER(vp), C.POINTER(i64)]
    lib.sccg_reconstruct_device.argtypes = [vp, vp, i64, vp, i64, vp, i64, vp, i64, C.POINTER(vp), C.POINTER(i64)]
    lib.sccg_decompress.argtypes = [vp, cp, i64, cp, i64, C.POINTER(vp), C.POINTER(i64)]
    lib.sccg_compress_into.argtypes = [vp, cp, i64, cp, i64, cp, i64, vp, i64, C.POINTER(i64), C.POINTER(C.c_int)]
    lib.sccg_reconstruct_into.argtypes = [vp, cp, i64, cp, i64, cp, i64, cp, i64, vp, i64, C.POINTER(i64)]
    lib.sccg_decompress_into.argtypes = [vp, cp, i64, cp, i64, vp, i64, C.POINTER(i64)]
    lib.sccg_decompress_part.argtypes = [vp, cp, i64, cp, i64, C.c_int, C.c_int, vp, i64, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64)]
    lib.sccg_shard_match.argtypes = [vp, cp, i64, cp, i64, i64, C.c_int, C.POINTER(ShardInfo)]
    lib.sccg_shard_write.argtypes = [vp, C.POINTER(ShardCarry), C.POINTER(vp), C.POINTER(i64), C.POINTER(vp), C.POINTER(i64)]
    lib.sccg_reference_set.argtypes = [vp, cp, i64]
    lib.sccg_reference_clear.argtypes = [vp]
    lib.sccg_compress_resident_into.argtypes = [vp, cp, i64, cp, i64, vp, i64, C.POINTER(i64), C.POINTER(C.c_int)]
    lib.sccg_decompress_resident_into.argtypes = [vp, cp, i64, vp, i64, C.POINTER(i64)]
    lib.sccg_compress_fasta.argtypes = [vp, cp, i64, cp, i64, C.POINTER(vp), C.POINTER(i64), C.POINTER(C.c_int)]
    lib.sccg_decompress_fasta.argtypes = [vp, cp, i64, cp, i64, C.POINTER(vp), C.POINTER(i64)]
    i32p, i64p = C.POINTER(C.c_int32), C.POINTER(i64)
    lib.sccg_pinned_alloc.restype = vp
    lib.sccg_pinned_alloc.argtypes = [i64]
    lib.sccg_pinned_free.argtypes = [vp]
    lib.sccg_pinned_free.restype = None
    lib.sccg_compress_fasta_into.argtypes = [vp, cp, i64, cp, i64, vp, i64, i64p, C.POINTER(C.c_int)]
    lib.sccg_decompress_fasta_into.argtypes = [vp, cp, i64, cp, i64, vp, i64, i64p]
    lib.sccg_decompress_stream.argtypes = [vp, cp, i64, cp, i64, SINK_FN, vp, i64p]
    lib.sccg_decompress_fasta_stream.argtypes = [vp, cp, i64, cp, i64, SINK_FN, vp, i64p]
    lib.sccg_extract.argtypes = [vp, cp, i64, cp, i64, vp, i64, vp, i64, i64p, i64p]
    lib.sccg_extract_fasta.argtypes = [vp, cp, i64, cp, i64, vp, i64, vp, i64, i64p, i64p]
    lib.sccg_extract_resident.argtypes = [vp, cp, i64, vp, i64, vp, i64, i64p, i64p]
    lib.sccg_archive_open.argtypes = [vp, cp, i64, C.POINTER(vp)]
    lib.sccg_archive_info.argtypes = [vp, i64p, C.POINTER(C.c_int), i64p]
    lib.sccg_archive_close.argtypes = [vp, vp]
    lib.sccg_archive_extract.argtypes = [vp, vp, i64, vp, i64, vp, i64, i64p]
    lib.sccg_archive_search.argtypes = [vp, vp, i64, vp, i64, cp, vp, i64, C.c_int, C.c_int, vp, i64, i64p]
    lib.sccg_archive_search_edits.argtypes = [vp, vp, i64, vp, i64, cp, vp, i64, C.c_int, C.c_int, vp, i64, i64p]
    lib.sccg_archive_variants.argtypes = [vp, vp, i64, vp, i64, vp, i64, i64p, vp, i64, i64p]
    lib.sccg_archive_liftover.argtypes = [vp, vp, i64, vp, i64, vp]
    lib.sccg_mgpu_unique_id.argtypes = [C.c_char_p]
    lib.sccg_mgpu_init.argtypes = [vp, C.c_char_p, C.c_int, C.c_int, C.POINTER(vp)]
    lib.sccg_mgpu_destroy.argtypes = [vp]
    lib.sccg_mgpu_destroy.restype = None
    lib.sccg_mgpu_assign.argtypes = [i64p, C.c_int, C.c_int, i32p]
    lib.sccg_mgpu_compress_item.argtypes = [vp, C.c_int32, cp, i64, cp, i64, cp, i64, i64p, C.POINTER(C.c_int)]
    lib.sccg_mgpu_compress_item_device.argtypes = [vp, C.c_int32, vp, i64, vp, i64, cp, i64, i64p, C.POINTER(C.c_int)]
    lib.sccg_mgpu_stash_device.argtypes = [vp, C.c_int32, vp, i64]
    lib.sccg_mgpu_gather.argtypes = [vp, vp, i64, i32p, i64p, i64p, C.c_int32, i32p, i64p]
    lib.sccg_mgpu_gather_device.argtypes = [vp, C.POINTER(vp), i32p, i64p, i64p, C.c_int32, i32p, i64p]
    lib.sccg_mgpu_compress_sharded.argtypes = [vp, cp, i64, cp, i64, cp, i64, vp, i64, i64p, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.sccg_mgpu_decompress_sharded.argtypes = [vp, cp, i64, cp, i64, vp, i64, i64p, i64p, i64p]
    _libs[key] = lib
    return lib


MGPU_ID_BYTES = 128


def mgpu_unique_id(lib_path: str | os.PathLike | None = None) -> bytes:
    """rendezvous token of a multi-GPU job (rank 0 calls this, everybody gets the bytes): sccg_mgpu_unique_id"""
    lib = load_library(lib_path)
    buf = C.create_string_buffer(MGPU_ID_BYTES)
    rc = lib.sccg_mgpu_unique_id(buf)
    if rc != SCCG_OK:
        raise SccgError(rc, lib.sccg_last_error().decode())
    return buf.raw


def mgpu_assign(lengths: list[int], world: int, lib_path: str | os.PathLike | None = None) -> list[int]:
    """LPT packing of pairs onto ranks (sccg_mgpu_assign) -> owner rank of every pair"""
    lib = load_library(lib_path)
    n = len(lengths)
    arr = (C.c_int64 * max(n, 1))(*lengths)
    own = (C.c_int32 * max(n, 1))()
    rc = lib.sccg_mgpu_assign(arr, n, world, own)
    if rc != SCCG_OK:
        raise SccgError(rc, lib.sccg_last_error().decode())
    return list(own[:n])


class Mgpu:
    """One rank of a multi-GPU job (sccg_mgpu, include/sccg.h): C++ host logic over NCCL."""

    def __init__(self, ctx: "Context", unique_id: bytes, rank: int, world: int):
        self.ctx, self.lib, self.rank, self.world = ctx, ctx.lib, rank, world
        h = C.c_void_p()
        rc = self.lib.sccg_mgpu_init(ctx.handle, unique_id, rank, world, C.byref(h))
        if rc != SCCG_OK:
            raise SccgError(rc, self.lib.sccg_last_error().decode())
        self.handle = h

    def close(self):
        if getattr(self, "handle", None):
            self.lib.sccg_mgpu_destroy(self.handle)
            self.handle = None

    def _check(self, rc: int):
        if rc != SCCG_OK:
            raise SccgError(rc, self.lib.sccg_last_error().decode())

    def compress_item(self, item: int, ref, tgt, header: bytes = b"") -> tuple[int, int]:
        """compress one pair of this rank (host buffers); its encoded image joins the outgoing streams -> (length, mode)"""
        n = C.c_int64(); mode = C.c_int()
        self._check(self.lib.sccg_mgpu_compress_item(self.handle, item, _as_char_p(ref), len(ref), _as_char_p(tgt), len(tgt), header, len(header),
                                                     C.byref(n), C.byref(mode)))
        return n.value, mode.value

    def compress_item_device(self, item: int, d_ref: int, ref_len: int, d_tgt: int, tgt_len: int, header: bytes = b"") -> tuple[int, int]:
        n = C.c_int64(); mode = C.c_int()
        self._check(self.lib.sccg_mgpu_compress_item_device(self.handle, item, d_ref, ref_len, d_tgt, tgt_len, header, len(header), C.byref(n), C.byref(mode)))
        return n.value, mode.value

    def gather(self, out_ptr: int = 0, out_cap: int = 0, max_items: int = 64 * 64, max_bytes: int = 1 << 26):
        """collective; rank 0 -> {item: (offset, length)} into the caller's buffer (out_ptr / out_cap), or {item: bytes} when no
        buffer is given; other ranks -> None"""
        ids = (C.c_int32 * max_items)(); offs = (C.c_int64 * max_items)(); lens = (C.c_int64 * max_items)()
        n = C.c_int32(); total = C.c_int64()
        own = None
        if self.rank == 0 and not out_ptr:
            out_cap = max_bytes
            own = C.create_string_buffer(out_cap)
            out_ptr = C.cast(own, C.c_void_p)
        rc = self.lib.sccg_mgpu_gather(self.handle, out_ptr, out_cap, ids, offs, lens, max_items, C.byref(n), C.byref(total))
        self._check(rc)
        if self.rank != 0:
            return None
        if own is not None:
            return {ids[k]: own.raw[offs[k]:offs[k] + lens[k]] for k in range(n.value)}
        return {ids[k]: (offs[k], lens[k]) for k in range(n.value)}

    def gather_device(self, max_items: int = 64 * 64):
        """collective; the gathered streams stay in rank 0's device memory -> rank 0: (device pointer, {item: (offset, length)}); others: None"""
        ids = (C.c_int32 * max_items)(); offs = (C.c_int64 * max_items)(); lens = (C.c_int64 * max_items)()
        n = C.c_int32(); total = C.c_int64(); d = C.c_void_p()
        self._check(self.lib.sccg_mgpu_gather_device(self.handle, C.byref(d), ids, offs, lens, max_items, C.byref(n), C.byref(total)))
        if self.rank != 0:
            return None
        return d.value or 0, {ids[k]: (offs[k], lens[k]) for k in range(n.value)}

    def compress_sharded(self, ref, tgt, header: bytes = b"", out_ptr: int = 0, out_cap: int = 0):
        """collective: one pair over all ranks by segment range -> rank 0: (image or its length, mode, sharded); others: (None, mode, sharded)"""
        n = C.c_int64(); mode = C.c_int(); sh = C.c_int()
        own = None
        if self.rank == 0 and not out_ptr:
            out_cap = len(tgt) * 2 + len(header) + 4096
            own = C.create_string_buffer(out_cap)
            out_ptr = C.cast(own, C.c_void_p)
        self._check(self.lib.sccg_mgpu_compress_sharded(self.handle, _as_char_p(ref), len(ref), _as_char_p(tgt), len(tgt), header, len(header),
                                                        out_ptr, out_cap, C.byref(n), C.byref(mode), C.byref(sh)))
        if self.rank != 0:
            return None, mode.value, bool(sh.value)
        return (own.raw[:n.value] if own is not None else n.value), mode.value, bool(sh.value)

    def decompress_sharded(self, ref_raw, intermediate: bytes, out_ptr: int, out_cap: int) -> tuple[int, int, int]:
        """this rank's piece of the reconstructed image -> (offset in the image, piece length, total length)"""
        off = C.c_int64(); n = C.c_int64(); total = C.c_int64()
        self._check(self.lib.sccg_mgpu_decompress_sharded(self.handle, _as_char_p(ref_raw), len(ref_raw), intermediate, len(intermediate),
                                                          out_ptr, out_cap, C.byref(off), C.byref(n), C.byref(total)))
        return off.value, n.value, total.value


class Archive:
    """An intermediate file opened on the device (sccg_archive_open, include/sccg.h): its decoder tables stay in device memory
    until close(), and Context.query extracts pieces of it.  Usable as a context manager."""

    def __init__(self, ctx: "Context", handle: int):
        self.ctx, self.handle = ctx, handle
        n = C.c_int64(); mode = C.c_int(); nbytes = C.c_int64()
        ctx._check(ctx.lib.sccg_archive_info(handle, C.byref(n), C.byref(mode), C.byref(nbytes)))
        self.seq_len, self.mode, self._device_bytes = n.value, mode.value, nbytes.value

    @property
    def device_bytes(self) -> int:
        """device memory the archive holds (sccg_archive_info): its tables, plus its lift table once a liftover call built it"""
        if self.handle:
            n = C.c_int64()
            self.ctx._check(self.ctx.lib.sccg_archive_info(self.handle, None, None, C.byref(n)))
            self._device_bytes = n.value
        return self._device_bytes

    def close(self):
        if self.handle:
            h, self.handle = self.handle, None
            self.ctx._archives.discard(self)
            if self.ctx.handle:
                self.ctx._check(self.ctx.lib.sccg_archive_close(self.ctx.handle, h))

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


class Context:
    """One sccg_ctx (one GPU).  Method names follow the reference's free functions."""

    def __init__(self, device: int = 0, lib_path: str | os.PathLike | None = None):
        self.lib = load_library(lib_path)
        self._archives: set[Archive] = set()
        self.ref_len = 0                            # len(R) of the resident reference (set_reference)
        self.handle = self.lib.sccg_create(device)
        if not self.handle:
            raise SccgError(SCCG_E_CUDA, self.lib.sccg_last_error().decode())

    def close(self):
        if getattr(self, "handle", None):
            for a in list(self._archives):          # sccg_destroy releases them
                a.handle = None
            self._archives.clear()
            self.lib.sccg_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc: int):
        if rc != SCCG_OK:
            raise SccgError(rc, self.lib.sccg_last_error().decode())

    def _take(self, ptr: C.c_void_p, n: int) -> bytes:
        data = C.string_at(ptr, n) if (ptr.value and n) else b""
        if ptr.value:
            self.lib.sccg_free(ptr)
        return data

    def version(self) -> str:
        return self.lib.sccg_version().decode()

    def profile(self) -> dict:
        p = Profile()
        self._check(self.lib.sccg_get_profile(self.handle, C.byref(p)))
        return p.as_dict()

    def download(self, d_ptr: int, n: int) -> bytes:
        """device buffer (as returned by *_device calls) -> host bytes"""
        buf = C.create_string_buffer(max(n, 1))
        self._check(self.lib.sccg_download(self.handle, d_ptr, n, buf))
        return buf.raw[:n]

    # compress_genome minus file I/O and 7z (compression.cpp:320-579)
    def compress(self, ref, tgt, header: bytes = b"") -> tuple[bytes, int]:
        """ref / tgt: bytes or C-contiguous uint8 numpy arrays (zero-copy)"""
        out = C.c_void_p(); n = C.c_int64(); mode = C.c_int()
        rc = self.lib.sccg_compress(self.handle, _as_char_p(ref), len(ref), _as_char_p(tgt), len(tgt), header, len(header), C.byref(out), C.byref(n), C.byref(mode))
        if rc == SCCG_E_STOI:
            raise SccgError(rc, self.lib.sccg_last_error().decode(), self._take(out, n.value))
        self._check(rc)
        return self._take(out, n.value), mode.value

    def compress_into(self, ref, tgt, header: bytes, out_ptr: int, out_cap: int) -> tuple[int, int]:
        """result written to the caller's (ideally page-locked) buffer -> (length, mode)"""
        n = C.c_int64(); mode = C.c_int()
        rc = self.lib.sccg_compress_into(self.handle, ref, len(ref), tgt, len(tgt), header, len(header), out_ptr, out_cap,
                                         C.byref(n), C.byref(mode))
        if rc == SCCG_E_STOI:                                   # the caller's buffer holds the pre-delta image (include/sccg.h)
            raise SccgError(rc, self.lib.sccg_last_error().decode(), C.string_at(out_ptr, n.value))
        self._check(rc)
        return n.value, mode.value

    def decompress_into(self, ref_raw, intermediate, out_ptr: int, out_cap: int) -> int:
        n = C.c_int64()
        self._check(self.lib.sccg_decompress_into(self.handle, ref_raw, len(ref_raw), intermediate, len(intermediate), out_ptr, out_cap, C.byref(n)))
        return n.value

    def compress_device(self, d_ref: int, ref_len: int, d_tgt: int, tgt_len: int, header: bytes = b"") -> tuple[int, int, int]:
        """device pointers in -> (device pointer of the encoded image, its length, mode)"""
        out = C.c_void_p(); n = C.c_int64(); mode = C.c_int()
        self._check(self.lib.sccg_compress_device(self.handle, d_ref, ref_len, d_tgt, tgt_len, header, len(header),
                                                  C.byref(out), C.byref(n), C.byref(mode)))
        return out.value or 0, n.value, mode.value

    # match_sequences (compression.cpp:36-179)
    def match_sequences(self, Sr: bytes, St: bytes, k: int, m: int, is_global: bool, offset: int = 0) -> list[Record]:
        recs = _Records()
        self._check(self.lib.sccg_match_sequences(self.handle, Sr, len(Sr), St, len(St), k, m, int(is_global), offset, C.byref(recs)))
        total = recs.lit_off[recs.n] if recs.n else 0
        lits = C.string_at(recs.lits, total) if total else b""
        out = [Record(recs.p[i], recs.l[i], lits[recs.lit_off[i]:recs.lit_off[i + 1]]) for i in range(recs.n)]
        self.lib.sccg_records_free(C.byref(recs))
        return out

    # reconstruct_genome (decompression.cpp:117-279)
    def reconstruct(self, ref: bytes, encoded: bytes, n_idx: bytes, low_idx: bytes) -> bytes:
        out = C.c_void_p(); n = C.c_int64()
        self._check(self.lib.sccg_reconstruct(self.handle, ref, len(ref), encoded, len(encoded), n_idx, len(n_idx),
                                              low_idx, len(low_idx), C.byref(out), C.byref(n)))
        return self._take(out, n.value)

    def reconstruct_device(self, d_ref: int, ref_len: int, d_enc: int, enc_len: int, d_n: int, n_len: int, d_low: int, low_len: int) -> tuple[int, int]:
        out = C.c_void_p(); n = C.c_int64()
        self._check(self.lib.sccg_reconstruct_device(self.handle, d_ref, ref_len, d_enc, enc_len, d_n, n_len, d_low, low_len,
                                                     C.byref(out), C.byref(n)))
        return out.value or 0, n.value

    def decompress_part(self, ref_raw, intermediate: bytes, part: int, n_parts: int, out_ptr: int = 0, out_cap: int = 0):
        """the part-th of n_parts pieces of the reconstructed file image -> (offset in the image, piece, total length);
        with out_ptr / out_cap the piece is written into the caller's (page-locked) buffer and its length is returned instead"""
        off = C.c_int64(); n = C.c_int64(); total = C.c_int64()
        if out_ptr:
            self._check(self.lib.sccg_decompress_part(self.handle, _as_char_p(ref_raw), len(ref_raw), intermediate, len(intermediate), part, n_parts,
                                                      out_ptr, out_cap, C.byref(off), C.byref(n), C.byref(total)))
            return off.value, n.value, total.value
        cap = len(ref_raw) * 2 + len(intermediate) * 2 + 4096            # generous: a piece is at most the whole image
        buf = C.create_string_buffer(cap)
        self._check(self.lib.sccg_decompress_part(self.handle, _as_char_p(ref_raw), len(ref_raw), intermediate, len(intermediate), part, n_parts,
                                                  C.cast(buf, C.c_void_p), cap, C.byref(off), C.byref(n), C.byref(total)))
        return off.value, buf.raw[:n.value], total.value

    # many targets against one reference: the reference stays in device memory (include/sccg.h)
    def set_reference(self, ref) -> None:
        """ref: bytes or a C-contiguous uint8 numpy array (raw symbols, as read_genomes_from_files yields them)"""
        self._check(self.lib.sccg_reference_set(self.handle, _as_char_p(ref), len(ref)))
        self.ref_len = len(ref)

    def clear_reference(self) -> None:
        self._check(self.lib.sccg_reference_clear(self.handle))
        self.ref_len = 0

    def compress_resident(self, tgt, header: bytes = b"", out_ptr: int = 0, out_cap: int = 0):
        """compress against the resident reference -> (file image, mode); with out_ptr / out_cap the image is written into
        the caller's (page-locked) buffer and (length, mode) is returned"""
        n = C.c_int64(); mode = C.c_int()
        if out_ptr:
            rc = self.lib.sccg_compress_resident_into(self.handle, _as_char_p(tgt), len(tgt), header, len(header), out_ptr, out_cap, C.byref(n), C.byref(mode))
            if rc == SCCG_E_STOI:
                raise SccgError(rc, self.lib.sccg_last_error().decode(), C.string_at(out_ptr, n.value))
            self._check(rc)
            return n.value, mode.value
        cap = 2 * len(tgt) + len(header) + 4096
        while True:
            buf = C.create_string_buffer(cap)
            rc = self.lib.sccg_compress_resident_into(self.handle, _as_char_p(tgt), len(tgt), header, len(header), C.cast(buf, C.c_void_p), cap, C.byref(n), C.byref(mode))
            if rc == SCCG_E_ARG and n.value > cap:              # too small: the required size came back
                cap = n.value
                continue
            if rc == SCCG_E_STOI:
                raise SccgError(rc, self.lib.sccg_last_error().decode(), buf.raw[:n.value])
            self._check(rc)
            return buf.raw[:n.value], mode.value

    def decompress_resident(self, intermediate: bytes, out_ptr: int = 0, out_cap: int = 0):
        """decompress against the resident reference -> file image (or its length with out_ptr / out_cap)"""
        n = C.c_int64()
        if out_ptr:
            self._check(self.lib.sccg_decompress_resident_into(self.handle, intermediate, len(intermediate), out_ptr, out_cap, C.byref(n)))
            return n.value
        cap = 4096
        while True:
            buf = C.create_string_buffer(cap)
            rc = self.lib.sccg_decompress_resident_into(self.handle, intermediate, len(intermediate), C.cast(buf, C.c_void_p), cap, C.byref(n))
            if rc == SCCG_E_ARG and n.value > cap:
                cap = n.value + 16
                continue
            self._check(rc)
            return buf.raw[:n.value]

    # one chromosome over several GPUs: segment-range shards (include/sccg.h, sharding.py)
    def shard_match(self, ref_slice, tgt_slice, seg_base: int, is_last: bool) -> dict:
        """ref_slice / tgt_slice: bytes, or C-contiguous uint8 numpy arrays (zero-copy; pin them for full PCIe speed)"""
        info = ShardInfo()
        self._check(self.lib.sccg_shard_match(self.handle, _as_char_p(ref_slice), len(ref_slice), _as_char_p(tgt_slice), len(tgt_slice),
                                              seg_base, int(is_last), C.byref(info)))
        return info.as_dict()

    def shard_write(self, carry: dict) -> tuple[bytes, bytes]:
        """-> (this shard's part of the lowercase-run line, its part of the body)"""
        cy = ShardCarry(**carry)
        low = C.c_void_p(); nl = C.c_int64(); body = C.c_void_p(); nb = C.c_int64()
        self._check(self.lib.sccg_shard_write(self.handle, C.byref(cy), C.byref(low), C.byref(nl), C.byref(body), C.byref(nb)))
        return self._take(low, nl.value), self._take(body, nb.value)

    # read_genomes_from_files on the device + compress_genome (compression.cpp:181-220, :320-579): raw FASTA file images in
    def compress_fasta(self, ref_file: bytes, tgt_file: bytes) -> tuple[bytes, int]:
        out = C.c_void_p(); n = C.c_int64(); mode = C.c_int()
        rc = self.lib.sccg_compress_fasta(self.handle, ref_file, len(ref_file), tgt_file, len(tgt_file), C.byref(out), C.byref(n), C.byref(mode))
        if rc == SCCG_E_STOI:
            raise SccgError(rc, self.lib.sccg_last_error().decode(), self._take(out, n.value))
        self._check(rc)
        return self._take(out, n.value), mode.value

    def decompress_fasta(self, ref_file: bytes, intermediate: bytes) -> bytes:
        out = C.c_void_p(); n = C.c_int64()
        self._check(self.lib.sccg_decompress_fasta(self.handle, ref_file, len(ref_file), intermediate, len(intermediate), C.byref(out), C.byref(n)))
        return self._take(out, n.value)

    def compress_fasta_into(self, ref_file, tgt_file, out_ptr: int, out_cap: int) -> tuple[int, int]:
        """FASTA file images in (ideally in page-locked memory), compressed_genome.txt image into the caller's buffer -> (length, mode)"""
        n = C.c_int64(); mode = C.c_int()
        self._check(self.lib.sccg_compress_fasta_into(self.handle, _as_char_p(ref_file), len(ref_file), _as_char_p(tgt_file), len(tgt_file), out_ptr, out_cap,
                                                      C.byref(n), C.byref(mode)))
        return n.value, mode.value

    def decompress_stream(self, ref, intermediate: bytes, fasta: bool = False) -> list[tuple[int, bytes]]:
        """streaming decompression (sccg_decompress_stream / sccg_decompress_fasta_stream) -> the pieces [(offset, bytes)] in the
        order the sink received them; ref: raw symbols, or the reference FASTA file image with fasta=True"""
        pieces = []

        def sink(user, off, data, n):
            pieces.append((off, C.string_at(data, n)))
            return 0
        cb = SINK_FN(sink)
        total = C.c_int64()
        fn = self.lib.sccg_decompress_fasta_stream if fasta else self.lib.sccg_decompress_stream
        self._check(fn(self.handle, _as_char_p(ref), len(ref), intermediate, len(intermediate), cb, None, C.byref(total)))
        assert sum(len(p) for _, p in pieces) == total.value
        return pieces

    # region extraction (include/sccg.h): D[start_0:end_0] + D[start_1:end_1] + ... of the decoded sequence D
    def _extract(self, call, regions, out_ptr: int, out_cap: int):
        import numpy as np
        reg = np.ascontiguousarray(np.asarray(regions, dtype=np.int64).reshape(-1, 2))     # sccg_region[] layout, no copy for int64 (n, 2)
        n = C.c_int64(-1); seq = C.c_int64(-1)
        rp = reg.ctypes.data if len(reg) else None

        def run(ptr, cap):
            rc = call(rp, len(reg), ptr, cap, C.byref(n), C.byref(seq))
            if rc != SCCG_OK:
                err = SccgError(rc, self.lib.sccg_last_error().decode())
                err.out_len, err.seq_len = n.value, seq.value      # required size / length of D, where the library set them
                raise err
            self.last_seq_len = seq.value
        if out_ptr:
            run(out_ptr, out_cap)
            return n.value
        lens = reg[:, 1] - reg[:, 0]
        cap = max(int(lens.sum()), 0) if len(reg) and bool((lens >= 0).all()) else 0
        buf = C.create_string_buffer(max(cap, 1))
        run(C.cast(buf, C.c_void_p), cap)
        return buf.raw[:n.value]

    def extract(self, ref_raw, intermediate: bytes, regions, out_ptr: int = 0, out_cap: int = 0):
        """regions: an (n, 2) int64 numpy array or a sequence of (start, end) pairs, 0-based half-open in the decoded sequence ->
        the concatenated pieces (bytes), or their total length when written into the caller's buffer (out_ptr / out_cap).
        The length of the decoded sequence is left in self.last_seq_len (and in SccgError.seq_len for a region past its end)."""
        return self._extract(lambda *t: self.lib.sccg_extract(self.handle, _as_char_p(ref_raw), len(ref_raw), intermediate, len(intermediate), *t),
                             regions, out_ptr, out_cap)

    def extract_fasta(self, ref_file, intermediate: bytes, regions, out_ptr: int = 0, out_cap: int = 0):
        """extract with the reference FASTA file image"""
        return self._extract(lambda *t: self.lib.sccg_extract_fasta(self.handle, _as_char_p(ref_file), len(ref_file), intermediate, len(intermediate), *t),
                             regions, out_ptr, out_cap)

    def extract_resident(self, intermediate: bytes, regions, out_ptr: int = 0, out_cap: int = 0):
        """extract against the resident reference (set_reference)"""
        return self._extract(lambda *t: self.lib.sccg_extract_resident(self.handle, intermediate, len(intermediate), *t), regions, out_ptr, out_cap)

    # archives (include/sccg.h): record files decoded once, then queried with pieces of any of them in one call
    def open_archive(self, intermediate: bytes) -> Archive:
        """open an intermediate file against the resident reference (set_reference)"""
        h = C.c_void_p()
        self._check(self.lib.sccg_archive_open(self.handle, intermediate, len(intermediate), C.byref(h)))
        a = Archive(self, h.value)
        self._archives.add(a)
        return a

    def query(self, archives, queries, out_ptr: int = 0, out_cap: int = 0):
        """archives: a sequence of Archive; queries: an (n, 4) int64 array (or a sequence of rows) of [archive index, start, end,
        strand], strand 1 being the reverse complement -> the concatenated pieces (bytes), or their total length when written
        into the caller's buffer (out_ptr / out_cap).  A too-small buffer raises SccgError with out_len = the required size."""
        import numpy as np
        q = np.ascontiguousarray(np.asarray(queries, dtype=np.int64).reshape(-1, 4))     # sccg_query[] layout
        arr = (C.c_void_p * max(len(archives), 1))(*[a.handle for a in archives])
        n = C.c_int64(-1)
        qp = q.ctypes.data if len(q) else None

        def run(ptr, cap):
            rc = self.lib.sccg_archive_extract(self.handle, arr if len(archives) else None, len(archives), qp, len(q), ptr, cap, C.byref(n))
            if rc != SCCG_OK:
                err = SccgError(rc, self.lib.sccg_last_error().decode())
                err.out_len = n.value
                raise err
        if out_ptr:
            run(out_ptr, out_cap)
            return n.value
        lens = q[:, 2] - q[:, 1]
        cap = max(int(lens.sum()), 0) if len(q) and bool((lens >= 0).all()) else 0
        buf = C.create_string_buffer(max(cap, 1))
        run(C.cast(buf, C.c_void_p), cap)
        return buf.raw[:n.value]

    _HIT = [("window", "<i8"), ("pos", "<i8"), ("pattern", "<i4"), ("strand", "<i4"), ("mismatches", "<i4"), ("reserved", "<i4")]
    _STRANDS = {"+": 1, "-": 2, "both": 3, 1: 1, 2: 2, 3: 3}

    def search(self, archives, patterns, windows=None, max_mismatches: int = 0, strands="both", count_only: bool = False):
        """every occurrence of the patterns (a sequence of bytes) with at most max_mismatches mismatches in windows of open
        archives (sccg_archive_search, include/sccg.h).  windows: an (n, 3) int64 array of [archive index, start, end], passed
        straight through; None searches the whole D of each archive, in order.  strands: "both", "+" or "-" (or 3, 1, 2).
        -> an (n, 5) int64 array of [window, pos, pattern, strand, mismatches] in (window, pos, pattern, strand) order, or the
        number of hits when count_only.  The hit buffer starts at 65,536 hits; a call that finds more runs once more with the
        exact count it reported."""
        import numpy as np
        if strands not in self._STRANDS:
            raise ValueError("strands must be 'both', '+' or '-'")
        if windows is None:
            windows = [(k, 0, a.seq_len) for k, a in enumerate(archives)]
        w = np.ascontiguousarray(np.asarray(windows, dtype=np.int64).reshape(-1, 3))      # sccg_window[] layout
        pats = [bytes(p) for p in patterns]
        off = np.zeros(len(pats) + 1, dtype=np.int64)
        off[1:] = np.cumsum([len(p) for p in pats]) if pats else []
        blob = b"".join(pats)
        arr = (C.c_void_p * max(len(archives), 1))(*[a.handle for a in archives])
        n = C.c_int64(-1)

        def run(out, cap):
            return self.lib.sccg_archive_search(self.handle, arr if len(archives) else None, len(archives), w.ctypes.data if len(w) else None,
                                                len(w), blob, off.ctypes.data if pats else None, len(pats), max_mismatches,
                                                self._STRANDS[strands], out, cap, C.byref(n))
        if count_only:
            self._check(run(None, 0))
            return n.value
        for cap in (65536, None):
            buf = np.zeros(n.value if cap is None else cap, dtype=self._HIT)
            rc = run(buf.ctypes.data if len(buf) else None, len(buf))
            if rc == SCCG_OK or not (cap is not None and rc == SCCG_E_ARG and n.value > cap):
                break
        self._check(rc)
        h = buf[:n.value]
        return np.stack([h["window"], h["pos"], h["pattern"].astype(np.int64), h["strand"].astype(np.int64),
                         h["mismatches"].astype(np.int64)], axis=1).reshape(-1, 5)

    _EDIT_HIT = [("window", "<i8"), ("start", "<i8"), ("end", "<i8"), ("pattern", "<i4"), ("strand", "<i4"), ("edits", "<i4"),
                 ("reserved", "<i4")]

    def search_edits(self, archives, patterns, windows=None, max_edits: int = 0, strands="both", count_only: bool = False):
        """every end of an alignment of the patterns within max_edits edits (substitutions, insertions, deletions) in windows of
        open archives (sccg_archive_search_edits, include/sccg.h); windows and strands as for search.  -> an (n, 6) int64 array
        of [window, start, end, pattern, strand, edits] in (window, end, pattern, strand) order, or the number of hits when
        count_only.  Hits are not clustered: every end within max_edits is reported.  Same buffer scheme as search."""
        import numpy as np
        if strands not in self._STRANDS:
            raise ValueError("strands must be 'both', '+' or '-'")
        if windows is None:
            windows = [(k, 0, a.seq_len) for k, a in enumerate(archives)]
        w = np.ascontiguousarray(np.asarray(windows, dtype=np.int64).reshape(-1, 3))      # sccg_window[] layout
        pats = [bytes(p) for p in patterns]
        off = np.zeros(len(pats) + 1, dtype=np.int64)
        off[1:] = np.cumsum([len(p) for p in pats]) if pats else []
        blob = b"".join(pats)
        arr = (C.c_void_p * max(len(archives), 1))(*[a.handle for a in archives])
        n = C.c_int64(-1)

        def run(out, cap):
            return self.lib.sccg_archive_search_edits(self.handle, arr if len(archives) else None, len(archives), w.ctypes.data if len(w) else None,
                                                      len(w), blob, off.ctypes.data if pats else None, len(pats), max_edits,
                                                      self._STRANDS[strands], out, cap, C.byref(n))
        if count_only:
            self._check(run(None, 0))
            return n.value
        for cap in (65536, None):
            buf = np.zeros(n.value if cap is None else cap, dtype=self._EDIT_HIT)
            rc = run(buf.ctypes.data if len(buf) else None, len(buf))
            if rc == SCCG_OK or not (cap is not None and rc == SCCG_E_ARG and n.value > cap):
                break
        self._check(rc)
        h = buf[:n.value]
        return np.stack([h["window"], h["start"], h["end"], h["pattern"].astype(np.int64), h["strand"].astype(np.int64),
                         h["edits"].astype(np.int64)], axis=1).reshape(-1, 6)

    _VARIANT = [("window", "<i8"), ("pos", "<i8"), ("end", "<i8"), ("d_start", "<i8"), ("d_end", "<i8"), ("alt_off", "<i8")]

    def variants(self, archives, windows=None, count_only: bool = False):
        """differences of open archives from the resident reference as normalised variant records (sccg_archive_variants,
        include/sccg.h).  windows: an (n, 3) int64 array of [archive index, start, end] in REFERENCE coordinates, passed
        straight through; None takes the whole reference for each archive, in order.  -> (records, alt): records an (n, 6)
        int64 array of [window, pos, end, d_start, d_end, alt_off] in (window, pos, d_start) order, alt the ALT bytes (record
        i's are alt[alt_off:alt_off + d_end - d_start]); or (number of records, ALT bytes) when count_only.  The buffers start
        at 65,536 records and 1 MiB; a call that needs more runs once more with the exact sizes it reported."""
        import numpy as np
        if windows is None:
            windows = [(k, 0, self.ref_len) for k in range(len(archives))]
        w = np.ascontiguousarray(np.asarray(windows, dtype=np.int64).reshape(-1, 3))      # sccg_window[] layout
        arr = (C.c_void_p * max(len(archives), 1))(*[a.handle for a in archives])
        n = C.c_int64(-1); na = C.c_int64(-1)

        def run(out, cap, alt, alt_cap):
            return self.lib.sccg_archive_variants(self.handle, arr if len(archives) else None, len(archives), w.ctypes.data if len(w) else None,
                                                  len(w), out, cap, C.byref(n), alt, alt_cap, C.byref(na))
        if count_only:
            self._check(run(None, 0, None, 0))
            return n.value, na.value
        caps = (65536, 1 << 20)
        for _ in range(2):
            buf = np.zeros(caps[0], dtype=self._VARIANT)
            alt = C.create_string_buffer(max(caps[1], 1))
            rc = run(buf.ctypes.data if len(buf) else None, len(buf), C.cast(alt, C.c_void_p), caps[1])
            if rc == SCCG_OK or not (rc == SCCG_E_ARG and (n.value > caps[0] or na.value > caps[1])):
                break
            caps = (n.value, na.value)
        self._check(rc)
        v = buf[:n.value]
        rec = np.stack([v[f] for f, _ in self._VARIANT], axis=1).reshape(-1, 6).astype(np.int64)
        return rec, alt.raw[:na.value]

    _LIFT_QUERY = [("archive", "<i8"), ("start", "<i8"), ("end", "<i8"), ("from", "<i4"), ("reserved", "<i4")]
    _LIFT = [("start", "<i8"), ("end", "<i8"), ("same", "<i8"), ("subst", "<i8"), ("records", "<i8"), ("flags", "<i4"), ("reserved", "<i4")]

    def liftover(self, archives, queries):
        """intervals lifted between the resident reference and open archives (sccg_archive_liftover, include/sccg.h).  queries:
        an (n, 4) int64 array of [archive index, start, end, from], from 0 for a reference interval lifted into the archive
        and 1 for an archive interval lifted onto the reference.  -> an (n, 6) int64 array of [start, end, same, subst,
        records, flags], one row per query in order.  The first call that names an archive builds its lift table."""
        import numpy as np
        q = np.asarray(queries, dtype=np.int64).reshape(-1, 4)
        t = np.zeros(len(q), dtype=self._LIFT_QUERY)                     # sccg_lift_query[] layout
        t["archive"], t["start"], t["end"] = q[:, 0], q[:, 1], q[:, 2]
        t["from"] = np.where((q[:, 3] < -2**31) | (q[:, 3] >= 2**31), -1, q[:, 3]).astype(np.int32)   # (out of range stays invalid)
        out = np.zeros(len(q), dtype=self._LIFT)
        arr = (C.c_void_p * max(len(archives), 1))(*[a.handle for a in archives])
        self._check(self.lib.sccg_archive_liftover(self.handle, arr if len(archives) else None, len(archives), t.ctypes.data if len(t) else None,
                                                   len(t), out.ctypes.data if len(out) else None))
        return np.stack([out[f].astype(np.int64) for f, _ in self._LIFT[:6]], axis=1).reshape(-1, 6)

    # decompress_genome (in-memory part) + reconstruct_genome + header line (decompression.cpp:66-110, :117-279, :322)
    def decompress(self, ref_raw: bytes, intermediate: bytes) -> bytes:
        out = C.c_void_p(); n = C.c_int64()
        self._check(self.lib.sccg_decompress(self.handle, ref_raw, len(ref_raw), intermediate, len(intermediate), C.byref(out), C.byref(n)))
        return self._take(out, n.value)
