"""Record-body tokens outside the canonical "(d,l)" text: checks shared by test_emu_token_grammar.py (CPU, SIMT emulator
build) and test_gpu_token_grammar.py (B200).

The reference reads a body token with find / substr / std::stoi (decompression.cpp:210-236, restated by orc_reconstruct): the
token ends at the first ')' after its '(', the delta is stoi from the byte after the '(' and the length is stoi from the byte
after the first ',' after the '('.  stoi skips leading isspace, takes one '+' or '-', any number of leading zeros, and stops
at the first non-digit.  The oracle's verdict is the expected value throughout, and every check asserts one invariant:
  - the library never returns bytes that differ from the oracle's;
  - it returns an error where the oracle decodes only for a body that holds a pinned class (INTEGRATION.md section 5), and
    then the error is SCCG_E_FORMAT;
  - where the oracle fails, the library fails too."""
import ctypes as C
import random
import re

import oracle_lib as ol
import sccg_b200
from cases import rnd
from test_emu_extract import PATHS, env, mixed_regions, seq_of

TOK_MAX = 25                    # csrc/sccg_decode.cuh: a token's ')' may lie at most TOK_MAX bytes after its '('
WS = [b" ", b"\t", b"\v", b"\f", b"\r"]     # the isspace bytes stoi skips ('\n' ends the body line of a file)
PINNED = ("negative_length", "long_token", "no_comma")


def py_stoi(s: bytes):
    """std::stoi on s -> int, or None where it throws"""
    m = re.match(rb"[ \t\n\v\f\r]*([+-]?)([0-9]+)", s)
    if not m:
        return None
    v = int(m.group(2)) * (-1 if m.group(1) == b"-" else 1)
    return v if -2 ** 31 <= v < 2 ** 31 else None


def pinned_class(body: bytes):
    """the pinned class of the first body token that falls in one, walking the body as the reference does; None if there
    is none (or the walk reaches a token without ')', on which the reference fails)"""
    i, n = 0, len(body)
    while i < n:
        if body[i] != ord("("):
            i += 1
            continue
        close = body.find(b")", i)
        if close < 0:
            return None
        comma = body.find(b",", i)
        if comma < 0 or comma > close:
            return "no_comma"            # the reference reads the length from a later ',' or from the body's first byte
        if close - i > TOK_MAX:
            return "long_token"          # beyond the look-back that decides a 16-byte chunk's entry state
        length = py_stoi(body[comma + 1:close])
        if length is not None and length < 0:
            return "negative_length"     # substr wraps it to "the rest of the reference" there
        i = close + 1
    return None


def first_difference(got: bytes, exp: bytes) -> str:
    k = next((i for i in range(min(len(got), len(exp))) if got[i] != exp[i]), min(len(got), len(exp)))
    return f"first difference at byte {k} (lengths {len(got)} / {len(exp)}): got {got[k:k + 24]!r}, expected {exp[k:k + 24]!r}"


def verdict(rc_o: int, exp: bytes, body: bytes, run, what: str):
    """run() against the oracle's verdict (rc_o, exp) on a stream whose record body is `body`"""
    pin = pinned_class(body)
    try:
        got = run()
    except sccg_b200.SccgError as e:
        if rc_o == 0:
            assert pin in PINNED, f"{what}: the oracle decodes {body[:80]!r} but the library failed: {e}"
            assert e.code == sccg_b200.SCCG_E_FORMAT, f"{what}: pinned class {pin} must be SCCG_E_FORMAT, got {e}"
        return None
    assert rc_o == 0, f"{what}: the oracle fails (rc {rc_o}) on {body[:80]!r}, the library returned bytes"
    assert pin is None, f"{what}: {body[:80]!r} holds a token of the pinned class {pin}, which must fail with SCCG_E_FORMAT"
    assert got == exp, f"{what} on {body[:80]!r}: " + first_difference(got, exp)
    return got


def check_reconstruct(ctx, ref, body, nlist=b"", low=b"", what="reconstruct"):
    rc_o, exp = ol.orc_reconstruct(ref, body, nlist, low)
    verdict(rc_o, exp, body, lambda: ctx.reconstruct(ref, body, nlist, low), what)
    return rc_o


# ------------------------------------------------------------------------------------------------ the deterministic table
TABLE_REF = rnd(500, "token grammar")

REPORTED = [b"AC(+5,3)GT", b"AC( 5,3)GT", b"AC(\t5,3)GT", b"AC(5, 3)GT", b"AC(5,+3)GT", b"AC(5 ,3)GT", b"AC(5,3 )GT",
            b"AC(5x,3)GT", b"AC(5,3x)GT", b"AC(00000000005,3)GT", b"AC(5,3)(+0,2)", b"(" + b" " * 4 + b"5,3)",
            b"(" + b" " * 20 + b"5,3)", b"(-0,3)", b"AC)GT(5,3)", b"AC,12-3)GT(5,3)"]


def number_forms(v: int, second: bool):
    """text forms of the number v that stoi reads as v (and a few it does not), with what may follow it inside a token"""
    s = b"%d" % v
    sign, digits = (b"-", s[1:]) if v < 0 else (b"", s)
    out = [s]
    out += [w + s for w in WS] + [b"  " + s, b" \t" + s]
    if v >= 0:
        out += [b"+" + s, b" +" + s]
    out += [sign + b"0" * k + digits for k in range(1, 13)]
    out += [s + w for w in WS]
    out += [s + b"x", s + b"-", s + b"+", s + b".5", s + b"A"]
    if second:
        out += [s + b",3", s + b",", s + b",,", s + b"(", s + b"(x"]
    return out


def token_table():
    """(body) rows: reported divergences, isspace / sign / leading zeros / trailing bytes on each number, the int limits,
    empty and broken numbers, tokens without ')' or ','"""
    rows = list(REPORTED)
    pre, post = b"(100,2)AC", b"GT(7,4)T"               # prev_abs_start 100: negative deltas stay inside the reference
    for d in (5, -5, 0):
        for f in number_forms(d, False):
            rows.append(pre + b"(" + f + b",3)" + post)
    for ln in (3, 0):
        for f in number_forms(ln, True):
            rows.append(pre + b"(5," + f + b")" + post)
    for d, ln in ((b"+0", b"3"), (b"-0", b"3"), (b"5", b"+0"), (b"5", b"-0"), (b"-0", b"-0"), (b"+0", b"+0")):
        rows.append(pre + b"(" + d + b"," + ln + b")" + post)
    limits = [b"2147483647", b"-2147483648", b"2147483648", b"-2147483649", b" 2147483647", b"+2147483647", b"0002147483647",
              b"-0002147483648", b"2147483647 ", b"\t-2147483648", b"+2147483648", b"00000000000000000002147483647"]
    # a length near INT_MAX at a position > 0 overflows `absolute_start + length` in int (:223), undefined behaviour in the
    # reference: the length limits go on tokens at position 0
    for x in limits:
        rows += [pre + b"(" + x + b",3)" + post, b"(" + x + b",3)", b"(0," + x + b")"]
    rows += [b"(10,5)(2147483647,1)", b"(2147483647,0)", b"(-2147483648,0)"]
    rows += [b"AC(,3)GT", b"AC(5,)GT", b"AC( ,3)GT", b"AC(+,3)GT", b"AC(- 5,3)GT", b"AC((5,3)GT", b"AC(5,(3)GT", b"AC(+-5,3)GT",
             b"AC(--5,3)GT", b"AC(5,--3)GT", b"AC(\n5,3)GT", b"AC(,)GT", b"AC()GT(5,3)", b"AC(5,3,)GT", b"AC(5,,3)GT"]
    rows += [b"AC(5,3", b"AC(5,", b"AC(", b"AC( 5", b"AC(+5,3 ", b"(7,2)AC(5,3", b"(7,2)(", b"(7,2)(5"]
    rows += [b"AC(5)GT,3)", b"AC(5)GT", b"12AC(5)GT", b"AC(5)GT(7,2)", b"7(5)", b"(5)", b"(5)(7,2)", b"3,(5)GT",
             b"AC(5)GT,+3)", b"AC(5)GT, 3x", b"AC(5,3)(9)TT,2)"]
    rows += [b"AC(5,-3)GT", b"AC(5, -3)GT", b"AC(5,-03)GT", b"AC(5,-3x)GT"]
    return rows


def check_table(ctx):
    decoded = 0
    for body in token_table():
        decoded += check_reconstruct(ctx, TABLE_REF, body, what="table") == 0
    assert decoded > 150                                    # most rows are input the reference decodes


# ------------------------------------------------------------------------------------------------ phases and lengths
NONCANON = [b"(+5,3)", b"( 5,3)", b"(\t5,3)", b"(5, 3)", b"(5,+3)", b"(5 ,3)", b"(5,3 )", b"(5x,3)", b"(5,3x)",
            b"(00000000005,3)", b"(5,2,3)", b"(+0005,\v3\f)", b"(5)", b"(5,-3)", b"(5,3", b"(-0,3)", b"(5,(3)"]
PADS = [lambda k: b"(" + b" " * k + b"5,3)", lambda k: b"(" + b"0" * k + b"5,3)", lambda k: b"(5," + b" " * k + b"3)",
        lambda k: b"(5," + b"0" * k + b"3)", lambda k: b"(5,3" + b" " * k + b")", lambda k: b"(5" + b" " * k + b",3)",
        lambda k: b"(5,3" + b"x" * k + b")"]
BLOCK = 4096                     # DEC_T * 16 bytes of record stream per CTA of dec_count_k / dec_emit_k


def placements(tok_len: int):
    """offsets of a token's '(' in the body: every phase of a 16-byte chunk (near the start, where the look-back is short,
    and with a full 32-byte look-back), and every offset at which the token crosses the 4,096-byte block border"""
    out = list(range(16)) + [32 + p for p in range(16)]
    out += range(BLOCK - tok_len - 1, BLOCK + 2)
    return out


def sweep_bodies():
    tail = b"ACG(7,4)" + rnd(20, "sweep tail") + b"(-3,5)"
    rows = []
    for tok in NONCANON:
        for at in placements(len(tok)):
            rows.append(rnd(at, ("sweep", at)) + tok + tail)
            if at >= 8:                                     # a canonical token right before: its ')' is in the look-back
                rows.append(rnd(at - 6, ("sweep", at)) + b"(40,1)" + tok + tail)
    for pad in PADS:
        for total in range(TOK_MAX - 3, TOK_MAX + 5):
            tok = pad(total - 5)
            assert len(tok) == total
            for at in placements(total):
                rows.append(rnd(at, ("pad", at)) + tok + tail)
    return rows


def check_sweep(ctx):
    long_refused = 0
    for body in sweep_bodies():
        check_reconstruct(ctx, TABLE_REF, body, what="sweep")
        long_refused += pinned_class(body) == "long_token"
    assert long_refused > 0


# ------------------------------------------------------------------------------------------------ seeded fuzzer
TOKEN = re.compile(rb"\((-?[0-9]+),(-?[0-9]+)\)")


def perturb(r: random.Random, s: bytes, second: bool) -> bytes:
    """another text of the number s that stoi reads as the same value"""
    sign, digits = (b"-", s[1:]) if s.startswith(b"-") else (b"", s)
    kind = r.randrange(5)
    if kind == 0:
        return b"".join(r.choice(WS) for _ in range(r.randint(1, 3))) + s
    if kind == 1:
        return (b"+" + s) if not sign else (r.choice(WS) + s)
    if kind == 2:
        return sign + b"0" * r.randint(1, 4) + digits
    if kind == 3:
        tails = [b" ", b"\t", b"\r", b"x", b"-", b"+", b"A", b"N"] + ([b",3", b",", b"("] if second else [])
        return s + r.choice(tails)
    return r.choice(WS) + (b"+" if not sign else b"") + s + b" "


def fuzz_body(r: random.Random, body: bytes, share: float = 0.2, long_tokens: int = 0) -> bytes:
    """rewrites a `share` of the canonical tokens of body, numbers kept; tokens stay within the look-back unless long_tokens
    of them are padded past it"""
    out, last = bytearray(), 0
    for m in TOKEN.finditer(body):
        out += body[last:m.start()]
        last = m.end()
        if r.random() >= share:
            out += m.group(0)
            continue
        d, ln = m.group(1), m.group(2)
        for _ in range(8):
            dd = perturb(r, d, False) if r.random() < 0.7 else d
            ll = perturb(r, ln, True) if r.random() < 0.7 else ln
            tok = b"(" + dd + b"," + ll + b")"
            if len(tok) <= TOK_MAX + 1:
                break
        else:
            tok = m.group(0)
        if long_tokens and r.random() < 0.05:
            tok = b"(" + b" " * (TOK_MAX + 3 - len(tok)) + tok[1:]       # TOK_MAX + 3 characters
            long_tokens -= 1
        out += tok
    out += body[last:]
    return bytes(out)


def compressed_streams(seed: int):
    """(prepared reference, body, N list, lowercase list) of orc_compress on a small local-mode pair with lowercase runs and
    on a small global-mode pair with N runs and lowercase runs"""
    from sccg_genome_compression_b200 import synth
    r = random.Random(repr(("streams", seed)))
    out = []
    for kind in ("local", "gap"):
        if kind == "local":
            ref, tgt = synth.local_pair(20_000 + 1000 * seed, synth.seed_for(2, 900 + seed))
        else:
            ref, tgt = synth.global_gap_pair(16_000 + 1000 * seed, 14_000, synth.seed_for(1, 900 + seed))
        t = bytearray(tgt.tobytes())
        for _ in range(6):
            a = r.randrange(len(t) - 200)
            n = r.randint(1, 150)
            t[a:a + n] = bytes(t[a:a + n]).lower()
            b = r.randrange(len(t) - 200)
            n = r.randint(1, 120)
            t[b:b + n] = b"N" * n
        ref = ref.tobytes()
        rc, inter, mode = ol.orc_compress(ref, bytes(t), b">fuzz")
        assert rc == 0
        header, low, nline, body = ol.split_intermediate(inter)
        out.append((ol.prepare_reference(ref, nline), body, b"" if nline == b"," else nline, low))
    return out


def fuzz_corpus(seeds):
    """canonical streams (orc_compress of synth pairs, test_emu_decode.make_record_stream) with a fifth of their tokens
    rewritten; every seventh stream also carries one token padded past the look-back"""
    from test_emu_decode import make_record_stream
    out = []
    for seed in seeds:
        streams = compressed_streams(seed) + [make_record_stream(1000 + seed)]
        for k, (ref, body, nlist, low) in enumerate(streams):
            r = random.Random(repr(("fuzz", seed, k)))
            out.append((ref, fuzz_body(r, body, 0.2, long_tokens=1 if (seed + k) % 7 == 0 else 0), nlist, low))
    return out


def check_fuzz(ctx, seeds):
    decoded = 0
    for ref, body, nlist, low in fuzz_corpus(seeds):
        decoded += check_reconstruct(ctx, ref, body, nlist, low, what="fuzz") == 0 and pinned_class(body) is None
    assert decoded >= len(seeds)                             # the corpus is not all errors


# ------------------------------------------------------------------------------------------------ every entry point
def entry_corpus():
    """a subset: reported bodies, a few padded tokens, a few fuzzed streams with N and lowercase run lists"""
    rows = [(TABLE_REF, b + b"TT(100,30)", b"", b"") for b in REPORTED]
    rows += [(TABLE_REF, b"(3,4)" + PADS[k % len(PADS)](TOK_MAX - 4 + k) + b"GG(50,20)", b"", b"") for k in range(5)]
    rows += [(TABLE_REF, b"(3,4)AC(5)GT,3)(20,9)", b"", b""), (TABLE_REF, b"(3,4)AC(5,-3)GT", b"", b"")]
    rows += fuzz_corpus([3])
    return rows


def check_entry_points(ctx, ref, body, nlist=b"", low=b"", parts=3):
    """reconstruct, decompress (default and pipelined in 4 KiB chunks with poisoned reference chunks), decompress_stream,
    decompress_part pieces, extract on every gather path, open_archive + query on both strands"""
    from test_emu_archive import both_strands
    from test_emu_archive import expect as query_expect
    check_reconstruct(ctx, ref, body, nlist, low)
    inter = b">tokens\n" + low + b"\n" + (nlist if nlist else b",") + b"\n" + body
    rc_o, image = ol.orc_decompress(ref, inter)
    v = lambda run, what, exp=image: verdict(rc_o, exp, body, run, what)
    v(lambda: ctx.decompress(ref, inter), "decompress")
    with env(SCCG_PIPE_CHUNK=4096, SCCG_PIPE_POISON=1):
        v(lambda: ctx.decompress(ref, inter), "decompress, 4 KiB chunks")
    v(lambda: b"".join(p for _, p in ctx.decompress_stream(ref, inter)), "decompress_stream")

    def by_parts():
        cap = len(image) + len(inter) + 4096                 # a piece is at most the whole image
        buf = C.create_string_buffer(cap)
        img, covered = None, 0
        for p in range(parts):
            off, n, total = ctx.decompress_part(ref, inter, p, parts, C.cast(buf, C.c_void_p).value, cap)
            img = img if img is not None else bytearray(total)
            img[off:off + n] = buf.raw[:n]
            covered += n
        assert covered == len(img)
        return bytes(img)
    v(by_parts, "decompress_part")
    D = seq_of(image) if rc_o == 0 else b""
    regs = mixed_regions(len(D), ("tok", body[:40])) if D else [(0, 0)]
    for path in PATHS:
        with env(SCCG_EXT_LANE_MIN=PATHS[path]):
            v(lambda: ctx.extract(ref, inter, regs), f"extract ({path})", b"".join(D[a:b] for a, b in regs))
    ctx.set_reference(ref)
    try:
        try:
            resident = ctx.decompress_resident(inter)
        except sccg_b200.SccgError as e1:
            try:
                ctx.open_archive(inter).close()
            except sccg_b200.SccgError as e2:
                assert e2.code == e1.code
            else:
                raise AssertionError(f"open_archive succeeded where decompress_resident failed ({e1}) on {body[:80]!r}")
            v(lambda: ctx.decompress_resident(inter), "decompress_resident")
            return
        assert verdict(rc_o, image, body, lambda: resident, "decompress_resident") == image
        with ctx.open_archive(inter) as a:
            assert a.seq_len == len(D)
            qs = both_strands(0, regs, ("tokq", body[:40])) if D else [(0, 0, 0, 0), (0, 0, 0, 1)]
            assert ctx.query([a], qs) == query_expect([D], qs)
    finally:
        ctx.clear_reference()


def check_entry_corpus(ctx):
    for ref, body, nlist, low in entry_corpus():
        check_entry_points(ctx, ref, body, nlist, low)


# ------------------------------------------------------------------------------------------------ our own round trip
ROUNDTRIP_PIECES = [b"(5, 3)", b"(5,+3)", b"(1,2,3)", b"(5,3x)", b"(5,\t3)"]


def piece_pair(piece: bytes, make_global: bool, n: int = 9000):
    """a near-identical pair whose target carries `piece` three times (global mode: after a 5 kb insertion)"""
    r = random.Random(repr(("piece", piece, make_global)))
    ref = rnd(n, ("pieceref", piece))
    t = bytearray(ref)
    for p in r.sample(range(n), n // 700):
        t[p] = r.choice(b"ACGT")
    if make_global:
        t[n // 4:n // 4] = rnd(5200, ("pieceins", piece))
    for at in (1000, n // 2, len(t) - 700):
        t[at:at + len(piece)] = piece
    return ref, bytes(t)


def roundtrip_pairs():
    from test_emu_compress import grammar_pair
    out = [(f"grammar_pair({s}, make_global={g})", *grammar_pair(s, make_global=g)) for s in range(24) for g in (False, True)]
    out += [(f"{p!r} {'global' if g else 'local'}", *piece_pair(p, g)) for p in ROUNDTRIP_PIECES for g in (False, True)]
    return out


def check_roundtrip(ctx, name, ref, tgt, header=b">round (trip) 1,2"):
    """ctx.decompress(ctx.compress(...)) equals orc_decompress of the same file, or fails where it fails -> oracle rc or None
    when the reference's compress throws already"""
    rc_c, inter_o, mode_o = ol.orc_compress(ref, tgt, header)
    if rc_c != 0:
        try:
            ctx.compress(ref, tgt, header)
        except sccg_b200.SccgError as e:
            assert e.code == sccg_b200.SCCG_E_STOI, name
            return None
        raise AssertionError(f"{name}: the reference's compress throws, the library's did not")
    inter, mode = ctx.compress(ref, tgt, header)
    assert (mode, inter) == (mode_o, inter_o), name
    rc_o, image = ol.orc_decompress(ref, inter)
    verdict(rc_o, image, ol.split_intermediate(inter)[3], lambda: ctx.decompress(ref, inter), f"round trip {name}")
    return rc_o


def check_roundtrips(ctx):
    decoded = {}
    for name, ref, tgt in roundtrip_pairs():
        decoded[name] = check_roundtrip(ctx, name, ref, tgt)
    for p in ROUNDTRIP_PIECES:                              # the reference decodes every one of these files
        for mode in ("local", "global"):
            assert decoded[f"{p!r} {mode}"] == 0, (p, mode)
    assert decoded["grammar_pair(10, make_global=True)"] == 0
