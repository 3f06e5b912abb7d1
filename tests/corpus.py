"""Shared seeded test inputs (mirrors the data shapes of LZ4Test.java:456-541 and SURVEY.md §8d)."""
import os
import random

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))

# LZ4Test.java:350-419 — malformed blocks
MALFORMED = [
    bytes([16, 42, 0, 0, 128] + [42] * 8),                      # offset 0: must not throw / hang (:351-361)
    bytes([96, 42, 43, 44, 45, 46, 47, 5, 0]),                   # ends with a match: must throw (:363-388)
    bytes([96, 42, 43, 44, 45, 46, 47, 5, 0, 1]),
    bytes([96, 42, 43, 44, 45, 46, 47, 5, 0, 1, 2]),
    bytes([96, 42, 43, 44, 45, 46, 47, 5, 0, 1, 2, 3]),
    bytes([96, 42, 43, 44, 45, 46, 47, 5, 0, 1, 2, 3, 4]),
    # exactly the arrays LZ4Test.java:390-397 builds: the 9 bytes above + a token of i literals + i zero bytes, i = 1..4
    bytes([96, 42, 43, 44, 45, 46, 47, 5, 0, 1 << 4, 0]),
    bytes([96, 42, 43, 44, 45, 46, 47, 5, 0, 2 << 4, 0, 0]),
    bytes([96, 42, 43, 44, 45, 46, 47, 5, 0, 3 << 4, 0, 0, 0]),
    bytes([96, 42, 43, 44, 45, 46, 47, 5, 0, 4 << 4, 0, 0, 0, 0]),
]


def blocks(checker, big=True):
    """(name, bytes) pairs: edge sizes, data shapes and synthetic corpora."""
    rng = random.Random(1234)
    out = [("empty", b"")]
    for n in (1, 4, 5, 11, 12, 13, 14, 20, 31, 32, 33, 63, 64, 65, 66, 100, 255, 270, 1000, 4096):
        out.append((f"rand3_{n}", bytes(rng.randrange(3) for _ in range(n))))
        out.append((f"urandom_{n}", rng.randbytes(n)))
        out.append((f"equal_{n}", b"a" * n))
    for n in (20000, 65535, 65536):
        out.append((f"equal_{n}", b"\x00" * n))
        out.append((f"urandom_{n}", rng.randbytes(n)))
    # a match at distance exactly 65535 (LZ4Test.java:465-475)
    head = rng.randbytes(40)
    out.append(("dist65535", head + bytes(rng.randrange(1, 255) for _ in range(65535 - 40)) + head + b"tail-literals"))
    # small alphabets, periodic data with periods around the copy-path thresholds
    for period in (1, 2, 3, 4, 7, 8, 15, 16, 31, 32, 33, 100, 127, 128, 129, 300):
        unit = rng.randbytes(period)
        out.append((f"period_{period}", (unit * (3000 // period + 2))[:3000] + rng.randbytes(7)))
    for mp, seed in ((0.2, 1), (0.5, 2), (0.8, 3), (0.95, 4)):
        for n in (777, 65536) if big else (777,):
            out.append((f"rdg_p{mp}_{n}", checker.datagen(n, mp, 0.0, seed).tobytes()))
    return out


def calgary_blocks(limit=4):
    """64 KiB cuts of the Calgary files book1, geo and pic (the reference's src/test-resources/calgary, which LZ4Test.java
    round-trips): the first `limit` (at most 4) of each file; geo is 102400 bytes long, so it has two.  Stored under
    tests/golden: book1@0, geo@0, geo@65536 and pic@0 as the reference's own LZ4 streams in calgary_lz4.json (checked
    against their recorded digests here), the next three cuts of book1 and of pic in calgary_cuts.xz."""
    import base64
    import hashlib
    import json
    import lzma
    from oracle import oracle as O
    assert limit <= 4
    port = O.Port()
    cuts = {}
    for b in json.load(open(os.path.join(HERE, "golden", "calgary_lz4.json")))["blocks"]:
        r, d = port.decompress_safe(base64.b64decode(b["fast_b64"]), b["len"])
        assert r == b["len"] and hashlib.sha256(d).hexdigest() == b["sha256"], b["name"]
        cuts[b["name"]] = d
    extra = lzma.decompress(open(os.path.join(HERE, "golden", "calgary_cuts.xz"), "rb").read())
    for k, name in enumerate(CALGARY_XZ_CUTS):
        cuts[name] = extra[k * 65536:(k + 1) * 65536]
    out = []
    for f, size in (("book1", 768771), ("geo", 102400), ("pic", 513216)):
        for i in range(0, min(size, limit * 65536), 65536):
            out.append((f"{f}@{i}", cuts[f"{f}@{i}"]))
    return out


CALGARY_XZ_CUTS = [f"{f}@{k * 65536}" for f in ("book1", "pic") for k in (1, 2, 3)]     # tests/golden/calgary_cuts.xz, in order


def codec_variants(c: bytes, n: int, rng: random.Random):
    """(stream, capacity) pairs around a compressed block `c` of `n` bytes: capacities off by a little, a cut and an
    extended stream, and 25 mutations (tests/test_oracle_pin.py's differential against the reference's decoders)"""
    variants = [(c, n), (c, n - 1), (c, n + 1), (c, n + 64), (c, 0), (c[:-1], n), (c + b"\0", n)]
    variants += [(m, rng.choice([n, n + 1, n + 70, max(0, n - 5)])) for m in mutate(c, rng, 25)]
    return [(cc, cap) for cc, cap in variants if cc]


def compress_caps(c: bytes):
    """output capacities around the size of a compressed block `c`: the limitedOutput thresholds (lz4.c:1085-1088)"""
    return (len(c) - 1, len(c), len(c) + 3, len(c) // 2)


def frame_header_len(f: bytes) -> int:
    """bytes of an LZ4 frame's header: magic, FLG, BD, the optional content size and dictionary ID, HC"""
    return 7 + (8 if f[4] & 0x08 else 0) + (4 if f[4] & 0x01 else 0)


class ReferenceFrames:
    """LZ4F_compressFrame's frames (the reference's writer) for the inputs the tests use, rebuilt without the reference:
    its frames differ from the restated writer's only in the header (it shrinks the block size ID to the input and
    writes no content size of 0), so each is the reference's recorded header in front of the restated writer's blocks,
    checked against the recorded digest of the reference's whole frame (tests/golden/ref_outputs.json)."""
    kind = "reference"

    def __init__(self, port, table):
        self.port, self.table = port, table

    def frame_compress(self, data, bs_code=7, flags=1) -> bytes:
        import hashlib
        e = self.table[f"{len(data)}/{bs_code}/{flags}"]
        f = self.port.frame_compress(data, bs_code, flags)
        g = bytes.fromhex(e["head"]) + f[frame_header_len(f):]
        assert hashlib.sha256(g).hexdigest() == e["sha256"], (len(data), bs_code, flags)
        return g


def mutate(c: bytes, rng: random.Random, k: int):
    """k corrupted variants of a compressed block (bit flips, byte sets, cuts, splices)."""
    outs = []
    for _ in range(k):
        b = bytearray(c)
        if not b:
            break
        for _ in range(rng.randrange(1, 4)):
            i = rng.randrange(len(b))
            m = rng.randrange(4)
            if m == 0:
                b[i] = rng.randrange(256)
            elif m == 1:
                b[i] ^= 1 << rng.randrange(8)
            elif m == 2:
                b[i] = 0xFF
            else:
                b[i] = 0
        outs.append(bytes(b))
    return outs


def pack(items, align=1, pad=0):
    """Concatenate byte strings into one uint8 array; returns (array, offsets u64, lengths i32)."""
    offs, lens, pos = [], [], 0
    for it in items:
        pos = (pos + align - 1) // align * align
        offs.append(pos)
        lens.append(len(it))
        pos += len(it) + pad
    buf = np.zeros(max(pos, 1) + 64, dtype=np.uint8)
    for o, it in zip(offs, items):
        buf[o:o + len(it)] = np.frombuffer(it, dtype=np.uint8)
    return buf, np.array(offs, dtype=np.uint64), np.array(lens, dtype=np.int32)


# ---- fixtures and data recipes of the reference's own tests
def issue12():
    """the regression input of https://github.com/jpountz/lz4-java/issues/12 as LZ4Test.java:488-539 uses it: bytes [9:] of
    the array literal (committed under tests/golden/issue12.json, extracted once from the reference's test source)"""
    import json
    raw = bytes.fromhex(json.load(open(os.path.join(HERE, "golden", "issue12.json")))["hex"])
    return raw[9:]


class JavaRandom:
    """java.util.Random (the 48-bit LCG of the Java SE specification), enough of it to rebuild the test data of
    LZ4FrameIOStreamTest.java: nextInt() and nextBytes()"""

    def __init__(self, seed: int):
        self.s = (seed ^ 0x5DEECE66D) & ((1 << 48) - 1)

    def next(self, bits: int) -> int:
        self.s = (self.s * 0x5DEECE66D + 0xB) & ((1 << 48) - 1)
        v = self.s >> (48 - bits)
        return v - (1 << bits) if v >= (1 << (bits - 1)) else v        # signed, like Java's int

    def next_int(self) -> int:
        return self.next(32)

    def next_bytes(self, n: int) -> bytes:
        out = bytearray()
        while len(out) < n:
            rnd = self.next_int() & 0xFFFFFFFF
            for _ in range(min(n - len(out), 4)):
                out.append(rnd & 0xFF); rnd >>= 8
        return bytes(out)


def frame_test_sizes():
    """LZ4FrameIOStreamTest.java:73-90: the fixed sizes + ten drawn from Random(78370789134L)"""
    sizes = [0, 1, 1 << 10, (1 << 10) + 1, 1 << 16, 1 << 17, 1 << 20]
    rnd = JavaRandom(78370789134)
    for _ in range(10):
        v = rnd.next_int()
        sizes.append(abs(v) % (1 << 22))                                 # Math.abs(rnd.nextInt()) % (1 << 22)
    return sizes


def frame_test_data(size: int) -> bytes:
    """LZ4FrameIOStreamTest.java:100-119: 1 KiB buffers of Random(5378L).nextBytes whose whole 32-bit words are then
    overwritten with 0xDEADBEEF (little-endian) — so only a final partial word keeps random bytes"""
    rnd = JavaRandom(5378)
    out = bytearray()
    remaining = size
    while remaining > 0:
        n = min(remaining, 1 << 10)
        buf = bytearray(rnd.next_bytes(n))
        for w in range(n // 4):
            buf[4 * w:4 * w + 4] = b"\xEF\xBE\xAD\xDE"
        out += buf
        remaining -= n
    return bytes(out)
