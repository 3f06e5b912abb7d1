"""Pins the CPU oracle (oracle/*.c restatements) to the reference: against the committed golden
vectors produced by the reference's own C (tests/golden/kat.json and ref_outputs.json).  CPU only."""
import hashlib
import json
import os
import random

import numpy as np
import pytest

import corpus

KAT = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "kat.json")))


def sha(b):
    return hashlib.sha256(bytes(b)).hexdigest()


def test_golden_datagen(port):
    for e in KAT["datagen"]:
        assert sha(port.datagen(e["size"], e["match_proba"], 0.0, e["seed"])) == e["sha256"], e


def test_golden_xxhash(port):
    stream = port.datagen(200000, 0.5, 0.0, 77).tobytes()
    for e in KAT["xxh"]:
        buf = stream[: e["len"]]
        assert port.xxh32(buf, e["seed"]) == e["xxh32"], e
        assert port.xxh64(buf, e["seed"] * 0x100000001) == e["xxh64"], e
    # python-xxhash (libxxhash 0.8) as an independent second witness
    xx = pytest.importorskip("xxhash")
    for n in (0, 5, 17, 4096, 100001):
        assert port.xxh32(stream[:n], 7) == xx.xxh32_intdigest(stream[:n], 7)
        assert port.xxh64(stream[:n], 7) == xx.xxh64_intdigest(stream[:n], 7)


def test_golden_xxhash_streaming(port):
    rng = random.Random(3)
    stream = port.datagen(200000, 0.5, 0.0, 77).tobytes()
    for e in KAT["xxh"][::3]:
        buf = stream[: e["len"]]
        cuts = sorted(rng.randint(0, len(buf)) for _ in range(4))
        chunks = [buf[a:b] for a, b in zip([0] + cuts, cuts + [len(buf)])]
        assert port.xxh_stream(32, chunks, e["seed"]) == e["xxh32"]
        assert port.xxh_stream(64, chunks, e["seed"] * 0x100000001) == e["xxh64"]


def test_golden_compress_bytes_and_roundtrip(port):
    """the restated compressor reproduces the reference's exact bytes (so ratio comparisons are
    against the reference's own parse), and both restated decoders invert it"""
    by_name = {e["name"]: e for e in KAT["compress"]}
    for name, d in corpus.blocks(port):
        e = by_name[name]
        assert sha(d) == e["in_sha256"], name
        c = port.compress(d)
        assert len(c) == e["clen"] and sha(c) == e["c_sha256"], name
        r, out = port.decompress_safe(c, len(d))
        assert r == len(d) and out == d, name
        r, out = port.decompress_fast(c, len(d))
        assert r == len(c) and out == d, name


def test_golden_malformed_codes(port):
    for e in KAT["malformed_safe"]:
        assert port.decompress_safe(bytes.fromhex(e["hex"]), e["cap"])[0] == e["ret"], e
    for e in KAT["malformed_fast"]:
        assert port.decompress_fast(bytes.fromhex(e["hex"]), e["n"])[0] == e["ret"], e


def test_compress_bound(port):
    assert port.compress_bound(65536) == 65809 and port.compress_bound(0) == 16
    assert port.compress_bound(0x7E000000) == 0x7E000000 + 0x7E000000 // 255 + 16
    assert port.compress_bound(0x7E000001) == 0 and port.compress_bound(-1) == 0


# ------------------------------------------------------------------ differential against the reference's recorded outputs
REF = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "ref_outputs.json")))


def test_ref_differential_codec(port):
    """the restated codec against what the reference's LZ4_compress_default / LZ4_decompress_safe / LZ4_decompress_fast
    returned for the same blocks, capacities and corrupted streams (tests/golden/ref_outputs.json)"""
    assert REF["lz4_version"] == KAT["lz4_version"]
    rng = random.Random(2)
    items = corpus.blocks(port, big=False) + corpus.calgary_blocks(2)
    assert [name for name, _ in items] == [e["name"] for e in REF["codec"]]
    bad = 0
    for (name, d), e in zip(items, REF["codec"]):
        c = port.compress(d)
        assert sha(c) == e["c_sha256"], name
        for cap, want in zip(corpus.compress_caps(c), e["caps"]):
            got = port.compress(d, cap)
            assert (None if got is None else sha(got)) == want, (name, cap)     # limitedOutput thresholds
        safe, fast, decoded = [], [], hashlib.sha256()
        for cc, cap in corpus.codec_variants(c, len(d), rng):
            r, out = port.decompress_safe(cc, cap)
            safe.append(r); decoded.update(out)
            if cap >= 0:
                r, out = port.decompress_fast(cc, cap)
                fast.append(r)
                if r >= 0:
                    decoded.update(out)
        bad += (safe != e["safe"]) + (fast != e["fast"]) + (decoded.hexdigest() != e["decoded_sha256"])
    assert bad == 0


def test_ref_differential_frames(port):
    """frames written by the restatement decode with the reference's LZ4F_decompress (its recorded verdict on these exact
    bytes) and the reference's LZ4F_compressFrame frames (corpus.ReferenceFrames) decode with the restatement"""
    frames = REF["frames"]
    ref = corpus.ReferenceFrames(port, frames)
    for n in (0, 1, 100, 65536, 65537, 300000, 5 << 20):
        data = port.datagen(n, 0.5, 0.0, n & 0xFF).tobytes()
        for bs in (4, 7):
            for flags in (0, 1, 3, 5, 7):
                e = frames[f"{n}/{bs}/{flags}"]
                f = port.frame_compress(data, bs, flags)
                assert sha(f) == e["port_sha256"] and e["ref_decodes"] == [n, sha(data)], (n, bs, flags)
                g = ref.frame_compress(data, bs, flags)
                r, out = port.frame_decompress(g, n + 16)
                assert r == n and out == data, (n, bs, flags, r)
    # concatenated + skippable frames (LZ4FrameIOStreamTest.java:253-309, 378-426)
    a, b = b"hello frame " * 1000, port.datagen(70000, 0.5, 0.0, 1).tobytes()
    skip = bytes([0x50, 0x2A, 0x4D, 0x18, 4, 0, 0, 0, 1, 2, 3, 4])
    cat = port.frame_compress(a, 4, 1) + skip + ref.frame_compress(b, 5, 1)
    r, out = port.frame_decompress(cat, len(a) + len(b))
    assert r == len(a) + len(b) and out == a + b
    bad = bytearray(port.frame_compress(b, 4, 1)); bad[-1] ^= 1          # content checksum mismatch
    assert port.frame_decompress(bytes(bad), len(b))[0] == -7


def test_container_restatements_roundtrip(port):
    """LZ4Block container and length-prefixed blocks: the restatements invert themselves and reject corruption"""
    rng = random.Random(8)
    for n in (0, 1, 63, 64, 1000, 65536, 65537, 300000):
        data = port.datagen(n, 0.5, 0.0, 3).tobytes()
        for bs in (64, 4096, 65536, 1 << 20):
            blob = port.lz4block_compress(data, bs)
            assert blob[:8] == b"LZ4Block" and blob[-21:-13] == b"LZ4Block"
            r, out = port.lz4block_decompress(blob, n)
            assert r == n and out == data, (n, bs)
            r, out = port.lz4block_decompress(blob + blob, 2 * n, False)       # concatenated streams (LZ4BlockStreamingTest.java:309-348)
            assert r == 2 * n and out == data + data
            r, out = port.lz4block_decompress(blob + b"trailing bytes", n)     # stopOnEmptyBlock (the default): the rest is not read
            assert r == n and out == data
            assert port.lz4block_decompress(blob[:-21], n)[0] == -1            # no end block: "Stream ended prematurely" (:192-198)
            assert port.lz4block_decompress(blob[:-21] + b"LZ4", n, False) == (n, data)   # ... quiet end when not stopping (:193-194)
        wl = port.with_length_compress(data)
        assert int.from_bytes(wl[:4], "little") == n
        r, out = port.with_length_decompress(wl, n)
        assert r == len(wl) and out == data
    noise = rng.randbytes(5000)
    blob = port.lz4block_compress(noise, 4096)
    assert blob[8] & 0xF0 == 0x10                                               # incompressible -> RAW method
    bad = bytearray(port.lz4block_compress(port.datagen(5000, 0.5, 0.0, 1).tobytes(), 4096)); bad[40] ^= 0x55
    assert port.lz4block_decompress(bytes(bad), 5000)[0] == -2
    assert port.lz4block_decompress(blob[:30], 5000)[0] == -1


def test_golden_calgary_streams(port):
    """real data: the reference's own fast and HC-9 streams of Calgary cuts (tests/golden/calgary_lz4.json) decode
    under the restated decoders to bytes with the recorded digest, and the restated fast compressor reproduces the
    reference's stream byte for byte"""
    import base64
    cal = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "calgary_lz4.json")))
    assert cal["lz4_version"] == 10904 and len(cal["blocks"]) == 6
    for b in cal["blocks"]:
        fast, hc = base64.b64decode(b["fast_b64"]), base64.b64decode(b["hc9_b64"])
        r, d = port.decompress_safe(fast, b["len"])
        assert r == b["len"] and sha(d) == b["sha256"], b["name"]
        r2, d2 = port.decompress_safe(hc, b["len"])
        assert r2 == b["len"] and d2 == d, b["name"]
        rf, df = port.decompress_fast(hc, b["len"])
        assert rf == len(hc) and df == d, b["name"]
        assert port.compress(d) == fast, b["name"]


def test_java_port_restatement_cross_checks(port):
    """SURVEY.md 8(a) C3/D3: the pure-Java backend restated (oracle/lz4_java_port_oracle.c; unpinned — no JVM here) is
    tied to the pinned C restatement the way LZ4Test.java:305-324 ties the backends to each other: every compressor's
    stream under every decompressor.  Also the vectors LZ4Test.java:350-419 expects EVERY backend to reject."""
    import base64
    items = corpus.blocks(port)
    cal = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "calgary_lz4.json")))["blocks"]
    items += [(b["name"], port.decompress_safe(base64.b64decode(b["fast_b64"]), b["len"])[1]) for b in cal]
    sizes_c = sizes_j = 0
    for name, d in items:
        d = bytes(d)
        cj = port.java_compress(d)
        assert cj is not None and len(cj) <= port.compress_bound(len(d)), name
        cc = port.compress(d)
        sizes_c += len(cc); sizes_j += len(cj)
        for c in (cj, cc):
            assert port.decompress_safe(c, len(d)) == (len(d), d), name                        # C decoders read both
            assert port.decompress_fast(c + bytes(16), len(d)) == (len(c), d), name
            assert port.java_decompress_safe(c, len(d)) == (len(d), d), name                   # Java decoders read both
            assert port.java_decompress_safe(c, len(d) + 50) == (len(d), d), name
            assert port.java_decompress_fast(c + bytes(16), len(d)) == (len(c), d), name
        if len(d) > 20:
            assert port.java_decompress_safe(cj, len(d) - 1)[0] < 0, name                      # LZ4Test.java:240-252
            assert port.java_decompress_fast(cj + bytes(16), len(d) - 1)[0] < 0 or len(d) < 14, name
        assert port.java_compress(d, max(0, len(cj) - 1)) is None or len(d) == 0, name        # maxDestLen is too small
    assert 0.9 < sizes_j / sizes_c < 1.1            # same family of parse: sizes within a few percent of each other
    # LZ4Test.java:350-361: offset 0 must neither throw nor hang, in any backend
    v0 = corpus.MALFORMED[0]
    assert port.java_decompress_safe(v0, 20)[0] == 13 and port.decompress_safe(v0, 20)[0] == 13
    assert port.java_decompress_fast(v0, 13)[0] == 13 and port.decompress_fast(v0 + bytes(8), 13)[0] == 13
    # LZ4Test.java:363-419: ending with a match / with fewer than 5 literals must throw, in every backend
    for v in corpus.MALFORMED[1:]:
        assert port.java_decompress_safe(v, 20)[0] < 0 and port.decompress_safe(v, 20)[0] < 0, v.hex()
        for n in (10, 20):
            assert port.java_decompress_fast(v, n)[0] < 0 and port.decompress_fast(v + bytes(32), n)[0] < 0, (v.hex(), n)


def test_reference_test_fixtures_on_the_checkers(port):
    """the reference's own fixed inputs: the issue-#12 regression array (LZ4Test.java:488-539) through both restated
    compressors and all restated decoders, and the frame test data of LZ4FrameIOStreamTest.java:73-119 (sizes from
    Random(78370789134L), bytes from Random(5378L) overwritten with 0xDEADBEEF words) through the frame container"""
    d = corpus.issue12()
    assert len(d) == 1510
    for c in (port.compress(d), port.java_compress(d)):
        assert port.decompress_safe(c, len(d)) == (len(d), d) and port.java_decompress_safe(c, len(d)) == (len(d), d)
        assert port.decompress_fast(c + bytes(8), len(d)) == (len(c), d)
    sizes = corpus.frame_test_sizes()
    assert sizes[:7] == [0, 1, 1 << 10, (1 << 10) + 1, 1 << 16, 1 << 17, 1 << 20] and len(sizes) == 17 and all(0 <= s < (1 << 22) for s in sizes)
    assert corpus.JavaRandom(42).next_int() == -1170105035                   # java.util.Random's documented sequence
    for n in sizes[:8]:
        data = corpus.frame_test_data(n)
        assert len(data) == n and data[:n // 4 * 4] == b"\xEF\xBE\xAD\xDE" * (n // 4)
        for flags in (0, 1, 7):
            assert port.frame_decompress(port.frame_compress(data, 4, flags), n + 8) == (n, data)
