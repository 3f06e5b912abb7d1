"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on the same seeded
inputs.  Decompression and hashes must be bit-exact (including negative return codes of the safe
decoder); compression must emit a valid LZ4 block that the oracle decodes back to the input."""
import os
import random

import numpy as np
import pytest

import corpus

pytestmark = pytest.mark.gpu


def _slots(lens, extra=0, align=16):
    caps = [int(x) + extra for x in lens]
    offs, pos = [], 0
    for c in caps:
        offs.append(pos)
        pos += (c + align - 1) // align * align + align
    return np.array(offs, dtype=np.uint64), np.array(caps, dtype=np.int32), pos + 64


@pytest.fixture
def decoder():
    """The library launches the batched decoders (decode_batch() in front of the sequential code); the sequential-only
    instantiation is exercised on the CPU emulator (tests/test_kernel_logic_cpu.py)."""
    return "batched"


def test_decompress_safe_exact(b200, checker, decoder):
    items = corpus.blocks(checker) + corpus.calgary_blocks()
    comp = [checker.compress(d) for _, d in items]
    src, soff, slen = corpus.pack(comp)
    doff, dcap, total = _slots([len(d) for _, d in items])
    dst = np.full(total, 0xAA, dtype=np.uint8)
    res = b200.batch.decompress_safe_batch_host(src, soff, slen, dst, doff, dcap)
    for k, (name, d) in enumerate(items):
        assert res[k] == len(d), (name, res[k], len(d))
        assert dst[int(doff[k]):int(doff[k]) + len(d)].tobytes() == d, name
        # nothing written past the slot capacity
        assert (dst[int(doff[k]) + len(d):int(doff[k]) + len(d) + 16] == 0xAA).all(), name


def test_decompress_fast_exact(b200, checker, decoder):
    items = corpus.blocks(checker) + corpus.calgary_blocks()
    comp = [checker.compress(d) for _, d in items]
    src, soff, slen = corpus.pack(comp)
    doff, dlen, total = _slots([len(d) for _, d in items])
    dst = np.full(total, 0xAA, dtype=np.uint8)
    res = b200.batch.decompress_fast_batch_host(src, soff, slen, dst, doff, dlen)
    for k, (name, d) in enumerate(items):
        assert res[k] == len(comp[k]), (name, res[k], len(comp[k]))       # bytes READ (LZ4Test.java:185)
        assert dst[int(doff[k]):int(doff[k]) + len(d)].tobytes() == d, name
        assert (dst[int(doff[k]) + len(d):int(doff[k]) + len(d) + 16] == 0xAA).all(), name


def test_decompress_safe_malformed_codes(b200, checker, decoder):
    """Same accept/reject set AND same negative codes as the reference (lz4.c:2337)."""
    rng = random.Random(99)
    cases = []                                           # (compressed bytes, capacity)
    for name, d in corpus.blocks(checker, big=False):
        c = checker.compress(d)
        n = len(d)
        for cap in (n, n - 1, n + 1, n + 7, n + 64, n + 100, max(0, n - 13), 0, n // 2):
            cases.append((c, cap))
        for cut in (1, 2, 3, 5, 8, 13):
            if len(c) > cut:
                cases.append((c[:-cut], n))
        cases.append((c + b"\0", n))
        cases.append((c + b"\x10\x41", n))
        for m in corpus.mutate(c, rng, 12):
            cases.append((m, rng.choice([n, n, n + 1, n - 1, n + 70, max(0, n - 5)])))
    for v in corpus.MALFORMED:
        for cap in (20, 64, 100, 200):
            cases.append((v, cap))
    cases = [(c, cap) for c, cap in cases if len(c) > 0]
    src, soff, slen = corpus.pack([c for c, _ in cases], pad=8)
    doff, dcap, total = _slots([cap for _, cap in cases])
    dst = np.zeros(total, dtype=np.uint8)
    res = b200.batch.decompress_safe_batch_host(src, soff, slen, dst, doff, dcap)
    negatives = 0
    for k, (c, cap) in enumerate(cases):
        want, out = checker.decompress_safe(c, cap)
        assert res[k] == want, (k, len(c), cap, int(res[k]), want, c[:24].hex())
        if want >= 0:
            assert dst[int(doff[k]):int(doff[k]) + want].tobytes() == out, k
        else:
            negatives += 1
    assert negatives > 100


def test_decompress_fast_malformed(b200, checker, decoder):
    rng = random.Random(7)
    cases = []
    for name, d in corpus.blocks(checker, big=False):
        c = checker.compress(d)
        n = len(d)
        for dl in (n, n - 1, n + 1, n + 5, max(0, n - 12)):          # LZ4Test.java:209-226
            if dl >= 0:          # a negative size is rejected in Java before the native call (SafeUtils.java:24-42)
                cases.append((c, dl))     # and is undefined behaviour inside the reference's unsafe decoder
        for m in corpus.mutate(c, rng, 6):
            cases.append((m, n))
    for v in corpus.MALFORMED:
        cases.append((v, 20))
    cases = [(c, dl) for c, dl in cases if len(c) > 0]
    # give every stream generous zero padding so the reference's unbounded reads stay defined
    padded = [c + bytes(dl + dl // 255 + 64) for c, dl in cases]
    src, soff, slen = corpus.pack(padded)
    doff, dlen, total = _slots([dl for _, dl in cases])
    dst = np.zeros(total, dtype=np.uint8)
    res = b200.batch.decompress_fast_batch_host(src, soff, slen, dst, doff, dlen)
    for k, (c, dl) in enumerate(cases):
        want, out = checker.decompress_fast(c, dl)
        assert res[k] == want, (k, len(c), dl, int(res[k]), want)
        if want >= 0:
            assert dst[int(doff[k]):int(doff[k]) + dl].tobytes() == out, k


def test_decompress_dependency_patterns(b200, checker, decoder):
    """Streams built to stress the batched decoder's match rounds: runs (offset 1), short periods, matches
    whose source is the previous sequence's output, long literal runs and long matches, all mixed."""
    rng = random.Random(4242)
    items = []
    for trial in range(24):
        parts = []
        while sum(map(len, parts)) < 30000 + 4000 * trial:
            kind = rng.randrange(7)
            if kind == 0:
                parts.append(bytes([rng.randrange(256)]) * rng.randrange(5, 700))                      # run
            elif kind == 1:
                pat = bytes(rng.randrange(256) for _ in range(rng.randrange(2, 9)))
                parts.append(pat * rng.randrange(3, 120))                                              # short period
            elif kind == 2:
                parts.append(bytes(rng.randrange(256) for _ in range(rng.randrange(1, 80))))           # literals
            elif kind == 3 and parts:
                prev = b"".join(parts[-3:])
                a = rng.randrange(len(prev)); parts.append(prev[a:a + rng.randrange(4, 60)])           # near copy
            elif kind == 4 and parts:
                whole = b"".join(parts)
                a = rng.randrange(len(whole)); parts.append(whole[a:a + rng.randrange(4, 400)])        # far copy
            elif kind == 5:
                pat = bytes(rng.randrange(256) for _ in range(rng.randrange(33, 200)))
                parts.append(pat * rng.randrange(2, 6))                                                # period >= 32
            else:
                parts.append(bytes(rng.randrange(4) for _ in range(rng.randrange(20, 300))))           # low entropy
        items.append(b"".join(parts))
    comp = [checker.compress(d) for d in items]
    src, soff, slen = corpus.pack(comp)
    doff, dcap, total = _slots([len(d) for d in items], extra=3)
    for fast in (False, True):
        dst = np.full(total, 0x55, dtype=np.uint8)
        if fast:
            lens = np.array([len(d) for d in items], dtype=np.int32)
            res = b200.batch.decompress_fast_batch_host(src, soff, slen, dst, doff, lens)
        else:
            res = b200.batch.decompress_safe_batch_host(src, soff, slen, dst, doff, dcap)
        for k, d in enumerate(items):
            assert res[k] == (len(comp[k]) if fast else len(d)), (decoder, fast, k, int(res[k]))
            assert dst[int(doff[k]):int(doff[k]) + len(d)].tobytes() == d, (decoder, fast, k)
            # bytes between the decoded length and the slot capacity are unspecified (as with the reference's wild
            # copies); nothing may be written past the capacity
            end = int(doff[k]) + (len(d) if fast else int(dcap[k]))
            assert (dst[end:end + 13] == 0x55).all(), (decoder, fast, k)


def test_decompress_long_sequence_then_short_ones_near_the_end(b200, checker, decoder):
    """Regression: a long match followed by many short sequences close to the end of the block — the batched decoder
    must count the long one against the output margin too (it once skipped the per-sequence check when the margin
    looked roomy at the start of a batch, accepted sequences inside the margin and walked past the end of the
    stream).  The fast decoder is given far more readable input than the stream holds, and what follows the stream
    looks like more LZ4 sequences (another block's stream) — what a caller with bound-sized slots that were used
    before hands over."""
    rng = random.Random(8080)
    items = []
    for trial in range(48):
        hist = bytes(rng.randrange(256) for _ in range(3000))
        parts = [hist]

        def short():                                                             # 1-6 literals + 5-12 byte match
            parts.append(bytes(rng.randrange(256) for _ in range(rng.randrange(1, 7))))
            a = rng.randrange(0, 2900); parts.append(hist[a:a + rng.randrange(5, 13)])
        for _ in range(rng.randrange(40, 90)): short()
        a = rng.randrange(0, 500)
        parts.append(bytes(rng.randrange(256) for _ in range(2))); parts.append(hist[a:a + rng.randrange(900, 2400)])   # the long one
        for _ in range(rng.randrange(30, 90)): short()
        parts.append(bytes(rng.randrange(256) for _ in range(rng.randrange(5, 40))))
        items.append(b"".join(parts))
    items.append(bytes(70000))                                                   # 640 bytes of input = most of the block
    items.append(bytes([7]) * 40000 + bytes(rng.randrange(256) for _ in range(300)) + bytes([9]) * 3000)
    comp = [checker.compress(d) for d in items]
    lens = np.array([len(d) for d in items], dtype=np.int32)
    src, soff, slen = corpus.pack(comp)
    doff, dcap, total = _slots([len(d) for d in items], align=64)
    dst = np.full(total + 4096, 0x55, dtype=np.uint8)
    res = b200.batch.decompress_safe_batch_host(src, soff, slen, dst, doff, dcap)
    for k, d in enumerate(items):
        assert res[k] == len(d) and dst[int(doff[k]):int(doff[k]) + len(d)].tobytes() == d, (decoder, "safe", k)
        assert (dst[int(doff[k]) + len(d):int(doff[k]) + len(d) + 16] == 0x55).all(), (decoder, "safe", k)
    padded = [c + comp[(k + 1) % len(comp)][9:3000] + bytes(64) for k, c in enumerate(comp)]
    src, soff, slen = corpus.pack(padded)
    dst = np.full(total + 4096, 0x55, dtype=np.uint8)
    res = b200.batch.decompress_fast_batch_host(src, soff, slen, dst, doff, lens)
    for k, d in enumerate(items):
        assert res[k] == len(comp[k]) and dst[int(doff[k]):int(doff[k]) + len(d)].tobytes() == d, (decoder, "fast", k)
        assert (dst[int(doff[k]) + len(d):int(doff[k]) + len(d) + 16] == 0x55).all(), (decoder, "fast", k)


@pytest.mark.parametrize("table", ["u16", "u32"])
def test_compress_roundtrip_through_oracle(b200, checker, table):
    """u16: blocks <= 64 KiB (three-warp kernel, 8192 x u16 table, lz4.c:1353); u32: any size (one warp, 4096 x u32, lz4.c:1356)"""
    items = corpus.blocks(checker) + corpus.calgary_blocks()
    if table == "u16":                      # 16-bit position table: caller promises blocks <= 64 KiB
        items = [(nm, d) for nm, d in items if len(d) <= 65536]
    _compress_roundtrip(b200, checker, items, 65536 if table == "u16" else 0, slack=1.10)


def test_compress_streams_against_the_pinned_ones(b200, checker):
    """tests/golden/fast_streams.json holds what the kernel source emits on the CPU emulator for the seeded corpus.  Two
    positions of one 128-position sub-round that hash alike store to the same table slot and "any winner is a valid
    position": WHICH one wins is the hardware's store arbitration (the emulator's differs), so on inputs with many equal
    4-byte sequences the GPU's parse may differ in a few sequences.  Pinned here: every stream is valid, its size is at most
    the emulator's + 5 % + 8 bytes, at least half of the streams are byte-identical, and two runs on the GPU agree."""
    import hashlib, json, os
    gold = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fast_streams.json")))["streams"]
    items = [(nm, d) for nm, d in corpus.blocks(checker) if nm in gold]
    assert len(items) == len(gold)
    src, soff, slen = corpus.pack([d for _, d in items], align=4)
    bounds = [b200.max_compressed_length(len(d)) for _, d in items]
    doff, dcap, total = _slots(bounds)
    runs = []
    for _ in range(2):
        dst = np.zeros(total + 64, dtype=np.uint8)
        res = b200.batch.compress_fast_batch_host(src, soff, slen, dst, doff, dcap, max_src_len=65536)
        runs.append((res.copy(), dst))
    assert (runs[0][0] == runs[1][0]).all() and (runs[0][1] == runs[1][1]).all(), "two GPU runs differ"
    res, dst = runs[0]
    same = 0
    for k, (nm, d) in enumerate(items):
        c = dst[int(doff[k]):int(doff[k]) + int(res[k])].tobytes()
        assert checker.decompress_safe(c, len(d)) == (len(d), d), nm
        assert int(res[k]) <= gold[nm]["c"] + gold[nm]["c"] // 20 + 8, (nm, int(res[k]), gold[nm]["c"])      # (often smaller: 17 % on RDG P=0.95)
        same += hashlib.sha256(c).hexdigest() == gold[nm]["sha256"]
    assert same >= len(items) // 2, same


def _compress_roundtrip(b200, checker, items, max_src_len, slack):
    src, soff, slen = corpus.pack([d for _, d in items])
    bounds = [b200.max_compressed_length(len(d)) for _, d in items]
    doff, dcap, total = _slots(bounds)
    dst = np.full(total, 0x55, dtype=np.uint8)
    res = b200.batch.compress_fast_batch_host(src, soff, slen, dst, doff, dcap, max_src_len=max_src_len)
    tot_c = tot_ref = 0
    for k, (name, d) in enumerate(items):
        assert 0 < res[k] <= bounds[k], (name, res[k])
        c = dst[int(doff[k]):int(doff[k]) + int(res[k])].tobytes()
        r, out = checker.decompress_safe(c, len(d))
        assert r == len(d) and out == d, (name, r, len(d))
        r2, out2 = checker.decompress_fast(c, len(d))
        assert r2 == len(c) and out2 == d, name
        assert dst[int(doff[k]) + bounds[k]] == 0x55, name           # nothing written past the slot
        tot_c += len(c)
        tot_ref += len(checker.compress(d))
    # same ballpark as the reference's ratio on this mixed corpus
    assert tot_c < slack * tot_ref, (tot_c, tot_ref)


def test_compress_large_blocks_u32_table(b200, checker):
    """blocks > 64 KiB use the 32-bit position table (lz4.c:1356 analogue)"""
    datas = [checker.datagen(n, 0.5, 0.0, 11).tobytes() for n in (65547, 100000, 262144, 1 << 20)]
    datas.append(b"\0" * 300000)
    src, soff, slen = corpus.pack(datas)
    bounds = [b200.max_compressed_length(len(d)) for d in datas]
    doff, dcap, total = _slots(bounds)
    dst = np.zeros(total, dtype=np.uint8)
    res = b200.batch.compress_fast_batch_host(src, soff, slen, dst, doff, dcap, max_src_len=0)
    for k, d in enumerate(datas):
        c = dst[int(doff[k]):int(doff[k]) + int(res[k])].tobytes()
        r, out = checker.decompress_safe(c, len(d))
        assert r == len(d) and out == d, k
        assert len(c) < 1.1 * len(checker.compress(d)) + 64


def test_compress_limited_output(b200, checker):
    """dst too small: 0 (-> LZ4Exception) or a valid smaller stream (LZ4Test.java:188-203)"""
    d = checker.datagen(20000, 0.5, 0.0, 5).tobytes()
    full = b200.LZ4Factory.b200Instance().fastCompressor().compress(d)
    for cap in (len(full) - 1, len(full) // 2, 10, 1, 0):
        out = bytearray(max(cap, 1))
        try:
            n = b200.LZ4Factory.b200Instance().fastCompressor().compress(d, 0, len(d), out, 0, cap)
        except b200.LZ4Exception:
            continue
        assert n <= cap
        r, o = checker.decompress_safe(bytes(out[:n]), len(d))
        assert o == d


def test_self_roundtrip_gpu_only(b200, checker):
    """compress on GPU -> decompress on GPU (both decoders), no CPU in the loop except the compare"""
    items = [(nm, d) for nm, d in corpus.blocks(checker) if len(d) <= 65536]
    src, soff, slen = corpus.pack([d for _, d in items])
    bounds = [b200.max_compressed_length(len(d)) for _, d in items]
    coff, ccap, ctotal = _slots(bounds)
    comp = np.zeros(ctotal, dtype=np.uint8)
    clen = b200.batch.compress_fast_batch_host(src, soff, slen, comp, coff, ccap, max_src_len=65536)
    doff, dcap, total = _slots(slen)
    out = np.zeros(total, dtype=np.uint8)
    r = b200.batch.decompress_safe_batch_host(comp, coff, clen, out, doff, dcap)
    assert (r == slen).all()
    out2 = np.zeros(total, dtype=np.uint8)
    r2 = b200.batch.decompress_fast_batch_host(comp, coff, ccap, out2, doff, slen)
    assert (r2 == clen).all()
    for k, (name, d) in enumerate(items):
        assert out[int(doff[k]):int(doff[k]) + len(d)].tobytes() == d, name
        assert out2[int(doff[k]):int(doff[k]) + len(d)].tobytes() == d, name


def test_compact_host(b200, checker):
    datas = [checker.datagen(65536, 0.5, 0.0, s).tobytes() for s in range(40)] + [b"", b"x", b"\0" * 5000]
    src, soff, slen = corpus.pack(datas)
    dst = np.zeros(sum(b200.max_compressed_length(len(d)) for d in datas) + 64, dtype=np.uint8)
    ooff, olen, total = b200.batch.compress_fast_compact_host(src, soff, slen, dst, max_src_len=65536)
    assert total == int(olen.sum())
    pos = 0
    for k, d in enumerate(datas):
        assert int(ooff[k]) == pos
        c = dst[pos:pos + int(olen[k])].tobytes()
        r, out = checker.decompress_safe(c, len(d))
        assert r == len(d) and out == d
        pos += int(olen[k])


def test_failed_pipeline_call_leaves_nothing_in_flight(b200):
    """A host-buffer call that fails after some chunks were queued (here: `dst_capacity too small for the packed stream`,
    found when the FIRST chunk retires while the next two are in flight) must drain them: the next call on the same
    thread would otherwise retire the stale chunks into its own result / offset arrays.  Three chunks are needed: chunks
    hold at most 65 536 blocks (tiny blocks reach that on a GPU), or B200LZ4_CHUNK_MB bytes (the emulator slice of
    the CPU suite sets it to 1 and uses 4 KiB blocks, since every emulated CTA costs milliseconds)."""
    chunk_mb = int(os.environ.get("B200LZ4_CHUNK_MB", "256"))
    if chunk_mb <= 4:
        bl = 4096; per_chunk = (chunk_mb << 20) // bl
    else:
        bl = 20; per_chunk = 65536
    n = 2 * per_chunk + 100
    cl = bl + 1 + (0 if bl < 15 else (bl - 15) // 255 + 1)                # random bytes: one literals-only sequence
    hdr = cl - bl
    rng = np.random.default_rng(77)
    src = rng.integers(0, 256, n * bl, dtype=np.uint8)
    soff, slen = b200.batch.uniform_layout(n, bl)
    small = np.zeros(1000, dtype=np.uint8)
    with pytest.raises(b200.B200Error, match="dst_capacity"):
        b200.batch.compress_fast_compact_host(src, soff, slen, small, max_src_len=65536)
    # found at the LAST chunk instead, while the payload copies of the earlier chunks are still draining
    with pytest.raises(b200.B200Error, match="dst_capacity"):
        b200.batch.compress_fast_compact_host(src, soff, slen, np.zeros(n * cl - 1, dtype=np.uint8), max_src_len=65536)
    # same thread, same streams: a short batch and then the full one must come back exact
    dst = np.zeros(n * cl + 64, dtype=np.uint8)
    ooff, olen, total = b200.batch.compress_fast_compact_host(src[:5 * bl], soff[:5], slen[:5], dst, max_src_len=65536)
    assert total == 5 * cl and (olen == cl).all() and (ooff == np.arange(5) * cl).all()
    ooff, olen, total = b200.batch.compress_fast_compact_host(src, soff, slen, dst, max_src_len=65536)
    assert total == n * cl and (olen == cl).all()
    assert (ooff == np.arange(n, dtype=np.uint64) * np.uint64(cl)).all()
    packed = dst[:total].reshape(n, cl)
    assert (packed[:, 0] == (min(bl, 15) << 4)).all() and (packed[:, hdr:] == src.reshape(n, bl)).all()
    # the slot-layout batch path after its own argument error (a dst slot out of order, found at the third chunk)
    coff, ccap = b200.batch.uniform_layout(n, cl)
    bad = coff.copy(); bad[2 * per_chunk + 50] = 0
    comp = np.zeros(n * cl, dtype=np.uint8)
    with pytest.raises(b200.B200Error, match="ascend"):
        b200.batch.compress_fast_batch_host(src, soff, slen, comp, bad, ccap, max_src_len=65536)
    clen = b200.batch.compress_fast_batch_host(src[:7 * bl], soff[:7], slen[:7], comp, coff[:7], ccap[:7], max_src_len=65536)
    assert (clen == cl).all() and (comp[:7 * cl].reshape(7, cl)[:, hdr:] == src[:7 * bl].reshape(7, bl)).all()


def test_xxhash_batches(b200, checker):
    rng = random.Random(5)
    bufs = [rng.randbytes(n) for n in list(range(0, 70)) + [255, 256, 257, 1000, 4096, 4097, 65536, 100001]]
    for align, pad in ((16, 0), (1, 3)):                 # TMA path (16-byte aligned) and direct path
        buf, off, ln = corpus.pack(bufs, align=align, pad=pad)
        for seed in (0, 0x9747B28C, 0xFFFFFFFF):
            h32 = b200.batch.xxh32_batch_host(buf, off, ln, seed)
            h64 = b200.batch.xxh64_batch_host(buf, off, ln, seed * 0x100000001)
            for k, bts in enumerate(bufs):
                assert int(h32[k]) == checker.xxh32(bts, seed), (align, len(bts), seed)
                assert int(h64[k]) == checker.xxh64(bts, seed * 0x100000001), (align, len(bts), seed)


def test_xxhash_uniform_4k(b200, checker):
    n = 3000
    data = np.frombuffer(random.Random(3).randbytes(n * 4096), dtype=np.uint8).copy()
    off, ln = b200.batch.uniform_layout(n, 4096)
    h64 = b200.batch.xxh64_batch_host(data, off, ln, 0)
    h32 = b200.batch.xxh32_batch_host(data, off, ln, 0x9747B28C)
    for k in range(0, n, 37):
        blk = data[k * 4096:(k + 1) * 4096]
        assert int(h64[k]) == checker.xxh64(blk, 0)
        assert int(h32[k]) == checker.xxh32(blk, 0x9747B28C)


def test_xxhash_long_streams(b200, checker):
    """a few long buffers take the one-warp-per-stream kernel: every alignment phase, every tail length"""
    rng = random.Random(21)
    blob = np.frombuffer(rng.randbytes(6 << 20), dtype=np.uint8).copy()
    offs, lens, pos = [], [], 0
    for k in range(9):
        pos += rng.randrange(0, 9)                                   # alignment phase 0..3 and beyond
        n = rng.choice([32768, 40000, 65536 + k, 300000 + 17 * k, 1 << 20]) + rng.randrange(0, 16)
        n = min(n, len(blob) - pos)
        offs.append(pos); lens.append(n); pos += n
    off = np.array(offs, dtype=np.uint64); ln = np.array(lens, dtype=np.int32)
    for seed in (0, 0x9747B28C):
        h = b200.batch.xxh32_batch_host(blob, off, ln, seed)
        h64 = b200.batch.xxh64_batch_host(blob, off, ln, seed)
        for k in range(len(offs)):
            assert int(h[k]) == checker.xxh32(blob[offs[k]:offs[k] + lens[k]], seed), (k, offs[k], lens[k])
            assert int(h64[k]) == checker.xxh64(blob[offs[k]:offs[k] + lens[k]], seed), (k, offs[k], lens[k])
    # the streaming states take the same warp loops for large updates
    f = b200.XXHashFactory.b200Instance()
    data = blob[3:3 + (1 << 20) + 5].tobytes()
    for mk, ref in ((f.newStreamingHash32, checker.xxh32), (f.newStreamingHash64, checker.xxh64)):
        h = mk(7)
        h.update(data, 0, 5); h.update(data, 5, 70001); h.update(data, 70006, len(data) - 70006)
        assert h.getValue() == ref(data, 7)
        h.close()


def test_xxhash_streaming(b200, checker):
    """random chunking + resets, like XXHash32Test.java:31-75"""
    rng = random.Random(11)
    f = b200.XXHashFactory.b200Instance()
    for bits, mk in ((32, f.newStreamingHash32), (64, f.newStreamingHash64)):
        for _ in range(6):
            data = rng.randbytes(rng.randrange(0, 5000))
            seed = rng.randrange(1 << 31)
            h = mk(seed)
            h.update(rng.randbytes(50))
            h.reset()
            pos = 0
            while pos < len(data):
                step = rng.randrange(1, 600)
                h.update(data, pos, min(step, len(data) - pos))
                pos += step
                if rng.random() < 0.3:
                    h.getValue()                       # digest must be callable mid-stream
            want = checker.xxh32(data, seed) if bits == 32 else checker.xxh64(data, seed)
            assert h.getValue() == want
            h.close()
            h.close()                                  # XXHash32Test.java:167-190 (testClose): closing twice is fine,
            for use in (h.getValue, h.reset, lambda: h.update(b"x")):     # any use afterwards is an AssertionError
                with pytest.raises(AssertionError):
                    use()


def test_factory_api_contract(b200, checker):
    """per-call contract of LZ4Test.java:170-256 through the mirrored API"""
    F = b200.LZ4Factory.b200Instance()
    comp, fast, safe = F.fastCompressor(), F.fastDecompressor(), F.safeDecompressor()
    for name, d in corpus.blocks(checker, big=False)[:40]:
        n = len(d)
        buf = bytearray(comp.maxCompressedLength(n))
        clen = comp.compress(d, 0, n, buf, 0, len(buf)) if n else comp.compress(b"", 0, 0, buf, 0, len(buf))
        c = bytes(buf[:clen])
        if n == 0:
            assert c == b"\x00"                                     # LZ4Test.java:111-114
        out = bytearray(n + 1)
        assert fast.decompress(c, 0, out, 0, n) == clen            # bytes read (:185)
        assert bytes(out[:n]) == d
        out = bytearray(n)
        assert safe.decompress(c, 0, clen, out, 0, n) == n         # bytes written (:232)
        assert bytes(out) == d
        if n > 0:
            with pytest.raises(b200.LZ4Exception):                  # destLen-1 must throw (:209-217)
                fast.decompress(c, 0, bytearray(n), 0, n - 1)
        with pytest.raises(b200.LZ4Exception):                      # srcLen+1 must throw (:240-245)
            safe.decompress(c + b"\x00", 0, clen + 1, bytearray(n + 8), 0, n)
    for v in corpus.MALFORMED[1:]:
        with pytest.raises(b200.LZ4Exception):
            safe.decompress(v, 0, len(v), bytearray(64), 0, 64)
    safe.decompress(corpus.MALFORMED[0], 0, len(corpus.MALFORMED[0]), bytearray(64), 0, 64)   # must not throw or hang


def test_jni_shim_through_fake_jnienv(b200, checker, tmp_path):
    """lz4-java_b200/jni/b200_jni.c compiled against tests/jni_fake/jni.h (no JDK here) and driven from C:
    byte[] / direct-buffer operands with offsets, return conventions, balanced critical sections."""
    import os
    import re
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "jni_harness")
    pkg = os.path.join(root, "lz4-java_b200")
    so = os.path.abspath(b200._native.SO_PATH)             # the library under test (libb200lz4.so unless the harness switched it)
    subprocess.run(["gcc", "-O1", "-I" + os.path.join(root, "tests", "jni_fake"), "-I" + os.path.join(root, "include"),
                    os.path.join(root, "tests", "jni_fake", "harness.c"), os.path.join(pkg, "jni", "b200_jni.c"),
                    so, "-Wl,-rpath," + os.path.dirname(so), "-o", exe], check=True)
    out = subprocess.run([exe], capture_output=True, text=True)
    assert out.returncode == 0 and out.stdout.startswith("ok"), out.stdout + out.stderr
    # the hashes printed by the harness must be the oracle's for the same generated bytes
    raw = bytearray(20007)
    s = 1
    for i in range(len(raw)):
        s = (s * 1103515245 + 12345) & 0xFFFFFFFF
        raw[i] = (i % 13) if (i % 97 < 60) else (s >> 24)
    m = re.search(r"xxh64=([0-9a-f]+) xxh32=([0-9a-f]+)", out.stdout)
    assert int(m.group(1), 16) == checker.xxh64(bytes(raw[7:]), 42)
    assert int(m.group(2), 16) == checker.xxh32(bytes(raw[7:]), 7)


def test_hc_compress_roundtrip_and_ratio(b200, checker):
    """LZ4 HC (level 9 class): valid stream, never worse than the fast parse, close to the reference's HC-9"""
    items = [(nm, d) for nm, d in corpus.blocks(checker) if len(d) in (0, 1, 12, 13, 64, 1000, 4096, 65536) or nm.startswith("period")]
    items += [(f"rdg256k_{mp}", checker.datagen(262144, mp, 0.0, 4).tobytes()) for mp in (0.2, 0.5, 0.8)]
    items += corpus.calgary_blocks(2)
    src, soff, slen = corpus.pack([d for _, d in items])
    bounds = [b200.max_compressed_length(len(d)) for _, d in items]
    doff, dcap, total = _slots(bounds)
    dst = np.zeros(total, dtype=np.uint8)
    res = b200.batch.compress_hc_batch_host(src, soff, slen, dst, doff, dcap, level=9)
    fast = b200.batch.compress_fast_batch_host(src, soff, slen, np.zeros(total, dtype=np.uint8), doff, dcap, max_src_len=0)
    ref_hc9 = _golden("ref_outputs.json")["hc9"]                     # LZ4_compress_HC(9)'s stream length for each block
    tot = tot_fast = tot_ref = 0
    for k, (name, d) in enumerate(items):
        assert 0 < res[k] <= bounds[k], (name, int(res[k]))
        c = dst[int(doff[k]):int(doff[k]) + int(res[k])].tobytes()
        r, out = checker.decompress_safe(c, len(d))
        assert r == len(d) and out == d, name
        tot += len(c); tot_fast += int(fast[k])
        tot_ref += ref_hc9[name]
    assert tot <= tot_fast, (tot, tot_fast)
    assert tot < 1.08 * tot_ref, (tot, tot_ref)
    # the single-block entry point the JNI shim binds, and level clamping of the factory (LZ4Factory.java:263-270)
    F = b200.LZ4Factory.b200Instance()
    d = items[-1][1]
    for lvl in (-5, 1, 9, 17, 99):
        c = F.highCompressor(lvl).compress(d)
        assert checker.decompress_safe(c, len(d))[1] == d


def test_frame_batch_decoder(b200, port):
    """LZ4 Frame container (config 3's driver): frames written by the oracle and by the reference's
    LZ4F_compressFrame (rebuilt from its recorded headers, corpus.ReferenceFrames) decode bit-exactly;
    every checksum / truncation error of LZ4FrameInputStream is reported with the oracle's code"""
    writers = [port, corpus.ReferenceFrames(port, _golden("ref_outputs.json")["frames"])]
    rng = random.Random(4)
    for w in writers:
        for n in (0, 1, 100, 65536, 65537, 300000, 9 << 20):
            data = port.datagen(n, 0.5, 0.0, n & 0xFF).tobytes() if n < (1 << 20) else (port.datagen(1 << 20, 0.5, 0.0, 3).tobytes() * 9)[:n]
            for bs in (4, 5, 7):
                for flags in (0, 1, 3, 5, 7):
                    f = w.frame_compress(data, bs, flags)
                    assert b200.decompress_frames(f, n + 8) == data, (w.kind, n, bs, flags)
    # incompressible data -> stored (raw) blocks (LZ4FrameOutputStream.java:215-222)
    noise = rng.randbytes(200000)
    assert b200.decompress_frames(port.frame_compress(noise, 4, 3), len(noise)) == noise
    # concatenated + skippable frames (LZ4FrameIOStreamTest.java:253-309, 378-426)
    a, b = b"hello frame " * 1000, port.datagen(70000, 0.5, 0.0, 1).tobytes()
    skip = bytes([0x50, 0x2A, 0x4D, 0x18, 4, 0, 0, 0, 1, 2, 3, 4])
    cat = port.frame_compress(a, 4, 1) + skip + port.frame_compress(b, 5, 7) + port.frame_compress(b"", 4, 1)
    assert b200.decompress_frames(cat, len(a) + len(b)) == a + b
    # error parity with the oracle's codes
    good = port.frame_compress(b, 4, 7)
    cases = {"truncated": good[:-3], "truncated2": good[:20], "magic": b"\x01\x02\x03\x04" + good[4:],
             "descriptor": good[:5] + bytes([good[5] ^ 0x10]) + good[6:], "content": good[:-1] + bytes([good[-1] ^ 1]),
             "payload": good[:40] + bytes([good[40] ^ 0xFF]) + good[41:], "empty": b""}
    for name, blob in cases.items():
        want = port.frame_decompress(blob, len(b))[0]
        assert want < 0, name
        with pytest.raises(b200.LZ4FrameError) as e:
            b200.decompress_frames(blob, len(b))
        assert e.value.code == want, (name, e.value.code, want)
    with pytest.raises(b200.LZ4FrameError) as e:
        b200.decompress_frames(good, len(b) - 1)
    assert e.value.code == -9


def test_frame_writer_and_lz4java_containers(b200, port):
    """(f)-2..4: frames / LZ4Block streams / length-prefixed blocks WRITTEN on the GPU path are read by the CPU
    restatements (and by the reference's LZ4F_decompress when available), and vice versa"""
    from oracle import oracle as O
    try:
        ref = O.Ref()
    except (FileNotFoundError, OSError):
        ref = None
    rng = random.Random(12)
    for n in (0, 1, 100, 65536, 65537, 300000, 3 << 20):
        data = port.datagen(n, 0.5, 0.0, n & 0xFF).tobytes()
        for bs, cc, bc, cs in ((4, True, False, False), (5, True, True, True), (7, False, False, False), (6, False, True, False)):
            f = b200.compress_frame(data, bs, cc, bc, cs)
            r, out = port.frame_decompress(f, n + 8)
            assert r == n and out == data, (n, bs)
            if ref is not None:
                r, out = ref.frame_decompress(f, n + 8)
                assert r == n and out == data, ("LZ4F_decompress", n, bs)
            assert b200.decompress_frames(f, n + 8) == data
        for blk in (64, 4096, 65536, 1 << 20):
            blob = b200.compress_lz4block(data, blk)
            r, out = port.lz4block_decompress(blob, n)
            assert r == n and out == data, (n, blk)
            assert b200.decompress_lz4block(port.lz4block_compress(data, blk), n) == data
            assert b200.decompress_lz4block(blob + blob, 2 * n, stop_on_empty_block=False) == data + data
            assert b200.decompress_lz4block(blob + blob, 2 * n) == data                     # stopOnEmptyBlock, the reference's default
            assert b200.decompress_lz4block(blob + b"not a block", n) == data
            assert b200.decompress_lz4block(blob[:-21] + b"LZ4", n, stop_on_empty_block=False) == data
            with pytest.raises(EOFError):
                b200.decompress_lz4block(blob[:-21], n)                                      # no end block (LZ4BlockInputStream.java:192-198)
        wl = b200.compress_with_length(data)
        assert port.with_length_decompress(wl, n) == (len(wl), data)
        assert b200.decompress_with_length(port.with_length_compress(data)) == data
    noise = rng.randbytes(200000)                                   # stored (raw) blocks
    assert port.frame_decompress(b200.compress_frame(noise, 4), len(noise))[1] == noise
    assert port.lz4block_decompress(b200.compress_lz4block(noise, 65536), len(noise))[1] == noise
    good = port.lz4block_compress(port.datagen(70000, 0.5, 0.0, 1).tobytes(), 65536)
    bad = bytearray(good); bad[50] ^= 0x41
    with pytest.raises(IOError):
        b200.decompress_lz4block(bytes(bad), 70000)
    with pytest.raises(EOFError):
        b200.decompress_lz4block(good[:100], 70000)


def test_decompress_fast_does_not_walk_past_the_stream(b200, checker, decoder):
    """The same regression, aimed: blocks ending  …long match, a few short sequences, 5-14 last literals, built so that
    the old batched walk (modelled on the CPU while writing this test) takes the final literal-only token for a full
    sequence in 6 of the 96 blocks; what follows each stream starts with the bytes 01 00 — a valid-looking offset —
    and continues with another block's sequences.  Added after the round's GPU budget was spent: its data was
    validated on the CPU instead — tests/test_kernel_logic_cpu.py runs the kernels' own source under a SIMT emulator,
    where the pre-fix source fails on exactly those six blocks (return -1 and a write past the output) and the fixed
    source passes."""
    rng = random.Random(8080)
    items = []
    for trial in range(96):
        hist = bytes(rng.randrange(256) for _ in range(3000))
        parts = [hist]

        def short():
            parts.append(bytes(rng.randrange(256) for _ in range(rng.randrange(1, 7))))
            a = rng.randrange(0, 2900); parts.append(hist[a:a + rng.randrange(5, 13)])
        for _ in range(rng.randrange(40, 90)): short()
        a = rng.randrange(0, 500)
        parts.append(bytes(rng.randrange(256) for _ in range(2))); parts.append(hist[a:a + rng.randrange(1100, 1700)])
        for _ in range(rng.randrange(3, 26)): short()
        parts.append(bytes(rng.randrange(256) for _ in range(rng.randrange(5, 15))))
        items.append(b"".join(parts))
    comp = [checker.compress(d) for d in items]
    lens = np.array([len(d) for d in items], dtype=np.int32)
    padded = [c + b"\x01\x00" + comp[(k + 1) % len(comp)][9:3000] + bytes(64) for k, c in enumerate(comp)]
    src, soff, slen = corpus.pack(padded)
    doff, dcap, total = _slots([len(d) for d in items], align=64)
    dst = np.full(total + 4096, 0x55, dtype=np.uint8)
    res = b200.batch.decompress_fast_batch_host(src, soff, slen, dst, doff, lens)
    for k, d in enumerate(items):
        assert res[k] == len(comp[k]), (decoder, k, int(res[k]), len(comp[k]))
        assert dst[int(doff[k]):int(doff[k]) + len(d)].tobytes() == d, (decoder, k)
        assert (dst[int(doff[k]) + len(d):int(doff[k]) + len(d) + 16] == 0x55).all(), (decoder, k)


def test_contexts_are_reused_across_threads(b200, checker):
    """LZ4Compressor instances are singletons used from any number of threads (LZ4Compressor.java:25): every thread gets
    its own streams and staging, and a thread that exits hands them to the next new thread instead of leaking them."""
    import threading
    lib = b200._native.lib()
    data = checker.datagen(3000, 0.5, 0.0, 9).tobytes()
    comp = b200.LZ4Factory.b200Instance().fastCompressor().compress(data)        # this thread's context exists now
    base = lib.b200lz4_context_count()
    errs = []

    def work(k):
        try:
            f = b200.LZ4Factory.b200Instance()
            c = f.fastCompressor().compress(data)
            assert c == comp
            assert f.fastDecompressor().decompress(c, destLen=len(data)) == data
            assert b200.XXHashFactory.b200Instance().hash64().hash(data, 0, len(data), k) == checker.xxh64(data, k)
        except Exception as e:      # noqa: BLE001
            errs.append(e)

    import time
    for k in range(8):                       # eight threads one after the other: they share one or two contexts
        t = threading.Thread(target=work, args=(k,)); t.start(); t.join()
        time.sleep(0.05)                     # join() returns before the OS thread has run its thread-exit hooks
    assert not errs, errs
    assert base <= lib.b200lz4_context_count() <= base + 3      # (0 new ones if earlier tests left idle contexts in the pool)
    ts = [threading.Thread(target=work, args=(k,)) for k in range(4)]    # four at once: at most four contexts alive
    for t in ts: t.start()
    for t in ts: t.join()
    assert not errs, errs
    assert lib.b200lz4_context_count() <= base + 3 + 4


def test_frames_sharded_by_frame(b200, port):
    """config 3's multi-GPU split: every rank decodes its own byte-balanced range of whole frames (here the ranks run one
    after the other on one GPU); the pieces concatenate to the single-rank result"""
    from lz4java_b200.sharding import frame_boundaries, shard_frames
    frames, plain = [], []
    for k in range(12):
        d = port.datagen(50000 + 40000 * (k % 4), 0.5, 0.0, 20 + k).tobytes()
        frames.append(port.frame_compress(d, 4 + k % 2, 1 + 2 * (k % 2))); plain.append(d)
    stream = b"".join(frames)
    whole = b200.decompress_frames(stream, sum(map(len, plain)))
    assert whole == b"".join(plain)
    bounds = frame_boundaries(stream)
    assert len(bounds) == len(frames)
    for world in (2, 8):
        got = b""
        for lo, hi in shard_frames([e - s for s, e in bounds], world):
            if hi > lo:
                got += b200.decompress_frames(stream[bounds[lo][0]:bounds[hi - 1][1]], sum(map(len, plain[lo:hi])))
        assert got == whole


def _golden(name):
    import json
    return json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name)))


def test_golden_vectors_on_gpu(b200, port, decoder):
    """The CUDA path against the COMMITTED outputs of the reference's own C (tests/golden/kat.json, generated from
    oracle/_ref by make_golden.py): XXH32/XXH64 values, the safe decoder's return code on every malformed vector x
    capacity, the fast decoder's, and — for every corpus block — decoding the stream whose digest the fixture records."""
    import hashlib
    kat = _golden("kat.json")
    stream = port.datagen(200000, 0.5, 0.0, 77)
    # hashes: one batch per seed over the prefixes
    for seed in (0, 0x9747B28C):
        ents = [e for e in kat["xxh"] if e["seed"] == seed]
        off = np.zeros(len(ents), dtype=np.uint64)
        ln = np.array([e["len"] for e in ents], dtype=np.int32)
        h32 = b200.batch.xxh32_batch_host(stream, off, ln, seed)
        h64 = b200.batch.xxh64_batch_host(stream, off, ln, seed * 0x100000001)
        for k, e in enumerate(ents):
            assert int(h32[k]) == e["xxh32"] and int(h64[k]) == e["xxh64"], e
    # malformed vectors: return codes recorded from the reference
    ms = kat["malformed_safe"]
    src, soff, slen = corpus.pack([bytes.fromhex(e["hex"]) for e in ms], pad=8)
    doff, dcap, total = _slots([e["cap"] for e in ms])
    res = b200.batch.decompress_safe_batch_host(src, soff, slen, np.zeros(total, dtype=np.uint8), doff, dcap)
    for k, e in enumerate(ms):
        assert int(res[k]) == e["ret"], e
    mf = kat["malformed_fast"]
    padded = [bytes.fromhex(e["hex"]) + bytes(e["n"] + 64) for e in mf]
    src, soff, slen = corpus.pack(padded)
    doff, dlen, total = _slots([e["n"] for e in mf])
    res = b200.batch.decompress_fast_batch_host(src, soff, slen, np.zeros(total, dtype=np.uint8), doff, dlen)
    for k, e in enumerate(mf):
        assert int(res[k]) == e["ret"], e
    # corpus blocks: the pinned restatement reproduces the reference's stream (digest in the fixture); the GPU decodes it
    items = corpus.blocks(port)
    assert [n for n, _ in items] == [e["name"] for e in kat["compress"]]
    comp = [port.compress(d) for _, d in items]
    for c, (_, d), e in zip(comp, items, kat["compress"]):
        assert hashlib.sha256(c).hexdigest() == e["c_sha256"] and hashlib.sha256(bytes(d)).hexdigest() == e["in_sha256"]
    src, soff, slen = corpus.pack(comp)
    doff, dcap, total = _slots([len(d) for _, d in items])
    dst = np.zeros(total, dtype=np.uint8)
    res = b200.batch.decompress_safe_batch_host(src, soff, slen, dst, doff, dcap)
    for k, e in enumerate(kat["compress"]):
        assert int(res[k]) == e["len"], e["name"]
        assert hashlib.sha256(dst[int(doff[k]):int(doff[k]) + e["len"]].tobytes()).hexdigest() == e["in_sha256"], e["name"]


def test_golden_calgary_on_gpu(b200, port, decoder):
    """real data that travels to the GPU box: the reference's fast and HC-9 streams of Calgary cuts decode on the GPU
    (safe and fast decoders) to bytes with the recorded digest; the GPU's own fast and HC streams of those bytes decode
    back under the CPU checker, and the GPU HC stream is smaller than the reference's FAST stream"""
    import base64
    import hashlib
    cal = _golden("calgary_lz4.json")["blocks"]
    for key in ("fast_b64", "hc9_b64"):
        comp = [base64.b64decode(b[key]) for b in cal]
        src, soff, slen = corpus.pack([c + bytes(64) for c in comp])
        slen_exact = np.array([len(c) for c in comp], dtype=np.int32)
        doff, dcap, total = _slots([b["len"] for b in cal])
        dst = np.zeros(total, dtype=np.uint8)
        res = b200.batch.decompress_safe_batch_host(src, soff, slen_exact, dst, doff, dcap)
        dst2 = np.zeros(total, dtype=np.uint8)
        res2 = b200.batch.decompress_fast_batch_host(src, soff, slen, dst2, doff, dcap)
        for k, b in enumerate(cal):
            assert int(res[k]) == b["len"] and int(res2[k]) == len(comp[k]), (key, b["name"])
            for out in (dst, dst2):
                assert hashlib.sha256(out[int(doff[k]):int(doff[k]) + b["len"]].tobytes()).hexdigest() == b["sha256"], (key, b["name"])
    if decoder != "batched":
        return
    plain = [dst[int(doff[k]):int(doff[k]) + b["len"]].tobytes() for k, b in enumerate(cal)]
    f = b200.LZ4Factory.b200Instance()
    for b, d in zip(cal, plain):
        c = f.fastCompressor().compress(d)
        assert port.decompress_safe(c, len(d)) == (len(d), d), b["name"]
        h = f.highCompressor(9).compress(d)
        assert port.decompress_safe(h, len(d)) == (len(d), d), b["name"]
        assert len(h) < len(base64.b64decode(b["fast_b64"])), (b["name"], len(h))


def test_multi_gpu_range_sharded_host_batches(b200, checker):
    """One process driving several GPUs (SURVEY.md 8e, the single-JVM case): the *_multi calls cut the block list into
    contiguous ranges, one worker thread + context per listed device, no exchange.  Output must be byte-identical to the
    single-GPU call whatever the device list is.  A one-GPU box lists device 0 several times (the shards then share the
    GPU but not their streams or staging); the emulator build pretends SIMT_DEVICES GPUs."""
    lib = b200._native.lib()
    ndev = lib.b200lz4_device_count()
    assert ndev >= 1
    lists = [1, [0, 0, 0], [0] * 7] + ([ndev, list(range(ndev))[::-1]] if ndev > 1 else [])
    if "sim" in os.environ.get("B200LZ4_TEST_SO", ""):          # emulator build (CPU suite): every launch costs seconds
        lists = [[0, 0, 0]] + ([list(range(ndev))[::-1]] if ndev > 1 else [])
    datas = [checker.datagen(rng_n, 0.5, 0.0, s).tobytes() for s, rng_n in enumerate([65536, 1, 0, 40000, 65536, 13, 70000, 5000, 65536, 300, 12, 65536, 100000])]
    src, soff, slen = corpus.pack(datas)
    coff, ccap, ctotal = _slots([b200.max_compressed_length(len(d)) for d in datas])
    want_c = np.zeros(ctotal, dtype=np.uint8)
    want_len = b200.batch.compress_fast_batch_host(src, soff, slen, want_c, coff, ccap)
    want_h32 = b200.batch.xxh32_batch_host(src, soff, slen, 7)
    want_h64 = b200.batch.xxh64_batch_host(src, soff, slen, 7)
    doff, dcap, dtotal = _slots([len(d) for d in datas])
    for devs in lists:
        comp = np.zeros(ctotal, dtype=np.uint8)
        clen = b200.batch.compress_fast_batch_host_multi(src, soff, slen, comp, coff, ccap, devs)
        assert (clen == want_len).all(), devs
        for k in range(len(datas)):
            o = int(coff[k])
            assert comp[o:o + int(clen[k])].tobytes() == want_c[o:o + int(clen[k])].tobytes(), (devs, k)
        out = np.zeros(dtotal, dtype=np.uint8)
        r = b200.batch.decompress_safe_batch_host_multi(comp, coff, clen, out, doff, dcap, devs)
        out2 = np.zeros(dtotal, dtype=np.uint8)
        r2 = b200.batch.decompress_fast_batch_host_multi(comp, coff, ccap, out2, doff, dcap, devs)
        for k, d in enumerate(datas):
            assert int(r[k]) == len(d) and int(r2[k]) == int(clen[k]), (devs, k)
            o = int(doff[k])
            assert out[o:o + len(d)].tobytes() == d and out2[o:o + len(d)].tobytes() == d, (devs, k)
        assert (b200.batch.xxh32_batch_host_multi(src, soff, slen, devs, 7) == want_h32).all()
        assert (b200.batch.xxh64_batch_host_multi(src, soff, slen, devs, 7) == want_h64).all()
    # packed output per shard: same bytes as the single-GPU compaction, shard by shard, at bases known in advance
    pk = np.zeros(ctotal, dtype=np.uint8)
    w_off, w_len, w_total = b200.batch.compress_fast_compact_host(src, soff, slen, pk)
    for devs in lists:
        nd = devs if isinstance(devs, int) else len(devs)
        pm = np.full(ctotal, 0x77, dtype=np.uint8)
        ooff, olen, sbase, stotal = b200.batch.compress_fast_compact_host_multi(src, soff, slen, pm, devs)
        assert (olen == w_len).all() and int(stotal.sum()) == w_total, devs
        for g in range(nd):
            lo, hi = len(datas) * g // nd, len(datas) * (g + 1) // nd
            want = b"".join(pk[int(w_off[i]):int(w_off[i]) + int(w_len[i])].tobytes() for i in range(lo, hi))
            assert int(stotal[g]) == len(want) and pm[int(sbase[g]):int(sbase[g]) + len(want)].tobytes() == want, (devs, g)
            if hi > lo:
                assert int(ooff[lo]) == int(sbase[g]), (devs, g)
    with pytest.raises(b200.B200Error, match="dst_capacity"):
        b200.batch.compress_fast_compact_host_multi(src, soff, slen, np.zeros(1000, dtype=np.uint8), [0, 0])
    # HC: same sharding (a few blocks: one CTA each)
    hc_want = np.zeros(ctotal, dtype=np.uint8)
    hc_len = b200.batch.compress_hc_batch_host(src, soff[:6], slen[:6], hc_want, coff[:6], ccap[:6])
    hc = np.zeros(ctotal, dtype=np.uint8)
    assert (b200.batch.compress_hc_batch_host_multi(src, soff[:6], slen[:6], hc, coff[:6], ccap[:6], [0, 0]) == hc_len).all()
    for k in range(6):
        o = int(coff[k])
        assert hc[o:o + int(hc_len[k])].tobytes() == hc_want[o:o + int(hc_len[k])].tobytes(), k
    # fewer blocks than devices, no blocks, and a device that does not exist
    two = b200.batch.compress_fast_batch_host_multi(src, soff[:2], slen[:2], np.zeros(ctotal, dtype=np.uint8), coff[:2], ccap[:2], [0] * 5)
    assert (two == want_len[:2]).all()
    assert len(b200.batch.xxh64_batch_host_multi(src, soff[:0], slen[:0], 3)) == 0
    with pytest.raises(b200.B200Error, match="device"):
        b200.batch.xxh32_batch_host_multi(src, soff, slen, [0, ndev + 5])
    # the calling thread keeps working on its own device afterwards
    assert (b200.batch.xxh32_batch_host(src, soff, slen, 7) == want_h32).all()


def test_cross_backend_with_the_java_port(b200, port, decoder):
    """LZ4Test.java:305-324 ties every compressor to every decompressor of every backend.  The pure-Java backend
    (LZ4Factory.safeInstance(), BASELINE configs[0]) is available here only as a restatement (oracle/lz4_java_port_oracle.c,
    unpinned): its streams must decode bit-exactly on the GPU with the right return values, and the GPU compressors'
    streams must be accepted by the Java decoders' rule set (decompress.template), which differs from lz4.c's."""
    items = [(n, bytes(d)) for n, d in corpus.blocks(port)]
    jcomp = [port.java_compress(d) for _, d in items]
    assert all(c is not None for c in jcomp)
    src, soff, slen = corpus.pack([c + bytes(64) for c in jcomp])
    exact = np.array([len(c) for c in jcomp], dtype=np.int32)
    doff, dcap, total = _slots([len(d) for _, d in items])
    out, out2 = np.zeros(total, dtype=np.uint8), np.zeros(total, dtype=np.uint8)
    r = b200.batch.decompress_safe_batch_host(src, soff, exact, out, doff, dcap)
    r2 = b200.batch.decompress_fast_batch_host(src, soff, slen, out2, doff, dcap)
    for k, (name, d) in enumerate(items):
        assert int(r[k]) == len(d) and int(r2[k]) == len(jcomp[k]), name
        o = int(doff[k])
        assert out[o:o + len(d)].tobytes() == d and out2[o:o + len(d)].tobytes() == d, name
    if decoder != "batched":
        return
    # the GPU compressors' streams under the Java decoders
    psrc, poff, plen = corpus.pack([d for _, d in items])
    coff, ccap, ctotal = _slots([b200.max_compressed_length(len(d)) for _, d in items])
    for fn in (b200.batch.compress_fast_batch_host, b200.batch.compress_hc_batch_host):
        comp = np.zeros(ctotal, dtype=np.uint8)
        clen = fn(psrc, poff, plen, comp, coff, ccap)
        for k, (name, d) in enumerate(items):
            c = comp[int(coff[k]):int(coff[k]) + int(clen[k])].tobytes()
            assert port.java_decompress_safe(c, len(d)) == (len(d), d), (fn.__name__, name)
            assert port.java_decompress_fast(c + bytes(16), len(d)) == (len(c), d), (fn.__name__, name)


def test_uncompress_worst_case_literal_only_blocks(b200, checker, decoder):
    """LZ4Test.java:89-154 (testUncompressWorstCase / testUncompressSafeWorstCase): hand-built literals-only blocks — one
    token, the 255-chain, the bytes — up to 100 KiB (longer than anything the compressors emit for 64 KiB blocks),
    including the seed the reference pins for lengths < 16"""
    rng = random.Random(0x69CCC652)
    lens = list(range(0, 18)) + [254, 255, 256, 269, 270, 271, 4096, 65535, 65536, 65537, 100 * 1024] + [rng.randrange(100 * 1024) for _ in range(6)]
    plain, comp = [], []
    for n in lens:
        d = bytes(rng.randrange(rng.choice([1, 2, 255, 256]) + 1) & 0xFF for _ in range(n))
        c = bytearray()
        if n >= 15:
            c.append(15 << 4); rest = n - 15
            while rest >= 255:
                c.append(255); rest -= 255
            c.append(rest)
        else:
            c.append(n << 4)
        plain.append(d); comp.append(bytes(c) + d)
    src, soff, slen = corpus.pack([c + bytes(32) for c in comp])
    exact = np.array([len(c) for c in comp], dtype=np.int32)
    doff, dcap, total = _slots(lens)
    out, out2 = np.zeros(total, dtype=np.uint8), np.zeros(total, dtype=np.uint8)
    r = b200.batch.decompress_safe_batch_host(src, soff, exact, out, doff, dcap)
    r2 = b200.batch.decompress_fast_batch_host(src, soff, slen, out2, doff, dcap)
    for k, d in enumerate(plain):
        assert (int(r[k]), int(r2[k])) == (len(d), len(comp[k])), (k, len(d))
        assert checker.decompress_safe(comp[k], len(d)) == (len(d), d)
        o = int(doff[k])
        assert out[o:o + len(d)].tobytes() == d and out2[o:o + len(d)].tobytes() == d, (k, len(d))


@pytest.mark.skipif("sim" in os.environ.get("B200LZ4_TEST_SO", ""), reason="8 GiB of hashing: not for the CPU emulator build")
def test_streaming_hash_past_4gb(b200, port):
    """XXHash64Test.java:149-170 / XXHash32Test.java (test4GB): a streaming state fed more than 2^32 bytes — XXH32 keeps
    its length modulo 2^32 (xxhash.c:437-563: total_len_32 + large_len), XXH64 a 64-bit one — checked against the CPU
    restatement fed the same chunks, with getValue() read (and required idempotent) along the way"""
    chunk = port.datagen((1 << 26) + 1000, 0.5, 0.0, 41)
    off, ln = 3, (1 << 26) + 1000 - 3 - 517
    view = chunk[off:off + ln]
    seed = 0x1234567
    h32, h64 = b200.StreamingXXHash32(seed), b200.StreamingXXHash64(seed * 0x100000001)
    import ctypes as C
    L = port.L
    s32 = C.create_string_buffer(L.orc_xxh32_state_size()); s64 = C.create_string_buffer(L.orc_xxh64_state_size())
    L.orc_xxh32_reset(s32, seed); L.orc_xxh64_reset(s64, seed * 0x100000001)
    total = 0
    while total < (1 << 32) + (1 << 27):
        h32.update(chunk, off, ln); h64.update(chunk, off, ln)
        L.orc_xxh32_update(s32, view.ctypes.data, ln); L.orc_xxh64_update(s64, view.ctypes.data, ln)
        total += ln
        if total > (1 << 32) - (1 << 27) or total < (1 << 28):
            assert h32.getValue() == L.orc_xxh32_digest(s32) == h32.getValue(), total
            assert h64.getValue() == L.orc_xxh64_digest(s64) == h64.getValue(), total
    h32.close(); h64.close()


def test_reference_test_fixtures_on_gpu(b200, port):
    """LZ4Test.testRoundtripIssue12 (the array at offset 9, LZ4Test.java:488-539) with the fast and the HC compressor, and
    the LZ4FrameIOStreamTest data recipe at all 17 of its sizes through the frame writer / reader and the LZ4Block
    container, each checked against the CPU checker in both directions"""
    import json
    raw = bytes.fromhex(json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "issue12.json")))["hex"])
    d = corpus.issue12()
    f = b200.LZ4Factory.b200Instance()
    for comp in (f.fastCompressor(), f.highCompressor(9)):
        dest = bytearray(comp.maxCompressedLength(len(d)) + 5)
        n = comp.compress(raw, 9, len(raw) - 9, dest, 5, len(dest) - 5)          # testRoundTrip(data, 9, data.length - 9)
        c = bytes(dest[5:5 + n])
        assert port.decompress_safe(c, len(d)) == (len(d), d)
        assert f.safeDecompressor().decompress(c, maxDestLen=len(d)) == d
        assert f.fastDecompressor().decompress(c, destLen=len(d)) == d
    for k, n in enumerate(corpus.frame_test_sizes()):
        data = corpus.frame_test_data(n)
        flags = (1, 0, 3, 7, 5)[k % 5]
        assert b200.decompress_frames(port.frame_compress(data, 4 + k % 4, flags), n + 8) == data, n
        fr = b200.compress_frame(data, 4 + (k + 1) % 4, content_checksum=bool(flags & 1), block_checksum=bool(flags & 2), content_size=bool(flags & 4))
        assert port.frame_decompress(fr, n + 8) == (n, data), n
        if n <= (1 << 20):
            assert b200.decompress_lz4block(b200.compress_lz4block(data, 1 << 16), n + 8) == data, n


# ---------------------------------------------------------------------------------------------- round-2 additions
def test_golden_skippable_frame(b200):
    """src/lz4/tests/goldenSamples/skip.bin, the reference's only golden file: a skippable frame decodes to nothing, alone
    and in front of / behind a real frame (LZ4FrameInputStream.java:154-173)"""
    import json, os
    blob = bytes.fromhex(json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "skip_bin.json")))["hex"])
    assert len(blob) == 38
    assert b200.decompress_frames(blob, 16) == b""
    data = bytes(range(256)) * 300
    f = b200.compress_frame(data, 4, True, False, False)
    assert b200.decompress_frames(blob + f + blob, len(data)) == data


@pytest.mark.parametrize("mp", [0.2, 0.5, 0.8])
def test_dev_pointer_entry_points_sweep(b200, checker, mp):
    """Every *_batch_dev entry point (what bench.py times) with device tensors on a NON-default stream, the sweep that found
    round 1's decoder bug: 16384 x 64 KiB blocks of RDG_genBuffer, bound-sized compressed slots that still hold the streams
    of ANOTHER corpus behind each stream's end, safe and fast decoders, against oracle/_ref: the reference decodes the
    GPU's streams, the GPU decodes the reference's streams, return codes for every block."""
    import torch
    from oracle import oracle as O
    n, bs = 16384, 65536
    dev = torch.device("cuda", 0)
    bound = b200.max_compressed_length(bs); stride = (bound + 15) // 16 * 16
    B = b200.batch
    threads = min(32, os.cpu_count() or 1)

    def corpus_of(p, seed):
        base = checker.datagen(2048 * bs, p, 0.0, seed)
        return np.tile(base, n // 2048)

    other = corpus_of(0.5 if mp != 0.5 else 0.8, 11)          # what the slots held before
    data = corpus_of(mp, 7)
    for k in range(n):                                          # make the tiled blocks distinct
        data[k * bs] ^= k & 0xFF; data[k * bs + 1] ^= (k >> 8) & 0xFF
    soff = torch.arange(n, device=dev, dtype=torch.int64) * bs
    slen = torch.full((n,), bs, device=dev, dtype=torch.int32)
    coff = torch.arange(n, device=dev, dtype=torch.int64) * stride
    ccap = torch.full((n,), bound, device=dev, dtype=torch.int32)
    st = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(st):
        d_src = torch.from_numpy(data).to(dev, non_blocking=False)
        comp = torch.zeros(n * stride, dtype=torch.uint8, device=dev)
        clen = torch.zeros(n, dtype=torch.int32, device=dev)
        res = torch.zeros(n, dtype=torch.int32, device=dev)
        out = torch.zeros(n * bs, dtype=torch.uint8, device=dev)
        d_other = torch.from_numpy(other).to(dev)
        B.compress_fast_batch_dev(d_other, soff, slen, comp, coff, ccap, clen, bs)      # stale streams in every slot
        B.compress_fast_batch_dev(d_src, soff, slen, comp, coff, ccap, clen, bs)
        B.decompress_safe_batch_dev(comp, coff, clen, out, soff, slen, res)
        st.synchronize()
        assert bool((clen > 0).all()) and bool((res == bs).all()) and bool(torch.equal(out, d_src)), "safe"
        out.zero_()
        B.decompress_fast_batch_dev(comp, coff, ccap, out, soff, slen, res)            # readable bytes = the whole slot
        st.synchronize()
        assert bool((res == clen).all()) and bool(torch.equal(out, d_src)), "fast"
        h_comp, h_clen = comp.cpu().numpy(), clen.cpu().numpy()
    # the reference decodes every GPU stream
    np_off = np.arange(n, dtype=np.uint64)
    back = np.zeros(n * bs, dtype=np.uint8)
    _, _, r = O.cpu_bench(checker, "dec_safe", h_comp, np_off * np.uint64(stride), h_clen.astype(np.int32), back,
                          np_off * np.uint64(bs), np.full(n, bs, dtype=np.int32), threads, 1)
    assert (r == bs).all() and (back == data).all(), "reference rejects a GPU stream"
    # the GPU decodes every reference stream (slots keep the GPU's longer/shorter streams behind them)
    ref_comp = h_comp.copy()
    _, _, rc = O.cpu_bench(checker, "compress", data, np_off * np.uint64(bs), np.full(n, bs, dtype=np.int32), ref_comp,
                           np_off * np.uint64(stride), np.full(n, bound, dtype=np.int32), threads, 1)
    assert (rc > 0).all()
    with torch.cuda.stream(st):
        comp.copy_(torch.from_numpy(ref_comp)); rlen = torch.from_numpy(rc.astype(np.int32)).to(dev)
        out.zero_(); B.decompress_safe_batch_dev(comp, coff, rlen, out, soff, slen, res); st.synchronize()
        assert bool((res == bs).all()) and bool(torch.equal(out, d_src)), "safe / reference streams"
        out.zero_(); B.decompress_fast_batch_dev(comp, coff, ccap, out, soff, slen, res); st.synchronize()
        assert bool((res == rlen).all()) and bool(torch.equal(out, d_src)), "fast / reference streams"
        # hashes through the device entry points, same stream
        h64 = torch.zeros(n, dtype=torch.int64, device=dev); h32 = torch.zeros(n, dtype=torch.int32, device=dev)
        B.xxh64_batch_dev(d_src, soff, slen, h64, 0); B.xxh32_batch_dev(d_src, soff, slen, h32, 0x9747B28C); st.synchronize()
        for k in (0, 1, n // 2, n - 1):
            blk = data[k * bs:(k + 1) * bs]
            assert (int(h64[k]) & (2 ** 64 - 1)) == checker.xxh64(blk, 0) and (int(h32[k]) & 0xFFFFFFFF) == checker.xxh32(blk, 0x9747B28C)
        # HC through its device entry point on a slice
        m = 64
        B.compress_hc_batch_dev(d_src, soff[:m], slen[:m], comp, coff[:m], ccap[:m], clen[:m], 9)
        out.zero_(); B.decompress_safe_batch_dev(comp, coff[:m], clen[:m], out, soff[:m], slen[:m], res[:m]); st.synchronize()
        assert bool((res[:m] == bs).all()) and bool(torch.equal(out[:m * bs], d_src[:m * bs])), "hc"


def test_negative_and_tiny_capacities(b200, checker):
    """dstCapacity < 0 is "no room" (0, nothing written), not a wrapped unsigned comparison (round-1 advisor finding);
    the reference returns 0 for every capacity below what it needs (lz4.c:1085-1088)"""
    d = checker.datagen(20000, 0.5, 0.0, 3).tobytes()
    src, soff, slen = corpus.pack([d, d, d, d])
    doff = np.arange(4, dtype=np.uint64) * np.uint64(32768)
    for max_src_len in (65536, 0):
        dst = np.full(4 * 32768, 0x55, dtype=np.uint8)
        need = int(b200.batch.compress_fast_batch_host(src, soff, slen, dst, doff, np.full(4, 32768, dtype=np.int32), max_src_len=max_src_len)[0])
        assert need > 0
        caps = np.array([-1, -(1 << 31), 0, need - 1], dtype=np.int32)
        dst = np.full(4 * 32768, 0x55, dtype=np.uint8)
        res = b200.batch.compress_fast_batch_host(src, soff, slen, dst, doff, caps, max_src_len=max_src_len)
        assert (res == 0).all(), res
        assert (dst[:3 * 32768] == 0x55).all()
    assert b200._native.lib().b200lz4_compress_default(src.ctypes.data, dst.ctypes.data, len(d), -1) == 0
    assert b200._native.lib().b200lz4_compress_HC(src.ctypes.data, dst.ctypes.data, len(d), -5, 9) == 0


def test_one_block_calls_leave_the_rest_of_dst_alone(b200, checker):
    """a decoder called with maxDestLen = "the rest of my buffer" must not clobber what lies further along (the reference
    only scribbles a few bytes past what it writes); compress likewise copies back exactly its output"""
    f = b200.LZ4Factory.b200Instance()
    a = checker.datagen(5000, 0.5, 0.0, 1).tobytes(); b = checker.datagen(7000, 0.5, 0.0, 2).tobytes()
    ca, cb = checker.compress(a), checker.compress(b)
    dest = bytearray(b"\xAA" * 20000)
    assert f.safeDecompressor().decompress(cb, 0, len(cb), dest, 5000, 15000) == len(b)      # block 2 first, further along
    assert f.safeDecompressor().decompress(ca, 0, len(ca), dest, 0, 20000) == len(a)         # block 1 with the whole buffer as room
    assert bytes(dest[:5000]) == a and bytes(dest[5000:12000]) == b and bytes(dest[12000:]) == b"\xAA" * 8000
    out = bytearray(b"\x33" * 30000)
    n = f.fastCompressor().compress(a, 0, len(a), out, 100, 20000)
    assert checker.decompress_safe(bytes(out[100:100 + n]), len(a)) == (len(a), a)
    assert bytes(out[:100]) == b"\x33" * 100 and bytes(out[100 + n:]) == b"\x33" * (30000 - 100 - n)


def test_error_offsets_beyond_a_million_are_decoder_errors(b200, checker):
    """-(offset)-1 of a corrupt 4 MiB frame block can be below -1000000: it must surface as "Error decoding offset N"
    (LZ4JNISafeDecompressor.java:40-42), not as a backend failure (the backend codes are INT_MIN + 1..3)"""
    d = checker.datagen(4 << 20, 0.2, 0.0, 5).tobytes()
    c = bytearray(checker.compress(d))
    assert len(c) > 3_000_000
    c = c[:len(c) - 7]                                          # cut inside the last literals: the error sits at the very end
    want, _ = checker.decompress_safe(bytes(c), len(d))
    assert want < -1_000_000
    src = np.frombuffer(bytes(c), dtype=np.uint8)
    dst = np.zeros(len(d), dtype=np.uint8)
    r = b200._native.lib().b200lz4_decompress_safe(src.ctypes.data, dst.ctypes.data, len(c), len(d))
    assert r == want
    with pytest.raises(b200.LZ4Exception) as e:
        b200.LZ4Factory.b200Instance().safeDecompressor().decompress(bytes(c), 0, len(c), bytearray(len(d)), 0, len(d))
    assert "offset" in str(e.value)


# ---- written after round 2's last visit to a GPU (DESIGN.md section 6): these ran on the emulator build only so far, so they come last
class _DevMem:
    """device buffers for tests that call the C ABI with raw device pointers: torch CUDA tensors on a GPU box, plain
    numpy arrays under the emulator build (its "device memory" is the host heap)"""

    def __init__(self):
        self.sim = "sim" in os.environ.get("B200LZ4_TEST_SO", "")
        if not self.sim:
            import torch
            self.torch = torch

    def up(self, arr, device=0):
        arr = np.ascontiguousarray(arr)
        if self.sim:
            return arr.copy()
        return self.torch.from_numpy(arr.view(np.uint8).reshape(-1)).to(self.torch.device("cuda", device))

    def zeros(self, nbytes, device=0):
        return self.up(np.zeros(max(nbytes, 16), dtype=np.uint8), device)

    def ptr(self, buf):
        return buf.ctypes.data if self.sim else buf.data_ptr()

    def down(self, buf, dtype=np.uint8):
        if not self.sim:
            self.torch.cuda.synchronize(buf.device)
            buf = buf.cpu().numpy()
        return buf.view(np.uint8).reshape(-1).view(dtype)


def _frame_of_pieces(port, pieces, bs_code, content_checksum=True, block_checksum=False, stored=()):
    """an LZ4 frame whose blocks are exactly `pieces` (what LZ4FrameOutputStream writes when flush() is called between
    writes, LZ4FrameOutputStream.java:204-251,268-277): short blocks anywhere, stored when they do not shrink or when asked"""
    hdr = bytes([0x60 | (0x10 if block_checksum else 0) | (0x04 if content_checksum else 0), bs_code << 4])
    out = bytearray(b"\x04\x22\x4d\x18" + hdr + bytes([(port.xxh32(hdr, 0) >> 8) & 0xFF]))
    for i, piece in enumerate(pieces):
        c = port.compress(piece)
        raw = i in stored or len(c) >= len(piece)
        payload = piece if raw else c
        out += (len(payload) | (0x80000000 if raw else 0)).to_bytes(4, "little") + payload
        if block_checksum:
            out += port.xxh32(payload, 0).to_bytes(4, "little")
    out += (0).to_bytes(4, "little")
    if content_checksum:
        out += port.xxh32(b"".join(pieces), 0).to_bytes(4, "little")
    return bytes(out)


def test_frames_written_with_flush(b200, port):
    """short blocks before the last one: the content checksum is folded across block boundaries that are not multiples
    of 16 on the device, the blocks are packed on the device, and a stream of tiny blocks asks for slots of its own size
    (not blockMaxSize each).  Against the restated reader (LZ4FrameInputStream.java:258-321)."""
    rng = random.Random(int(os.environ.get("B200_SEED", 77)))
    base = port.datagen(1 << 20, 0.5, 0.0, 9).tobytes()
    for trial in range(int(os.environ.get("B200_TRIALS", 4 if "sim" in os.environ.get("B200LZ4_TEST_SO", "") else 12))):   # (the emulator build takes seconds per launch)
        bs_code = rng.choice((4, 5, 6, 7))
        bs = 1 << (8 + 2 * bs_code)
        sizes = [rng.choice((1, 3, 5, 15, 16, 17, 31, 100, 4097, 65535, min(bs, 65536), min(bs, 200000))) for _ in range(rng.randrange(1, 40))]
        if trial == 0:
            sizes = [5] * 300                                     # nothing but 5-byte stored blocks
        if trial == 1:
            sizes = [bs, 7, bs, bs, 1, 16, 33]
        pieces = []
        for n in sizes:
            o = rng.randrange(0, len(base) - n) if n < len(base) else 0
            pieces.append(rng.randbytes(n) if rng.random() < 0.2 else (base * (n // len(base) + 1))[o:o + n])
        stored = {i for i in range(len(pieces)) if rng.random() < 0.15}
        f = _frame_of_pieces(port, pieces, bs_code, content_checksum=trial % 3 != 2, block_checksum=bool(trial & 1), stored=stored)
        want = b"".join(pieces)
        r, out = port.frame_decompress(f, len(want) + 8)
        assert r == len(want) and out == want, trial                # the builder writes what the restated reader accepts
        assert b200.decompress_frames(f, len(want) + 8) == want, (trial, sizes)
        both = f + port.frame_compress(base[:70000], 4, 1) + f       # gapped and contiguous frames in one call
        assert b200.decompress_frames(both, 2 * len(want) + 70000) == want + base[:70000] + want, trial
        if trial % 3 != 2 and want:
            bad = bytearray(f); bad[-1] ^= 0x40                      # content checksum of a gapped frame
            with pytest.raises(b200.LZ4FrameError) as e:
                b200.decompress_frames(bytes(bad), len(want) + 8)
            assert e.value.code == -7, trial
        if want:
            with pytest.raises(b200.LZ4FrameError) as e:
                b200.decompress_frames(f, len(want) - 1)
            assert e.value.code == -9
    # slots: 300 five-byte stored blocks in a 4 MiB-block frame need kilobytes, not 300 x 4 MiB
    import ctypes
    from importlib import import_module
    N = import_module(b200.__name__ + "._native")
    f = np.frombuffer(_frame_of_pieces(port, [b"12345"] * 300, 7, stored=set(range(300))), dtype=np.uint8)
    slot, err = ctypes.c_uint64(0), ctypes.c_int(0)
    ix = N.lib().b200lz4f_index_create(f.ctypes.data, len(f), ctypes.byref(slot), ctypes.byref(err))
    assert ix and err.value == 0 and slot.value == 300 * 16, (err.value, slot.value)
    offs = np.zeros(300, dtype=np.uint64)
    N.lib().b200lz4f_index_block_offsets(ix, offs.ctypes.data)
    assert (offs == np.arange(300, dtype=np.uint64) * 16).all()
    N.lib().b200lz4f_index_free(ix)
    # the device entry point on a gapped frame: every check passes, -11 says "read the blocks one by one", and the blocks are
    # where b200lz4f_index_block_offsets says, block_len_out bytes each
    pieces = [base[:65536], base[100:107], base[7:65543], b"", base[5:38], rng.randbytes(300)]
    pieces = [p for p in pieces if p]
    f = np.frombuffer(_frame_of_pieces(port, pieces, 4, content_checksum=True, block_checksum=True), dtype=np.uint8)
    M = _DevMem()
    ix = N.lib().b200lz4f_index_create(f.ctypes.data, len(f), ctypes.byref(slot), ctypes.byref(err))
    assert ix and err.value == 0
    nb = N.lib().b200lz4f_index_blocks(ix)
    assert nb == len(pieces) and N.lib().b200lz4f_index_frames(ix) == 1
    d_src, d_slots = M.up(np.concatenate([f, np.zeros(64, dtype=np.uint8)])), M.zeros(slot.value + 64)
    foff, flen, blen = np.zeros(1, dtype=np.uint64), np.zeros(1, dtype=np.uint64), np.zeros(nb, dtype=np.int32)
    rc = N.lib().b200lz4f_decode_dev(ix, M.ptr(d_src), M.ptr(d_slots), foff.ctypes.data, flen.ctypes.data, blen.ctypes.data, None)
    assert rc == -11 and int(flen[0]) == sum(map(len, pieces)) and [int(x) for x in blen] == [len(p) for p in pieces]
    offs = np.zeros(nb, dtype=np.uint64)
    N.lib().b200lz4f_index_block_offsets(ix, offs.ctypes.data)
    got = M.down(d_slots)
    for o, p in zip(offs, pieces):
        assert got[int(o):int(o) + len(p)].tobytes() == p
    bad = f.copy(); bad[-1] ^= 1                                   # the content checksum is verified BEFORE -11 is returned
    ix2 = N.lib().b200lz4f_index_create(bad.ctypes.data, len(bad), ctypes.byref(slot), ctypes.byref(err))
    d_bad = M.up(np.concatenate([bad, np.zeros(64, dtype=np.uint8)]))
    assert N.lib().b200lz4f_decode_dev(ix2, M.ptr(d_bad), M.ptr(d_slots), None, None, None, None) == -7
    N.lib().b200lz4f_index_free(ix); N.lib().b200lz4f_index_free(ix2)
    # the host path on a gapped frame with a stored block makes six launches, all counted: descriptor hash, block hashes,
    # stored-block gather, decode, chained content hash, and the gather that packs the blocks
    f = _frame_of_pieces(port, pieces, 4, content_checksum=True, block_checksum=True, stored={1})
    N.lib().b200lz4_launch_count_reset()
    assert b200.decompress_frames(f, sum(map(len, pieces))) == b"".join(pieces)
    assert N.lib().b200lz4_launch_count() == 6


def test_frame_index_free_keeps_the_current_device(b200, port):
    """an index decoded on GPU 0 and freed while GPU 1 is current releases its device state on GPU 0 and leaves GPU 1 current"""
    import ctypes
    M = _DevMem()
    if M.sim or M.torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    L = b200._native.lib()
    data = port.datagen(200000, 0.5, 0.0, 3).tobytes()
    f = np.frombuffer(port.frame_compress(data, 4, 3), dtype=np.uint8)
    slot, err = ctypes.c_uint64(0), ctypes.c_int(0)
    ix = L.b200lz4f_index_create(f.ctypes.data, len(f), ctypes.byref(slot), ctypes.byref(err))
    assert ix and err.value == 0
    try:
        M.torch.cuda.set_device(0)
        d_src, d_slots = M.up(np.concatenate([f, np.zeros(64, dtype=np.uint8)]), 0), M.zeros(slot.value + 64, 0)
        assert L.b200lz4f_decode_dev(ix, M.ptr(d_src), M.ptr(d_slots), None, None, None, None) == len(data)
        assert M.down(d_slots)[:len(data)].tobytes() == data
        M.zeros(16, 1)                                              # GPU 1 has a context, so the current device is CUDA's own
        M.torch.cuda.set_device(1)
        L.b200lz4f_index_free(ix)
        assert M.torch.cuda.current_device() == 1
    finally:
        M.torch.cuda.set_device(0)


def test_container_writers_with_the_high_compressor(b200, port):
    """LZ4FrameOutputStream / LZ4BlockOutputStream take the compressor as an argument (LZ4FrameOutputStream.java:132-133,
    LZ4BlockOutputStream.java:96,124); with highCompressor(level) the containers must still be read by the sequential readers
    (restated, and the reference's LZ4F_decompress when it is there), and must not come out larger than with the fast one."""
    from oracle import oracle as O
    try:
        ref = O.Ref()
    except (FileNotFoundError, OSError):
        ref = None
    sim = "sim" in os.environ.get("B200LZ4_TEST_SO", "")
    for n in ((1, 70000) if sim else (0, 1, 65536, 200000, 1500000)):
        data = port.datagen(n, 0.5, 0.0, 5).tobytes()
        for level in ((9,) if sim else (1, 9, 17)):
            f_fast, f_hc = b200.compress_frame(data, 4, True, True, True), b200.compress_frame(data, 4, True, True, True, hc_level=level)
            assert len(f_hc) <= len(f_fast), (n, level)
            assert port.frame_decompress(f_hc, n + 8) == (n, data), (n, level)
            if ref is not None:
                assert ref.frame_decompress(f_hc, n + 8) == (n, data), ("LZ4F_decompress", n, level)
            assert b200.decompress_frames(f_hc, n + 8) == data
            b_fast, b_hc = b200.compress_lz4block(data, 1 << 16), b200.compress_lz4block(data, 1 << 16, hc_level=level)
            assert len(b_hc) <= len(b_fast), (n, level)
            assert port.lz4block_decompress(b_hc, n) == (n, data), (n, level)
            assert b200.decompress_lz4block(b_hc, n) == data
    noise = random.Random(3).randbytes(70000)                       # does not shrink: stored blocks either way
    assert b200.compress_frame(noise, 4, hc_level=9) == b200.compress_frame(noise, 4)
    assert b200.compress_lz4block(noise, 1 << 16, hc_level=9) == b200.compress_lz4block(noise, 1 << 16)


def test_read_single_frame_and_expected_content_size(b200, port):
    """LZ4FrameIOStreamTest.java:310-426: a frame written with its content size reports it (getExpectedContentSize), one
    written without reports -1; with readSingleFrame the reader stops behind the first non-skippable frame -- four
    concatenated copies yield one -- and says how far it read; what follows that frame is not even looked at."""
    import ctypes
    data = port.datagen(300000, 0.5, 0.0, 77).tobytes()
    with_size = b200.compress_frame(data, 7, True, False, True)
    without = b200.compress_frame(data, 7, True, False, False)
    assert b200.expected_content_size(with_size) == len(data)                      # :326-329
    assert b200.expected_content_size(port.frame_compress(data, 4, 5)) == len(data)
    assert b200.expected_content_size(without) == -1                               # :348-351
    assert b200.decompress_frames(with_size, len(data), read_single_frame=True) == data
    four = without * 4                                                              # :379-420
    assert b200.decompress_frames(four, 4 * len(data)) == data * 4
    assert b200.decompress_frames(four, 4 * len(data), read_single_frame=True) == data
    assert b200.expected_content_size(four) == -1
    skip = bytes([0x5A, 0x2A, 0x4D, 0x18, 3, 0, 0, 0, 9, 9, 9])
    lead = skip + skip + with_size + b"\x00garbage that is not a frame"
    assert b200.decompress_frames(lead, len(data), read_single_frame=True) == data  # skippable frames do not count as "the" frame
    assert b200.expected_content_size(lead) == len(data)
    with pytest.raises(b200.LZ4FrameError) as e:
        b200.decompress_frames(lead, len(data))                                     # ... the multi-frame reader trips over the rest
    assert e.value.code == -2
    L = b200._native.lib()
    buf = np.frombuffer(lead, dtype=np.uint8); out = np.zeros(len(data), dtype=np.uint8); used = ctypes.c_size_t(0)
    assert L.b200lz4f_decompress_host_single(buf.ctypes.data, len(buf), out.ctypes.data, len(out), ctypes.byref(used)) == len(data)
    assert used.value == 2 * len(skip) + len(with_size) and out.tobytes() == data
    assert b200.expected_content_size(skip) == -1                                   # only skippable frames: no frame, no error (:141-147)
    assert b200.decompress_frames(skip, 10, read_single_frame=True) == b""
    for bad, code in ((b"", -1), (skip + b"\x04\x22", -1), (b"\x04\x22\x4d\x18\x60", -1), (b"\x01\x02\x03\x04rest", -2),
                      (with_size[:4] + bytes([with_size[4] ^ 0x80]) + with_size[5:], -10),
                      (with_size[:7] + bytes([with_size[7] ^ 1]) + with_size[8:], -3)):      # a bit of the content size: descriptor hash
        with pytest.raises(b200.LZ4FrameError) as e:
            b200.expected_content_size(bad)
        assert e.value.code == code, (bad[:12], e.value.code, code)


def test_frame_errors_come_in_stream_order(b200, port):
    """LZ4FrameInputStream is a stream: of several things wrong with a container it reports the FIRST one it meets
    (descriptor hash, then block by block checksum and decode, then at the EndMark content checksum before content size,
    LZ4FrameInputStream.java:208-216, 264-273, 298-311), and a container cut short or malformed further on still fails
    on an earlier checksum first.  One to three random faults per container, against the restated sequential reader."""
    rng = random.Random(2024)
    base = port.datagen(1 << 18, 0.5, 0.0, 21).tobytes()
    sim = "sim" in os.environ.get("B200LZ4_TEST_SO", "")
    seen = {}
    for trial in range(int(os.environ.get("B200_TRIALS", 60 if sim else 400))):
        frames = []
        for _ in range(rng.randrange(1, 4)):
            pieces = [base[o:o + n] for o, n in ((rng.randrange(0, 100000), rng.choice((1, 40, 700, 5000, 65536))) for _ in range(rng.randrange(0, 5)))]
            if rng.random() < 0.5:
                body = b"".join(pieces)
                frames.append(port.frame_compress(body, rng.choice((4, 5)), rng.randrange(8)))   # flags: content checksum, block checksums, content size
            else:
                frames.append(_frame_of_pieces(port, pieces, rng.choice((4, 5)), content_checksum=rng.random() < 0.7, block_checksum=rng.random() < 0.5,
                                               stored={i for i in range(len(pieces)) if rng.random() < 0.2}))
        blob = bytearray(b"".join(frames))
        total = 1 << 20
        for _ in range(rng.randrange(1, 4)):
            kind = rng.randrange(4)
            if kind == 0 and len(blob) > 8:
                del blob[rng.randrange(len(blob) - 8, len(blob)):]                   # cut short near the end
            elif kind == 1 and len(blob) > 1:
                del blob[rng.randrange(1, len(blob)):]                               # cut short anywhere
            elif blob:
                i = rng.randrange(len(blob)); blob[i] ^= 1 << rng.randrange(8)       # one flipped bit
        want, out = port.frame_decompress(bytes(blob), total)
        if want >= 0:
            assert b200.decompress_frames(bytes(blob), total) == out, trial
            seen["ok"] = seen.get("ok", 0) + 1
            continue
        with pytest.raises(b200.LZ4FrameError) as e:
            b200.decompress_frames(bytes(blob), total)
        assert e.value.code == want, (trial, e.value.code, want, bytes(blob).hex() if len(blob) < 400 else len(blob))
        seen[want] = seen.get(want, 0) + 1
    assert len([k for k in seen if k != "ok"]) >= (4 if sim else 6), seen              # the sweep met most of the codes
    # the same for lz4-java's own container (LZ4BlockInputStream.java:191-264): premature end vs "Stream is corrupted" vs our -9
    seen = {}
    for trial in range(int(os.environ.get("B200_TRIALS", 60 if sim else 400))):
        body = b"".join(base[o:o + n] for o, n in ((rng.randrange(0, 100000), rng.choice((1, 40, 700, 5000, 70000))) for _ in range(rng.randrange(0, 4))))
        if rng.random() < 0.2:
            body += rng.randbytes(3000)                                              # a stored block
        blob = bytearray(port.lz4block_compress(body, rng.choice((64, 4096, 65536))))
        for _ in range(rng.randrange(1, 4)):
            kind = rng.randrange(3)
            if kind == 0 and len(blob) > 1:
                del blob[rng.randrange(1, len(blob)):]
            elif blob:
                i = rng.randrange(len(blob)); blob[i] ^= 1 << rng.randrange(8)
        stop = rng.random() < 0.7
        cap = len(body) + rng.choice((0, 0, 8, -1000))
        cap = max(cap, 0)
        want, out = port.lz4block_decompress(bytes(blob), cap, stop)
        if want >= 0:
            assert b200.decompress_lz4block(bytes(blob), cap, stop_on_empty_block=stop) == out, trial
            seen["ok"] = seen.get("ok", 0) + 1
            continue
        with pytest.raises((EOFError, IOError)) as e:
            b200.decompress_lz4block(bytes(blob), cap, stop_on_empty_block=stop)
        got = -1 if isinstance(e.value, EOFError) else (-2 if "corrupted" in str(e.value) else -9)
        assert got == want, (trial, got, want, str(e.value))
        seen[want] = seen.get(want, 0) + 1
    assert len(seen) >= 3, seen


def test_device_side_compaction_and_stitch(b200, checker):
    """(f)-4 with everything in HBM: each shard's blocks are compressed into bound-sized slots, packed on the device
    (b200lz4_compact_dev) and the packed shards are stitched into one stream by peer copies at offsets computed from the
    shard totals (b200lz4_stitch_shards_dev).  The stitched stream must be byte-identical to what one GPU packs for the whole
    batch (b200lz4_compress_fast_compact_host), block offsets included.  A one-GPU box lists device 0 for every shard
    (device-to-device copies); the emulator build pretends SIMT_DEVICES GPUs; a multi-GPU box uses them all."""
    import ctypes
    L = b200._native.lib()
    M = _DevMem()
    ndev = L.b200lz4_device_count()
    assert ndev >= 1
    datas = [checker.datagen(n, 0.5, 0.0, s).tobytes() for s, n in enumerate([65536, 1, 0, 40000, 65536, 13, 70000, 5000, 65536, 300, 12, 65536, 100000])]
    src, soff, slen = corpus.pack(datas)
    want = np.zeros(sum(b200.max_compressed_length(len(d)) + 16 for d in datas), dtype=np.uint8)
    w_off, w_len, w_total = b200.batch.compress_fast_compact_host(src, soff, slen, want)
    for shard_devs in ([0], [0, 0, 0], [g % ndev for g in range(5)], list(range(ndev))[::-1]):
        k = len(shard_devs)
        bufs, totals, offs_all = [], [], []
        for g, dv in enumerate(shard_devs):
            lo, hi = len(datas) * g // k, len(datas) * (g + 1) // k
            assert L.b200lz4_set_device(dv) == 0
            if not M.sim:
                M.torch.cuda.set_device(dv)
            n = hi - lo
            coff, ccap, ctotal = _slots([b200.max_compressed_length(len(d)) for d in datas[lo:hi]])
            d_src, d_soff, d_slen = M.up(src, dv), M.up(soff[lo:hi], dv), M.up(slen[lo:hi], dv)
            d_coff, d_ccap = M.up(coff, dv), M.up(ccap, dv)
            d_slots, d_clen = M.zeros(ctotal, dv), M.zeros(4 * n, dv)
            d_pack, d_poff, d_tot = M.zeros(ctotal, dv), M.zeros(8 * n, dv), M.zeros(8, dv)
            if n:
                assert L.b200lz4_compress_fast_batch_dev(M.ptr(d_src), M.ptr(d_soff), M.ptr(d_slen), M.ptr(d_slots), M.ptr(d_coff), M.ptr(d_ccap),
                                                         M.ptr(d_clen), n, 0, None) == 0
            assert L.b200lz4_compact_dev(M.ptr(d_slots), M.ptr(d_coff), M.ptr(d_clen), M.ptr(d_pack), M.ptr(d_poff), M.ptr(d_tot), n, None) == 0
            tot = int(M.down(d_tot, np.uint64)[0])
            clen = M.down(d_clen, np.int32)[:n]
            assert (clen == w_len[lo:hi]).all() and tot == int(clen.sum()), (shard_devs, g)
            bufs.append(d_pack); totals.append(tot); offs_all.append(M.down(d_poff, np.uint64)[:n].copy())
        dst_dev = shard_devs[-1]
        d_out = M.zeros(sum(totals) + 32, dst_dev)
        ptrs = (ctypes.c_void_p * k)(*[M.ptr(b) for b in bufs])
        devs = (ctypes.c_int * k)(*shard_devs)
        tot = np.asarray(totals, dtype=np.uint64); pos = np.zeros(k, dtype=np.uint64)
        assert L.b200lz4_stitch_shards_dev(ptrs, devs, tot.ctypes.data, k, M.ptr(d_out), dst_dev, sum(totals) + 32, pos.ctypes.data) == 0
        got = M.down(d_out)
        assert sum(totals) == w_total and got[:w_total].tobytes() == want[:w_total].tobytes(), shard_devs
        assert (got[w_total:w_total + 32] == 0).all()
        where = np.concatenate([o + p for o, p in zip(offs_all, pos)])
        assert (where == w_off).all(), shard_devs
        # too small a destination is refused before anything is copied
        assert L.b200lz4_stitch_shards_dev(ptrs, devs, tot.ctypes.data, k, M.ptr(d_out), dst_dev, sum(totals) - 1, None) == b200._native.E_ARG
    assert L.b200lz4_set_device(0) == 0
    if not M.sim:
        M.torch.cuda.set_device(0)
