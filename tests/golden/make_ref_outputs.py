"""Generates tests/golden/ref_outputs.json and tests/golden/calgary_cuts.xz from the REFERENCE's own C, so that the tests
which compare against it run without it:

    make -C oracle REF=<lz4-java checkout>          # builds oracle/_ref/liblz4ref.so from its lz4 1.9.4 sources
    python tests/golden/make_ref_outputs.py <lz4-java checkout>

ref_outputs.json holds, for the inputs the tests use:
  codec   per block of corpus.blocks(big=False) + corpus.calgary_blocks(2): the digest of LZ4_compress_default's stream, of
          its output at the capacities of corpus.compress_caps (null where it refuses), and LZ4_decompress_safe's /
          LZ4_decompress_fast's return codes on corpus.codec_variants of that stream, with one digest over the bytes they
          decoded (tests/test_oracle_pin.py::test_ref_differential_codec)
  frames  per "<input length>/<block size ID>/<flags>": the digest of the restated writer's frame and what LZ4F_decompress
          made of it, and LZ4F_compressFrame's header and the digest of its whole frame (corpus.ReferenceFrames)
  hc9     LZ4_compress_HC level 9 stream lengths of the blocks tests/test_gpu_parity.py::test_hc_compress_roundtrip_and_ratio
          compresses
calgary_cuts.xz holds the 64 KiB cuts of corpus.CALGARY_XZ_CUTS, taken from <checkout>/src/test-resources/calgary."""
import hashlib
import json
import lzma
import os
import random
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))
from oracle import oracle as O      # noqa: E402
import corpus                       # noqa: E402


def sha(b):
    return hashlib.sha256(bytes(b)).hexdigest()


def frame_inputs(port):
    """(length -> bytes, block size IDs, flags) of the frames test_ref_differential_frames and test_frame_batch_decoder write"""
    for n in (0, 1, 100, 65536, 65537, 300000, 5 << 20, 9 << 20):
        if n == 9 << 20:
            data = (port.datagen(1 << 20, 0.5, 0.0, 3).tobytes() * 9)[:n]
        else:
            data = port.datagen(n, 0.5, 0.0, n & 0xFF).tobytes()
        yield data, ((4, 7) if n == 5 << 20 else (4, 5, 7)), (0, 1, 3, 5, 7)
    yield port.datagen(70000, 0.5, 0.0, 1).tobytes(), (5,), (1,)


def main(reference):
    R, P = O.Ref(), O.Port()
    assert R.version() == 10904, "the fixtures come from lz4 1.9.4"
    base = os.path.join(reference, "src", "test-resources", "calgary")
    cuts = []
    for name in corpus.CALGARY_XZ_CUTS:
        f, at = name.split("@")
        cuts.append(open(os.path.join(base, f), "rb").read()[int(at):int(at) + 65536])
        assert len(cuts[-1]) == 65536
    open(os.path.join(HERE, "calgary_cuts.xz"), "wb").write(lzma.compress(b"".join(cuts), preset=9 | lzma.PRESET_EXTREME))
    for name, d in corpus.calgary_blocks(4):                       # the stored cuts are the files' bytes
        f, at = name.split("@")
        assert d == open(os.path.join(base, f), "rb").read()[int(at):int(at) + 65536], name

    out = {"lz4_version": R.version(), "codec": [], "frames": {}, "hc9": {}}
    rng = random.Random(2)
    for name, d in corpus.blocks(R, big=False) + corpus.calgary_blocks(2):
        c = R.compress(d)
        caps = [R.compress(d, cap) for cap in corpus.compress_caps(c)]
        e = {"name": name, "c_sha256": sha(c), "caps": [None if x is None else sha(x) for x in caps], "safe": [], "fast": []}
        decoded = hashlib.sha256()
        for cc, cap in corpus.codec_variants(c, len(d), rng):
            r, o = R.decompress_safe(cc, cap)
            e["safe"].append(r); decoded.update(o)
            if cap >= 0:
                r, o = R.decompress_fast(cc, cap)
                e["fast"].append(r)
                if r >= 0:
                    decoded.update(o)
        e["decoded_sha256"] = decoded.hexdigest()
        out["codec"].append(e)

    for data, bss, flagss in frame_inputs(P):
        n = len(data)
        for bs in bss:
            for flags in flagss:
                f, g = P.frame_compress(data, bs, flags), R.frame_compress(data, bs, flags)
                r, o = R.frame_decompress(f, n + 16)
                assert r == n and o == data, (n, bs, flags)
                head = g[:corpus.frame_header_len(g)]
                assert head + f[corpus.frame_header_len(f):] == g, (n, bs, flags)
                out["frames"][f"{n}/{bs}/{flags}"] = {"port_sha256": sha(f), "ref_decodes": [r, sha(o)], "head": head.hex(), "sha256": sha(g)}

    items = [(nm, d) for nm, d in corpus.blocks(P) if len(d) in (0, 1, 12, 13, 64, 1000, 4096, 65536) or nm.startswith("period")]
    items += [(f"rdg256k_{mp}", P.datagen(262144, mp, 0.0, 4).tobytes()) for mp in (0.2, 0.5, 0.8)]
    items += corpus.calgary_blocks(2)
    for nm, d in items:
        h = R.compress_hc(d, 9)
        assert R.decompress_safe(h, len(d)) == (len(d), d), nm
        out["hc9"][nm] = len(h)

    p = os.path.join(HERE, "ref_outputs.json")
    json.dump(out, open(p, "w"), indent=0)
    print("wrote", p, os.path.getsize(p), "bytes and calgary_cuts.xz", os.path.getsize(os.path.join(HERE, "calgary_cuts.xz")), "bytes")


if __name__ == "__main__":
    main(sys.argv[1])
