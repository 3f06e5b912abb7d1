"""C-ABI checks that need no GPU: the library loads, exports every symbol include/b200lz4.h declares,
pure-arithmetic entry points work, and compute entry points fail LOUDLY (no CPU fallback) without a device."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    txt = open(os.path.join(ROOT, "include", "b200lz4.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(b200(?:lz4|xxh(?:32|64))_?\w*)\s*\(", txt)))


def test_every_header_symbol_is_exported_and_bound(b200):
    lib = b200._native.lib()
    names = header_functions()
    assert len(names) >= 35
    bound = {n for n, _, _ in b200._native.SYMBOLS}
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/b200lz4.h but not exported"
        assert n in bound, f"{n} exported but not bound in _native.SYMBOLS"
    assert lib.b200lz4_version() == 100


def test_compress_bound_matches_reference_formula(b200, port):
    lib = b200._native.lib()
    rng = np.random.default_rng(1)
    for n in [0, 1, 254, 255, 256, 65536, 0x7E000000, 0x7E000001, -1] + [int(x) for x in rng.integers(0, 1 << 30, 50)]:
        assert lib.b200lz4_compressBound(n) == port.compress_bound(n)
    # LZ4Utils.maxCompressedLength == LZ4_compressBound for valid lengths (LZ4Test.java:80-87)
    for n in (0, 1, 65536, 1 << 30):
        assert b200.max_compressed_length(n) == port.compress_bound(n)
    with pytest.raises(ValueError):
        b200.max_compressed_length(-1)
    with pytest.raises(ValueError):
        b200.max_compressed_length(0x7E000000)


def _no_gpu(b200):
    return b200._native.lib().b200lz4_device_count() < 0


def test_no_device_is_loud(b200, port):
    """without a usable GPU the product raises; it never computes on the CPU"""
    if not _no_gpu(b200):
        pytest.skip("a CUDA device is present")
    lib = b200._native.lib()
    src = np.zeros(100, dtype=np.uint8)
    dst = np.zeros(200, dtype=np.uint8)
    assert lib.b200lz4_compress_default(src.ctypes.data, dst.ctypes.data, 100, 200) == b200._native.E_NODEVICE
    assert "cuda" in b200._native.last_error().lower()
    with pytest.raises(b200.B200Error):
        b200.LZ4Factory.b200Instance()
    with pytest.raises(b200.B200Error):
        b200.batch.xxh32_batch_host(src, [0], [100])
    with pytest.raises(b200.B200Error):
        b200.XXHashFactory.b200Instance()
    # the hash calls return the VALUE: the failure travels in b200lz4_last_status(), and the mirror raises on it
    assert lib.b200xxh32(src.ctypes.data, 100, 0) == 0 and lib.b200lz4_last_status() == b200._native.E_NODEVICE
    assert lib.b200xxh64(src.ctypes.data, 100, 0) == 0 and lib.b200lz4_last_status() == b200._native.E_NODEVICE
    with pytest.raises(b200.B200Error):
        b200.xxhash.XXHash32().hash(src.tobytes(), 0, 100, 0)
    with pytest.raises(b200.B200Error):
        b200.xxhash.XXHash64().hash(src.tobytes(), 0, 100, 0)
    # the frame and container calls return the same code, and leave their own status and message behind (not an earlier
    # call's: each check starts from an argument error's); the frame writer writes no frame with a missing checksum
    E = b200._native.E_NODEVICE
    out = np.zeros(64, dtype=np.uint8)
    frame = np.frombuffer(port.frame_compress(b"a small frame", 4, 1), dtype=np.uint8)
    size = ctypes.c_int64(0)
    calls = [lambda flags=flags: lib.b200lz4f_compress_host(src.ctypes.data, 0, out.ctypes.data, len(out), 4, flags) for flags in (0, 1, 5)]
    calls += [lambda: lib.b200lz4f_decompress_host(frame.ctypes.data, len(frame), out.ctypes.data, len(out)),
              lambda: lib.b200lz4f_expected_content_size(frame.ctypes.data, len(frame), ctypes.byref(size)),
              lambda: lib.b200lz4block_compress_host(src.ctypes.data, 1, out.ctypes.data, len(out), 1 << 16)]
    for i, call in enumerate(calls):
        lib.b200xxh32(src.ctypes.data, 1 << 31, 0)
        assert lib.b200lz4_last_status() == b200._native.E_ARG
        assert call() == E, i
        msg = b200._native.last_error()
        assert lib.b200lz4_last_status() == E and msg and "invalid argument" not in msg, (i, msg)
    with pytest.raises(b200.B200Error):
        b200.compress_frame(b"")


def test_product_does_not_import_oracle():
    """the package may not reference oracle/ in any way (checker is test infrastructure only)"""
    pkg = os.path.join(ROOT, "lz4-java_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp", ".java")):
                txt = open(os.path.join(dp, f), errors="ignore").read()
                assert "oracle" not in txt.lower().replace("test oracle", ""), os.path.join(dp, f)


def test_product_loader_has_no_library_switch(b200, monkeypatch):
    """the package loads its own libb200lz4.so and nothing else: no environment variable can point it at another
    library (the emulator build of tests/simt is reachable only through tests/conftest.py / tools/_variant.py)"""
    pkg = os.path.join(ROOT, "lz4-java_b200")
    for f in os.listdir(pkg):
        if f.endswith(".py"):
            txt = open(os.path.join(pkg, f)).read()
            assert "os.environ" not in txt and "getenv" not in txt, f
    if not os.environ.get("B200LZ4_TEST_SO"):
        assert os.path.samefile(b200._native.SO_PATH, os.path.join(pkg, "libb200lz4.so"))


def test_java_natives_have_shim_symbols_and_shim_calls_are_in_the_header():
    """No JDK here, so the three layers are checked textually: every `native` method of the two Java JNI enums has its
    Java_<class>_<method> definition in jni/b200_jni.c (JNI name mangling: '_' -> '_1'), and every b200* function the shim
    calls is declared in include/b200lz4.h"""
    shim = open(os.path.join(ROOT, "lz4-java_b200", "jni", "b200_jni.c")).read()
    java = os.path.join(ROOT, "lz4-java_b200", "java", "net", "jpountz")
    n = 0
    for rel, cls in (("lz4/LZ4B200JNI.java", "net_jpountz_lz4_LZ4B200JNI"), ("xxhash/XXHashB200JNI.java", "net_jpountz_xxhash_XXHashB200JNI")):
        for m in re.findall(r"native\s+\w+\s+(\w+)\(", open(os.path.join(java, rel)).read()):
            assert re.search(r"\bJava_" + cls + "_" + m.replace("_", "_1") + r"\b", shim), (rel, m)
            n += 1
    assert n >= 32
    defined = set(re.findall(r"\bJava_(\w+)\b", shim))
    assert len(defined) == n, "a Java_ symbol in the shim has no native declaration"
    declared = set(header_functions())
    for call in set(re.findall(r"\b(b200(?:lz4|xxh(?:32|64))_?\w*)\s*\(", shim)):
        assert call in declared, call


def test_library_exports_nothing_but_the_header():
    """nm -D: the dynamic symbol table holds the C ABI of include/b200lz4.h and nothing else — no tuning knobs (round 1 had
    process-global ints a test could flip under every other thread's feet), no kernel stubs, no internal launch layer"""
    import re, subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run(["nm", "-D", "--defined-only", os.path.join(root, "lz4-java_b200", "libb200lz4.so")],
                         capture_output=True, text=True, check=True).stdout
    exported = {l.split()[-1] for l in out.splitlines() if l.strip()}
    declared = set(re.findall(r"\b(b200[A-Za-z0-9_]*)\s*\(", open(os.path.join(root, "include", "b200lz4.h")).read()))
    assert exported == declared, (sorted(exported - declared), sorted(declared - exported))
