#!/usr/bin/env python
"""bench.py — the measurement contract for the LZ4 block hot path on B200.

One "step" = one pass of the hot path over one batch of independent 64 KiB blocks:
fast-compress the whole batch, then fast-decompress it again (LZ4Factory.fastCompressor()
+ fastDecompressor(), BASELINE.json configs[1]).  `value` = uncompressed GiB processed per
second by that round trip, inputs resident in HBM, timed with CUDA events on the launching
stream, max over ranks.  Extra keys break the step into its compress and decompress halves,
give the compression ratio next to the reference's, the HBM roofline of the dominant kernel,
an end-to-end number through the C ABI with HOST buffers, and the reference's own CPU path
timed on this box's host cores.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                  [--blocks B]      # blocks per GPU (default 1048576 = BASELINE configs[1])
                  [--dump-outputs DIR]   # the last timed step's outputs as .npy, to compare two builds

Multi-GPU: one process per GPU (torchrun), contiguous block ranges per rank, no collective
on the data path (SURVEY.md §8e); only the timing is all-reduced (max) over ranks.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# the host-buffer pipeline runs 3 streams per calling thread; with the default 8 hardware queues two threads'
# H2D / kernel / D2H chains pick up false dependencies (measured: 172 vs 123 ms per overlapped call)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

try:
    FULL_AFFINITY = os.sched_getaffinity(0)          # before any rank pins itself to a NUMA node
except Exception:
    FULL_AFFINITY = None
BLOCK = 65536
METRIC = "lz4_fast_compress_plus_decompress_64KiB_blocks"
UNIT = "GiB/s"
GIB = float(1 << 30)


def env_int(name, default):
    return int(os.environ.get(name, default))


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            pass
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------ corpus
def host_corpus(chk, nblocks: int, seed: int = 2):
    """The reference's own synthetic generator (`lz4 -b` default: RDG_genBuffer P=0.50), cut at 64 KiB."""
    return chk.datagen(nblocks * BLOCK, 0.5, 0.0, seed)


def cpu_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_quota():
    for p in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            return open(p).read().strip()
        except Exception:
            pass
    return None


def quota_cpus():
    """CPUs the cgroup lets this container burn (cpu.max 'quota period'), or None when unlimited / unknown."""
    q = cpu_quota()
    try:
        a, b = q.split()[:2]
        return max(1, -(-int(a) // int(b)))
    except Exception:
        return None


def thread_candidates():
    """Thread counts tried for the CPU legs, so the reference gets its best operating point on this box: every
    hardware thread, one per physical core, and — where a cgroup quota is far below the visible CPUs (oversubscribed
    threads then lose time to CFS throttling) — the quota and twice the quota."""
    n = cpu_threads()
    c = {n, max(1, n // 2)}
    q = quota_cpus()
    if q and q < n:
        c |= {min(n, q), min(n, 2 * q)}
    return sorted(c, reverse=True)


def host_memory_budget():
    """bytes of host memory this container may still use: min(cgroup limit - usage, MemAvailable); None if unknown"""
    avail = None
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable:"):
                avail = int(line.split()[1]) * 1024
    except Exception:
        pass
    for lim_p, use_p in (("/sys/fs/cgroup/memory.max", "/sys/fs/cgroup/memory.current"),
                         ("/sys/fs/cgroup/memory/memory.limit_in_bytes", "/sys/fs/cgroup/memory/memory.usage_in_bytes")):
        try:
            lim = open(lim_p).read().strip()
            if lim != "max" and int(lim) < (1 << 60):
                room = int(lim) - int(open(use_p).read().strip())
                avail = room if avail is None else min(avail, room)
        except Exception:
            pass
    return avail


def cpu_roundtrip(chk, data, nblocks, threads, passes=3):
    """compress + fast-decompress `nblocks` blocks on `threads` host threads with the CPU library.
    Returns dict with GiB/s for each half, the round trip, and the ratio."""
    import numpy as np
    from oracle import oracle as O
    bound = chk.compress_bound(BLOCK)
    stride = (bound + 15) // 16 * 16
    soff = np.arange(nblocks, dtype=np.uint64) * np.uint64(BLOCK)
    slen = np.full(nblocks, BLOCK, dtype=np.int32)
    coff = np.arange(nblocks, dtype=np.uint64) * np.uint64(stride)
    ccap = np.full(nblocks, bound, dtype=np.int32)
    comp = np.empty(nblocks * stride, dtype=np.uint8)
    out = np.empty(nblocks * BLOCK, dtype=np.uint8)
    tc, tcm, clen = O.cpu_bench(chk, "compress", data, soff, slen, comp, coff, ccap, threads, passes)
    td, tdm, dres = O.cpu_bench(chk, "dec_fast", comp, coff, ccap, out, soff, slen, threads, passes)
    assert (dres == clen).all() and (out == data[: nblocks * BLOCK]).all(), "CPU round trip mismatch"
    nbytes = nblocks * BLOCK
    return {"compress_gibs": nbytes / tc / GIB, "decompress_gibs": nbytes / td / GIB,
            "roundtrip_gibs": nbytes / (tc + td) / GIB, "ratio": nbytes / float(clen.sum()),
            "t_compress_s": tc, "t_decompress_s": td}


# ------------------------------------------------------------------------------------------ reference arm
def run_reference(args):
    rank = env_int("RANK", 0)
    if rank != 0:
        return 0
    from oracle import oracle as O
    chk = O.best_available()
    nblocks = args.ref_blocks
    data = host_corpus(chk, nblocks)
    # pick the thread count that serves the reference best on this box (all SMT threads vs one per core)
    cands = thread_candidates()
    threads = max(cands, key=lambda t: cpu_roundtrip(chk, data, nblocks, t, passes=1)["roundtrip_gibs"])
    # W warm-up + K timed steps; each step = one bounded-sample round trip (best of 1 pass inside)
    for _ in range(args.warmup):
        cpu_roundtrip(chk, data, nblocks, threads, passes=1)
    t0 = time.perf_counter()
    rs = [cpu_roundtrip(chk, data, nblocks, threads, passes=1) for _ in range(args.steps)]
    wall = time.perf_counter() - t0
    tsum = sum(r["t_compress_s"] + r["t_decompress_s"] for r in rs)
    nbytes = nblocks * BLOCK
    value = nbytes * args.steps / tsum / GIB
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * tsum / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": f"{nblocks} x 64 KiB blocks (bounded sample of configs[1]), RDG_genBuffer P=0.50 seed=2, "
                               "LZ4_compress_default + LZ4_decompress_fast on host cores", "threads": threads, "cpu_quota": cpu_quota()},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": chk.kind,
                         "sample": f"{nblocks} blocks = {nbytes / GIB:.1f} GiB per step, {args.steps} steps",
                         "compress_gibs": sum(r["compress_gibs"] for r in rs) / len(rs),
                         "decompress_gibs": sum(r["decompress_gibs"] for r in rs) / len(rs),
                         "ratio": rs[0]["ratio"]},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "wall_s": wall,
    }
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------ NUMA
def numa_bind(local):
    """Pin this process (its pinned allocations follow by first touch) to the CPUs of the NUMA node GPU `local` hangs off.
    Round 1's 8-GPU end-to-end run scaled 0.355 with ranks floating over both sockets.  Best effort; returns what it did."""
    try:
        import torch
        bus = None
        try:
            import pynvml
            pynvml.nvmlInit()
            bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(local)).busId
            bus = bus.decode() if isinstance(bus, bytes) else bus
        except Exception:
            bus = subprocess.run(["nvidia-smi", f"--id={local}", "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                                 capture_output=True, text=True, timeout=20).stdout.strip()
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:                       # 00000000:1b:00.0 -> 0000:1b:00.0
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return {"gpu_pci": bus, "node": None, "note": "no NUMA node reported"}
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus |= set(range(int(a), int(b or a) + 1))
        mine = os.sched_getaffinity(0) & cpus
        if mine:
            os.sched_setaffinity(0, mine)
        return {"gpu_pci": bus, "node": node, "cpus": len(mine)}
    except Exception as e:          # noqa: BLE001
        return {"node": None, "note": f"not bound: {e}"}


def timed(fn, iters, warm, torch):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) / 1e3)
    return min(ts), sorted(ts)[len(ts) // 2]


def reduce_max(torch, dist, dev, world, *vals):
    t = torch.tensor(list(vals), device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(x) for x in t.tolist()]


# ------------------------------------------------------------------------------------------ secondary configs (BASELINE configs[2..4])
def run_config5(args, L, chk, torch, dist, dev, rank, world, local, peak):
    """configs[4]: XXH64 over 100 M x 4 KiB buffers on 8 B200 = 12.5 M buffers (51.2 GB) per GPU, weak scaling; seeds 0 and
    0x9747b28c (lz4-java's default, LZ4BlockOutputStream.java:56); xxhash.c:855-879, stripe loop :832-837"""
    n = args.xxh_buffers
    data = torch.empty(n * 4096, dtype=torch.uint8, device=dev)
    g = torch.Generator(device=dev); g.manual_seed(1234 + rank)
    base = torch.randint(0, 256, (1 << 28,), dtype=torch.uint8, device=dev, generator=g)
    for i in range(0, n * 4096, 1 << 28):
        data[i:i + (1 << 28)] = base[: min(1 << 28, n * 4096 - i)]
    idx = torch.arange(n, device=dev, dtype=torch.int64) + rank * n
    v = data.view(n, 4096)
    for k in range(8):
        v[:, k] ^= ((idx >> (8 * k)) & 0xFF).to(torch.uint8)     # every buffer distinct
    del base
    off = torch.arange(n, device=dev, dtype=torch.int64) * 4096
    ln = torch.full((n,), 4096, device=dev, dtype=torch.int32)
    o64 = torch.zeros(n, device=dev, dtype=torch.int64)
    o32 = torch.zeros(n, device=dev, dtype=torch.int32)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    if world > 1:
        dist.barrier()
    it = max(5, int(0.6 / max(n * 4104 / (peak * 1e9), 1e-4)))           # about 0.6 s per leg: the clock sampler needs that long
    t64, _ = timed(lambda: L.batch.xxh64_batch_dev(data, off, ln, o64, 0), it, 3, torch)
    t64b, _ = timed(lambda: L.batch.xxh64_batch_dev(data, off, ln, o64, 0x9747B28C), it, 1, torch)
    t32, _ = timed(lambda: L.batch.xxh32_batch_dev(data, off, ln, o32, 0x9747B28C), it, 1, torch)
    clocks = sampler.stop() if rank == 0 else None
    import random
    rng = random.Random(5 + rank)
    picks = [0, 1, n - 1] + [rng.randrange(n) for _ in range(253)]
    L.batch.xxh64_batch_dev(data, off, ln, o64, 0)
    for k in picks:                                                  # sampled _ref check, outside the timed region
        b = data[k * 4096:(k + 1) * 4096].cpu().numpy()
        if (int(o64[k].item()) & (2 ** 64 - 1)) != chk.xxh64(b, 0) or (int(o32[k].item()) & 0xFFFFFFFF) != chk.xxh32(b, 0x9747B28C):
            raise SystemExit("bench: config5 hash mismatch against the CPU checker")
    t64, t64b, t32 = reduce_max(torch, dist, dev, world, t64, t64b, t32)
    del data, v
    torch.cuda.empty_cache()
    by = n * (4096 + 8)
    return {"metric": "xxh64_4KiB_buffers", "value": by * world / t64 / 1e9, "unit": "GB/s",
            "workload": f"{n} x 4 KiB buffers per GPU (configs[4]: 100 M over 8 GPUs = 12.5 M per GPU), seed 0",
            "buffers_per_gpu": n, "seed_0x9747b28c_GBps": by * world / t64b / 1e9, "xxh32_GBps": n * 4100 * world / t32 / 1e9,
            "roofline": {"bound": "hbm", "kernel": "xxh_batch_kernel<64>", "achieved": by / t64 / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": by / t64 / 1e9 / peak, "algorithmic_bytes_per_launch": by, "note": "len + 8 per buffer; a read-only stream can exceed a copy-measured peak"},
            "clocks": clocks, "verified": "256 sampled buffers per GPU bit-exact vs the CPU checker (XXH64 seed 0, XXH32 seed 0x9747b28c)"}


def run_config3(args, L, chk, torch, dist, dev, rank, world, local, peak):
    """configs[2]: LZ4FrameInputStream decode (LZ4FrameInputStream.java:132-321; content checksum :264-273) of 16 GiB of
    4 MiB independent-block frames + XXH32 content checksum over 8 B200, sharded by FRAME = 32 frames of 64 MiB per GPU"""
    import numpy as np
    lib = L._native.lib()
    nframes, fsize = args.frames, 64 << 20
    ndistinct = min(4, nframes)                                      # 4 x 40 MiB of compressed frames cycle: larger than L2
    originals = [chk.datagen(fsize, 0.5, 0.0, 31 + 7 * rank + j) for j in range(ndistinct)]
    frames = [np.frombuffer(chk.frame_compress(o, 7, 1), dtype=np.uint8) for o in originals]      # bsID 7 = 4 MiB, content checksum
    host = np.concatenate([frames[i % ndistinct] for i in range(nframes)])
    slot = ctypes.c_uint64(); err = ctypes.c_int()
    index = lib.b200lz4f_index_create(host.ctypes.data, len(host), ctypes.byref(slot), ctypes.byref(err))
    if not index:
        raise SystemExit(f"bench: config3 index error {err.value}")
    d_src = torch.from_numpy(host).to(dev)
    d_slots = torch.empty(slot.value + 16, dtype=torch.uint8, device=dev)
    foff = np.zeros(nframes, dtype=np.uint64); flen = np.zeros(nframes, dtype=np.uint64)
    st = torch.cuda.current_stream().cuda_stream
    total = nframes * fsize

    def run():
        r = lib.b200lz4f_decode_dev(index, d_src.data_ptr(), d_slots.data_ptr(), foff.ctypes.data, flen.ctypes.data, None, st)
        if r != total:
            raise SystemExit(f"bench: config3 decode returned {r}")
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    if world > 1:
        dist.barrier()
    t, _ = timed(run, 5, 2, torch)
    clocks = sampler.stop() if rank == 0 else None
    for i in (0, 1, nframes - 1):                                    # decoded bytes against the original
        got = d_slots[int(foff[i]):int(foff[i]) + fsize]
        if not torch.equal(got.cpu(), torch.from_numpy(originals[i % ndistinct])):
            raise SystemExit("bench: config3 decoded bytes differ from the original")
    # end to end from (pinned) host memory through the one-call API
    pin_in = torch.from_numpy(host).pin_memory(); pin_out = torch.empty(total, dtype=torch.uint8).pin_memory()
    te = 1e30
    for _ in range(3):
        t1 = time.perf_counter()
        r = lib.b200lz4f_decompress_host(pin_in.data_ptr(), len(host), pin_out.data_ptr(), total)
        te = min(te, time.perf_counter() - t1)
    if r != total or not torch.equal(pin_out[:fsize], torch.from_numpy(originals[0])):
        raise SystemExit("bench: config3 host path mismatch")
    blocks = int(lib.b200lz4f_index_blocks(index))
    lib.b200lz4f_index_free(index)
    t, te = reduce_max(torch, dist, dev, world, t, te)
    csize = len(host)
    del d_src, d_slots, pin_in, pin_out
    torch.cuda.empty_cache()
    algo = csize + 2 * total                                         # C read, N written, N read again by the content hash
    return {"metric": "lz4_frame_decode_4MiB_blocks_content_xxh32", "value": total * world / t / GIB, "unit": "GiB/s",
            "workload": f"{nframes} frames x 64 MiB per GPU (configs[2]: 256 frames = 16 GiB over 8 GPUs, sharded by frame), "
                        "4 MiB independent blocks, content checksum, frames written by the reference's LZ4F_compressFrame, RDG P=0.50",
            "frames_per_gpu": nframes, "blocks_per_gpu": blocks, "e2e_host_GiBps": total * world / te / GIB,
            "roofline": {"bound": "hbm", "kernel": "lz4_decompress_safe_kernel + xxh32_long_kernel", "achieved": algo / t / 1e9, "peak": peak,
                         "unit": "GB/s", "frac": algo / t / 1e9 / peak, "algorithmic_bytes_per_launch": algo,
                         "note": "C + 2N: the content hash is a second pass over the decoded bytes; one warp per 4 MiB block and one per frame "
                                 "(XXH32 is four serial chains per stream) bound this far below HBM"},
            "clocks": clocks, "verified": "3 frames per GPU compared with the original bytes; header + content checksums verified on the device"}


def run_config4(args, L, chk, torch, dist, dev, rank, world, local, peak):
    """configs[3]: LZ4_compress_HC level 9 (lz4hc.c:958-973) over 256 K x 256 KiB blocks = 64 GiB on one B200, ratio next to
    the reference's on the same bytes.  The pass is sized to about a minute: the stated 262 144 blocks when the kernel's rate
    allows, else the largest power of two that fits (stated in `workload`)."""
    import numpy as np
    bs = 262144
    base_n = 256
    host = chk.datagen(base_n * bs, 0.5, 0.0, 4 + rank)
    base = torch.from_numpy(host).to(dev)
    bound = L.max_compressed_length(bs); stride = (bound + 15) // 16 * 16

    def arena(nblk):
        src = base.repeat((nblk + base_n - 1) // base_n)[: nblk * bs].contiguous() if nblk > base_n else base[: nblk * bs]
        soff = torch.arange(nblk, device=dev, dtype=torch.int64) * bs
        slen = torch.full((nblk,), bs, device=dev, dtype=torch.int32)
        return src, soff, slen
    # calibration on 2048 blocks (the compressed slots are reused modulo 4096 blocks: HC output is write-only here)
    nslots = 4096
    comp = torch.empty(nslots * stride, dtype=torch.uint8, device=dev)

    def hc(nblk, src, soff, slen, clen):
        for lo in range(0, nblk, nslots):
            m = min(nslots, nblk - lo)
            coff = torch.arange(m, device=dev, dtype=torch.int64) * stride
            ccap = torch.full((m,), bound, device=dev, dtype=torch.int32)
            L.batch.compress_hc_batch_dev(src, soff[lo:lo + m], slen[lo:lo + m], comp, coff, ccap, clen[lo:lo + m], 9)
    src, soff, slen = arena(2048)
    clen = torch.zeros(2048, device=dev, dtype=torch.int32)
    tcal, _ = timed(lambda: hc(2048, src, soff, slen, clen), 1, 1, torch)
    rate = 2048 * bs / tcal
    want = args.hc_blocks
    nblk = want
    while nblk > 2048 and nblk * bs / rate > args.hc_seconds:
        nblk //= 2
    if world > 1:
        nb = torch.tensor([nblk], device=dev, dtype=torch.int64); dist.all_reduce(nb, op=dist.ReduceOp.MIN); nblk = int(nb.item())
    # the 64 GiB source does not fit beside nothing else only because of tiling cost: index the 64 MiB base by offsets instead
    soff = (torch.arange(nblk, device=dev, dtype=torch.int64) % base_n) * bs
    slen = torch.full((nblk,), bs, device=dev, dtype=torch.int32)
    clen = torch.zeros(nblk, device=dev, dtype=torch.int32)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    if world > 1:
        dist.barrier()
    t, _ = timed(lambda: hc(nblk, base, soff, slen, clen), 1, 0, torch)
    clocks = sampler.stop() if rank == 0 else None
    csum = int(clen.sum().item())
    if not bool((clen > 0).all().item()):
        raise SystemExit("bench: config4 HC refused a block")
    # sampled _ref check: the last sub-batch's first blocks decode with the reference, ratio of the reference on the same bytes
    lo = (nblk - 1) // nslots * nslots
    for k in range(0, min(4, nblk - lo)):
        c = comp[k * stride: k * stride + int(clen[lo + k].item())].cpu().numpy()
        b = int(soff[lo + k].item())
        r, o = chk.decompress_safe(c, bs)
        if r != bs or o != host[b:b + bs].tobytes():
            raise SystemExit("bench: CPU checker rejects an HC block")
    ref_c = sum(len(chk.compress_hc(host[i * bs:(i + 1) * bs], 9)) for i in range(16)) if hasattr(chk, "compress_hc") else None
    ours16 = None
    if ref_c:
        c16 = torch.zeros(16, device=dev, dtype=torch.int32)
        hc(16, base, torch.arange(16, device=dev, dtype=torch.int64) * bs, slen[:16], c16)
        ours16 = 16 * bs / float(c16.sum().item())
    (t,) = reduce_max(torch, dist, dev, world, t)
    algo = nblk * bs + csum
    del comp, base
    torch.cuda.empty_cache()
    return {"metric": "lz4_hc9_compress_256KiB_blocks", "value": nblk * bs * world / t / GIB, "unit": "GiB/s",
            "workload": f"{nblk} x 256 KiB blocks per GPU (configs[3] states 262144 = 64 GiB on one GPU; "
                        f"{'stated size' if nblk == want else 'largest power of two within the time budget of %d s' % args.hc_seconds}), "
                        "LZ4_compress_HC level 9, RDG P=0.50, blocks addressed into a 64 MiB base corpus",
            "blocks_per_gpu": nblk, "ratio": nblk * bs / csum, "reference_hc9_ratio_first16": (16 * bs / ref_c) if ref_c else None,
            "ours_ratio_first16": ours16,
            "roofline": {"bound": "hbm", "kernel": "lz4hc_compress_kernel<11,32>", "achieved": algo / t / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": algo / t / 1e9 / peak, "algorithmic_bytes_per_launch": algo,
                         "note": "N + C; the kernel is latency-bound (one CTA per SM holds the 128 KiB candidate rings), the HBM fraction is tiny by construction"},
            "clocks": clocks, "verified": "4 blocks re-decoded by the CPU checker; ratio next to LZ4_compress_HC(9) on the same 16 blocks"}


def run_single_block(L, chk):
    """What a caller who only swaps the factory gets: ONE 64 KiB block per call through b200lz4_compress_default /
    b200lz4_decompress_safe / b200xxh64 (H2D + launch + D2H + sync each), next to the reference's own per-call time
    (net_jpountz_lz4_LZ4JNI.c:75,216; XXHashJNI.c)."""
    import numpy as np
    lib = L._native.lib()
    d = chk.datagen(BLOCK, 0.5, 0.0, 9)
    c_ref = chk.compress(d.tobytes())
    out = {}

    def worker(nthreads, iters):
        res = [None] * nthreads

        def body(i):
            src = d.copy(); bound = L.max_compressed_length(BLOCK)
            comp = np.zeros(bound, dtype=np.uint8); back = np.zeros(BLOCK, dtype=np.uint8)
            n = lib.b200lz4_compress_default(src.ctypes.data, comp.ctypes.data, BLOCK, bound)      # warm: context + staging
            assert n > 0
            t0 = time.perf_counter()
            for _ in range(iters):
                n = lib.b200lz4_compress_default(src.ctypes.data, comp.ctypes.data, BLOCK, bound)
            t1 = time.perf_counter()
            for _ in range(iters):
                r = lib.b200lz4_decompress_safe(comp.ctypes.data, back.ctypes.data, n, BLOCK)
            t2 = time.perf_counter()
            for _ in range(iters):
                h = lib.b200xxh64(src.ctypes.data, BLOCK, 0)
            t3 = time.perf_counter()
            assert r == BLOCK and (back == src).all() and (h & (2 ** 64 - 1)) == chk.xxh64(src, 0)
            res[i] = ((t1 - t0) / iters, (t2 - t1) / iters, (t3 - t2) / iters)
        ths = [threading.Thread(target=body, args=(i,)) for i in range(nthreads)]
        for t in ths: t.start()
        for t in ths: t.join()
        return [sum(r[k] for r in res) / nthreads * 1e6 for k in range(3)]
    for nt in (1, 16):
        us = worker(nt, 200 if nt == 1 else 60)
        out[f"threads_{nt}"] = {"compress_us_per_call": us[0], "decompress_safe_us_per_call": us[1], "xxh64_us_per_call": us[2],
                                "compress_calls_per_s": nt * 1e6 / us[0], "decompress_calls_per_s": nt * 1e6 / us[1]}
    # the reference's own functions, one thread, same block
    t0 = time.perf_counter()
    for _ in range(200):
        chk.compress(d.tobytes())
    tc = (time.perf_counter() - t0) / 200 * 1e6
    t0 = time.perf_counter()
    for _ in range(200):
        chk.decompress_safe(c_ref, BLOCK)
    td = (time.perf_counter() - t0) / 200 * 1e6
    out["reference_one_thread"] = {"compress_us_per_call": tc, "decompress_safe_us_per_call": td,
                                   "note": "through the Python checker binding (adds a few microseconds of its own)"}
    out["note"] = ("one 64 KiB block per call = H2D + launch + D2H + two syncs: tens of microseconds of fixed cost, slower than the CPU; "
                   "the batch entry points (LZ4B200Batch) are how the GPU pays off")
    return out


def run_e2e_multi(args, L, host, ngpus):
    """ONE process (the JVM's shape) drives all GPUs: b200lz4_compress_fast_compact_host_multi then
    b200lz4_decompress_fast_batch_host_multi over pinned host buffers, worker threads pinned to each GPU's NUMA node."""
    import numpy as np
    import torch
    B = L.batch
    n = min(args.e2e_blocks, args.blocks) * ngpus
    room = host_memory_budget()
    bound = L.max_compressed_length(BLOCK)
    if room is not None:
        fit = int(0.4 * room / (2 * BLOCK + bound + 16))
        if fit < n:
            n = max(4096 * ngpus, fit // (4096 * ngpus) * 4096 * ngpus)
    nbytes = n * BLOCK
    # Host buffers: plain pages, each GPU's share FIRST TOUCHED by a thread pinned to that GPU's NUMA node (the pages land
    # there), then registered with CUDA in one piece.  With every buffer on one socket the same call measured 37.8 GiB/s.
    stride = (bound + 15) // 16 * 16
    src = np.empty(nbytes, dtype=np.uint8); comp = np.empty(n * stride, dtype=np.uint8); out = np.empty(nbytes, dtype=np.uint8)
    keep = os.sched_getaffinity(0)
    if FULL_AFFINITY:
        os.sched_setaffinity(0, FULL_AFFINITY)         # this rank pinned itself to ITS GPU's node: the one-process leg spans all of them

    def touch(g):
        try:
            if FULL_AFFINITY:
                os.sched_setaffinity(0, FULL_AFFINITY)
            numa_bind(g)
        except Exception:
            pass
        lo, hi = n * g // ngpus, n * (g + 1) // ngpus
        for b in range(lo * BLOCK, hi * BLOCK, len(host)):
            e = min(hi * BLOCK, b + len(host)); src[b:e] = host[: e - b]
        out[lo * BLOCK:hi * BLOCK] = 0
        comp[lo * stride:hi * stride] = 0
    ths = [threading.Thread(target=touch, args=(g,)) for g in range(ngpus)]
    for t in ths: t.start()
    for t in ths: t.join()
    lib = L._native.lib()
    for a in (src, comp, out):
        L._native.check(lib.b200lz4_host_register(a.ctypes.data, a.nbytes))
    soff, slen = B.uniform_layout(n, BLOCK)
    devs = list(range(ngpus))
    best = 1e30
    for k in range(3):
        t0 = time.perf_counter()
        ooff, olen, shard_base, shard_total = B.compress_fast_compact_host_multi(src, soff, slen, comp, devs, BLOCK)
        res = B.decompress_fast_batch_host_multi(comp, ooff, olen, out, soff, slen, devs)
        dt = time.perf_counter() - t0
        if k:
            best = min(best, dt)
    assert (res == olen).all() and (out == src).all(), "e2e_multi round trip mismatch"
    for a in (src, comp, out):
        lib.b200lz4_host_unregister(a.ctypes.data)
    os.sched_setaffinity(0, keep)
    return {"value": nbytes / best / GIB, "unit": UNIT, "gpus": ngpus, "blocks": n,
            "sample": f"{n} blocks from ONE process over {ngpus} GPUs: b200lz4_compress_fast_compact_host_multi + "
                      "b200lz4_decompress_fast_batch_host_multi; host buffers first-touched per GPU on its NUMA node and registered "
                      "(cudaHostRegister), library workers pinned likewise; wall clock, best of 2 after a warm-up call"}


# ------------------------------------------------------------------------------------------ B200 arm
def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG", "WARN")          # keep NCCL's version banner off stdout (one JSON line)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = numa_bind(local) if not args.no_numa else {"node": None, "note": "--no-numa"}

    import lz4java_b200 as L
    from oracle import oracle as O
    lib = L._native.lib()
    L._native.check(lib.b200lz4_set_device(local))
    B = L.batch

    nblk = args.blocks                       # per GPU (weak scaling: every rank gets the same range size)
    nbytes = nblk * BLOCK
    bound = L.max_compressed_length(BLOCK)
    stride = (bound + 15) // 16 * 16        # 65 824: 16-byte aligned compressed slots (SURVEY.md §8d)

    # ---- corpus: 1 GiB of RDG P=0.50 (seed 2 + rank) on the host, uploaded once, tiled across HBM with a
    # per-block perturbation of the first 8 bytes so blocks are distinct (ratio unchanged)
    chk = O.best_available()
    base_blocks = min(nblk, 16384)
    host = host_corpus(chk, base_blocks, seed=2 + rank)
    base = torch.from_numpy(host).to(dev)
    src = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    reps = (nblk + base_blocks - 1) // base_blocks
    for r in range(reps):
        lo = r * base_blocks * BLOCK
        hi = min(nbytes, lo + base_blocks * BLOCK)
        src[lo:hi] = base[: hi - lo]
    idx = torch.arange(nblk, device=dev, dtype=torch.int64) + rank * nblk
    v = src.view(nblk, BLOCK)
    for k in range(8):
        v[:, k] ^= ((idx >> (8 * k)) & 0xFF).to(torch.uint8)
    del base, idx

    soff = torch.arange(nblk, device=dev, dtype=torch.int64) * BLOCK
    slen = torch.full((nblk,), BLOCK, device=dev, dtype=torch.int32)
    coff = torch.arange(nblk, device=dev, dtype=torch.int64) * stride
    ccap = torch.full((nblk,), bound, device=dev, dtype=torch.int32)
    comp = torch.empty(nblk * stride, dtype=torch.uint8, device=dev)
    clen = torch.zeros(nblk, device=dev, dtype=torch.int32)
    dres = torch.zeros(nblk, device=dev, dtype=torch.int32)
    h_before = torch.zeros(nblk, device=dev, dtype=torch.int64)
    h_after = torch.zeros(nblk, device=dev, dtype=torch.int64)
    B.xxh64_batch_dev(src, soff, slen, h_before, 0)        # checksum of every original block

    # decompression writes back into the source range: a correct round trip leaves it bit-identical,
    # which the checksum-of-checksums below proves; a third 64 GiB buffer would not fit next to
    # src + compressed slots in 180 GB.
    def step(ev=None):
        B.compress_fast_batch_dev(src, soff, slen, comp, coff, ccap, clen, BLOCK)
        if ev is not None:
            ev.record()
        B.decompress_fast_batch_dev(comp, coff, ccap, src, soff, slen, dres)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    lib.b200lz4_launch_count_reset()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    mids = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    e0.record()
    for k in range(args.steps):
        starts[k].record()
        step(mids[k])
    e1.record()
    barrier()
    launches = int(lib.b200lz4_launch_count())
    clocks = sampler.stop() if rank == 0 else None
    total_ms = e0.elapsed_time(e1)
    t_comp_ms = sum(starts[k].elapsed_time(mids[k]) for k in range(args.steps)) / args.steps
    t_step_ms = total_ms / args.steps
    t_dec_ms = t_step_ms - t_comp_ms

    # ---- correctness of what was timed (outside the timed region)
    csum = int(clen.sum().item())
    ok = bool((clen > 0).all().item()) and bool((dres == clen).all().item())
    B.xxh64_batch_dev(src, soff, slen, h_after, 0)
    ok = ok and bool(torch.equal(h_before, h_after))
    if not ok:
        raise SystemExit("bench: GPU round trip is not bit-exact — number invalid")
    # a sample of compressed blocks must decode with the CPU checker too
    for b in (0, nblk // 2, nblk - 1):
        c = comp[b * stride: b * stride + int(clen[b].item())].cpu().numpy()
        r, o = chk.decompress_safe(c, BLOCK)
        if r != BLOCK or o != src[b * BLOCK:(b + 1) * BLOCK].cpu().numpy().tobytes():
            raise SystemExit("bench: CPU checker rejects a GPU-compressed block")
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, "" if world == 1 else f"_rank{rank}", nblk, bound, stride, clen, dres, comp, src)

    # ---- max over ranks (device time)
    tt = torch.tensor([t_step_ms, t_comp_ms, t_dec_ms], device=dev, dtype=torch.float64)
    cs = torch.tensor([float(csum)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dist.all_reduce(cs, op=dist.ReduceOp.SUM)
    t_step_ms, t_comp_ms, t_dec_ms = (float(x) for x in tt.tolist())
    total_bytes = nbytes * world
    total_comp = float(cs.item())
    value = total_bytes / (t_step_ms / 1e3) / GIB

    # ---- end to end through the C ABI with HOST (pinned) buffers: H2D + kernels + D2H inside the timed region
    del src, comp, v
    torch.cuda.empty_cache()
    e2e = run_e2e(args, L, dev, host, rank, world)

    # ---- the in-process multi-GPU API (one JVM, all GPUs), the secondary configurations, the one-block latency
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    e2e_multi = None
    if world > 1 and not args.no_secondary:
        if rank == 0:
            try:
                e2e_multi = run_e2e_multi(args, L, host, world)
            except Exception as e:          # noqa: BLE001
                e2e_multi = {"error": str(e)[:300]}
        dist.barrier()
    # None of these may take the headline down with it: a leg that fails (its own checks raise SystemExit) is reported as
    # {"error": ...} under its key and the line is still printed.  The frame leg runs last: it is the only one with a second
    # kernel polling the first, so if anything can leave the context unusable it is that one.
    single = None
    if rank == 0 and not args.no_secondary and not args.only:
        try:
            single = run_single_block(L, chk)
        except (Exception, SystemExit) as e:        # noqa: BLE001
            single = {"error": str(e)[:300]}
    secondary = {}
    if not args.no_secondary:
        for key, fn in (("config5_xxh64", run_config5), ("config4_hc9", run_config4), ("config3_frame", run_config3)):
            if args.only and key.split("_")[0] not in args.only.split(","):
                continue
            try:
                secondary[key] = fn(args, L, chk, torch, dist, dev, rank, world, local, peak)
            except (Exception, SystemExit) as e:    # noqa: BLE001
                secondary[key] = {"error": str(e)[:300]}
                print(f"bench: {key} failed on rank {rank}: {e}", file=sys.stderr, flush=True)
            if isinstance(secondary[key], dict) and "error" in secondary[key]:
                try:
                    torch.cuda.empty_cache()        # (the failed leg's buffers went with its frames)
                except Exception:                   # noqa: BLE001
                    pass

    if rank == 0:
        peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if "hbm_gbs" in peaks else "6650 GB/s (of fallback)"
        algo_bytes = nbytes + csum                                  # N + C per compress launch (this rank)
        achieved = algo_bytes / (t_comp_ms / 1e3) / 1e9
        traffic = None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "compress_traffic.json")))
            if tj.get("blocks") == nblk and tj.get("kernel", "").startswith("lz4_compress_wide"):
                traffic = tj["dram_bytes_per_launch"]
        except Exception:
            pass
        cpu = None
        if world == 1 and not args.no_cpu:
            n_cpu = args.cpu_blocks
            cdata = host if base_blocks >= n_cpu else host_corpus(chk, n_cpu, seed=2)
            # all hardware threads, and one thread per physical core (SMT off-load): keep the better
            cands = thread_candidates()
            runs = [(cpu_roundtrip(chk, cdata, n_cpu, t, passes=3), t) for t in cands]
            r, threads = max(runs, key=lambda x: x[0]["roundtrip_gibs"])
            cpu = {"value": r["roundtrip_gibs"], "unit": UNIT, "cores": threads, "kind": chk.kind,
                   "tried_threads": {str(t): rr["roundtrip_gibs"] for rr, t in runs}, "cpu_quota": cpu_quota(),
                   "sample": f"{n_cpu} blocks = {n_cpu * BLOCK / GIB:.2f} GiB of the same corpus, best of 3 passes, "
                             f"{threads} pthreads, LZ4_compress_default + LZ4_decompress_fast",
                   "compress_gibs": r["compress_gibs"], "decompress_gibs": r["decompress_gibs"], "ratio": r["ratio"]}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": t_step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": {"workload": f"{nblk} x 64 KiB independent blocks per GPU (BASELINE configs[1]), "
                                   "fast compress + fast decompress, RDG_genBuffer P=0.50 tiled from 1 GiB",
                       "blocks_per_gpu": nblk, "block_bytes": BLOCK, "hash_log": 13, "numa": numa,
                       "l2": "inputs (64 GiB per GPU) larger than L2; no flush needed", "parallelism": f"range-shard x{world}"},
            "compress_gibs": total_bytes / (t_comp_ms / 1e3) / GIB,
            "decompress_gibs": total_bytes / (t_dec_ms / 1e3) / GIB,
            "ratio": total_bytes / total_comp,
            "roofline": {"bound": "hbm", "kernel": "lz4_compress_wide_kernel<13> (3 warps per block)", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "frac_of_nominal_8TBs": achieved / 8000.0,
                         "traffic": traffic, "algorithmic_bytes_per_launch": algo_bytes, "peak_source": peak_src,
                         "decompress_achieved": algo_bytes / (t_dec_ms / 1e3) / 1e9},
            "cpu_baseline": cpu, "e2e": e2e, "e2e_multi": e2e_multi, "gpu_launches": launches, "clocks": clocks,
            "config3_frame": secondary.get("config3_frame"), "config4_hc9": secondary.get("config4_hc9"),
            "config5_xxh64": secondary.get("config5_xxh64"), "single_block": single,
            "verified": "xxh64 of every block before == after all steps; 3 blocks re-decoded by the CPU checker",
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def dump_outputs(out_dir, suffix, nblk, bound, stride, clen, dres, comp, dec):
    """What the last timed step handed its caller, as float32 .npy files (every value is an integer below 2^24, so exact):
    the compressed length of every block, the decompressor's return value (bytes read) for every block, and for a fixed
    seeded sample of 64 blocks their compressed streams (zero past each stream's length, in slots of compressBound bytes)
    and their decompressed bytes.  About 42 MB at the default 1 M blocks."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    pick = np.sort(np.random.default_rng(0).choice(nblk, size=min(64, nblk), replace=False))
    lens = clen.cpu().numpy()
    streams = comp.view(nblk, stride)[pick, :bound].cpu().numpy().astype(np.float32)
    streams[np.arange(bound)[None, :] >= lens[pick][:, None]] = 0
    arrays = {"compressed_lengths": lens, "decompress_results": dres.cpu().numpy(), "sample_block_index": pick,
              "sample_compressed": streams, "sample_decompressed": dec.view(nblk, BLOCK)[pick].cpu().numpy()}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), a.astype(np.float32))


def run_e2e(args, L, dev, host, rank, world):
    """Same step through the public C-ABI batch calls with pinned HOST buffers (what a JNI caller with
    DirectByteBuffers does): b200lz4_compress_fast_compact_host then b200lz4_decompress_fast_batch_host.

    Two schedules are timed over the same K steps:
      * serial     — compress(k) then decompress(k), one host thread (each call alone is PCIe-bound in ONE direction);
      * pipelined  — two host threads (the library keeps streams/staging per thread): decompress(k) overlaps
                     compress(k+1), so both PCIe directions carry payload at once.  This is the reported `value`."""
    import queue
    import threading
    import numpy as np
    import torch
    import torch.distributed as dist
    B = L.batch
    n = min(args.e2e_blocks, args.blocks)
    bound = L.max_compressed_length(BLOCK)
    # the e2e leg pins 2 x 64 KiB + 2 x bound bytes of host memory per block and per rank: keep all ranks of this node
    # together under 40 % of what the container may still use (an 8-rank run must not drive the box out of memory)
    room = host_memory_budget()
    if room is not None:
        local_world = env_int("LOCAL_WORLD_SIZE", world)
        fit = int(0.4 * room / max(1, local_world) / (2 * BLOCK + 2 * bound))
        if fit < n:
            n = max(4096, fit // 4096 * 4096)
    if world > 1:                                   # every rank runs the same sample size
        nn = torch.tensor([n], device=dev, dtype=torch.int64)
        dist.all_reduce(nn, op=dist.ReduceOp.MIN)
        n = int(nn.item())
    nbytes = n * BLOCK
    src_t = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    comp_t = [torch.empty(n * bound, dtype=torch.uint8).pin_memory() for _ in range(2)]     # double-buffered between the threads
    out_t = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    src, comp, out = src_t.numpy(), [c.numpy() for c in comp_t], out_t.numpy()
    reps = (nbytes + len(host) - 1) // len(host)
    for r in range(reps):
        lo = r * len(host); hi = min(nbytes, lo + len(host))
        src[lo:hi] = host[: hi - lo]
    soff, slen = B.uniform_layout(n, BLOCK)
    lib = L._native.lib()
    local = int(os.environ.get("LOCAL_RANK", 0))

    def step_serial(k):
        ooff, olen, total = B.compress_fast_compact_host(src, soff, slen, comp[k & 1], BLOCK)
        res = B.decompress_fast_batch_host(comp[k & 1], ooff, olen, out, soff, slen)
        return olen, total, res

    for k in range(max(1, min(args.warmup, 2))):
        step_serial(k)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for k in range(args.steps):
        olen, total, res = step_serial(k)
    dt_serial = time.perf_counter() - t0
    assert (res == olen).all() and (out == src).all(), "e2e round trip mismatch"

    # pipelined: producer thread compresses step k into comp[k&1]; consumer decompresses it
    q_full, q_free = queue.Queue(), queue.Queue()
    q_free.put(0); q_free.put(1)
    state = {"err": None, "last": None}

    go = threading.Event(); ready = threading.Event()

    def producer():
        try:
            L._native.check(lib.b200lz4_set_device(local))
            B.compress_fast_compact_host(src, soff, slen, comp[0], BLOCK)    # untimed: this thread's streams + staging buffers
            ready.set(); go.wait()
            for k in range(args.steps):
                buf = q_free.get()
                ooff, olen, total = B.compress_fast_compact_host(src, soff, slen, comp[buf], BLOCK)
                q_full.put((buf, ooff, olen, total))
        except Exception as e:          # noqa: BLE001
            state["err"] = e
        q_full.put(None)

    th = threading.Thread(target=producer)
    th.start()
    ready.wait()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    go.set()
    while True:
        item = q_full.get()
        if item is None:
            break
        buf, ooff, olen, total = item
        res = B.decompress_fast_batch_host(comp[buf], ooff, olen, out, soff, slen)
        state["last"] = (olen, total, res)
        q_free.put(buf)
    th.join()
    dt_pipe = time.perf_counter() - t0
    if state["err"] is not None:
        raise state["err"]
    olen, total, res = state["last"]
    assert (res == olen).all() and (out == src).all(), "pipelined e2e round trip mismatch"

    t = torch.tensor([dt_pipe, dt_serial], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dt_pipe, dt_serial = (float(x) for x in t.tolist())
    per_step_h2d = nbytes + total + 2 * n * 28          # payload both ways + descriptors
    per_step_d2h = total + nbytes + 2 * n * 28
    return {"value": nbytes * world * args.steps / dt_pipe / GIB, "unit": UNIT,
            "h2d_bytes_per_step": int(per_step_h2d), "d2h_bytes_per_step": int(per_step_d2h),
            "serial_value": nbytes * world * args.steps / dt_serial / GIB,
            "sample": f"{n} blocks per GPU per step through b200lz4_compress_fast_compact_host + "
                      "b200lz4_decompress_fast_batch_host, pinned host buffers, wall clock (max over ranks); value = two host "
                      "threads (decompress of step k overlaps compress of step k+1), serial_value = one thread"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--blocks", type=int, default=1 << 20, help="blocks per GPU")
    ap.add_argument("--e2e-blocks", type=int, default=1 << 16, help="blocks per GPU per e2e step (4 GiB)")
    ap.add_argument("--cpu-blocks", type=int, default=1 << 14, help="blocks in the cpu_baseline sample (1 GiB)")
    ap.add_argument("--ref-blocks", type=int, default=1 << 15, help="blocks per step for --impl reference (2 GiB)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip configs[2..4], the one-block latency and the in-process multi-GPU leg")
    ap.add_argument("--only", default="", help="development: run only these secondary configs, e.g. config3,config5")
    ap.add_argument("--no-numa", action="store_true", help="do not pin the rank to its GPU's NUMA node")
    ap.add_argument("--xxh-buffers", type=int, default=12_500_000, help="config 5: 4 KiB buffers per GPU")
    ap.add_argument("--frames", type=int, default=32, help="config 3: 64 MiB frames per GPU")
    ap.add_argument("--hc-blocks", type=int, default=1 << 18, help="config 4: 256 KiB blocks per GPU")
    ap.add_argument("--hc-seconds", type=int, default=60, help="config 4: time budget of the timed pass")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the last timed step computed to DIR/<name>.npy (float32; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the outputs of --impl b200")
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
