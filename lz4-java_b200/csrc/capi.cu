// capi.cu — the C ABI of libb200lz4.so (include/b200lz4.h): device selection, per-thread
// streams and staging, the one-block-per-call entry points the JNI shim binds, and the batch
// entry points (device-resident and host-buffer, the latter as a 3-slot H2D / kernel / D2H
// pipeline).  No codec or hash arithmetic happens on the host: everything is a kernel launch.
#include "../../include/b200lz4.h"
#include "kernels.h"

#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>
#if defined(__linux__) && !defined(B200_HOST_SIM)
#include <sched.h>
#define B200_HAVE_AFFINITY 1
#endif

namespace b200 {

std::atomic<unsigned long long> g_launches{0};
static thread_local char tl_err[256] = "";
static thread_local int tl_status = 0;          // B200LZ4_E_* of the last value-returning call (hashes, digests) on this thread
static thread_local int tl_device = -1;          // -1: not chosen yet (defaults to device 0)

int fail_cuda(cudaError_t e, const char* where)
{
    snprintf(tl_err, sizeof tl_err, "%s: %s", where, cudaGetErrorString(e));
    if (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver || e == cudaErrorInitializationError)
        return tl_status = B200LZ4_E_NODEVICE;
    return tl_status = B200LZ4_E_CUDA;
}
int fail_arg(const char* what) { snprintf(tl_err, sizeof tl_err, "invalid argument: %s", what); return tl_status = B200LZ4_E_ARG; }

static int ensure_device()
{
    int cnt = 0;
    cudaError_t e = cudaGetDeviceCount(&cnt);
    if (e != cudaSuccess) return fail_cuda(e, "cudaGetDeviceCount");
    if (cnt <= 0) { snprintf(tl_err, sizeof tl_err, "no CUDA device"); return tl_status = B200LZ4_E_NODEVICE; }
    if (tl_device < 0) {
        // no b200lz4_set_device() on this thread yet: adopt the thread's CURRENT device (0 on a fresh thread) instead of
        // forcing device 0, so a caller that already selected a GPU (torch.cuda.set_device, cudaSetDevice) and hands
        // us device pointers / its stream does not find its current device switched under it
        int cur = 0;
        if (cudaGetDevice(&cur) != cudaSuccess || cur < 0 || cur >= cnt) cur = 0;
        tl_device = cur;
    }
    CK(cudaSetDevice(tl_device));
    return 0;
}

// ---------------------------------------------------------------------------------------------
// A buffer that grows on demand, in device or in pinned host memory.  The old buffer is freed before the new one is
// allocated.
enum Mem { DEVICE, PINNED };
struct Buf { uint8_t* p = nullptr; size_t cap = 0; };

static int grow(Buf& b, Mem mem, size_t need, size_t grown)
{
    if (need <= b.cap) return 0;
    if (b.p) CK(mem == PINNED ? cudaFreeHost(b.p) : cudaFree(b.p));
    b.p = nullptr; b.cap = 0;
    CK(mem == PINNED ? cudaHostAlloc(&b.p, grown, cudaHostAllocDefault) : cudaMalloc(&b.p, grown));
    b.cap = grown;
    return 0;
}
static size_t staging_size(size_t need) { return need + (need >> 2) + 4096; }

// A slot's descriptor arrays, [total | soff | doff | xoff] u64 then [slen | dcap | res] i32, in either copy (pinned or device).
struct Desc {
    uint64_t *total, *soff, *doff, *xoff;
    int32_t *slen, *dcap, *res;
    void* hash;                                        // per-buffer digests of a hash batch
};
static Desc desc_view(uint8_t* base, size_t nb)
{
    uint64_t* const u = (uint64_t*)base + 2;          // total and its pad take 16 bytes
    int32_t* const i = (int32_t*)(u + 3 * nb);
    return Desc{ (uint64_t*)base, u, u + nb, u + 2 * nb,
                 i, i + nb, i + 2 * nb,
                 u + nb };                             // hash: a hash batch has no dst slots, its digests take doff's place
}

// A pipeline slot: one stream, device staging for a chunk of blocks and pinned descriptor arrays.
struct Slot {
    cudaStream_t st = nullptr;
    cudaEvent_t done = nullptr;
    Buf src, dst;                                      // device
    Buf aux;                                           // device: compacted output (compact_host only)
    Buf out;                                           // pinned bounce for scattered dst slots
    bool scatter = false;                              // retire must copy out -> caller slots
    cudaEvent_t drained = nullptr; bool draining = false;
    Buf h_desc, d_desc; size_t desc_blocks = 0;        // descriptors: one pinned and one device copy
    size_t i0 = 0, i1 = 0;            // block range in flight
    bool busy = false;
    Desc host() const { return desc_view(h_desc.p, desc_blocks); }
    Desc dev() const { return desc_view(d_desc.p, desc_blocks); }
    static size_t desc_bytes(size_t nb) { return 16 + nb * (3 * 8 + 3 * 4); }
};

static constexpr int    NSLOTS = 3;
static size_t chunk_span_init() { const char* e = getenv("B200LZ4_CHUNK_MB"); size_t mb = e ? (size_t)atol(e) : 256; if (mb < 1) mb = 1; return mb << 20; }
static const size_t CHUNK_SPAN = chunk_span_init();    // bytes of src (and of dst) per pipeline chunk: >= 4096 64-KiB blocks,
                                                           // i.e. at least two full waves of warps on 148 SMs per launch
static constexpr size_t CHUNK_BLOCKS = 1 << 16;

struct Ctx {
    int device = -1;
    Slot slot[NSLOTS];
    ~Ctx() { /* process teardown frees device memory; explicit frees would race CUDA shutdown */ }
};

// Contexts (streams + staging) are owned by one thread at a time.  A thread keeps one per device it has used; when
// the thread exits they go to a process-wide idle pool and the next new thread on that device picks them up, so a
// server that churns threads (or a thread that alternates devices) does not grow device memory without bound.  No CUDA
// call happens at thread exit (nothing here can race the runtime's own teardown); the pool itself is never destroyed.
static std::atomic<int> g_contexts{0};
struct CtxPool { std::mutex mu; std::vector<Ctx*> idle; };
static CtxPool& ctx_pool() { static CtxPool* p = new CtxPool(); return *p; }
struct ThreadCtxs {
    std::vector<Ctx*> mine;
    ~ThreadCtxs()
    {
        if (mine.empty()) return;
        CtxPool& p = ctx_pool();
        std::lock_guard<std::mutex> g(p.mu);
        for (Ctx* c : mine) p.idle.push_back(c);
    }
};
static thread_local ThreadCtxs tl_ctxs;
static thread_local Ctx* tl_ctx = nullptr;          // the context of tl_device (cache of the lookup below)

static int get_ctx(Ctx** out)
{
    int rc = ensure_device();
    if (rc) return rc;
    if (tl_ctx && tl_ctx->device != tl_device) tl_ctx = nullptr;        // device switched on this thread
    if (!tl_ctx) {
        for (Ctx* c : tl_ctxs.mine) if (c->device == tl_device) { tl_ctx = c; break; }
    }
    if (!tl_ctx) {
        CtxPool& p = ctx_pool();
        std::lock_guard<std::mutex> g(p.mu);
        for (size_t k = 0; k < p.idle.size(); k++)
            if (p.idle[k]->device == tl_device) { tl_ctx = p.idle[k]; p.idle.erase(p.idle.begin() + (long)k); break; }
        if (tl_ctx) tl_ctxs.mine.push_back(tl_ctx);
    }
    if (!tl_ctx) {
        Ctx* c = new (std::nothrow) Ctx();
        if (!c) return fail_arg("out of host memory");
        c->device = tl_device;
        for (int s = 0; s < NSLOTS; s++) {
            cudaError_t e = cudaStreamCreateWithFlags(&c->slot[s].st, cudaStreamNonBlocking);
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->slot[s].done, cudaEventDisableTiming);
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->slot[s].drained, cudaEventDisableTiming);
            if (e != cudaSuccess) {
                for (int t = 0; t <= s; t++) {
                    if (c->slot[t].st) cudaStreamDestroy(c->slot[t].st);
                    if (c->slot[t].done) cudaEventDestroy(c->slot[t].done);
                    if (c->slot[t].drained) cudaEventDestroy(c->slot[t].drained);
                }
                delete c;
                return fail_cuda(e, "creating the pipeline streams");
            }
        }
        tl_ctxs.mine.push_back(c);
        tl_ctx = c;
        g_contexts.fetch_add(1, std::memory_order_relaxed);
    }
    *out = tl_ctx;
    return 0;
}

// A pipeline call that fails half way (a CUDA error, or an argument error found at a later chunk) must not leave
// chunks in flight: the next call on this thread would retire them into ITS result array with the old block indices.
// The guard waits for whatever was queued and clears the slots' bookkeeping unless the call ran to completion.
struct PipelineGuard {
    Ctx* c; bool completed = false;
    ~PipelineGuard()
    {
        if (completed) return;
        for (Slot& s : c->slot) {
            if (s.busy || s.draining) cudaStreamSynchronize(s.st);       // result of the wait is irrelevant here
            s.busy = false; s.draining = false; s.scatter = false;
        }
    }
};

static int slot_reserve(Slot& s, size_t src_bytes, size_t dst_bytes, size_t nblocks, size_t aux_bytes = 0)
{
    if (s.draining) { CK(cudaEventSynchronize(s.drained)); s.draining = false; }
    int rc = grow(s.aux, DEVICE, aux_bytes, staging_size(aux_bytes));
    if (!rc) rc = grow(s.src, DEVICE, src_bytes, staging_size(src_bytes));
    if (!rc) rc = grow(s.dst, DEVICE, dst_bytes, staging_size(dst_bytes));
    if (!rc && nblocks > s.desc_blocks) {
        const size_t nb = (nblocks + (nblocks >> 1) + 64 + 1) & ~size_t(1);    // even: keeps the i32 arrays 8-byte aligned
        s.desc_blocks = 0;
        rc = grow(s.d_desc, DEVICE, Slot::desc_bytes(nb), Slot::desc_bytes(nb));
        if (!rc) rc = grow(s.h_desc, PINNED, Slot::desc_bytes(nb), Slot::desc_bytes(nb));
        if (!rc) s.desc_blocks = nb;
    }
    return rc;
}

enum Op { OP_COMPRESS_FAST, OP_COMPRESS_HC, OP_DEC_SAFE, OP_DEC_FAST };

static cudaError_t launch_op(Op op, const BatchArgs& a, int param, cudaStream_t st)
{
    g_launches.fetch_add(1, std::memory_order_relaxed);
    switch (op) {
    case OP_COMPRESS_FAST: return launch_compress_fast(a, param, st);
    case OP_COMPRESS_HC:   return launch_compress_hc(a, param, st);
    case OP_DEC_SAFE:      return launch_decompress_safe(a, st);
    default:               return launch_decompress_fast(a, st);
    }
}

static uint64_t nonneg(int32_t v) { return v > 0 ? (uint64_t)v : 0; }

// A pipeline chunk: blocks [i0, i1), their source bytes [s_lo, s_hi) and destination slots [d_lo, d_hi).
struct Chunk {
    size_t i0, i1; uint64_t s_lo, s_hi, d_lo, d_hi;
    size_t nb() const { return i1 - i0; }
    size_t s_span() const { return (size_t)(s_hi - s_lo); }
    size_t d_span() const { return (size_t)(d_hi - d_lo); }
};

// Cuts the chunk that starts at block i0: one block at least, otherwise at most CHUNK_BLOCKS blocks and CHUNK_SPAN bytes of
// source and, when the blocks have destination slots (dst_off), of destination.  Blocks ascend in both, and destination
// slots do not overlap.  A negative length or capacity spans no bytes; the kernel reports it as that block's error.
static int cut_chunk(Chunk& ch, size_t i0, size_t n, const uint64_t* src_off, const int32_t* src_len,
                     const uint64_t* dst_off, const int32_t* dst_cap, const char* order_error)
{
    const uint64_t d0 = dst_off ? dst_off[i0] : 0;
    ch = Chunk{ i0, i0, src_off[i0], src_off[i0], d0, d0 };
    for (size_t i = i0; i < n && i - i0 < CHUNK_BLOCKS; i++) {
        if (src_off[i] < ch.s_lo || (dst_off && dst_off[i] < ch.d_hi)) return fail_arg(order_error);
        const uint64_t s_hi = std::max(ch.s_hi, src_off[i] + nonneg(src_len[i]));
        const uint64_t d_hi = dst_off ? std::max(ch.d_hi, dst_off[i] + nonneg(dst_cap[i])) : 0;
        if (i > i0 && (s_hi - ch.s_lo > CHUNK_SPAN || d_hi - ch.d_lo > CHUNK_SPAN)) break;
        ch.s_hi = s_hi; ch.d_hi = d_hi; ch.i1 = i + 1;
    }
    return 0;
}

// Writes the chunk's source descriptors and queues the descriptor and source copies; the caller has written its own
// descriptors.  The source keeps its 16-byte phase on the device, so aligned inputs stay aligned.
static int upload(Slot& s, const Chunk& ch, const uint8_t* src_base, const uint64_t* src_off, const int32_t* src_len)
{
    const size_t phase = (size_t)((uintptr_t)(src_base + ch.s_lo) & 15);
    const Desc h = s.host();
    for (size_t k = 0; k < ch.nb(); k++) {
        h.soff[k] = src_off[ch.i0 + k] - ch.s_lo + phase;
        h.slen[k] = src_len[ch.i0 + k];
    }
    CK(cudaMemcpyAsync(s.d_desc.p, s.h_desc.p, Slot::desc_bytes(s.desc_blocks), cudaMemcpyHostToDevice, s.st));
    if (ch.s_span()) CK(cudaMemcpyAsync(s.src.p + phase, src_base + ch.s_lo, ch.s_span(), cudaMemcpyHostToDevice, s.st));
    return 0;
}

// The 3-slot H2D / kernel / D2H pipeline under every host-buffer batch.  Chunks go round the slots.  Before a slot takes a
// chunk, the one it holds is finished: wait for its `done`, then retire(s) hands its results to the caller.  stage(s, ch)
// reserves staging and queues the chunk's copies and launches on s.st.  At the end every slot is finished and every
// `drained` copy (started by a retire) awaited.  A call that fails half way drains what it queued (PipelineGuard).
template <class Stage, class Retire>
static int run_pipeline(size_t n, const uint64_t* src_off, const int32_t* src_len, const uint64_t* dst_off,
                        const int32_t* dst_cap, const char* order_error, Stage stage, Retire retire)
{
    Ctx* c; int rc = get_ctx(&c); if (rc) return rc;
    PipelineGuard guard{ c };
    auto finish = [&](Slot& s) -> int {
        if (!s.busy) return 0;
        CK(cudaEventSynchronize(s.done));
        const int r = retire(s); if (r) return r;
        s.busy = false;
        return 0;
    };
    int cur = 0;
    for (size_t i0 = 0; i0 < n; cur = (cur + 1) % NSLOTS) {
        Chunk ch;
        rc = cut_chunk(ch, i0, n, src_off, src_len, dst_off, dst_cap, order_error); if (rc) return rc;
        Slot& s = c->slot[cur];
        rc = finish(s); if (rc) return rc;
        rc = stage(s, ch); if (rc) return rc;
        CK(cudaEventRecord(s.done, s.st));
        s.busy = true; s.i0 = ch.i0; s.i1 = ch.i1;
        i0 = ch.i1;
    }
    for (int k = 0; k < NSLOTS; k++) { rc = finish(c->slot[(cur + k) % NSLOTS]); if (rc) return rc; }
    for (Slot& s : c->slot) if (s.draining) { CK(cudaEventSynchronize(s.drained)); s.draining = false; }
    guard.completed = true;
    return 0;
}

// Host-buffer batch of one codec op.  Blocks ascend in src and dst.
static int host_batch(Op op, const uint8_t* src_base, const uint64_t* src_off, const int32_t* src_len,
                      uint8_t* dst_base, const uint64_t* dst_off, const int32_t* dst_cap,
                      int32_t* result, size_t n, int param)
{
    if (n == 0) return 0;
    if (!src_base || !src_off || !src_len || !dst_base || !dst_off || !dst_cap || !result) return fail_arg("null pointer");
    auto stage = [&](Slot& s, const Chunk& ch) -> int {
        const size_t nb = ch.nb(), d_span = ch.d_span();
        int rc = slot_reserve(s, ch.s_span() + 16, d_span + 16, nb); if (rc) return rc;
        const size_t d_phase = (size_t)((uintptr_t)(dst_base + ch.d_lo) & 15);
        const Desc h = s.host(), d = s.dev();
        for (size_t k = 0; k < nb; k++) {
            h.doff[k] = dst_off[ch.i0 + k] - ch.d_lo + d_phase;
            h.dcap[k] = dst_cap[ch.i0 + k];
        }
        rc = upload(s, ch, src_base, src_off, src_len); if (rc) return rc;
        BatchArgs a{ s.src.p, d.soff, d.slen, s.dst.p, d.doff, d.dcap, d.res, nb };
        CK(launch_op(op, a, param, s.st));
        CK(cudaMemcpyAsync(h.res, d.res, nb * sizeof(int32_t), cudaMemcpyDeviceToHost, s.st));
        if (!d_span) return 0;
        if (n == 1) {
            // one block per call (the JNI shim's shape): the caller's bytes behind the result stay untouched, like in the
            // reference (a decoder called with maxDestLen = "rest of my buffer" must not clobber what lies further along),
            // and no stale staging bytes of another call leave the device.  Costs one more round trip of a few bytes.
            CK(cudaStreamSynchronize(s.st));
            const int32_t r = h.res[0];
            const size_t produced = op == OP_DEC_FAST ? (r >= 0 ? d_span : 0) : (size_t)(r > 0 ? r : 0);
            if (produced) CK(cudaMemcpyAsync(dst_base + ch.d_lo, s.dst.p + d_phase, std::min(produced, d_span), cudaMemcpyDeviceToHost, s.st));
            return 0;
        }
        // when the dst slots are back to back (the normal layout) one DMA lands straight in the caller's memory; otherwise
        // the span goes to a pinned bounce buffer and retire scatters the slots, so caller bytes BETWEEN non-adjacent slots
        // are never touched
        bool contiguous = true;
        uint64_t end = ch.d_lo;
        for (size_t i = ch.i0; i < ch.i1 && contiguous; i++) {
            contiguous = dst_off[i] == end;
            end = dst_off[i] + nonneg(dst_cap[i]);
        }
        if (contiguous) {
            CK(cudaMemcpyAsync(dst_base + ch.d_lo, s.dst.p + d_phase, d_span, cudaMemcpyDeviceToHost, s.st));
        } else {
            rc = grow(s.out, PINNED, d_span, staging_size(d_span)); if (rc) return rc;
            CK(cudaMemcpyAsync(s.out.p, s.dst.p + d_phase, d_span, cudaMemcpyDeviceToHost, s.st));
            s.scatter = true;
        }
        return 0;
    };
    auto retire = [&](Slot& s) -> int {
        memcpy(result + s.i0, s.host().res, (s.i1 - s.i0) * sizeof(int32_t));
        if (s.scatter) {
            const uint64_t d_lo = dst_off[s.i0];
            for (size_t k = s.i0; k < s.i1; k++)
                if (dst_cap[k] > 0) memcpy(dst_base + dst_off[k], s.out.p + (dst_off[k] - d_lo), (size_t)dst_cap[k]);
        }
        s.scatter = false;
        return 0;
    };
    return run_pipeline(n, src_off, src_len, dst_off, dst_cap, "blocks must ascend and not overlap in dst", stage, retire);
}

template <typename W>
static int hash_host_batch(const uint8_t* base, const uint64_t* off, const int32_t* len, uint64_t seed,
                           W* out, size_t n)
{
    if (n == 0) return 0;
    if (!base || !off || !len || !out) return fail_arg("null pointer");
    auto stage = [&](Slot& s, const Chunk& ch) -> int {
        const size_t nb = ch.nb(), span = ch.s_span();
        int rc = slot_reserve(s, span + 16, 16, nb); if (rc) return rc;
        rc = upload(s, ch, base, off, len); if (rc) return rc;
        const Desc d = s.dev();
        const bool long_bufs = span / nb >= XXH_LONG_AVG;
        g_launches.fetch_add(1, std::memory_order_relaxed);
        if (sizeof(W) == 4) CK((long_bufs ? launch_xxh32_long : launch_xxh32)(s.src.p, d.soff, d.slen, (uint32_t)seed, (uint32_t*)d.hash, nb, s.st));
        else                CK((long_bufs ? launch_xxh64_long : launch_xxh64)(s.src.p, d.soff, d.slen, seed, (uint64_t*)d.hash, nb, s.st));
        CK(cudaMemcpyAsync(s.host().hash, d.hash, nb * sizeof(W), cudaMemcpyDeviceToHost, s.st));
        return 0;
    };
    auto retire = [&](Slot& s) -> int { memcpy(out + s.i0, s.host().hash, (s.i1 - s.i0) * sizeof(W)); return 0; };
    return run_pipeline(n, off, len, nullptr, nullptr, "buffers must ascend", stage, retire);
}

// one block, host buffers: the n = 1 case of the host batch path
static int one_block(Op op, const char* src, int src_len, char* dst, int dst_cap, int param)
{
    const uint64_t zero = 0;
    int32_t res = 0;
    static const char dummy = 0;
    if (!src) src = &dummy;
    char local_dst = 0;
    if (!dst) { dst = &local_dst; if (dst_cap > 0) return fail_arg("dst is NULL"); }
    int rc = host_batch(op, (const uint8_t*)src, &zero, &src_len, (uint8_t*)dst, &zero, &dst_cap, &res, 1, param);
    if (rc) return rc;
    return res;
}

// one buffer, host memory: the n = 1 case of the host hash batch
template <typename W>
static W one_hash(const void* input, size_t len, uint64_t seed)
{
    const uint64_t zero = 0; int32_t l = (int32_t)len; W out = 0; static const char dummy = 0;
    tl_status = 0;
    if (len > 0x7FFFFFFFu) { fail_arg("len > 2^31-1"); return 0; }
    if (hash_host_batch<W>((const uint8_t*)(input ? input : &dummy), &zero, &l, seed, &out, 1)) return 0;
    return out;
}

// Pin the calling WORKER thread to the CPUs of the NUMA node its GPU hangs off (sysfs: the PCI device's numa_node and the
// node's cpulist).  Staging and descriptor buffers a worker allocates then land on that node (first touch), and its DMA
// descriptors are written by a core next to the root complex.  Round 1's 8-GPU end-to-end run scaled 0.355 with every
// thread floating over both sockets.  Best effort: any failure leaves the thread where it was.
static void bind_worker_to_device_node(int device)
{
#ifdef B200_HAVE_AFFINITY
    char bus[32] = "";
    if (cudaDeviceGetPCIBusId(bus, sizeof bus, device) != cudaSuccess) return;
    for (char* q = bus; *q; q++) if (*q >= 'A' && *q <= 'Z') *q = char(*q - 'A' + 'a');
    char path[160];
    snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/numa_node", bus);
    FILE* f = fopen(path, "r"); if (!f) return;
    int node = -1; const int got = fscanf(f, "%d", &node); fclose(f);
    if (got != 1 || node < 0) return;
    snprintf(path, sizeof path, "/sys/devices/system/node/node%d/cpulist", node);
    f = fopen(path, "r"); if (!f) return;
    char list[1024] = ""; const bool ok = fgets(list, sizeof list, f) != nullptr; fclose(f);
    if (!ok) return;
    cpu_set_t want; CPU_ZERO(&want);
    for (char* q = list; *q; ) {                                   // "0-31,64-95"
        char* e; const long a = strtol(q, &e, 10); if (e == q) break;
        long b = a; q = e;
        if (*q == '-') { b = strtol(q + 1, &e, 10); q = e; }
        for (long c = a; c <= b && c < CPU_SETSIZE; c++) CPU_SET((int)c, &want);
        if (*q == ',') q++; else break;
    }
    cpu_set_t cur;
    if (sched_getaffinity(0, sizeof cur, &cur) != 0) return;
    cpu_set_t both; CPU_AND(&both, &cur, &want);                   // never widen what the process was given (cgroups, taskset)
    if (CPU_COUNT(&both) > 0) sched_setaffinity(0, sizeof both, &both);
#else
    (void)device;
#endif
}

// ---- one process, several GPUs: contiguous block ranges, one worker thread (own device, own context) per GPU
template <class ShardFn>
static int run_sharded(size_t n, const int* devices, int ndev, ShardFn shard)
{
    if (ndev < 1 || ndev > 64) return fail_arg("ndev must be 1..64");
    int cnt = b200lz4_device_count();
    if (cnt < 0) return cnt;
    for (int g = 0; g < ndev; g++) {
        const int d = devices ? devices[g] : g;
        if (d < 0 || d >= cnt) return fail_arg("device index in devices[]");
    }
    std::vector<int> rc((size_t)ndev, 0);
    std::vector<std::string> msg((size_t)ndev);
    std::vector<std::thread> th;
    auto body = [&](int g) {
        const size_t lo = n * (size_t)g / (size_t)ndev, hi = n * (size_t)(g + 1) / (size_t)ndev;
        if (hi == lo) return;
        int r = b200lz4_set_device(devices ? devices[g] : g);       // thread-local: this worker's device
        if (r == 0 && g > 0) bind_worker_to_device_node(devices ? devices[g] : g);      // (shard 0 runs on the caller's thread: its affinity is the caller's business)
        if (r == 0) r = shard(lo, hi - lo);
        rc[(size_t)g] = r;
        if (r) msg[(size_t)g] = tl_err;
    };
    try {
        for (int g = 1; g < ndev; g++) th.emplace_back(body, g);
    } catch (...) {
        for (auto& t : th) t.join();
        return fail_arg("cannot start a worker thread");
    }
    const int my_device = tl_device;
    int my_cuda_device = -1;
    if (cudaGetDevice(&my_cuda_device) != cudaSuccess) my_cuda_device = -1;
    body(0);                                                        // shard 0 runs on the calling thread
    for (auto& t : th) t.join();
    tl_device = my_device;                                          // the caller keeps its device, in the library and in CUDA
    if (my_cuda_device >= 0) cudaSetDevice(my_cuda_device);
    for (int g = 0; g < ndev; g++)
        if (rc[(size_t)g]) {
            snprintf(tl_err, sizeof tl_err, "device %d: %s", devices ? devices[g] : g, msg[(size_t)g].c_str());
            return tl_status = rc[(size_t)g];
        }
    return 0;
}

static int multi_host_batch(Op op, const uint8_t* src_base, const uint64_t* src_off, const int32_t* src_len,
                            uint8_t* dst_base, const uint64_t* dst_off, const int32_t* dst_cap,
                            int32_t* result, size_t n, int param, const int* devices, int ndev)
{
    if (n == 0) return 0;
    if (!src_base || !src_off || !src_len || !dst_base || !dst_off || !dst_cap || !result) return fail_arg("null pointer");
    return run_sharded(n, devices, ndev, [&](size_t lo, size_t cnt) {
        return host_batch(op, src_base, src_off + lo, src_len + lo, dst_base, dst_off + lo, dst_cap + lo, result + lo, cnt, param);
    });
}

} // namespace b200

using namespace b200;

extern "C" {

int b200lz4_version(void) { return B200LZ4_VERSION; }

int b200lz4_device_count(void)
{
    int cnt = 0;
    cudaError_t e = cudaGetDeviceCount(&cnt);
    if (e != cudaSuccess) return fail_cuda(e, "cudaGetDeviceCount");
    return cnt;
}

int b200lz4_set_device(int device)
{
    int cnt = b200lz4_device_count();
    if (cnt < 0) return cnt;
    if (device < 0 || device >= cnt) return fail_arg("device index");
    tl_device = device;
    CK(cudaSetDevice(device));
    return 0;
}

const char* b200lz4_last_error(void) { return tl_err; }
int b200lz4_last_status(void) { return tl_status; }

int b200lz4_host_register(void* p, size_t bytes)
{
    int rc = ensure_device(); if (rc) return rc;
    CK(cudaHostRegister(p, bytes, cudaHostRegisterPortable));
    return 0;
}
int b200lz4_host_unregister(void* p)
{
    int rc = ensure_device(); if (rc) return rc;
    CK(cudaHostUnregister(p));
    return 0;
}

int b200lz4_compressBound(int n)
{   // pure size arithmetic (lz4.h:212); LZ4Utils.maxCompressedLength must equal it (LZ4Test.java:80-87)
    return ((unsigned)n > 0x7E000000u) ? 0 : n + n / 255 + 16;
}

int b200lz4_compress_default(const char* src, char* dst, int srcSize, int dstCapacity)
{
    if (srcSize < 0 || (unsigned)srcSize > 0x7E000000u || dstCapacity < 0) return 0;  // lz4.c:1324; no room at all
    return one_block(OP_COMPRESS_FAST, src, srcSize, dst, dstCapacity, srcSize <= 65536 ? 65536 : 0);
}
int b200lz4_compress_HC(const char* src, char* dst, int srcSize, int dstCapacity, int level)
{
    if (srcSize < 0 || (unsigned)srcSize > 0x7E000000u || dstCapacity < 0) return 0;
    return one_block(OP_COMPRESS_HC, src, srcSize, dst, dstCapacity, level);
}
int b200lz4_decompress_safe(const char* src, char* dst, int compressedSize, int dstCapacity)
{
    if (!src || dstCapacity < 0) return -1;                                           // lz4.c:1953
    if (compressedSize < 0) return -1;
    return one_block(OP_DEC_SAFE, src, compressedSize, dst, dstCapacity, 0);
}
int b200lz4_decompress_fast_bounded(const char* src, int srcAvail, char* dst, int originalSize)
{
    if (!src || originalSize < 0 || srcAvail < 0) return -1;
    return one_block(OP_DEC_FAST, src, srcAvail, dst, originalSize, 0);
}

uint32_t b200xxh32(const void* input, size_t len, uint32_t seed) { return one_hash<uint32_t>(input, len, seed); }
uint64_t b200xxh64(const void* input, size_t len, uint64_t seed) { return one_hash<uint64_t>(input, len, seed); }

// ---- streaming state: device-resident struct + a pinned staging area, one stream per handle
struct StreamHandle {
    int bits; int device; void* d_state; Buf buf; cudaStream_t st; void* h_out;
};
static void* stream_create(int bits, uint64_t seed)
{
    if (ensure_device()) return nullptr;
    StreamHandle* h = new (std::nothrow) StreamHandle();
    if (!h) return nullptr;
    h->bits = bits; h->device = tl_device;
    if (cudaStreamCreateWithFlags(&h->st, cudaStreamNonBlocking) != cudaSuccess ||
        cudaMalloc(&h->d_state, bits == 32 ? sizeof(Xxh32State) : sizeof(Xxh64State)) != cudaSuccess ||
        cudaHostAlloc(&h->h_out, 8, cudaHostAllocDefault) != cudaSuccess) { fail_cuda(cudaGetLastError(), "stream_create"); delete h; return nullptr; }
    g_launches.fetch_add(1, std::memory_order_relaxed);
    if (bits == 32) launch_xxh32_stream((Xxh32State*)h->d_state, XXH_OP_RESET, (uint32_t)seed, nullptr, 0, h->st);
    else            launch_xxh64_stream((Xxh64State*)h->d_state, XXH_OP_RESET, seed, nullptr, 0, h->st);
    return h;
}
static void stream_reset(void* hv, uint64_t seed)
{
    StreamHandle* h = (StreamHandle*)hv; if (!h) return;
    cudaSetDevice(h->device);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    if (h->bits == 32) launch_xxh32_stream((Xxh32State*)h->d_state, XXH_OP_RESET, (uint32_t)seed, nullptr, 0, h->st);
    else               launch_xxh64_stream((Xxh64State*)h->d_state, XXH_OP_RESET, seed, nullptr, 0, h->st);
}
static int stream_update(void* hv, const void* input, size_t len)
{
    StreamHandle* h = (StreamHandle*)hv; if (!h) return fail_arg("null state");
    if (len == 0) return 0;
    CK(cudaSetDevice(h->device));
    if (len > h->buf.cap) {
        CK(cudaStreamSynchronize(h->st));
        const int rc = grow(h->buf, DEVICE, len, len + (len >> 1) + 4096); if (rc) return rc;
    }
    CK(cudaMemcpyAsync(h->buf.p, input, len, cudaMemcpyHostToDevice, h->st));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    if (h->bits == 32) CK(launch_xxh32_stream((Xxh32State*)h->d_state, XXH_OP_UPDATE, 0, h->buf.p, len, h->st));
    else               CK(launch_xxh64_stream((Xxh64State*)h->d_state, XXH_OP_UPDATE, 0, h->buf.p, len, h->st));
    CK(cudaStreamSynchronize(h->st));          // the caller may reuse `input` as soon as we return
    return 0;
}
static uint64_t stream_digest(void* hv)
{
    tl_status = 0;
    StreamHandle* h = (StreamHandle*)hv; if (!h) { fail_arg("null state"); return 0; }
    cudaSetDevice(h->device);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    if (h->bits == 32) {
        launch_xxh32_stream((Xxh32State*)h->d_state, XXH_OP_DIGEST, 0, nullptr, 0, h->st);
        cudaMemcpyAsync(h->h_out, &((Xxh32State*)h->d_state)->digest, 4, cudaMemcpyDeviceToHost, h->st);
    } else {
        launch_xxh64_stream((Xxh64State*)h->d_state, XXH_OP_DIGEST, 0, nullptr, 0, h->st);
        cudaMemcpyAsync(h->h_out, &((Xxh64State*)h->d_state)->digest, 8, cudaMemcpyDeviceToHost, h->st);
    }
    cudaError_t e = cudaStreamSynchronize(h->st);
    if (e != cudaSuccess) { fail_cuda(e, "stream_digest"); return 0; }
    return h->bits == 32 ? (uint64_t)*(uint32_t*)h->h_out : *(uint64_t*)h->h_out;
}
static void stream_free(void* hv)
{
    StreamHandle* h = (StreamHandle*)hv; if (!h) return;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->st);
    cudaFree(h->d_state); if (h->buf.p) cudaFree(h->buf.p); cudaFreeHost(h->h_out); cudaStreamDestroy(h->st);
    delete h;
}

void*    b200xxh32_create(uint32_t seed) { return stream_create(32, seed); }
void     b200xxh32_reset(void* s, uint32_t seed) { stream_reset(s, seed); }
int      b200xxh32_update(void* s, const void* in, size_t len) { return stream_update(s, in, len); }
uint32_t b200xxh32_digest(void* s) { return (uint32_t)stream_digest(s); }
void     b200xxh32_free(void* s) { stream_free(s); }
void*    b200xxh64_create(uint64_t seed) { return stream_create(64, seed); }
void     b200xxh64_reset(void* s, uint64_t seed) { stream_reset(s, seed); }
int      b200xxh64_update(void* s, const void* in, size_t len) { return stream_update(s, in, len); }
uint64_t b200xxh64_digest(void* s) { return stream_digest(s); }
void     b200xxh64_free(void* s) { stream_free(s); }

// ---- device-resident batches
#define DEV_BATCH(OP, PARAM) \
    int rc = ensure_device(); if (rc) return rc; \
    if (n > 0xFFFFFFFFull) return fail_arg("n"); \
    BatchArgs a{ src_base, src_off, src_len, dst_base, dst_off, dst_cap, result, n }; \
    CK(launch_op(OP, a, PARAM, (cudaStream_t)stream)); \
    return 0;

int b200lz4_compress_fast_batch_dev(const uint8_t* src_base, const uint64_t* src_off, const int32_t* src_len,
                                    uint8_t* dst_base, const uint64_t* dst_off, const int32_t* dst_cap,
                                    int32_t* result, size_t n, int max_src_len, void* stream)
{ DEV_BATCH(OP_COMPRESS_FAST, max_src_len) }
int b200lz4_compress_hc_batch_dev(const uint8_t* src_base, const uint64_t* src_off, const int32_t* src_len,
                                  uint8_t* dst_base, const uint64_t* dst_off, const int32_t* dst_cap,
                                  int32_t* result, size_t n, int level, void* stream)
{ DEV_BATCH(OP_COMPRESS_HC, level) }
int b200lz4_decompress_safe_batch_dev(const uint8_t* src_base, const uint64_t* src_off, const int32_t* src_len,
                                      uint8_t* dst_base, const uint64_t* dst_off, const int32_t* dst_cap,
                                      int32_t* result, size_t n, void* stream)
{ DEV_BATCH(OP_DEC_SAFE, 0) }
int b200lz4_decompress_fast_batch_dev(const uint8_t* src_base, const uint64_t* src_off, const int32_t* src_len,
                                      uint8_t* dst_base, const uint64_t* dst_off, const int32_t* dst_cap,
                                      int32_t* result, size_t n, void* stream)
{ DEV_BATCH(OP_DEC_FAST, 0) }

int b200xxh32_batch_dev(const uint8_t* base, const uint64_t* off, const int32_t* len, uint32_t seed, uint32_t* out, size_t n, void* stream)
{
    int rc = ensure_device(); if (rc) return rc;
    g_launches.fetch_add(1, std::memory_order_relaxed);
    CK(launch_xxh32(base, off, len, seed, out, n, (cudaStream_t)stream));
    return 0;
}
int b200xxh64_batch_dev(const uint8_t* base, const uint64_t* off, const int32_t* len, uint64_t seed, uint64_t* out, size_t n, void* stream)
{
    int rc = ensure_device(); if (rc) return rc;
    g_launches.fetch_add(1, std::memory_order_relaxed);
    CK(launch_xxh64(base, off, len, seed, out, n, (cudaStream_t)stream));
    return 0;
}

// ---- device-resident packing and the cross-GPU stitch (SURVEY.md 8e "optional next", (f)-4)
int b200lz4_compact_dev(const uint8_t* slots, const uint64_t* slot_off, const int32_t* lens, uint8_t* out, uint64_t* out_off,
                        uint64_t* total, size_t n, void* stream)
{
    int rc = ensure_device(); if (rc) return rc;
    if (n > 0xFFFFFFFFull) return fail_arg("n");
    if (!total || (n && (!slots || !slot_off || !lens || !out || !out_off))) return fail_arg("null pointer");
    if (n == 0) { CK(cudaMemsetAsync(total, 0, sizeof(uint64_t), (cudaStream_t)stream)); return 0; }
    g_launches.fetch_add(2, std::memory_order_relaxed);
    CK(launch_compact(slots, slot_off, lens, out, out_off, total, n, (cudaStream_t)stream));
    return 0;
}

int b200lz4_stitch_shards_dev(const void* const* shard_ptr, const int* shard_dev, const uint64_t* shard_total, int nshard,
                              void* dst, int dst_dev, size_t dst_capacity, uint64_t* shard_pos)
{
    if (nshard < 1 || nshard > 64) return fail_arg("nshard must be 1..64");
    if (!shard_ptr || !shard_dev || !shard_total || !dst) return fail_arg("null pointer");
    int cnt = b200lz4_device_count();
    if (cnt < 0) return cnt;
    if (dst_dev < 0 || dst_dev >= cnt) return fail_arg("dst_dev");
    uint64_t acc = 0;
    std::vector<uint64_t> pos((size_t)nshard);
    for (int g = 0; g < nshard; g++) {
        if (shard_dev[g] < 0 || shard_dev[g] >= cnt) return fail_arg("device index in shard_dev[]");
        if (shard_total[g] && !shard_ptr[g]) return fail_arg("null shard");
        pos[(size_t)g] = acc; acc += shard_total[g];
        if (shard_pos) shard_pos[g] = pos[(size_t)g];
    }
    if (acc > dst_capacity) return fail_arg("dst_capacity must hold the sum of shard_total[]");
    int my_cuda_device = -1;
    if (cudaGetDevice(&my_cuda_device) != cudaSuccess) my_cuda_device = -1;
    // one copy per shard, each on a stream of its SOURCE device, so the links into dst_dev are all busy at once
    std::vector<cudaStream_t> st((size_t)nshard, nullptr);
    cudaError_t err = cudaSuccess; const char* where = "";
    for (int g = 0; g < nshard && err == cudaSuccess; g++) {
        if (!shard_total[g]) continue;
        if ((err = cudaSetDevice(shard_dev[g])) != cudaSuccess) { where = "cudaSetDevice"; break; }
        if (shard_dev[g] != dst_dev) {
            int can = 0;
            if (cudaDeviceCanAccessPeer(&can, shard_dev[g], dst_dev) == cudaSuccess && can) {
                const cudaError_t e = cudaDeviceEnablePeerAccess(dst_dev, 0);        // direct NVLink/PCIe stores; without it the copy is staged
                if (e != cudaSuccess) (void)cudaGetLastError();                      // (already enabled, or not possible: either way the copy below works)
            }
        }
        if ((err = cudaStreamCreateWithFlags(&st[(size_t)g], cudaStreamNonBlocking)) != cudaSuccess) { st[(size_t)g] = nullptr; where = "cudaStreamCreate"; break; }
        uint8_t* to = (uint8_t*)dst + pos[(size_t)g];
        err = shard_dev[g] == dst_dev ? cudaMemcpyAsync(to, shard_ptr[g], shard_total[g], cudaMemcpyDeviceToDevice, st[(size_t)g])
                                      : cudaMemcpyPeerAsync(to, dst_dev, shard_ptr[g], shard_dev[g], shard_total[g], st[(size_t)g]);
        where = "peer copy";
    }
    for (int g = 0; g < nshard; g++) {
        if (!st[(size_t)g]) continue;
        cudaSetDevice(shard_dev[g]);
        const cudaError_t e = cudaStreamSynchronize(st[(size_t)g]);
        if (err == cudaSuccess && e != cudaSuccess) { err = e; where = "cudaStreamSynchronize"; }
        cudaStreamDestroy(st[(size_t)g]);
    }
    if (my_cuda_device >= 0) cudaSetDevice(my_cuda_device);
    if (err != cudaSuccess) return fail_cuda(err, where);
    return 0;
}

// ---- host-buffer batches
int b200lz4_compress_fast_batch_host(const uint8_t* src_base, const uint64_t* src_off, const int32_t* src_len,
                                     uint8_t* dst_base, const uint64_t* dst_off, const int32_t* dst_cap,
                                     int32_t* result, size_t n, int max_src_len)
{ return host_batch(OP_COMPRESS_FAST, src_base, src_off, src_len, dst_base, dst_off, dst_cap, result, n, max_src_len); }
int b200lz4_compress_hc_batch_host(const uint8_t* src_base, const uint64_t* src_off, const int32_t* src_len,
                                   uint8_t* dst_base, const uint64_t* dst_off, const int32_t* dst_cap,
                                   int32_t* result, size_t n, int level)
{ return host_batch(OP_COMPRESS_HC, src_base, src_off, src_len, dst_base, dst_off, dst_cap, result, n, level); }
int b200lz4_decompress_safe_batch_host(const uint8_t* src_base, const uint64_t* src_off, const int32_t* src_len,
                                       uint8_t* dst_base, const uint64_t* dst_off, const int32_t* dst_cap,
                                       int32_t* result, size_t n)
{ return host_batch(OP_DEC_SAFE, src_base, src_off, src_len, dst_base, dst_off, dst_cap, result, n, 0); }
int b200lz4_decompress_fast_batch_host(const uint8_t* src_base, const uint64_t* src_off, const int32_t* src_avail,
                                       uint8_t* dst_base, const uint64_t* dst_off, const int32_t* dst_len,
                                       int32_t* result, size_t n)
{ return host_batch(OP_DEC_FAST, src_base, src_off, src_avail, dst_base, dst_off, dst_len, result, n, 0); }
int b200xxh32_batch_host(const uint8_t* base, const uint64_t* off, const int32_t* len, uint32_t seed, uint32_t* out, size_t n)
{ return hash_host_batch<uint32_t>(base, off, len, seed, out, n); }
int b200xxh64_batch_host(const uint8_t* base, const uint64_t* off, const int32_t* len, uint64_t seed, uint64_t* out, size_t n)
{ return hash_host_batch<uint64_t>(base, off, len, seed, out, n); }

int b200lz4_compress_fast_compact_host(const uint8_t* src_base, const uint64_t* src_off, const int32_t* src_len,
                                       uint8_t* dst_base, size_t dst_capacity, uint64_t* out_off,
                                       int32_t* result, size_t n, int max_src_len, uint64_t* total)
{
    if (total) *total = 0;
    if (n == 0) return 0;
    if (!src_base || !src_off || !src_len || !dst_base || !out_off || !result) return fail_arg("null pointer");
    // each block compresses into a slot of its aligned bound; the compaction kernel then packs the chunk's streams
    auto stage = [&](Slot& s, const Chunk& ch) -> int {
        const size_t nb = ch.nb();
        uint64_t slots = 0;
        for (size_t i = ch.i0; i < ch.i1; i++) slots += lz4_slot_bytes(src_len[i]);
        int rc = slot_reserve(s, ch.s_span() + 16, (size_t)slots + 16, nb, (size_t)slots + 16); if (rc) return rc;
        const Desc h = s.host(), d = s.dev();
        uint64_t pos = 0;
        for (size_t k = 0; k < nb; k++) {
            h.doff[k] = pos;
            h.dcap[k] = (int32_t)lz4_bound(src_len[ch.i0 + k]);
            pos += lz4_slot_bytes(src_len[ch.i0 + k]);
        }
        rc = upload(s, ch, src_base, src_off, src_len); if (rc) return rc;
        BatchArgs a{ s.src.p, d.soff, d.slen, s.dst.p, d.doff, d.dcap, d.res, nb };
        CK(launch_op(OP_COMPRESS_FAST, a, max_src_len, s.st));
        g_launches.fetch_add(2, std::memory_order_relaxed);
        CK(launch_compact(s.dst.p, d.doff, d.res, s.aux.p, d.xoff, d.total, nb, s.st));
        CK(cudaMemcpyAsync(s.h_desc.p, s.d_desc.p, Slot::desc_bytes(s.desc_blocks), cudaMemcpyDeviceToHost, s.st));
        return 0;
    };
    // the chunk's packed size is known: start the payload copy at the running offset
    uint64_t running = 0;
    auto retire = [&](Slot& s) -> int {
        const Desc h = s.host();
        const uint64_t tot = *h.total;
        if (running + tot > dst_capacity) return fail_arg("dst_capacity too small for the packed stream");
        if (tot) CK(cudaMemcpyAsync(dst_base + running, s.aux.p, (size_t)tot, cudaMemcpyDeviceToHost, s.st));
        CK(cudaEventRecord(s.drained, s.st)); s.draining = true;
        const size_t nb = s.i1 - s.i0;
        memcpy(result + s.i0, h.res, nb * sizeof(int32_t));
        for (size_t k = 0; k < nb; k++) out_off[s.i0 + k] = running + h.xoff[k];
        running += tot;
        return 0;
    };
    const int rc = run_pipeline(n, src_off, src_len, nullptr, nullptr, "blocks must ascend", stage, retire);
    if (rc) return rc;
    if (total) *total = running;
    return 0;
}

int b200lz4_compress_fast_batch_host_multi(const uint8_t* src_base, const uint64_t* src_off, const int32_t* src_len,
                                           uint8_t* dst_base, const uint64_t* dst_off, const int32_t* dst_cap,
                                           int32_t* result, size_t n, int max_src_len, const int* devices, int ndev)
{ return multi_host_batch(OP_COMPRESS_FAST, src_base, src_off, src_len, dst_base, dst_off, dst_cap, result, n, max_src_len, devices, ndev); }
int b200lz4_compress_hc_batch_host_multi(const uint8_t* src_base, const uint64_t* src_off, const int32_t* src_len,
                                         uint8_t* dst_base, const uint64_t* dst_off, const int32_t* dst_cap,
                                         int32_t* result, size_t n, int level, const int* devices, int ndev)
{ return multi_host_batch(OP_COMPRESS_HC, src_base, src_off, src_len, dst_base, dst_off, dst_cap, result, n, level, devices, ndev); }
int b200lz4_decompress_safe_batch_host_multi(const uint8_t* src_base, const uint64_t* src_off, const int32_t* src_len,
                                             uint8_t* dst_base, const uint64_t* dst_off, const int32_t* dst_cap,
                                             int32_t* result, size_t n, const int* devices, int ndev)
{ return multi_host_batch(OP_DEC_SAFE, src_base, src_off, src_len, dst_base, dst_off, dst_cap, result, n, 0, devices, ndev); }
int b200lz4_decompress_fast_batch_host_multi(const uint8_t* src_base, const uint64_t* src_off, const int32_t* src_avail,
                                             uint8_t* dst_base, const uint64_t* dst_off, const int32_t* dst_len,
                                             int32_t* result, size_t n, const int* devices, int ndev)
{ return multi_host_batch(OP_DEC_FAST, src_base, src_off, src_avail, dst_base, dst_off, dst_len, result, n, 0, devices, ndev); }
int b200lz4_compress_fast_compact_host_multi(const uint8_t* src_base, const uint64_t* src_off, const int32_t* src_len,
                                             uint8_t* dst_base, size_t dst_capacity, uint64_t* out_off,
                                             int32_t* result, size_t n, int max_src_len, const int* devices, int ndev,
                                             uint64_t* shard_base, uint64_t* shard_total)
{
    if (ndev < 1 || ndev > 64) return fail_arg("ndev must be 1..64");
    for (int g = 0; g < ndev; g++) { if (shard_base) shard_base[g] = 0; if (shard_total) shard_total[g] = 0; }
    if (n == 0) return 0;
    if (!src_base || !src_off || !src_len || !dst_base || !out_off || !result) return fail_arg("null pointer");
    // region of shard g: the aligned bounds of its blocks, laid end to end (prefix sums at the shard boundaries only)
    std::vector<uint64_t> base((size_t)ndev + 1, 0);
    {
        uint64_t acc = 0; int g = 0;
        for (size_t i = 0; i <= n; i++) {
            while (g <= ndev && i == n * (size_t)g / (size_t)ndev) base[(size_t)g++] = acc;
            if (i < n) acc += lz4_slot_bytes(src_len[i]);
        }
        if (acc > dst_capacity) return fail_arg("dst_capacity must hold the aligned bounds of all blocks");
    }
    return run_sharded(n, devices, ndev, [&](size_t lo, size_t cnt) {
        int g = 0;
        while (n * (size_t)(g + 1) / (size_t)ndev <= lo) g++;                  // which shard this range is
        uint64_t total = 0;
        int rc = b200lz4_compress_fast_compact_host(src_base, src_off + lo, src_len + lo, dst_base + base[(size_t)g],
                                                    (size_t)(base[(size_t)g + 1] - base[(size_t)g]), out_off + lo, result + lo, cnt,
                                                    max_src_len, &total);
        if (rc) return rc;
        for (size_t i = lo; i < lo + cnt; i++) out_off[i] += base[(size_t)g];
        if (shard_base) shard_base[g] = base[(size_t)g];
        if (shard_total) shard_total[g] = total;
        return 0;
    });
}
int b200xxh32_batch_host_multi(const uint8_t* base, const uint64_t* off, const int32_t* len, uint32_t seed,
                               uint32_t* out, size_t n, const int* devices, int ndev)
{
    if (n == 0) return 0;
    if (!base || !off || !len || !out) return fail_arg("null pointer");
    return run_sharded(n, devices, ndev, [&](size_t lo, size_t cnt) { return hash_host_batch<uint32_t>(base, off + lo, len + lo, seed, out + lo, cnt); });
}
int b200xxh64_batch_host_multi(const uint8_t* base, const uint64_t* off, const int32_t* len, uint64_t seed,
                               uint64_t* out, size_t n, const int* devices, int ndev)
{
    if (n == 0) return 0;
    if (!base || !off || !len || !out) return fail_arg("null pointer");
    return run_sharded(n, devices, ndev, [&](size_t lo, size_t cnt) { return hash_host_batch<uint64_t>(base, off + lo, len + lo, seed, out + lo, cnt); });
}

int b200lz4_context_count(void) { return g_contexts.load(std::memory_order_relaxed); }
uint64_t b200lz4_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }
void     b200lz4_launch_count_reset(void) { g_launches.store(0, std::memory_order_relaxed); }

} // extern "C"
