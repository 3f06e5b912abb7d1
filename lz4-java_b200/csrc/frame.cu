// frame.cu — LZ4 Frame batch decoder: LZ4FrameInputStream semantics (reference:
// src/java/net/jpountz/lz4/LZ4FrameInputStream.java:132-321; format src/lz4/doc/lz4_Frame_format.md)
// for a buffer holding any number of concatenated frames (skippable frames included).
//
// The stream adapter in the reference is strictly sequential: one block in flight, one XXH32 state per
// frame.  Here the host only INDEXES the container (magic / FLG / BD / block sizes: O(#blocks), no
// payload byte is touched), and the payload work is three batched launches on the device:
//   1. XXH32 over every frame descriptor (header checksum byte) and, if present, every block payload
//      (block checksums)                                            -> xxh_batch_kernel<32>
//   2. safe-decompress of every compressed block into its slot; stored blocks are copied
//                                                                   -> lz4_decompress_safe_kernel, gather
//   3. XXH32 over every frame's decoded content (content checksum)  -> xxh32_frames_chained_kernel: one warp per frame,
//      beside the decoder on a second stream, taking each block as soon as it is decoded
// Blocks of one frame are decoded in parallel because lz4-java only writes independent blocks
// (LZ4FrameOutputStream.java:58,361-363; dependent blocks are rejected like the reference does).
#include "../../include/b200lz4.h"
#include "kernels.h"
#include <cstring>
#include <new>
#include <type_traits>
#include <vector>

namespace b200 {

cudaError_t launch_gather(const uint8_t* src, const uint64_t* src_off, const int32_t* lens,
                          uint8_t* dst, const uint64_t* dst_off, size_t n, cudaStream_t st);

static inline uint32_t rd32(const uint8_t* p) { return p[0] | (p[1] << 8) | (p[2] << 16) | ((uint32_t)p[3] << 24); }

struct FrameRec {
    uint64_t desc_off; int32_t desc_len; uint8_t hc_byte; uint8_t flg; uint32_t bs;
    uint64_t content_size; bool has_size;
    size_t first_block, nblocks;
    uint32_t content_checksum; bool has_checksum;
    uint64_t out_off;                   // slot-layout start of this frame's content
    bool complete;                      // read up to its EndMark (and content checksum); false: the container breaks off inside it
};

struct BlockRec { uint64_t src_off; uint32_t size; bool raw; uint32_t checksum; bool has_checksum; size_t frame; uint64_t out_off; uint32_t cap; };

struct FrameIndex {
    std::vector<FrameRec> frames;
    std::vector<BlockRec> blocks;
    uint64_t slot_bytes = 0;            // device bytes needed for the slot layout (upper bound of the decoded size)
    int tail_err = 0;                   // the container's own error, behind everything indexed (reported after what precedes it)
    std::vector<size_t> comp_ix, raw_ix, bsum_ix, fsum_ix;      // compressed / stored blocks, blocks and frames with a checksum
    std::vector<uint8_t> h_blob;        // the descriptor arrays (FrameDesc), built once
    // device state, all of it on `device` or none of it (create_device_state / release_device_state)
    int device = -1;
    uint8_t* d_blob = nullptr;          // the device copy of h_blob
    cudaStream_t st2 = nullptr; cudaEvent_t e1 = nullptr, e2 = nullptr;   // the checksum warps run beside the decoder
};

// The descriptor arrays of an index, in its host blob or in the device copy: every array starts on 16 bytes.
struct FrameDesc {
    uint64_t *c_soff, *c_doff; int32_t *c_slen, *c_dcap, *c_res;        // compressed blocks
    uint64_t *r_soff, *r_doff; int32_t *r_len;                          // stored blocks
    uint64_t *h_off; int32_t *h_len; uint32_t *h_out;                   // frame descriptors (header checksums)
    uint64_t *b_off; int32_t *b_len; uint32_t *b_out;                   // block checksums
    uint32_t *f_first, *f_nblk, *f_out;                                 // content checksums (chained to the decoder: xxhash.cu)
    int32_t *k_comp, *k_rawlen; uint64_t *k_off;                        // per block: index among the compressed blocks (-1: stored), stored size, slot
};
// base == nullptr only measures the layout: *bytes receives the blob's size.
static FrameDesc desc_view(uint8_t* base, const FrameIndex& ix, size_t* bytes = nullptr)
{
    const size_t nc = ix.comp_ix.size(), nr = ix.raw_ix.size(), nbs = ix.bsum_ix.size(), nfs = ix.fsum_ix.size();
    const size_t nf = ix.frames.size(), nb = ix.blocks.size();
    size_t o = 0;
    auto take = [&](auto*& p, size_t count) {
        p = base ? reinterpret_cast<std::remove_reference_t<decltype(p)>>(base + o) : nullptr;
        o = (o + count * sizeof *p + 15) & ~size_t(15);
    };
    FrameDesc d;
    take(d.c_soff, nc); take(d.c_doff, nc); take(d.c_slen, nc); take(d.c_dcap, nc); take(d.c_res, nc);
    take(d.r_soff, nr); take(d.r_doff, nr); take(d.r_len, nr);
    take(d.h_off, nf); take(d.h_len, nf); take(d.h_out, nf);
    take(d.b_off, nbs); take(d.b_len, nbs); take(d.b_out, nbs);
    take(d.f_first, nfs); take(d.f_nblk, nfs); take(d.f_out, nfs);
    take(d.k_comp, nb); take(d.k_rawlen, nb); take(d.k_off, nb);
    if (bytes) *bytes = o;
    return d;
}

// LZ4FrameInputStream.nextFrameInfo / readHeader / readBlock as a pure index pass.  The reader is a stream: it hands out the
// bytes of every frame before a malformed spot and fails THERE, after any checksum or decode error that lies earlier.  So an
// error behind at least one indexed frame is not returned here: it is kept in ix.tail_err, what precedes it is decoded and
// verified like any other input (the blocks of a frame cut short included -- that frame has no content checks), and
// decode_dev reports the first error in stream order.
static int index_frames(const uint8_t* src, size_t n, FrameIndex& ix, bool single = false, size_t* consumed = nullptr)
{
    size_t ip = 0; bool seen = false;
    int err = 0;
    FrameRec f{};
    auto stop = [&](int code) { err = code; };
    while (ip < n && !err) {
        if (n - ip < 4) { stop(-1); break; }
        const uint32_t magic = rd32(src + ip); ip += 4;
        if ((magic >> 4) == (0x184D2A50u >> 4)) {                               // skippable (:154,162-173)
            if (n - ip < 4) { stop(-1); break; }
            const uint32_t sz = rd32(src + ip); ip += 4;
            if (n - ip < sz) { stop(-1); break; }
            ip += sz; seen = true; continue;
        }
        if (magic != 0x184D2204u) { stop(-2); break; }                          // (:151)
        f = FrameRec{};
        f.desc_off = ip;
        if (n - ip < 3) { stop(-1); break; }
        f.flg = src[ip++]; const uint8_t bd = src[ip++];
        if ((f.flg >> 6) != 1 || (f.flg & 2) || !(f.flg & 0x20) || (f.flg & 1)) { stop(-10); break; }   // version, reserved, B.Indep, dictID
        if ((bd & 0x8F) || (bd >> 4) < 4) { stop(-10); break; }
        f.bs = 1u << (8 + 2 * (bd >> 4));
        f.has_size = f.flg & 8;
        if (f.has_size) { if (n - ip < 9) { stop(-1); break; } f.content_size = (uint64_t)rd32(src + ip) | ((uint64_t)rd32(src + ip + 4) << 32); ip += 8; }
        if (n - ip < 1) { stop(-1); break; }
        f.desc_len = (int32_t)(ip - f.desc_off);
        f.hc_byte = src[ip++];
        f.first_block = ix.blocks.size();
        f.out_off = ix.slot_bytes;
        for (;;) {                                                              // readBlock (:258-321)
            if (n - ip < 4) { stop(-1); break; }
            const uint32_t word = rd32(src + ip); ip += 4;
            const uint32_t sz = word & 0x7FFFFFFFu;
            if (sz == 0) break;                                                 // EndMark
            if (sz > f.bs) { stop(-4); break; }
            BlockRec b{}; b.src_off = ip; b.size = sz; b.raw = word >> 31; b.frame = ix.frames.size();
            if (n - ip < sz) { stop(-1); break; }
            ip += sz;
            b.has_checksum = f.flg & 0x10;
            if (b.has_checksum) { if (n - ip < 4) { stop(-1); break; } b.checksum = rd32(src + ip); ip += 4; }
            // the slot: a stored block needs its own size, a compressed one cannot decode to more than 255 bytes per byte
            // (one length byte adds at most 255) -- so a stream of tiny flushed blocks asks for what it can fill, not for
            // blockMaxSize each.  Full blocks keep exactly bs: a frame without short blocks in the middle stays contiguous.
            const uint64_t room = b.raw ? sz : std::min<uint64_t>(f.bs, 255ull * sz);
            b.cap = (uint32_t)room;
            b.out_off = ix.slot_bytes; ix.slot_bytes += room >= f.bs ? f.bs : ((room + 15) & ~15ull);
            ix.blocks.push_back(b);
        }
        f.nblocks = ix.blocks.size() - f.first_block;
        f.complete = !err;
        f.has_checksum = !err && (f.flg & 4);
        if (f.has_checksum) {
            if (n - ip < 4) { stop(-1); f.complete = false; f.has_checksum = false; }
            else { f.content_checksum = rd32(src + ip); ip += 4; }
        }
        if (!f.complete) f.has_size = false;
        ix.frames.push_back(f); seen = true;
        if (single) break;                                                      // readSingleFrame (:83-91, 327, 346): the rest is not read
    }
    if (consumed) *consumed = ip;
    if (err) {
        if (ix.frames.empty()) return err;                                      // nothing lies before the error
        ix.tail_err = err;
        return 0;
    }
    return seen ? 0 : -1;
}

static int build_descriptors(FrameIndex& ix)
{
    for (size_t i = 0; i < ix.blocks.size(); i++) {
        (ix.blocks[i].raw ? ix.raw_ix : ix.comp_ix).push_back(i);
        if (ix.blocks[i].has_checksum) ix.bsum_ix.push_back(i);
    }
    for (size_t f = 0; f < ix.frames.size(); f++) if (ix.frames[f].has_checksum) ix.fsum_ix.push_back(f);
    size_t bytes = 0;
    desc_view(nullptr, ix, &bytes);
    ix.h_blob.resize(bytes);
    const FrameDesc h = desc_view(ix.h_blob.data(), ix);
    for (size_t k = 0; k < ix.blocks.size(); k++) h.k_off[k] = ix.blocks[k].out_off;
    for (size_t k = 0; k < ix.fsum_ix.size(); k++) {
        const FrameRec& fr = ix.frames[ix.fsum_ix[k]];
        if (fr.first_block > 0xFFFFFFFFull || fr.nblocks > 0xFFFFFFFFull) return -10;
        h.f_first[k] = (uint32_t)fr.first_block; h.f_nblk[k] = (uint32_t)fr.nblocks;
    }
    for (size_t k = 0; k < ix.comp_ix.size(); k++) {
        const BlockRec& b = ix.blocks[ix.comp_ix[k]];
        h.k_comp[ix.comp_ix[k]] = (int32_t)k;
        h.c_soff[k] = b.src_off; h.c_doff[k] = b.out_off; h.c_slen[k] = (int32_t)b.size; h.c_dcap[k] = (int32_t)b.cap;
    }
    for (size_t k = 0; k < ix.raw_ix.size(); k++) {
        const BlockRec& b = ix.blocks[ix.raw_ix[k]];
        h.k_comp[ix.raw_ix[k]] = -1; h.k_rawlen[ix.raw_ix[k]] = (int32_t)b.size;
        h.r_soff[k] = b.src_off; h.r_doff[k] = b.out_off; h.r_len[k] = (int32_t)b.size;
    }
    for (size_t f = 0; f < ix.frames.size(); f++) { h.h_off[f] = ix.frames[f].desc_off; h.h_len[f] = ix.frames[f].desc_len; }
    for (size_t k = 0; k < ix.bsum_ix.size(); k++) {
        const BlockRec& b = ix.blocks[ix.bsum_ix[k]];
        h.b_off[k] = b.src_off; h.b_len[k] = (int32_t)b.size;
    }
    return 0;
}

// Releases the index's device state on ix.device; the caller's current device stays current.
static void release_device_state(FrameIndex& ix)
{
    if (!ix.d_blob) return;
    int cur = -1;
    if (cudaGetDevice(&cur) != cudaSuccess) cur = -1;
    cudaSetDevice(ix.device);
    cudaFree(ix.d_blob);
    if (ix.st2) cudaStreamDestroy(ix.st2);
    if (ix.e1) cudaEventDestroy(ix.e1);
    if (ix.e2) cudaEventDestroy(ix.e2);
    ix.d_blob = nullptr; ix.st2 = nullptr; ix.e1 = nullptr; ix.e2 = nullptr;
    if (cur >= 0) cudaSetDevice(cur);
}

// Creates it on the current device `dev`: the blob's device copy, the checksum stream and its two events, all or none.
static int create_device_state(FrameIndex& ix, int dev)
{
    ix.device = dev;
    cudaError_t e = cudaMalloc(&ix.d_blob, ix.h_blob.size() + 16);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ix.st2, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ix.e1, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ix.e2, cudaEventDisableTiming);
    if (e == cudaSuccess) return 0;
    release_device_state(ix);
    return fail_cuda(e, "creating the frame index's device state");
}

// What one host-buffer decode holds, released when the call returns: nothing is kept between calls.
struct HostDecode {
    FrameIndex* ix = nullptr;
    uint8_t *d_src = nullptr, *d_slots = nullptr, *d_tmp = nullptr;
    cudaStream_t st = nullptr;
    ~HostDecode()
    {
        if (d_tmp) cudaFree(d_tmp);
        if (d_src) cudaFree(d_src);
        if (d_slots) cudaFree(d_slots);
        if (st) cudaStreamDestroy(st);
        b200lz4f_index_free(ix);
    }
};

} // namespace b200

using namespace b200;

extern "C" {

static void* index_create(const uint8_t* src_host, size_t n, bool single, uint64_t* slot_bytes, size_t* consumed, int* err)
{
    FrameIndex* ix = new (std::nothrow) FrameIndex();
    if (!ix) { const int rc = fail_arg("out of host memory"); if (err) *err = rc; return nullptr; }
    int rc = src_host ? index_frames(src_host, n, *ix, single, consumed) : -1;
    if (rc == 0) rc = build_descriptors(*ix);
    if (rc) { delete ix; if (err) *err = rc; return nullptr; }
    if (slot_bytes) *slot_bytes = ix->slot_bytes;
    if (err) *err = 0;
    return ix;
}

void* b200lz4f_index_create(const uint8_t* src_host, size_t n, uint64_t* slot_bytes, int* err)
{ return index_create(src_host, n, false, slot_bytes, nullptr, err); }
void* b200lz4f_index_create_single(const uint8_t* src_host, size_t n, uint64_t* slot_bytes, size_t* src_consumed, int* err)
{ return index_create(src_host, n, true, slot_bytes, src_consumed, err); }

// getExpectedContentSize / isExpectedContentSizeDefined (:416-445): the content size the first non-skippable frame declares,
// -1 when it declares none or when there is no frame at all; the descriptor hash is verified like nextFrameInfo does.
int b200lz4f_expected_content_size(const uint8_t* src, size_t n, int64_t* content_size)
{
    if (!src || !content_size) return fail_arg("null pointer");
    *content_size = -1;
    size_t ip = 0; bool seen = false;
    for (;;) {
        if (n - ip < 4) return (seen && n == ip) ? 0 : -1;                      // clean end behind skippable frames: "no frame" (:141-147)
        const uint32_t magic = rd32(src + ip); ip += 4;
        if ((magic >> 4) == (0x184D2A50u >> 4)) {
            if (n - ip < 4) return -1;
            const uint32_t sz = rd32(src + ip); ip += 4;
            if (n - ip < sz) return -1;
            ip += sz; seen = true; continue;
        }
        if (magic != 0x184D2204u) return -2;
        const size_t desc = ip;
        if (n - ip < 2) return -1;
        const uint8_t flg = src[ip++], bd = src[ip++];
        if ((flg >> 6) != 1 || (flg & 2) || !(flg & 0x20) || (flg & 1)) return -10;
        if ((bd & 0x8F) || (bd >> 4) < 4) return -10;
        uint64_t size = 0;
        if (flg & 8) { if (n - ip < 8) return -1; size = (uint64_t)rd32(src + ip) | ((uint64_t)rd32(src + ip + 4) << 32); ip += 8; }
        if (n - ip < 1) return -1;
        const uint32_t h = b200xxh32(src + desc, ip - desc, 0);
        const int st = b200lz4_last_status();
        if (st) return st;
        if (((h >> 8) & 0xFF) != src[ip]) return -3;
        if (flg & 8) *content_size = (int64_t)size;
        return 0;
    }
}

void b200lz4f_index_free(void* index)
{
    FrameIndex* ix = (FrameIndex*)index;
    if (!ix) return;
    release_device_state(*ix);
    delete ix;
}

// Decode every indexed frame: d_src holds the container bytes, d_slots (>= slot_bytes) receives block b at its slot
// (b200lz4f_index_block_offsets; full blocks of one frame lie back to back).  On success frame_off[f] / frame_len[f] (host
// arrays, may be NULL) describe each frame's content, one run inside d_slots when no block was flushed short mid-frame;
// otherwise -11 is returned after every check has passed and the caller reads block by block (the host path below does).
// Returns total decoded bytes or a negative code.
int64_t b200lz4f_decode_dev(void* index, const uint8_t* d_src, uint8_t* d_slots, uint64_t* frame_off, uint64_t* frame_len,
                            int32_t* block_len_out, void* stream)
{
    FrameIndex& ix = *(FrameIndex*)index;
    cudaStream_t st = (cudaStream_t)stream;
    int dev = 0;
    const cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) { fail_cuda(e, "cudaGetDevice"); return B200LZ4_E_NODEVICE; }
    if (ix.d_blob && ix.device != dev) release_device_state(ix);
    if (!ix.d_blob) { const int rc = create_device_state(ix, dev); if (rc) return rc; }
    const FrameDesc h = desc_view(ix.h_blob.data(), ix), d = desc_view(ix.d_blob, ix);
    const size_t nc = ix.comp_ix.size(), nr = ix.raw_ix.size(), nbs = ix.bsum_ix.size(), nfs = ix.fsum_ix.size(), nf = ix.frames.size();
    CK(cudaMemcpyAsync(ix.d_blob, ix.h_blob.data(), ix.h_blob.size(), cudaMemcpyHostToDevice, st));
    if (nc) CK(cudaMemsetAsync(d.c_res, 0x80, nc * 4, st));                 // FRAME_RES_PENDING
    // 1. header + block checksums
    g_launches.fetch_add(1, std::memory_order_relaxed);
    CK(launch_xxh32(d_src, d.h_off, d.h_len, 0, d.h_out, nf, st));
    if (nbs) {
        // few long payloads: one warp per stream; many short ones: one lane per buffer (xxhash.cu)
        uint64_t sum = 0; for (size_t b : ix.bsum_ix) sum += ix.blocks[b].size;
        g_launches.fetch_add(1, std::memory_order_relaxed);
        CK((sum / nbs >= XXH_LONG_AVG ? launch_xxh32_long : launch_xxh32)(d_src, d.b_off, d.b_len, 0, d.b_out, nbs, st));
    }
    // 2. stored blocks are copied, then every compressed block is decoded; 3. one warp per frame folds the blocks into the
    // content checksum as the decoder hands them over (second stream; the decode kernel is launched FIRST and waits for nobody)
    if (nr) {
        g_launches.fetch_add(1, std::memory_order_relaxed);
        CK(launch_gather(d_src, d.r_soff, d.r_len, d_slots, d.r_doff, nr, st));
    }
    CK(cudaEventRecord(ix.e1, st));
    if (nc) {
        BatchArgs a{ d_src, d.c_soff, d.c_slen, d_slots, d.c_doff, d.c_dcap, d.c_res, nc };
        g_launches.fetch_add(1, std::memory_order_relaxed);
        CK(launch_decompress_safe(a, st));
    }
    if (nfs) {
        CK(cudaStreamWaitEvent(ix.st2, ix.e1, 0));
        g_launches.fetch_add(1, std::memory_order_relaxed);
        CK(launch_xxh32_frames_chained(d_slots, d.k_off, d.f_first, d.f_nblk, d.k_comp, d.k_rawlen, d.c_res, d.f_out, nfs, ix.st2));
        CK(cudaEventRecord(ix.e2, ix.st2));
        CK(cudaStreamWaitEvent(st, ix.e2, 0));
    }
    if (nc) CK(cudaMemcpyAsync(h.c_res, d.c_res, nc * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(h.h_out, d.h_out, nf * 4, cudaMemcpyDeviceToHost, st));
    if (nbs) CK(cudaMemcpyAsync(h.b_out, d.b_out, nbs * 4, cudaMemcpyDeviceToHost, st));
    if (nfs) CK(cudaMemcpyAsync(h.f_out, d.f_out, nfs * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));

    // the verdict, in the order the stream reader meets things: frame by frame -- descriptor hash (:208-216), then block by
    // block its checksum (:298-303) and its decode (:307-311), then at the EndMark content checksum (:266-269) and size (:270-272)
    std::vector<int32_t> bsum_of(ix.blocks.size(), -1), fsum_of(nf, -1);
    for (size_t k = 0; k < nbs; k++) bsum_of[ix.bsum_ix[k]] = (int32_t)k;
    for (size_t k = 0; k < nfs; k++) fsum_of[ix.fsum_ix[k]] = (int32_t)k;
    std::vector<int32_t> blen(ix.blocks.size());
    int64_t total = 0; bool gaps = false;
    for (size_t f = 0; f < nf; f++) {
        const FrameRec& fr = ix.frames[f];
        if (((h.h_out[f] >> 8) & 0xFF) != fr.hc_byte) return -3;
        uint64_t len = 0;
        for (size_t k = 0; k < fr.nblocks; k++) {
            const size_t b = fr.first_block + k;
            const BlockRec& br = ix.blocks[b];
            if (bsum_of[b] >= 0 && h.b_out[bsum_of[b]] != br.checksum) return -5;
            int32_t l = (int32_t)br.size;
            if (!br.raw) { l = h.c_res[h.k_comp[b]]; if (l < 0) return -6; }   // LZ4Exception -> IOException
            blen[b] = l;
            if (k + 1 < fr.nblocks && (uint32_t)l != fr.bs) gaps = true;          // a short block in the middle of a frame
            len += (uint64_t)l;
        }
        if (fsum_of[f] >= 0 && h.f_out[fsum_of[f]] != fr.content_checksum) return -7;
        if (fr.has_size && fr.content_size != len) return -8;
        if (frame_off) frame_off[f] = fr.out_off;
        if (frame_len) frame_len[f] = len;
        total += (int64_t)len;
    }
    if (ix.tail_err) return ix.tail_err;                    // the container breaks off / is malformed behind all that
    if (block_len_out) memcpy(block_len_out, blen.data(), blen.size() * sizeof(int32_t));
    return gaps ? -11 : total;                              // -11: everything verified, but read the blocks one by one
}

size_t b200lz4f_index_frames(void* index) { return ((FrameIndex*)index)->frames.size(); }
size_t b200lz4f_index_blocks(void* index) { return ((FrameIndex*)index)->blocks.size(); }
void b200lz4f_index_block_offsets(void* index, uint64_t* block_off)
{
    const FrameIndex& ix = *(FrameIndex*)index;
    for (size_t b = 0; b < ix.blocks.size(); b++) block_off[b] = ix.blocks[b].out_off;
}

// Whole thing with HOST buffers: index, upload, decode, download frame by frame into one contiguous stream.
static int64_t decompress_host(const uint8_t* src, size_t n, uint8_t* dst, size_t dst_capacity, bool single, size_t* consumed)
{
    int err = 0; uint64_t slot_bytes = 0;
    HostDecode c;
    c.ix = (FrameIndex*)index_create(src, n, single, &slot_bytes, consumed, &err);
    if (!c.ix) return err;
    const FrameIndex& ix = *c.ix;
    std::vector<uint64_t> foff(ix.frames.size()), flen(ix.frames.size());
    std::vector<int32_t> blen(ix.blocks.size());
    if (b200lz4_device_count() <= 0) return B200LZ4_E_NODEVICE;           // a failed query has set the message
    CK(cudaStreamCreateWithFlags(&c.st, cudaStreamNonBlocking));
    CK(cudaMalloc(&c.d_src, n + 16));
    CK(cudaMalloc(&c.d_slots, slot_bytes + 16));
    CK(cudaMemcpyAsync(c.d_src, src, n, cudaMemcpyHostToDevice, c.st));
    const int64_t rc = b200lz4f_decode_dev(c.ix, c.d_src, c.d_slots, foff.data(), flen.data(), blen.data(), c.st);
    if (rc < 0 && rc != -11) return rc;
    uint64_t pos = 0;
    if (rc >= 0) {
        // contiguous frames: one copy per frame
        for (size_t f = 0; f < ix.frames.size(); f++) {
            if (pos + flen[f] > dst_capacity) return -9;
            if (flen[f]) CK(cudaMemcpyAsync(dst + pos, c.d_slots + foff[f], flen[f], cudaMemcpyDeviceToHost, c.st));
            pos += flen[f];
        }
    } else {
        // short blocks in mid-frame (everything is verified already): the device packs the blocks, one copy brings them back
        const size_t nb = ix.blocks.size();
        std::vector<uint64_t> from(nb), to(nb);
        for (size_t b = 0; b < nb; b++) { from[b] = ix.blocks[b].out_off; to[b] = pos; pos += (uint64_t)blen[b]; }
        if (pos > dst_capacity) return -9;
        if (pos) {
            // d_tmp: [from | to] u64, [len] i32, then the packed bytes; every part starts on 16 bytes
            const size_t offs_bytes = (nb * 8 + 15) & ~size_t(15), lens_bytes = (nb * 4 + 15) & ~size_t(15);
            CK(cudaMalloc(&c.d_tmp, 2 * offs_bytes + lens_bytes + pos + 16));
            uint64_t* const d_from = (uint64_t*)c.d_tmp;
            uint64_t* const d_to = (uint64_t*)(c.d_tmp + offs_bytes);
            int32_t* const d_len = (int32_t*)(c.d_tmp + 2 * offs_bytes);
            uint8_t* const d_out = c.d_tmp + 2 * offs_bytes + lens_bytes;
            CK(cudaMemcpyAsync(d_from, from.data(), nb * 8, cudaMemcpyHostToDevice, c.st));
            CK(cudaMemcpyAsync(d_to, to.data(), nb * 8, cudaMemcpyHostToDevice, c.st));
            CK(cudaMemcpyAsync(d_len, blen.data(), nb * 4, cudaMemcpyHostToDevice, c.st));
            g_launches.fetch_add(1, std::memory_order_relaxed);
            CK(launch_gather(c.d_slots, d_from, d_len, d_out, d_to, nb, c.st));
            CK(cudaMemcpyAsync(dst, d_out, pos, cudaMemcpyDeviceToHost, c.st));
            CK(cudaStreamSynchronize(c.st));
        }
    }
    CK(cudaStreamSynchronize(c.st));
    return (int64_t)pos;
}

int64_t b200lz4f_decompress_host(const uint8_t* src, size_t n, uint8_t* dst, size_t dst_capacity)
{ return decompress_host(src, n, dst, dst_capacity, false, nullptr); }
// LZ4FrameInputStream(in, readSingleFrame = true): the first non-skippable frame only; *src_consumed = where it ended
int64_t b200lz4f_decompress_host_single(const uint8_t* src, size_t n, uint8_t* dst, size_t dst_capacity, size_t* src_consumed)
{ return decompress_host(src, n, dst, dst_capacity, true, src_consumed); }

} // extern "C"
