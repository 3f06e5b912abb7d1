// containers.cu — the containers lz4-java wraps around the block codec, as whole-buffer batch calls:
//   * LZ4 Frame writer     — LZ4FrameOutputStream.writeHeader/writeBlock/writeEndMark
//                            (src/java/net/jpountz/lz4/LZ4FrameOutputStream.java:178-251)
//   * "LZ4Block" container — LZ4BlockOutputStream.flushBufferedData/finish (:203-266) and
//                            LZ4BlockInputStream.refill (LZ4BlockInputStream.java:191-264)
//   * length-prefixed block — LZ4CompressorWithLength / LZ4DecompressorWithLength
// The reference does these one block per native call; here the host only lays out headers and the
// payload work (block compression / decompression, every XXH32) goes through the batch entry points,
// i.e. the CUDA kernels.  No hashing or codec arithmetic runs on the host.
#include "../../include/b200lz4.h"
#include "kernels.h"
#include <cstring>
#include <memory>
#include <new>
#include <vector>

static inline void put32(uint8_t* p, uint32_t v) { p[0] = (uint8_t)v; p[1] = (uint8_t)(v >> 8); p[2] = (uint8_t)(v >> 16); p[3] = (uint8_t)(v >> 24); }
static inline uint32_t get32(const uint8_t* p) { return p[0] | (p[1] << 8) | (p[2] << 16) | ((uint32_t)p[3] << 24); }

// Both writers' blocks: [0, n) cut into bs-byte blocks and compressed with the writer's compressor argument (LZ4FrameOutputStream /
// LZ4BlockOutputStream take any LZ4Compressor): hc_level 0 = the fast compressor, packed output; 1..17 = LZ4_compress_HC at that
// level into bound-sized slots.  Then put(src_off, src_len, payload, size, raw) for each block in order; raw: stored as it is,
// because compressing did not shrink it.
template <class Put>
static int write_blocks(const uint8_t* src, size_t n, size_t bs, int hc_level, Put put)
{
    const size_t nb = (n + bs - 1) / bs;
    if (nb == 0) return 0;
    std::vector<uint64_t> soff(nb), coff(nb);
    std::vector<int32_t> slen(nb), ccap(nb), clen(nb);
    size_t tmp_cap = 0;
    for (size_t i = 0; i < nb; i++) {
        soff[i] = i * bs; slen[i] = (int32_t)(n - i * bs < bs ? n - i * bs : bs);
        coff[i] = tmp_cap; ccap[i] = (int32_t)b200::lz4_bound(slen[i]);         // HC: the block's slot (the fast compressor packs, setting coff)
        tmp_cap += b200::lz4_slot_bytes(slen[i]);
    }
    std::unique_ptr<uint8_t[]> tmp(new (std::nothrow) uint8_t[tmp_cap]);
    if (!tmp) return b200::fail_arg("out of host memory");
    uint64_t total = 0;
    const int rc = hc_level <= 0
        ? b200lz4_compress_fast_compact_host(src, soff.data(), slen.data(), tmp.get(), tmp_cap, coff.data(), clen.data(), nb, bs <= 65536 ? 65536 : 0, &total)
        : b200lz4_compress_hc_batch_host(src, soff.data(), slen.data(), tmp.get(), coff.data(), ccap.data(), clen.data(), nb, hc_level);
    if (rc) return rc;
    for (size_t i = 0; i < nb; i++) {
        const bool raw = clen[i] <= 0 || clen[i] >= slen[i];
        put(soff[i], slen[i], raw ? src + soff[i] : tmp.get() + coff[i], raw ? (uint32_t)slen[i] : (uint32_t)clen[i], raw);
    }
    return 0;
}

extern "C" {

size_t b200lz4f_compress_bound(size_t n, int bsCode)
{
    if (bsCode < 4 || bsCode > 7) return 0;
    const size_t bs = (size_t)1 << (8 + 2 * bsCode), nb = (n + bs - 1) / bs;
    return 4 + 2 + 8 + 1 + nb * 8 + n + 4 + 4;
}

// flags: bit0 content checksum, bit1 block checksums, bit2 content size.  Returns bytes written or a negative code.
int64_t b200lz4f_compress_host_hc(const uint8_t* src, size_t n, uint8_t* dst, size_t cap, int bsCode, int flags, int hc_level)
{
    if (bsCode < 4 || bsCode > 7) return b200::fail_arg("bsCode must be 4..7");
    if (cap < b200lz4f_compress_bound(n, bsCode)) return -9;
    const size_t bs = (size_t)1 << (8 + 2 * bsCode);
    size_t o = 0;
    put32(dst, 0x184D2204u); o = 4;
    const size_t hdr = o;
    dst[o++] = (uint8_t)((1 << 6) | (1 << 5) | ((flags & 2) ? 1 << 4 : 0) | ((flags & 4) ? 1 << 3 : 0) | ((flags & 1) ? 1 << 2 : 0));
    dst[o++] = (uint8_t)(bsCode << 4);
    if (flags & 4) { put32(dst + o, (uint32_t)n); put32(dst + o + 4, (uint32_t)((uint64_t)n >> 32)); o += 8; }
    const uint32_t hh = b200xxh32(dst + hdr, o - hdr, 0);                        // descriptor checksum (:187)
    int st = b200lz4_last_status();
    if (st) return st;
    dst[o++] = (uint8_t)((hh >> 8) & 0xFF);
    std::vector<uint64_t> poff; std::vector<int32_t> plen;
    int rc = write_blocks(src, n, bs, hc_level, [&](uint64_t, int32_t, const uint8_t* payload, uint32_t size, bool raw) {
        put32(dst + o, size | (raw ? 0x80000000u : 0u)); o += 4;                 // writeBlock (:199-235), stored when it does not shrink (:215-222)
        memcpy(dst + o, payload, size);
        poff.push_back(o); plen.push_back((int32_t)size); o += size;
        if (flags & 2) o += 4;                                                   // block checksum slot, filled below
    });
    if (rc) return rc;
    if (flags & 2) {
        std::vector<uint32_t> sums(poff.size());
        rc = b200xxh32_batch_host(dst, poff.data(), plen.data(), 0, sums.data(), poff.size());
        if (rc) return rc;
        for (size_t i = 0; i < sums.size(); i++) put32(dst + poff[i] + plen[i], sums[i]);
    }
    put32(dst + o, 0); o += 4;                                                   // EndMark (:243-245)
    if (flags & 1) {
        if (n > 0x7FFFFFFFull) return -10;
        const uint32_t h = b200xxh32(src, n, 0);                                 // content checksum (:246-249)
        st = b200lz4_last_status();
        if (st) return st;
        put32(dst + o, h); o += 4;
    }
    return (int64_t)o;
}
int64_t b200lz4f_compress_host(const uint8_t* src, size_t n, uint8_t* dst, size_t cap, int bsCode, int flags)
{ return b200lz4f_compress_host_hc(src, n, dst, cap, bsCode, flags, 0); }

// ---------------------------------------------------------------- "LZ4Block" container
static const uint8_t LZ4BLOCK_MAGIC[8] = { 'L', 'Z', '4', 'B', 'l', 'o', 'c', 'k' };
enum { LZ4BLOCK_HEADER = 8 + 1 + 4 + 4 + 4, METHOD_RAW = 0x10, METHOD_LZ4 = 0x20 };
static const uint32_t LZ4BLOCK_SEED = 0x9747b28cu;                               // LZ4BlockOutputStream.java:56

static int lz4block_level(int blockSize)                                        // LZ4BlockOutputStream.java:58-70
{
    int lvl = 0; while ((1 << lvl) < blockSize) lvl++;                           // 32 - numberOfLeadingZeros(blockSize - 1)
    lvl -= 10; return lvl < 0 ? 0 : lvl;
}

size_t b200lz4block_compress_bound(size_t n, int blockSize)
{
    if (blockSize < 64 || blockSize > (1 << 25)) return 0;
    const size_t nb = (n + blockSize - 1) / blockSize;
    return (nb + 1) * LZ4BLOCK_HEADER + n + nb * 16 + n / 255;
}

int64_t b200lz4block_compress_host_hc(const uint8_t* src, size_t n, uint8_t* dst, size_t cap, int blockSize, int hc_level)
{
    if (blockSize < 64 || blockSize > (1 << 25)) return b200::fail_arg("blockSize must be 64..2^25");
    if (cap < b200lz4block_compress_bound(n, blockSize)) return -9;
    const int level = lz4block_level(blockSize);
    size_t o = 0;
    std::vector<uint64_t> soff, sum_at; std::vector<int32_t> slen;
    int rc = write_blocks(src, n, (size_t)blockSize, hc_level, [&](uint64_t src_off, int32_t src_len, const uint8_t* payload, uint32_t size, bool raw) {
        memcpy(dst + o, LZ4BLOCK_MAGIC, 8);                                      // flushBufferedData (:203-227)
        dst[o + 8] = (uint8_t)((raw ? METHOD_RAW : METHOD_LZ4) | level);
        put32(dst + o + 9, size); put32(dst + o + 13, (uint32_t)src_len);
        memcpy(dst + o + LZ4BLOCK_HEADER, payload, size);
        soff.push_back(src_off); slen.push_back(src_len); sum_at.push_back(o + 17);   // checksum slot, filled below
        o += LZ4BLOCK_HEADER + size;
    });
    if (rc) return rc;
    std::vector<uint32_t> sums(soff.size());
    rc = b200xxh32_batch_host(src, soff.data(), slen.data(), LZ4BLOCK_SEED, sums.data(), soff.size());   // checksum of the ORIGINAL bytes
    if (rc) return rc;
    for (size_t i = 0; i < sums.size(); i++) put32(dst + sum_at[i], sums[i] & 0x0FFFFFFFu);   // Checksum view keeps 28 bits (StreamingXXHash32.java:106)
    memcpy(dst + o, LZ4BLOCK_MAGIC, 8);                                          // finish(): empty block (:255-266)
    dst[o + 8] = (uint8_t)(METHOD_RAW | level);
    put32(dst + o + 9, 0); put32(dst + o + 13, 0); put32(dst + o + 17, 0);
    o += LZ4BLOCK_HEADER;
    return (int64_t)o;
}
int64_t b200lz4block_compress_host(const uint8_t* src, size_t n, uint8_t* dst, size_t cap, int blockSize)
{ return b200lz4block_compress_host_hc(src, n, dst, cap, blockSize, 0); }

// Decodes an LZ4Block stream the way LZ4BlockInputStream reads it.  stopOnEmptyBlock != 0 (the reference's default, :100-104):
// reading ends at the first empty block, whatever follows is left alone (*srcConsumed says where), and a stream that ends
// before one is "Stream ended prematurely" (:192-198).  stopOnEmptyBlock == 0: empty blocks are stepped over, concatenated
// streams continue, and the end of src at (or inside) a header ends the stream quietly (:193-194, tryReadFully).
// Returns decoded bytes; -1 premature end, -2 "Stream is corrupted", -9 dst too small.
int64_t b200lz4block_decompress_host(const uint8_t* src, size_t n, uint8_t* dst, size_t cap, int stopOnEmptyBlock, size_t* srcConsumed)
{
    std::vector<uint64_t> soff, doff; std::vector<int32_t> savail, dlen, csz; std::vector<uint32_t> want;
    std::vector<uint64_t> hoff; std::vector<int32_t> hlen;
    size_t ip = 0, op = 0;
    int64_t tail = 0;                    // what is wrong with the container itself, behind the blocks collected so far: the reader
                                         // would have decoded and checked THOSE first, so their verdict comes first
    for (;;) {                                                                   // refill (:191-264)
        if (n - ip < LZ4BLOCK_HEADER) { if (stopOnEmptyBlock) tail = -1; else ip = n; break; }
        if (memcmp(src + ip, LZ4BLOCK_MAGIC, 8) != 0) { tail = -2; break; }
        const int token = src[ip + 8], method = token & 0xF0, level = 10 + (token & 0x0F);
        if (method != METHOD_RAW && method != METHOD_LZ4) { tail = -2; break; }
        const int32_t clen = (int32_t)get32(src + ip + 9), olen = (int32_t)get32(src + ip + 13);
        const uint32_t check = get32(src + ip + 17);
        if (olen > (1 << level) || olen < 0 || clen < 0 || (olen == 0 && clen != 0) || (olen != 0 && clen == 0) ||
            (method == METHOD_RAW && olen != clen)) { tail = -2; break; }
        ip += LZ4BLOCK_HEADER;
        if (olen == 0) { if (check != 0) { tail = -2; break; } if (stopOnEmptyBlock) break; continue; }   // empty block (:225-233)
        if (n - ip < (size_t)clen) { tail = -1; break; }
        if (cap - op < (size_t)olen) { tail = -9; break; }
        if (method == METHOD_RAW) memcpy(dst + op, src + ip, (size_t)olen);
        else { soff.push_back(ip); savail.push_back(clen); doff.push_back(op); dlen.push_back(olen); csz.push_back(clen); }
        hoff.push_back(op); hlen.push_back(olen); want.push_back(check);
        ip += (size_t)clen; op += (size_t)olen;
    }
    // per block the reader decodes, compares the consumed length, then the checksum -- all "Stream is corrupted" (:236-262)
    if (!soff.empty()) {
        std::vector<int32_t> res(soff.size());
        int rc = b200lz4_decompress_fast_batch_host(src, soff.data(), savail.data(), dst, doff.data(), dlen.data(), res.data(), soff.size());
        if (rc) return rc;
        for (size_t i = 0; i < res.size(); i++) if (res[i] != csz[i]) return -2;  // compressedLen != compressedLen2 (:247-250)
    }
    if (!hoff.empty()) {
        std::vector<uint32_t> sums(hoff.size());
        int rc = b200xxh32_batch_host(dst, hoff.data(), hlen.data(), LZ4BLOCK_SEED, sums.data(), hoff.size());
        if (rc) return rc;
        for (size_t i = 0; i < sums.size(); i++) if ((sums[i] & 0x0FFFFFFFu) != want[i]) return -2;
    }
    if (tail) return tail;
    if (srcConsumed) *srcConsumed = ip;
    return (int64_t)op;
}

// ---------------------------------------------------------------- length-prefixed block (LZ4CompressorWithLength.java:45-50)
int b200lz4_compress_with_length(const char* src, char* dst, int srcSize, int dstCapacity)
{
    if (dstCapacity < 4) return 0;
    const int r = b200lz4_compress_default(src, dst + 4, srcSize, dstCapacity - 4);
    if (r <= 0) return r;
    put32((uint8_t*)dst, (uint32_t)srcSize);
    return r + 4;
}
int b200lz4_decompressed_length(const char* src) { return (int)get32((const uint8_t*)src); }   // LZ4DecompressorWithLength.java:52-54
// fast-decompressor flavour: returns bytes read (incl. the 4-byte prefix) or < 0 (LZ4DecompressorWithLength.java:125-131)
int b200lz4_decompress_with_length(const char* src, int srcAvail, char* dst, int dstCapacity)
{
    if (srcAvail < 4) return -1;
    const int n = b200lz4_decompressed_length(src);
    if (n < 0 || n > dstCapacity) return -1;
    const int r = b200lz4_decompress_fast_bounded(src + 4, srcAvail - 4, dst, n);
    return r < 0 ? r : r + 4;
}

} // extern "C"
