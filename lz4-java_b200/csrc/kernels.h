// kernels.h — internal launch interface between the C-ABI layer (capi.cu) and the kernels.
#pragma once
#include <atomic>
#include <cstddef>
#include <cstdint>
#ifdef B200_HOST_SIM
#include "simt.h"
#else
#include <cuda_runtime.h>
#endif

namespace b200 {

// One batch of independent LZ4 blocks (or hash buffers); every pointer is a device pointer.
struct BatchArgs {
    const uint8_t*  src_base;
    const uint64_t* src_off;
    const int32_t*  src_len;    // compress: bytes to compress; safe: compressed size; fast: readable bytes
    uint8_t*        dst_base;
    const uint64_t* dst_off;
    const int32_t*  dst_cap;    // compress/safe: capacity; fast: exact decoded size
    int32_t*        result;
    size_t          n;
};

cudaError_t launch_decompress_safe(const BatchArgs& a, cudaStream_t st);
cudaError_t launch_decompress_fast(const BatchArgs& a, cudaStream_t st);
cudaError_t launch_compress_fast(const BatchArgs& a, int max_src_len, cudaStream_t st);
cudaError_t launch_compress_hc(const BatchArgs& a, int level, cudaStream_t st);
cudaError_t launch_xxh32(const uint8_t* base, const uint64_t* off, const int32_t* len, uint32_t seed,
                         uint32_t* out, size_t n, cudaStream_t st);
// One warp per buffer: for a few long streams (frame content checksums).
cudaError_t launch_xxh32_long(const uint8_t* base, const uint64_t* off, const int32_t* len, uint32_t seed,
                              uint32_t* out, size_t n, cudaStream_t st);
// frame content checksums chained to the block decoder (frame.cu): one warp per frame follows the decoder's result words
static constexpr int32_t FRAME_RES_PENDING = int32_t(0x80808080);      // what cudaMemset(0x80) leaves; no decoder result looks like it
cudaError_t launch_xxh32_frames_chained(const uint8_t* slots, const uint64_t* blk_off, const uint32_t* f_first, const uint32_t* f_nblk,
                                        const int32_t* blk_comp, const int32_t* blk_rawlen, const int32_t* c_res,
                                        uint32_t* out, size_t n, cudaStream_t st);
cudaError_t launch_xxh64(const uint8_t* base, const uint64_t* off, const int32_t* len, uint64_t seed,
                         uint64_t* out, size_t n, cudaStream_t st);
// average buffer length from which the one-warp-per-buffer kernels (launch_xxh*_long) win
static constexpr uint64_t XXH_LONG_AVG = 32768;

// streaming hash: one device-resident state per handle, updated by a single-warp kernel
struct Xxh32State { uint64_t total; uint32_t v[4]; uint8_t mem[16]; uint32_t memsize; uint32_t seed; uint32_t digest; };
struct Xxh64State { uint64_t total; uint64_t v[4]; uint8_t mem[32]; uint32_t memsize; uint32_t pad; uint64_t seed; uint64_t digest; };
cudaError_t launch_xxh32_stream(Xxh32State* st, int op, uint32_t seed, const uint8_t* data, size_t len, cudaStream_t s);
cudaError_t launch_xxh64_stream(Xxh64State* st, int op, uint64_t seed, const uint8_t* data, size_t len, cudaStream_t s);
enum { XXH_OP_RESET = 0, XXH_OP_UPDATE = 1, XXH_OP_DIGEST = 2 };

cudaError_t launch_xxh64_long(const uint8_t* base, const uint64_t* off, const int32_t* len, uint64_t seed,
                              uint64_t* out, size_t n, cudaStream_t st);

// prefix-sum compaction of variable-length outputs (compact_host path)
cudaError_t launch_compact(const uint8_t* slots, const uint64_t* slot_off, const int32_t* lens,
                           uint8_t* out, uint64_t* out_off, uint64_t* total, size_t n, cudaStream_t st);

// LZ4_compressBound (lz4.h:212) of one block, a negative length counting as 0, and the block's slot in the packed layouts
// (compact_host staging, the HC container writers): the bound rounded up to 16 bytes.
static inline uint64_t lz4_bound(int32_t len) { const uint64_t n = len > 0 ? (uint64_t)len : 0; return n + n / 255 + 16; }
static inline uint64_t lz4_slot_bytes(int32_t len) { return (lz4_bound(len) + 15) & ~uint64_t(15); }

// Host-side state of the library, defined in capi.cu and shared by the host files (capi.cu, frame.cu, containers.cu).
extern std::atomic<unsigned long long> g_launches;          // kernel launches of every entry point, any thread (b200lz4_launch_count)
// Record what went wrong for b200lz4_last_error / b200lz4_last_status and return the code: B200LZ4_E_NODEVICE or _E_CUDA
// (fail_cuda), B200LZ4_E_ARG (fail_arg).
int fail_cuda(cudaError_t e, const char* where);
int fail_arg(const char* what);
#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return b200::fail_cuda(e_, #call); } while (0)

} // namespace b200
