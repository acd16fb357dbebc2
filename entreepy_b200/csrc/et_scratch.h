// Layouts of the device scratch blocks: the decoder's (status words and arrays) and the pack's.  Each block is
// declared once, by one function that both sizes it and hands out its arrays.  Plain C++17 without CUDA headers,
// so that tests/test_scratch_layout.py can compile it with g++ and check the layouts on the CPU.
#pragma once
#include <cstddef>
#include <cstdint>

namespace et {

constexpr int kChunkThreads = 256;  // chunks per CTA of the per-thread decoder

// Parts of a chunk that the lane write walk decodes side by side (et_lanes.inc).  MEASURED (r2, text-1G, all else equal):
// two parts 0.996 ms per decode, four parts 1.012 ms - the write walk gains (wait stalls down, issue slots 59 -> 68 %) what
// the count walk loses to recording three boundaries per chunk instead of one (four reconvergence points per chunk).
#ifndef ET_WRITE_CHAINS
#define ET_WRITE_CHAINS 2
#endif
// What the count walk records for the write walk per chunk: 18 bits per boundary.
#if ET_WRITE_CHAINS == 2
typedef uint32_t mid_t;
#else
typedef uint64_t mid_t;
#endif

constexpr uint32_t kMaxStates = 16;                  // most entries of a chunk's transfer function (longest code of such a dictionary)
constexpr uint32_t kSegChunks = 16, kSegThreads = 256;  // transfer functions: chunks per composing thread, threads per block
constexpr uint32_t kGroupRegions = 1024;             // lane decoder: regions per group of the symbol scan

constexpr size_t kScratchAlign = 128;

// Lays arrays out one after another.  A null base only counts: the size and the pointers come from the same calls.
struct Carve {
    uint8_t *base = nullptr;
    size_t bytes = 0;
    template <class T>
    T *take(size_t count, size_t align = kScratchAlign) {
        bytes = (bytes + align - 1) & ~(align - 1);
        T *p = base ? reinterpret_cast<T *>(base + bytes) : nullptr;
        bytes += count * sizeof(T);
        return p;
    }
};

// The decoder's status words, at the start of its scratch.  Cleared (all 64 bytes) before every decode; the host reads
// back the first kDecodeStatusReadBack bytes.
struct DecodeStatus {
    uint32_t pad;
    uint32_t error_flags;      // kErrInvalidCode: a bit pattern that is no code
    unsigned long long total;  // symbols found
    uint32_t changed;          // a check found an entry that was not the true one
    uint32_t max_sum;          // lane decoder: symbols of the largest region
    uint32_t entry;            // first codeword of chunk 0, bits past the chunk grid
    uint32_t exit;             // first codeword boundary at or after the end of the last chunk, bits past that end
    uint32_t work_count;       // lane decoder: regions on the repair list (device only)
    uint32_t spare[7];
};
static_assert(sizeof(DecodeStatus) == 64, "one 64-byte clear covers the status words");
static_assert(offsetof(DecodeStatus, max_sum) == offsetof(DecodeStatus, changed) + 4, "one 8-byte clear resets changed and max_sum");
static_assert(offsetof(DecodeStatus, exit) == offsetof(DecodeStatus, entry) + 4, "entry and exit are written as a pair (DecArgs::entry_exit)");
constexpr size_t kDecodeStatusReadBack = offsetof(DecodeStatus, work_count);

// log2 of the entries per chunk of the transfer tables for a code whose chunks can be entered at `states` bit offsets;
// 0: no transfer functions (fewer than two states, or more than kMaxStates).
inline uint32_t transfer_log2(uint32_t states) {
    if (states < 2 || states > kMaxStates) return 0;
    uint32_t s = 1;
    while ((1u << s) < states) ++s;
    return s;
}

// The decoder's scratch for n chunks.  Arrays a path does not use are null.
struct DecodeLayout {
    DecodeStatus *status = nullptr;
    unsigned long long *block_prefix = nullptr;  // [n_blocks] scan of the symbols per block of chunks (lanes: per region)
    uint32_t *count = nullptr;                   // [n]
    uint16_t *start_off = nullptr;               // [n]
    uint16_t *exit_off = nullptr;                // [n]
    // lane-interleaved decoder (regions of 32 chunks)
    mid_t *mid = nullptr;                        // [n]
    unsigned long long *group_prefix = nullptr;  // [n_groups + 1]
    uint32_t *work = nullptr;                    // [n_blocks + 8]
    uint32_t *edge = nullptr;                    // [n_blocks + 8]
    uint32_t *rsum = nullptr;                    // [n_blocks + 8]
    uint8_t *self_listed = nullptr;              // [n_blocks]
    // per-thread decoder, codes that take transfer functions
    uint8_t *tr_exit = nullptr;                  // [n << tr_log2]
    uint16_t *tr_cnt = nullptr;                  // [n << tr_log2]
    unsigned long long *seg_prefix = nullptr;    // [seg_blocks * kSegThreads]
    unsigned long long *block_map = nullptr;     // [seg_blocks]
    uint64_t n_blocks = 0;
    uint32_t tr_log2 = 0;
    uint64_t seg_blocks = 0;
    size_t bytes = 0;
};

inline DecodeLayout decode_layout(void *base, uint64_t n, bool lanes, uint32_t transfer_states) {
    DecodeLayout L;
    Carve c{static_cast<uint8_t *>(base)};
    L.n_blocks = lanes ? (n + 31) / 32 : (n + kChunkThreads - 1) / kChunkThreads;
    L.status = c.take<DecodeStatus>(1);
    L.block_prefix = c.take<unsigned long long>(L.n_blocks);
    L.count = c.take<uint32_t>(n);
    L.start_off = c.take<uint16_t>(n);
    L.exit_off = c.take<uint16_t>(n);
    if (lanes) {
        L.mid = c.take<mid_t>(n);
        L.group_prefix = c.take<unsigned long long>((L.n_blocks + kGroupRegions - 1) / kGroupRegions + 1);
        L.work = c.take<uint32_t>(L.n_blocks + 8);
        L.edge = c.take<uint32_t>(L.n_blocks + 8);
        L.rsum = c.take<uint32_t>(L.n_blocks + 8);
        L.self_listed = c.take<uint8_t>(L.n_blocks);
    } else if ((L.tr_log2 = transfer_log2(transfer_states)) != 0) {
        L.seg_blocks = (n + kSegChunks * kSegThreads - 1) / (kSegChunks * kSegThreads);
        L.tr_exit = c.take<uint8_t>(n << L.tr_log2);
        L.tr_cnt = c.take<uint16_t>(n << L.tr_log2);
        L.seg_prefix = c.take<unsigned long long>(L.seg_blocks * kSegThreads);
        L.block_map = c.take<unsigned long long>(L.seg_blocks);
    }
    L.bytes = c.bytes;
    return L;
}

// The pack's scratch for num_tiles tiles of 4096 symbols.  The wide kernel uses one slot per tile; the lane-run path
// one per region of 2048 symbols (two per tile, and pass A's slabs may touch two more).  The single pass keeps its
// look-back descriptors where the two-pass path keeps run_bits: neither uses the other's.  The arrays follow each other at
// their elements' alignment (16 bytes for ticket, tile_state and run_bits): MEASURED (text-1G, B200 at 1000 W), putting
// every array on a 128-byte boundary made the pack 2 % slower (0.809 -> 0.826 ms) with the same kernels.
struct PackLayout {
    uint32_t *ticket = nullptr;                  // [4] tile counter (16 bytes cleared)
    unsigned long long *tile_state = nullptr;    // [slots] wide kernel: look-back descriptors; all: last bit + 1 of each slot
    uint8_t *seam_head = nullptr;                // [slots]
    uint8_t *seam_tail = nullptr;                // [slots]
    uint32_t *tile_bits = nullptr;               // [slots] two passes: bits of the earlier regions of the same group
    unsigned long long *group_prefix = nullptr;  // [(slots + 7) / 8] two passes: bits before each group
    uint16_t *run_bits = nullptr;                // [32 * slots] two passes: bits of every run of 64 symbols
    unsigned long long *tile_desc = nullptr;     // [slots] single pass: look-back descriptors
    size_t bytes = 0;
};

inline PackLayout pack_layout(void *base, uint32_t num_tiles) {
    PackLayout L;
    Carve c{static_cast<uint8_t *>(base)};
    const size_t slots = (size_t)num_tiles * 2 + 2;
    L.ticket = c.take<uint32_t>(4, 16);
    L.tile_state = c.take<unsigned long long>(slots, 16);
    L.group_prefix = c.take<unsigned long long>((slots + 7) / 8, 8);
    L.tile_bits = c.take<uint32_t>(slots, 4);
    L.seam_head = c.take<uint8_t>(slots, 1);
    L.seam_tail = c.take<uint8_t>(slots, 1);
    Carve single = c;
    L.tile_desc = single.take<unsigned long long>(slots, 16);
    L.run_bits = c.take<uint16_t>(slots * 32, 16);
    L.bytes = c.bytes > single.bytes ? c.bytes : single.bytes;
    return L;
}

}  // namespace et
