// Layouts of the device scratch blocks: the decoder's (status words and arrays) and the pack's.  Each block is
// declared once, by one function that both sizes it and hands out its arrays.  Plain C++17 without CUDA headers,
// so that tests/test_scratch_layout.py can compile it with g++ and check the layouts on the CPU.
#pragma once
#include <cstddef>
#include <cstdint>

#include "et_internal.h"

namespace et {

constexpr int kChunkThreads = 256;  // chunks per CTA of the per-thread decoder

// What the count walk records for the write walk per chunk: where its second part begins (18 bits, et_lanes.inc).
typedef uint32_t mid_t;

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
// one per region of 2048 symbols (two per tile, and pass A's slabs may touch two more).  The arrays follow each other at
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
    L.run_bits = c.take<uint16_t>(slots * 32, 16);
    L.bytes = c.bytes;
    return L;
}

// ---------------------------------------------------------------- batched decode (et_decode_batch_dev)
// A batch is decoded in groups of streams; a group's tables and chunk arrays share one scratch block.
constexpr uint32_t kBatchGroupItems = 512;           // streams per group: bounds the per-stream tables (48 KB each)
constexpr uint64_t kBatchGroupBytes = 256ull << 20;  // stream bytes per group (a longer stream is a group of its own): bounds the chunk arrays
constexpr size_t kBatchHeadBytes = 4096;             // front of a stream the host parses the dictionary from, as et_decode_dev does
constexpr uint32_t kBatchWorkWords = 32;             // per stream: slot counter and slot windows of the table build
constexpr size_t kBatchSlots = kLutSize + (kMaxSubTables << kSubBits);  // per stream: marker-window slots, second-level tables

struct BatchSource {  // the front of a stream: p[0, min(n, kBatchHeadBytes)) is gathered for the host
    const uint8_t *p;
    uint64_t n;
};
struct BatchTile {  // kChunkThreads chunks of one stream, from its chunk `first`
    uint32_t item, first;
};
struct BatchItemStatus {
    unsigned long long total;  // symbols found
    uint32_t error_flags;      // kErrInvalidCode
    uint32_t changed;          // the final check found a chunk whose entry was not its left neighbour's exit
};
struct BatchStatus {
    uint32_t changed;        // some stream's entries moved (the sync rounds, the final check)
    uint32_t entry_exit[2];  // written by the scan, not used
    uint32_t pad;
};

// The scratch of one group: `items` streams on the per-thread chunk path with `tiles` tiles, `chunks` chunks and
// `node_words` words of tries in all.  The arrays come in four runs: cleared before the group (status .. work), the
// heads (sources, heads), uploaded with one copy (args .. nodes), device only.  A pinned host buffer of host_bytes
// carved the same way mirrors the first three; the host reads back status .. item_status with one copy.
struct BatchLayout {
    BatchStatus *status = nullptr;           // [1]
    BatchItemStatus *item_status = nullptr;  // [items]
    uint32_t *work = nullptr;                // [items * kBatchWorkWords]
    BatchSource *sources = nullptr;          // [items]
    uint8_t *heads = nullptr;                // [items * kBatchHeadBytes]
    uint8_t *args = nullptr;                 // [items * args_bytes] the decoder's arguments per stream
    BatchTile *tiles = nullptr;              // [tiles]
    uint32_t *nodes = nullptr;               // [node_words] every stream's trie
    uint32_t *lut = nullptr;                 // [items * 2 * kLutSize] clut | wlut per stream
    uint16_t *slots = nullptr;               // [items * kBatchSlots]
    unsigned long long *tile_sums = nullptr; // [tiles + 1] symbols per tile, scanned in place; [tiles] = the group's total
    uint32_t *count = nullptr;               // [chunks]
    uint16_t *start_off = nullptr;           // [chunks]
    uint16_t *exit_off = nullptr;            // [chunks]
    size_t clear_bytes = 0;                  // status .. work, from the start of the block
    size_t status_bytes = 0;                 // status .. item_status
    size_t upload_begin = 0, upload_end = 0; // args .. nodes
    size_t host_bytes = 0;                   // status .. nodes
    size_t bytes = 0;
};

inline BatchLayout batch_layout(void *base, uint32_t items, size_t args_bytes, uint64_t tiles, uint64_t node_words, uint64_t chunks) {
    BatchLayout L;
    Carve c{static_cast<uint8_t *>(base)};
    L.status = c.take<BatchStatus>(1);
    L.item_status = c.take<BatchItemStatus>(items);
    L.status_bytes = c.bytes;
    L.work = c.take<uint32_t>((size_t)items * kBatchWorkWords);
    L.clear_bytes = c.bytes;
    L.sources = c.take<BatchSource>(items);
    L.heads = c.take<uint8_t>((size_t)items * kBatchHeadBytes);
    L.args = c.take<uint8_t>((size_t)items * args_bytes);
    L.upload_begin = c.bytes - (size_t)items * args_bytes;
    L.tiles = c.take<BatchTile>(tiles);
    L.nodes = c.take<uint32_t>(node_words);
    L.upload_end = L.host_bytes = c.bytes;
    L.lut = c.take<uint32_t>((size_t)items * 2 * kLutSize);
    L.slots = c.take<uint16_t>((size_t)items * kBatchSlots);
    L.tile_sums = c.take<unsigned long long>(tiles + 1);
    L.count = c.take<uint32_t>(chunks);
    L.start_off = c.take<uint16_t>(chunks);
    L.exit_off = c.take<uint16_t>(chunks);
    L.bytes = c.bytes;
    return L;
}

// ---------------------------------------------------------------- batched encode (et_encode_batch_dev)
// Groups follow the decode batch's rule (kBatchGroupItems streams, kBatchGroupBytes of text).  The histograms run over
// tiles of kEncHistTileBytes of one stream; the pack numbers the regions of 2048 symbols of every stream of the group
// one after another and runs over tiles of kEncTileRegions regions of one stream.
constexpr uint32_t kEncHistTileBytes = 16384;  // text per CTA of the batched histogram (a multiple of 16)
constexpr uint32_t kEncTileRegions = 16;       // regions per CTA of the batched pack (pass B: one per warp)
constexpr uint32_t kEncPrefixGroup = 1024;     // regions per group of the scan (region_prefix_kernel)

struct EncHistTile {  // bytes [lo, hi) of base[0, kEncHistTileBytes) belong to stream `item` (base 16-byte aligned)
    const uint8_t *base;
    uint32_t lo, hi;
    uint32_t item, pad;
};

// The scratch of one encode group: `items` streams, `hist_tiles` histogram tiles; `packed` of them reach the batched pack
// with `header_bytes` of headers, `tiles` pack tiles and `regions` regions in all.  Four runs: the counts (cleared, read
// back), the histogram tiles (uploaded before the histogram), args .. tiles (uploaded with one copy before the pack),
// device only.  A pinned host buffer of host_bytes carved the same way mirrors the first three.
struct EncBatchLayout {
    unsigned long long *counts = nullptr;        // [items * 256]
    EncHistTile *hist_tiles = nullptr;           // [hist_tiles]
    uint8_t *args = nullptr;                     // [packed * args_bytes] the pack's arguments per stream
    uint32_t *tables = nullptr;                  // [packed * 512] narrow pack tables: 256 x {code, len}
    uint8_t *headers = nullptr;                  // [header_bytes]
    BatchTile *tiles = nullptr;                  // [tiles] kEncTileRegions regions of one stream, from its region `first`
    uint16_t *run_bits = nullptr;                // [regions * 32] bits of every run of 64 symbols
    uint32_t *region_bits = nullptr;             // [regions] a region's bits, then the bits before it inside its scan group
    unsigned long long *group_prefix = nullptr;  // [(regions + kEncPrefixGroup - 1) / kEncPrefixGroup] bits before each scan group
    unsigned long long *region_end = nullptr;    // [regions] last bit + 1 of each region, in its stream's body
    uint8_t *seam_head = nullptr;                // [regions]
    uint8_t *seam_tail = nullptr;                // [regions]
    size_t counts_bytes = 0;                     // counts, from the start of the block
    size_t hist_begin = 0, hist_end = 0;         // hist_tiles
    size_t upload_begin = 0, upload_end = 0;     // args .. tiles
    size_t host_bytes = 0;                       // counts .. tiles
    size_t bytes = 0;
};

inline EncBatchLayout enc_batch_layout(void *base, uint32_t items, uint64_t hist_tiles, uint32_t packed, size_t args_bytes,
                                       uint64_t header_bytes, uint64_t tiles, uint64_t regions) {
    EncBatchLayout L;
    Carve c{static_cast<uint8_t *>(base)};
    L.counts = c.take<unsigned long long>((size_t)items * 256);
    L.counts_bytes = c.bytes;
    L.hist_tiles = c.take<EncHistTile>(hist_tiles);
    L.hist_begin = c.bytes - hist_tiles * sizeof(EncHistTile);
    L.hist_end = c.bytes;
    L.args = c.take<uint8_t>((size_t)packed * args_bytes);
    L.upload_begin = c.bytes - (size_t)packed * args_bytes;
    L.tables = c.take<uint32_t>((size_t)packed * 512);
    L.headers = c.take<uint8_t>(header_bytes);
    L.tiles = c.take<BatchTile>(tiles);
    L.upload_end = L.host_bytes = c.bytes;
    L.run_bits = c.take<uint16_t>(regions * 32);
    L.region_bits = c.take<uint32_t>(regions);
    L.group_prefix = c.take<unsigned long long>((regions + kEncPrefixGroup - 1) / kEncPrefixGroup);
    L.region_end = c.take<unsigned long long>(regions);
    L.seam_head = c.take<uint8_t>(regions);
    L.seam_tail = c.take<uint8_t>(regions);
    L.bytes = c.bytes;
    return L;
}

}  // namespace et
