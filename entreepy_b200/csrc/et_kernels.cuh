// Launch wrappers for the sm_100a kernels (definitions in et_hist.cu, et_pack.cu, et_unpack.cu).
#pragma once
#include <cuda_runtime.h>

#include "et_internal.h"
#include "et_scratch.h"

namespace et {

// ---------------------------------------------------------------- K1
constexpr int kHistThreads = 512;
// counts (device, 256 x u64) must be zeroed by the caller; the kernel adds into it.
cudaError_t launch_histogram(const uint8_t *d_in, size_t n, unsigned long long *d_counts, int num_sms,
                             cudaStream_t stream);

// ---------------------------------------------------------------- K2
constexpr int kPackThreads = 256;
constexpr int kPackItems = 16;  // symbols per thread per tile (one 16-byte load)
constexpr int kPackTileSyms = kPackThreads * kPackItems;

struct PackGeometry {
    const uint8_t *in_aligned;  // d_in rounded down to 16 bytes
    uint32_t misalign;          // d_in - in_aligned
    uint64_t v_end;             // misalign + n (virtual end)
    uint32_t num_tiles;
};
PackGeometry pack_geometry(const void *d_in, size_t n);

// Device scratch the pack kernels need (pack_layout(), et_scratch.h).
size_t pack_scratch_bytes(const PackGeometry &g);

// d_tables: narrow -> 256 x {code, len} (u32 pairs); wide -> 256 x u64 codes followed by 256 x u8 lengths.
// max_len: longest code (sizes the bit image of a warp on the narrow path).
// bits_ctas_per_sm: from pack_init_device() (0: ask the runtime at every call).
cudaError_t launch_pack(const PackGeometry &g, const void *d_tables, bool wide, uint32_t max_len, uint8_t *d_out, uint32_t bit_phase,
                        void *scratch_base, int num_sms,
                        cudaStream_t stream, int *launches, bool single_pass = false, int bits_ctas_per_sm = 0);
// Once per context: lets the pack kernels use all of an SM's shared memory and reads how many CTAs of pass A fit an SM
// (both used to be asked of the runtime at every call, a few microseconds each with the GPU waiting).
cudaError_t pack_init_device(int max_smem, int *bits_ctas_per_sm);

// ---------------------------------------------------------------- K3-K5 (chunked self-synchronising decoder)
constexpr int kSubseqBits = 128;    // a piece: the unit the stream is read in (one 16-byte load)

// Where the stream sits relative to the 16-byte grid the pieces are cut on.  All bit
// positions are relative to body_aligned.
struct UnpackGeometry {
    const uint8_t *body_aligned;  // 16-byte aligned base
    uint64_t byte_lo, byte_hi;    // readable bytes: [byte_lo, byte_hi)
    uint64_t own_begin_bit;       // symbols that begin in [own_begin_bit, own_end_bit) are decoded
    uint64_t own_end_bit;
    uint64_t end_bit;             // no code may extend past this bit (end of the stream / of the readable range)
    bool head_known;              // head_bit is a true codeword boundary (else the first entry is a guess)
    uint64_t head_bit;
};
UnpackGeometry unpack_geometry(const void *d_body, size_t body_bytes);
// A shard: d_range 16-byte aligned, own_begin_byte a multiple of 16, own_end_byte a multiple of 16
// unless the stream ends there; range_bytes >= own_end_byte + 32 unless the stream ends there.
// head_bit < 0: the first codeword boundary is unknown (found by run-up from the bytes before own_begin_byte).
UnpackGeometry unpack_geometry_shard(const void *d_range, size_t range_bytes, size_t own_begin_byte, size_t own_end_byte,
                                     long long head_bit);

constexpr uint32_t kErrInvalidCode = 2u;

// Per-context decoder settings: device properties read once by unpack_init_device() and the knobs of
// et_ctx_set_tuning().
struct UnpackTuning {
    long long lane_min_bytes = -1;  // bodies of at least this many bytes take the lane-interleaved decoder (-1: default)
    int debug = 0;
    int max_smem = 0;  // cudaDevAttrMaxSharedMemoryPerBlockOptin
    int num_sms = 0;
    int sync_warps = 0;             // > 0: warps per CTA of the count walk (default: as many as fit)
    int write_warps = 0;            // > 0: warps per CTA of the write walk (default: as many as fit)
    int no_transfer = 0;            // non-zero: slowly synchronising codes take the repair rounds instead of transfer functions
    int pack_single_pass = 0;       // non-zero: the encoder packs in ONE pass with a decoupled look-back (measured slower, see et_pack.cu)
    int pack_bits_ctas = 0;         // CTAs of pack pass A per SM (pack_init_device)
    void *d_lane_tables = nullptr;  // device-built tables of the lane-interleaved decoder
};
cudaError_t unpack_init_device(int device, UnpackTuning *tune);
void unpack_free_device(UnpackTuning *tune);

// Chunk size for this stream (bytes per thread) and the device scratch the decoder needs (decode_layout(), et_scratch.h).
uint32_t unpack_chunk_bytes(const UnpackGeometry &g, const UnpackTuning &tune, uint32_t min_length, uint32_t max_length);
size_t unpack_scratch_bytes(const UnpackGeometry &g, uint32_t chunk_bytes, uint32_t transfer_states);
// Writes min(total, max_symbols) bytes to d_out.  Blocks on the stream between check rounds; on return the
// stream is idle and h_status (pinned host memory) holds the status words the decode ended with (DecodeStatus:
// error flags, symbols found, entry used by the first chunk, exit of the last chunk).
// d_slots: slot of every marker window (kLutSize x u16) followed by the second-level tables (launch_build_tables).
// *rounds_out = passes over the chunk entries it took (2 = the guesses plus one repair round sufficed).
// fixed_len: the dictionary is a complete code whose codes all have this many bits (0: it is not) — such a
// stream never re-synchronises, but every chunk's entry follows from the first one in closed form.
// transfer_states: > 0 for codes that synchronise slowly (lengths within 2 bits of each other): the number of bit
// offsets at which a chunk can be entered (= the longest code); the per-thread path then tabulates every chunk's
// transfer function and scans instead of running repair rounds.
cudaError_t launch_unpack(const UnpackGeometry &g, uint32_t chunk_bytes, const uint32_t *d_clut, const uint32_t *d_wlut,
                          const uint32_t *d_nodes, const uint16_t *d_slots, uint8_t *d_out, uint64_t max_symbols, void *scratch_base,
                          DecodeStatus *h_status, cudaStream_t stream, const UnpackTuning &tune, uint32_t fixed_len, uint32_t transfer_states,
                          int *launches, uint32_t *rounds_out);

// The decoder's first-level tables (et_internal.h) from the uploaded trie, on the device.
cudaError_t launch_build_tables(const uint32_t *d_nodes, uint32_t *d_clut, uint16_t *d_slots, uint32_t *d_work, cudaStream_t stream,
                                int *launches);

// ---------------------------------------------------------------- synthetic input generator
cudaError_t launch_synth(uint8_t *d_out, size_t n, uint64_t seed, uint64_t first_index, const uint32_t *d_thresholds,
                         cudaStream_t stream);

}  // namespace et
