/*
 * entreepy_b200.h — C ABI of the B200-native Huffman compress/decompress path.
 *
 * Drop-in boundary for typio/entreepy's codec seam.  The reference has no FFI layer; its
 * narrowest seam is the two public functions
 *     encode(allocator, text, out_writer, std_out, flags) !usize      (src/encode.zig:25)
 *     decode(allocator, compressed_text, out_writer, std_out, flags) !usize (src/decode.zig:13)
 * called from src/main.zig:202,204 and src/test.zig:15,26.  A Zig (or any other) host binds
 * the entry points below with `extern fn` and keeps those two signatures (INTEGRATION.md).
 *
 * Conventions: plain pointers and sizes only, no exceptions cross the boundary, every entry
 * point returns an et_status.  A context is thread-compatible (one caller at a time).
 * There is NO CPU fallback: entry points that compute on the stream fail with
 * ET_ERR_NO_DEVICE / ET_ERR_CUDA when no sm_100 device is usable.
 */
#ifndef ENTREEPY_B200_H
#define ENTREEPY_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ET_ABI_VERSION 1

#if defined(__GNUC__)
#define ET_API __attribute__((visibility("default")))
#else
#define ET_API
#endif

/* ------------------------------------------------------------------ status codes */
typedef enum et_status {
    ET_OK = 0,
    ET_ERR_QUEUE_EMPTY = 1,   /* empty input: QueueError.QueueEmpty, queue.zig:28 via encode.zig:138 */
    ET_ERR_NO_SPACE = 2,      /* NoSpaceLeft: output > caller capacity or > reference scratch (encode.zig:253-254) */
    ET_ERR_OUT_OF_MEMORY = 3, /* error.OutOfMemory (host or device allocation) */
    ET_ERR_CUDA = 4,          /* a CUDA call failed; et_last_error() has the text */
    ET_ERR_NO_DEVICE = 5,     /* no CUDA device / not sm_100: there is no CPU fallback */
    ET_ERR_CORRUPT = 6,       /* .et stream cannot be parsed / is not a prefix code */
    ET_ERR_TOO_LARGE = 7,     /* n > 2^32-1: body length field is 4 bytes (encode.zig:279, decode.zig:36-42) */
    ET_ERR_UNSUPPORTED = 8,   /* e.g. dictionary code length > 32 on decode (decode.zig:49 holds [32]u8) */
    ET_ERR_INVALID_ARG = 9
} et_status;

/* ------------------------------------------------------------------ flags
 * EncodeFlags (encode.zig:9-14) / DecodeFlags (decode.zig:7-11). */
#define ET_FLAG_WRITE_OUTPUT 0x1u /* write_output */
#define ET_FLAG_PRINT_OUTPUT 0x2u /* print_output: decode streams the text to the output fd (decode.zig:189) */
#define ET_FLAG_DEBUG 0x4u        /* debug: dictionary dump, "bits in output", "time taken" (encode.zig:27,205-211,320) */
/* extensions (not in the reference) */
#define ET_FLAG_QUIET 0x100u             /* suppress the "X => Y" stderr summary (encode.zig:334, decode.zig:217) */
#define ET_FLAG_NO_SCRATCH_LIMIT 0x200u  /* lift the reference's 7200+n scratch bound (encode.zig:253) */
/* decode: the input validation the reference leaves as a TODO (main.zig:199).  With the flag a dictionary that is
 * not a complete prefix code, or a body too short for body_len symbols, is ET_ERR_CORRUPT before anything is
 * decoded.  Without it acceptance follows the reference: whatever parses is decoded (when two dictionary
 * entries collide the shorter code wins, as decode.zig:181 tries lengths from the shortest up). */
#define ET_FLAG_VALIDATE 0x400u
#define ET_FLAG_TIMING 0x800u            /* *_dev calls: record per-stage CUDA events (et_ctx_last_stage_ms), print nothing */

/* ------------------------------------------------------------------ code tables */
/* Code{data:u32,length:u8}, encode.zig:141-144.  data keeps only the low 32 path bits. */
typedef struct et_code {
    uint32_t data;
    uint8_t length;
} et_code;

typedef struct et_codebook {
    et_code code[256];    /* dictionary[256], encode.zig:146; length 0 = symbol has no code */
    uint32_t n_symbols;   /* leaves that entered the tree (symbols_length, encode.zig:79) */
    uint32_t n_entries;   /* codes with length > 0 (encode.zig:270-273) */
    uint32_t min_length;  /* over entries; 0 when n_entries == 0 */
    uint32_t max_length;
    uint64_t body_bits;   /* sum count*length: bits the body occupies before the final pad */
} et_codebook;

/* Parsed .et dictionary (decode.zig:34-141).  `in` handed to the parser is file[4..]. */
typedef struct et_dictionary {
    uint32_t n_entries;    /* entries read: in[0] + 1 as u8 (decode.zig:34), fewer when the bytes ran out first */
    uint32_t body_len;     /* symbols to decode, BE u32 (decode.zig:36-42) */
    uint64_t body_offset;  /* byte offset of the body inside `in` (decode.zig:136,156) */
    uint8_t symbol[256];
    uint8_t length[256];
    uint64_t code[256];
    uint32_t min_length, max_length;
    uint32_t truncated;    /* the stream ended inside the dictionary: the body is empty (decode.zig:66,135-140) */
} et_dictionary;

typedef struct et_ctx et_ctx;

/* ------------------------------------------------------------------ context */
ET_API int et_abi_version(void);
ET_API const char *et_strerror(int status);
/* Creates a context on CUDA device `device` (streams, device scratch, pinned staging). */
ET_API int et_ctx_create(int device, et_ctx **out);
ET_API void et_ctx_destroy(et_ctx *ctx);
ET_API const char *et_last_error(const et_ctx *ctx);
/* fd that plays the role of the reference's `std_out` argument (default 1). */
ET_API int et_ctx_set_output_fd(et_ctx *ctx, int fd);
/* Kernels launched by this context since creation (bench.py's gpu_launches). */
ET_API uint64_t et_ctx_kernel_launches(const et_ctx *ctx);
/* Milliseconds the last et_encode_dev / et_decode_dev call spent per stage, measured with
 * CUDA events on the launching stream.  encode: [0]=histogram kernel + 2 KiB read-back,
 * [1]=host codebook/header, [2]=pack + seam fix-up kernels.  decode: [0]=header read-back and
 * dictionary parse, [1]=table upload, [2]=decode kernels.  [3]=0.  et_histogram_dev: [0]=kernel + read-back.
 * et_encode_dev / et_decode_dev fill it only when ET_FLAG_TIMING or ET_FLAG_DEBUG was passed. */
ET_API int et_ctx_last_stage_ms(const et_ctx *ctx, float ms[4]);

/* Passes over the chunk entries in the last decode: 2 = the guessed entries plus one repair round were enough
 * (self-synchronising streams); more = that many fixpoint rounds were needed (slowly synchronising codes). */
ET_API uint32_t et_ctx_last_decode_rounds(const et_ctx *ctx);

/* Tuning knobs of a context (tests and benchmarks; the defaults are what production wants).  The environment
 * variables ET_LANE_MIN_BYTES and ET_DEBUG_LANES seed the first two when the context is created. */
#define ET_TUNE_LANE_MIN_BYTES 1 /* bodies of at least this many bytes take the lane-interleaved decoder; -1 = default */
#define ET_TUNE_DEBUG 2          /* bit 0: lane decoder timings per decode on stderr; bit 1: host time of the phases of a sharded call (rank 0) */
#define ET_TUNE_NO_TRANSFER 5     /* non-zero: slowly synchronising codes are decoded with repair rounds (round 1's way) instead of
                                     the scan of per-chunk transfer functions */
/* Keys 3, 4 and 6 are retired (they selected measured-and-rejected kernel variants) and must not be reused. */
ET_API int et_ctx_set_tuning(et_ctx *ctx, int key, long long value);

/* Pinned host memory for full-rate host<->device copies in et_encode/et_decode. */
ET_API int et_alloc_pinned(size_t bytes, void **out);
ET_API void et_free_pinned(void *p);

/* ------------------------------------------------------------------ host-only steps (no GPU) */
/* E2-E4: sort (encode.zig:54-74, incl. the saturating u8 index), two-queue tree
 * (encode.zig:82-138, queue.zig:9-43) and code assignment (encode.zig:141-214).
 * ET_ERR_QUEUE_EMPTY when every count is zero. */
ET_API int et_build_codebook(const uint64_t counts[256], et_codebook *cb);
/* E5: header bytes 0..H-1 (encode.zig:261-299): magic e7 c0 de, version 01, entries-1,
 * n mod 2^32 BE, bit-packed (symbol,len,code) records, zero pad to a byte. */
ET_API size_t et_header_size(const et_codebook *cb);
ET_API int et_write_header(const et_codebook *cb, uint64_t n, uint8_t *out, size_t cap, size_t *header_len);
/* E7: the reference's scratch size 7200 + n (encode.zig:253-254). */
ET_API size_t et_encode_bound(size_t n);
/* D1+D2: parse file[4..] (decode.zig:34-141). */
ET_API int et_parse_header(const uint8_t *in_after_magic, size_t n, et_dictionary *dict);

/* ------------------------------------------------------------------ E1: histogram (kernel K1) */
/* encode.zig:43-47.  Host-buffer and device-buffer forms. `stream` is a cudaStream_t
 * (NULL = the context's own stream). */
ET_API int et_histogram(et_ctx *ctx, const uint8_t *in, size_t n, uint64_t counts[256]);
ET_API int et_histogram_dev(et_ctx *ctx, const void *d_in, size_t n, uint64_t counts[256], void *stream);

/* ------------------------------------------------------------------ encode / decode */
/* encode.zig:25.  Writes the complete .et file into out[0..*out_len).  Without
 * ET_FLAG_WRITE_OUTPUT nothing is written but *out_len is still the file size
 * (encode.zig:319,336). */
ET_API int et_encode(et_ctx *ctx, const uint8_t *in, size_t n, uint8_t *out, size_t cap, size_t *out_len, uint32_t flags);
/* decode.zig:13.  `in` is file[4..] exactly as main.zig:204 / test.zig:26 pass it.
 * *out_len = bytes written (0 on a dry run, decode.zig:187,219).  The text is min(body_len, symbols the body holds)
 * symbols; when that is more than `cap`, the decoders (this one, et_decode_dev and the batch) return ET_ERR_NO_SPACE
 * with *out_len = 0 and the first `cap` bytes of the text written to out. */
ET_API int et_decode(et_ctx *ctx, const uint8_t *in_after_magic, size_t n, uint8_t *out, size_t cap, size_t *out_len,
              uint32_t flags);
/* Same, input and output resident in device memory (no PCIe bulk copies). */
ET_API int et_encode_dev(et_ctx *ctx, const void *d_in, size_t n, void *d_out, size_t cap, size_t *out_len, uint32_t flags,
                  void *stream);
ET_API int et_decode_dev(et_ctx *ctx, const void *d_in_after_magic, size_t n, void *d_out, size_t cap, size_t *out_len,
                  uint32_t flags, void *stream);

/* Batched device decode: many independent streams in one call, for workloads of many small .et objects, where a call
 * per stream would spend its time on launches and host synchronisations.  Item i ends with the status, *out_len and
 * d_out bytes that et_decode_dev(ctx, d_in, n, d_out, cap, &out_len, flags, stream) would give it, including every
 * failure (corrupt dictionary or body, ET_FLAG_VALIDATE rejections, ET_ERR_NO_SPACE, truncated dictionaries, dry
 * runs); a failing item does not affect the others.  Items may share d_in.  Returns ET_OK once every item has its
 * status; fails only for invalid arguments (items == NULL with count > 0: ET_ERR_INVALID_ARG) or a CUDA error or
 * allocation failure, whose status is then also written into every item not yet finished.  count == 0 is ET_OK.
 * Streams that et_decode_dev decodes with the per-thread chunk kernels are decoded together, with a fixed number of
 * launches per group of up to 512 streams; longer bodies (lane decoder) and slowly synchronising codes that take
 * transfer functions are decoded one by one after them.  ET_FLAG_TIMING: et_ctx_last_stage_ms covers the whole call
 * ([0] heads and parse, [1] tables, [2] decode kernels); et_ctx_last_decode_rounds is the largest over the batch. */
typedef struct et_batch_item {
    const void *d_in; /* device memory, any alignment: file[4..] of one stream (decode) | one text (encode) */
    size_t n;
    void *d_out;      /* device memory, any alignment: the text (decode) | the whole .et file (encode) */
    size_t cap;
    size_t out_len;   /* out: bytes written (decode) | the file size, also on a dry run (encode) */
    int status;       /* out: et_status of this item */
} et_batch_item;
ET_API int et_decode_batch_dev(et_ctx *ctx, et_batch_item *items, size_t count, uint32_t flags, void *stream);

/* Batched device encode: many independent texts in one call, the other direction of et_decode_batch_dev.  Item i ends
 * with the status, *out_len and d_out bytes that et_encode_dev(ctx, d_in, n, d_out, cap, &out_len, flags, stream) would
 * give it, including every failure (d_in == NULL with n > 0 or ET_FLAG_WRITE_OUTPUT with d_out == NULL:
 * ET_ERR_INVALID_ARG; n == 0: ET_ERR_QUEUE_EMPTY; n > 2^32-1: ET_ERR_TOO_LARGE, before any byte is read;
 * ET_ERR_NO_SPACE) and dry runs (*out_len = the file size, nothing written); a failing item does not affect the others.
 * Items may share d_in.  Call-level behaviour as et_decode_batch_dev's.  Texts are handled in groups of up to 512 texts
 * and 256 MiB: per group one histogram launch, one synchronise, the codebooks and headers on the host, one upload and a
 * fixed number of pack launches.  Texts whose codes are longer than 32 bits, and texts of at least 256 MiB, are
 * encoded one by one after their group, as et_encode_dev encodes them.  ET_FLAG_TIMING or ET_FLAG_DEBUG:
 * et_ctx_last_stage_ms covers the whole call ([0] histograms and counts read-back, [1] host codebooks, headers and
 * upload, [2] pack kernels); nothing is printed. */
ET_API int et_encode_batch_dev(et_ctx *ctx, et_batch_item *items, size_t count, uint32_t flags, void *stream);

/* ------------------------------------------------------------------ sharded path (SURVEY §8e) */
/* One .et stream across several GPUs: each rank owns a contiguous byte range of the text
 * (encode) or of the body (decode); the host exchanges only the 2 KiB histogram, one bit
 * count and one byte per rank (encode) and three words per rank (decode).
 *
 * Encode shard: pack d_in[0..n) with `cb` so that its first code bit lands at bit
 * `bit_phase` (0..7) of d_out[0]; bits before it are left zero, so the seam byte of two
 * adjacent shards is the OR of their two copies.  shard_bits = et_shard_bits(local counts, cb).
 * *out_bytes = ceil((bit_phase + shard_bits) / 8). */
ET_API int et_pack_shard_dev(et_ctx *ctx, const void *d_in, size_t n, const et_codebook *cb, uint32_t bit_phase,
                      uint64_t shard_bits, void *d_out, size_t cap, size_t *out_bytes, void *stream);
/* Bits a shard with these local counts occupies under `cb` (the cross-GPU scan input). */
ET_API uint64_t et_shard_bits(const uint64_t counts[256], const et_codebook *cb);
/* Decode shard.  d_range (16-byte aligned) holds range_bytes of the body; the symbols that BEGIN
 * in its bytes [own_begin_byte, own_end_byte) are decoded to d_out.  own_begin_byte is a multiple
 * of 32; own_end_byte is a multiple of 32 followed by at least 32 bytes of look-ahead, or equals
 * range_bytes when the stream ends there.  head_bit >= 0: bit (from d_range) of a known codeword
 * boundary in the first 64 bits of the owned part; head_bit < 0: unknown — the decoder
 * synchronises on the bytes before own_begin_byte (give it >= 32) and reports what it found.
 * *entry_bit = where the first owned codeword began, *exit_bit = first codeword boundary at or
 * after own_end_byte*8 (both from d_range): rank r's entry must equal rank r-1's exit, which the
 * host checks after one all-gather; a rank whose entry was wrong calls again with head_bit.
 * ET_ERR_NO_SPACE when the shard holds more than `cap` symbols (*n_symbols is then the number found). */
ET_API int et_unpack_shard_dev(et_ctx *ctx, const void *d_range, size_t range_bytes, size_t own_begin_byte,
                        size_t own_end_byte, const et_dictionary *dict, int64_t head_bit, void *d_out, size_t cap,
                        uint64_t *n_symbols, uint64_t *entry_bit, uint64_t *exit_bit, void *stream);

/* ------------------------------------------------------------------ sharded path, the whole protocol of one rank */
/* The exchanges of the sharded path are all-gathers of a few hundred bytes per rank.  An et_comm carries them:
 * over NCCL (libnccl.so.2 is opened at run time; rank 0 makes an id with et_comm_unique_id and hands it to the
 * others by whatever means the host program has), or through a host callback. */
#define ET_COMM_ID_BYTES 128 /* = NCCL_UNIQUE_ID_BYTES */
typedef struct et_comm et_comm;
/* Gathers `bytes` from every rank: send -> recv[rank * bytes] on all ranks (host memory).  0 = ok. */
typedef int (*et_allgather_fn)(void *user, const void *send, void *recv, size_t bytes);
ET_API int et_comm_unique_id(uint8_t out[ET_COMM_ID_BYTES]);
ET_API int et_comm_create_nccl(et_ctx *ctx, const uint8_t id[ET_COMM_ID_BYTES], int rank, int world, et_comm **out);
ET_API int et_comm_create_callback(et_ctx *ctx, int rank, int world, et_allgather_fn fn, void *user, et_comm **out);
ET_API void et_comm_destroy(et_comm *comm);

typedef struct et_shard_encoded {
    uint64_t n_total;      /* bytes of the whole text (sum of the ranks' n_local) */
    uint64_t total_bytes;  /* size of the whole .et file */
    uint64_t body_bytes;
    uint64_t bit_offset;   /* bit of the body at which this rank's first code sits (the cross-GPU exclusive scan) */
    uint64_t first_byte;   /* body byte index of d_out[0] */
    uint64_t local_bytes;  /* bytes this rank wrote: d_out[0 .. local_bytes) */
    uint64_t own_lo, own_hi; /* body bytes [own_lo, own_hi) are final in this rank's buffer: the .et file is the header
                                followed by every rank's d_out[own_lo - first_byte .. own_hi - first_byte) in rank order */
    uint32_t header_len;
    uint8_t header[4096];  /* magic .. dictionary pad: the same on every rank */
} et_shard_encoded;
/* encode() of SURVEY §8e for one rank: histogram of the rank's slice, ONE all-gather (histograms, text heads,
 * lengths), codebook + header + bit-offset scan on every rank alike, pack at the final bit position, seam byte.
 * d_out needs ceil((7 + bits of the slice) / 8) bytes; n_local + 16 is what the 7200+n bound guarantees. */
ET_API int et_encode_sharded_dev(et_ctx *ctx, et_comm *comm, const void *d_in, size_t n_local, void *d_out, size_t cap,
                          et_shard_encoded *res, uint32_t flags, void *stream);

typedef struct et_shard_decoded {
    uint64_t n_local;  /* valid symbols in d_out */
    uint64_t offset;   /* position of the first of them in the text */
    uint64_t body_len; /* symbols of the whole stream (the header's length field) */
    uint32_t rounds;   /* 1 = every rank's guessed entry was right */
} et_shard_decoded;
/* decode() of SURVEY §8e for one rank.  header_after_magic: the .et bytes after the magic up to the body (every rank
 * has them); d_range / own_*_byte as for et_unpack_shard_dev; starts_body: this rank's share begins with the body
 * (its first codeword is known).  Ranks whose share is empty pass own_begin_byte == own_end_byte.  One all-gather
 * per round; a rank whose guessed entry was not its left neighbour's exit decodes again from there. */
ET_API int et_decode_sharded_dev(et_ctx *ctx, et_comm *comm, const uint8_t *header_after_magic, size_t header_len, const void *d_range,
                          size_t range_bytes, size_t own_begin_byte, size_t own_end_byte, int starts_body, void *d_out, size_t cap,
                          et_shard_decoded *res, uint32_t flags, void *stream);

/* ------------------------------------------------------------------ synthetic inputs (bench/test utility) */
/* out[i] = smallest s with thresholds[s] > (splitmix64(seed + first_index + i) >> 32);
 * same definition as entreepy_b200/synth.py on the CPU. */
ET_API int et_synth_dev(et_ctx *ctx, void *d_out, size_t n, uint64_t seed, uint64_t first_index,
                 const uint32_t thresholds[256], void *stream);

#ifdef __cplusplus
}
#endif
#endif /* ENTREEPY_B200_H */
