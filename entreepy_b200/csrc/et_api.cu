// C-ABI layer (include/entreepy_b200.h): context, orchestration of the kernels, host<->device
// staging.  Mirrors encode() (encode.zig:25) and decode() (decode.zig:13) behaviour: sizes,
// error mapping, dry-run results and the text the reference prints.
#include <unistd.h>

#include <algorithm>
#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "et_kernels.cuh"

using namespace et;

constexpr size_t kMaxHeaderBytes = 4096;

// The small fixed block of a context; the device copy and its pinned host mirror share this layout.
struct SmallBlock {
    alignas(128) unsigned long long counts[256];
    alignas(128) uint8_t pack_tables[2048 + 256];      // narrow: 256 x {code, len} u32 | wide: 256 x u64 codes, 256 x u8 lengths
    alignas(128) uint32_t lut[2 * kLutSize];            // clut | wlut
    alignas(128) uint32_t nodes[kMaxTrieNodes];         // the dictionary's trie
    alignas(128) uint16_t slots[kLutSize + (kMaxSubTables << kSubBits)];  // slot of a marker window | second-level tables
    alignas(128) uint32_t thresholds[256];              // et_synth_dev
    alignas(128) DecodeStatus status;                   // host copy: what the last decode read back
    alignas(128) uint32_t table_work[32];               // slot counter + slot windows of launch_build_tables
    alignas(128) uint8_t header[kMaxHeaderBytes];       // header staging
};

struct ncclUniqueIdBytes {  // layout of ncclUniqueId (nccl.h): passed by value to ncclCommInitRank
    char b[ET_COMM_ID_BYTES];
};

struct et_ctx {
    int device = 0;
    int num_sms = 0;
    cudaStream_t stream = nullptr;       // context-owned stream (used when the caller passes none)
    cudaStream_t copy_stream = nullptr;  // second stream for overlapped host copies (uploads)
    cudaStream_t copy_stream2 = nullptr; // third stream: downloads, so that both directions of the link run at once
    cudaEvent_t ev[8] = {};
    // device scratch, grown on demand
    void *d_scratch = nullptr;
    size_t scratch_cap = 0;
    SmallBlock *d_small = nullptr;  // fixed block: counts, tables, LUT, trie, thresholds
    SmallBlock *h_small = nullptr;  // pinned mirror of d_small: staging of the header, counts and decode status
    // bulk staging for the host-buffer entry points
    uint8_t *d_in = nullptr, *d_out = nullptr;
    size_t d_in_cap = 0, d_out_cap = 0;
    int out_fd = 1;
    uint64_t launches = 0;
    float stage_ms[4] = {0, 0, 0, 0};
    uint32_t last_decode_rounds = 0;  // passes over the chunk entries in the last decode (2 = guesses + one repair round sufficed)
    UnpackTuning tune;                // device properties + et_ctx_set_tuning() knobs
    UnpackTrie *trie = nullptr;       // host scratch of the dictionary parser (80 KB: not on the stack)
    uint8_t *h_batch = nullptr;       // pinned mirror of a batch group's scratch (et_batch.inc), grown on demand
    size_t h_batch_cap = 0;
    uint32_t fixed_len = 0;           // the uploaded decoder tables are a complete code whose codes all have this length (0: not so)
    char err[512] = {0};
};

namespace {

int fail(et_ctx *ctx, int status, const char *fmt, ...) {
    if (ctx) {
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(ctx->err, sizeof ctx->err, fmt, ap);
        va_end(ap);
    }
    return status;
}

#define ET_CUDA(ctx, call)                                                                        \
    do {                                                                                          \
        cudaError_t e_ = (call);                                                                  \
        if (e_ != cudaSuccess)                                                                    \
            return fail(ctx, e_ == cudaErrorMemoryAllocation ? ET_ERR_OUT_OF_MEMORY : ET_ERR_CUDA, \
                        "%s: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__);     \
    } while (0)

int ensure_scratch(et_ctx *ctx, size_t bytes) {
    if (bytes <= ctx->scratch_cap) return ET_OK;
    if (ctx->d_scratch) cudaFree(ctx->d_scratch);
    ctx->d_scratch = nullptr;
    ctx->scratch_cap = 0;
    const size_t want = bytes + bytes / 4 + 4096;
    ET_CUDA(ctx, cudaMalloc(&ctx->d_scratch, want));
    ctx->scratch_cap = want;
    return ET_OK;
}
int ensure_bulk(et_ctx *ctx, uint8_t **buf, size_t *cap, size_t bytes) {
    if (bytes <= *cap) return ET_OK;
    if (*buf) cudaFree(*buf);
    *buf = nullptr;
    *cap = 0;
    const size_t want = ((bytes + 4096) + 255) & ~(size_t)255;
    ET_CUDA(ctx, cudaMalloc(reinterpret_cast<void **>(buf), want));
    *cap = want;
    return ET_OK;
}

void fd_printf(int fd, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    const int n = vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (n > 0) (void)!write(fd, buf, (size_t)std::min<int>(n, (int)sizeof buf - 1));
}

// encode.zig:205-211: leaves in the order the explicit stack visits them (left before
// right), i.e. ascending code order; "{c} {} - " then the code bits.
void print_dictionary(int fd, const et_codebook &cb) {
    std::vector<int> syms;
    for (int s = 0; s < 256; ++s)
        if (cb.code[s].length > 0) syms.push_back(s);
    auto key = [&](int s) {
        const et_code &c = cb.code[s];
        const unsigned len = std::min<unsigned>(c.length, 32);
        return len ? ((uint64_t)c.data << (32 - len)) & 0xFFFFFFFFull : 0ull;
    };
    std::sort(syms.begin(), syms.end(), [&](int a, int b) { return key(a) < key(b); });
    for (int s : syms) {
        std::string line;
        line.push_back((char)s);
        line += " " + std::to_string(s) + " - ";
        const et_code &c = cb.code[s];
        for (unsigned j = c.length; j > 0; --j) line.push_back(((c.data >> ((j - 1) & 31u)) & 1u) ? '1' : '0');
        line.push_back('\n');
        (void)!write(fd, line.data(), line.size());
    }
}

void print_summary(double from, double to) {  // encode.zig:328-334 / decode.zig:211-217 (stderr)
    char a[64], b[64];
    format_file_size(a, sizeof a, from);
    format_file_size(b, sizeof b, to);
    fprintf(stderr, "%s => %s\n", a, b);
}

struct StageTimer {
    et_ctx *ctx;
    cudaStream_t s;
    bool on;
    void mark(int i) {
        if (on) cudaEventRecord(ctx->ev[i], s);
    }
    void finish(int n_marks) {
        ctx->stage_ms[0] = ctx->stage_ms[1] = ctx->stage_ms[2] = ctx->stage_ms[3] = 0.f;
        if (!on) return;
        for (int i = 0; i + 1 < n_marks && i < 4; ++i) cudaEventElapsedTime(&ctx->stage_ms[i], ctx->ev[i], ctx->ev[i + 1]);
    }
    // The end of a batch group's stages (marks 0..2 made): adds the times between the marks to ms[0..2].
    cudaError_t add_group(float *ms) {
        if (!on) return cudaSuccess;
        mark(3);
        const cudaError_t e = cudaEventSynchronize(ctx->ev[3]);
        if (e != cudaSuccess) return e;
        for (int k = 0; k < 3; ++k) {
            float t = 0.f;
            cudaEventElapsedTime(&t, ctx->ev[k], ctx->ev[k + 1]);
            ms[k] += t;
        }
        return cudaSuccess;
    }
};

// Histogram of a device buffer into host counts (blocks until the counts are on the host).
int histogram_dev(et_ctx *ctx, const void *d_in, size_t n, uint64_t counts[256], cudaStream_t s) {
    unsigned long long *d_counts = ctx->d_small->counts;
    ET_CUDA(ctx, cudaMemsetAsync(d_counts, 0, 2048, s));
    ET_CUDA(ctx, launch_histogram(static_cast<const uint8_t *>(d_in), n, d_counts, ctx->num_sms, s));
    if (n) ctx->launches += 1;
    ET_CUDA(ctx, cudaMemcpyAsync(ctx->h_small->counts, d_counts, sizeof ctx->h_small->counts, cudaMemcpyDeviceToHost, s));
    ET_CUDA(ctx, cudaStreamSynchronize(s));
    std::memcpy(counts, ctx->h_small->counts, sizeof ctx->h_small->counts);
    return ET_OK;
}

// Upload pack tables for `cb`; returns whether the wide kernel is needed.
int upload_pack_tables(et_ctx *ctx, const et_codebook &cb, bool *wide, cudaStream_t s) {
    PackTables t;
    const int rc = make_pack_tables(cb, &t);
    if (rc != ET_OK) return fail(ctx, rc, "code length %u cannot be emitted", cb.max_length);
    uint8_t *h = ctx->h_small->pack_tables;
    size_t bytes;
    if (t.narrow_ok) {
        std::memcpy(h, t.narrow, 2048);
        bytes = 2048;
    } else {
        std::memcpy(h, t.wide_code, 2048);
        std::memcpy(h + 2048, t.wide_len, 256);
        bytes = 2304;
    }
    *wide = !t.narrow_ok;
    ET_CUDA(ctx, cudaMemcpyAsync(ctx->d_small->pack_tables, h, bytes, cudaMemcpyHostToDevice, s));
    return ET_OK;
}

int pack_dev(et_ctx *ctx, const void *d_in, size_t n, const et_codebook &cb, uint32_t bit_phase, uint8_t *d_body,
             cudaStream_t s) {
    bool wide = false;
    int rc = upload_pack_tables(ctx, cb, &wide, s);
    if (rc != ET_OK) return rc;
    const PackGeometry g = pack_geometry(d_in, n);
    rc = ensure_scratch(ctx, pack_scratch_bytes(g));
    if (rc != ET_OK) return rc;
    int launches = 0;
    ET_CUDA(ctx, launch_pack(g, ctx->d_small->pack_tables, wide, cb.max_length, d_body, bit_phase, ctx->d_scratch, ctx->num_sms, s,
                             &launches, ctx->tune.pack_bits_ctas));
    ctx->launches += (uint64_t)launches;
    return ET_OK;
}

struct EncodePlan {
    et_codebook cb;
    size_t header_len = 0, total = 0;
};

// The file of `plan` to d_out: the header through the pinned staging, then the body behind it (pack_dev); returns once
// the stream has finished (the staging is free again).  tm (or null): marks 2 and 3 around the pack.
int write_encoded_dev(et_ctx *ctx, const void *d_in, size_t n, const EncodePlan &plan, uint8_t *d_out, cudaStream_t s, StageTimer *tm) {
    uint8_t *h_header = ctx->h_small->header;
    size_t hl = 0;
    int rc = et_write_header(&plan.cb, n, h_header, kMaxHeaderBytes, &hl);  // E5
    if (rc != ET_OK) return fail(ctx, rc, "header");
    ET_CUDA(ctx, cudaMemcpyAsync(d_out, h_header, hl, cudaMemcpyHostToDevice, s));
    if (tm) tm->mark(2);
    rc = pack_dev(ctx, d_in, n, plan.cb, 0, d_out + hl, s);  // E6
    if (rc != ET_OK) return rc;
    if (tm) tm->mark(3);
    ET_CUDA(ctx, cudaStreamSynchronize(s));
    return ET_OK;
}

// Everything between the histogram and the pack: codebook, sizes, capacity checks.
int plan_encode(et_ctx *ctx, const uint64_t counts[256], size_t n, size_t cap, uint32_t flags, EncodePlan *p) {
    const int rc = et_build_codebook(counts, &p->cb);
    if (rc != ET_OK) return fail(ctx, rc, "empty input: QueueEmpty (encode.zig:138)");
    p->header_len = et_header_size(&p->cb);
    p->total = p->header_len + (size_t)((p->cb.body_bits + 7) >> 3);
    if (p->header_len > kMaxHeaderBytes) return fail(ctx, ET_ERR_UNSUPPORTED, "header of %zu bytes", p->header_len);
    if (!(flags & ET_FLAG_NO_SCRATCH_LIMIT) && p->total > et_encode_bound(n))
        return fail(ctx, ET_ERR_NO_SPACE, "NoSpaceLeft: %zu bytes exceed the reference scratch of 7200+n (encode.zig:253)",
                    p->total);
    if ((flags & ET_FLAG_WRITE_OUTPUT) && p->total > cap)
        return fail(ctx, ET_ERR_NO_SPACE, "NoSpaceLeft: output needs %zu bytes, capacity %zu", p->total, cap);
    return ET_OK;
}

}  // namespace

// ====================================================================== context
extern "C" int et_abi_version(void) { return ET_ABI_VERSION; }

extern "C" const char *et_strerror(int status) {
    switch (status) {
        case ET_OK: return "ok";
        case ET_ERR_QUEUE_EMPTY: return "QueueEmpty (empty input)";
        case ET_ERR_NO_SPACE: return "NoSpaceLeft";
        case ET_ERR_OUT_OF_MEMORY: return "OutOfMemory";
        case ET_ERR_CUDA: return "CUDA error";
        case ET_ERR_NO_DEVICE: return "no usable CUDA device (there is no CPU fallback)";
        case ET_ERR_CORRUPT: return "corrupt .et stream";
        case ET_ERR_TOO_LARGE: return "input longer than 2^32-1 bytes";
        case ET_ERR_UNSUPPORTED: return "unsupported";
        case ET_ERR_INVALID_ARG: return "invalid argument";
    }
    return "unknown status";
}

extern "C" int et_ctx_create(int device, et_ctx **out) {
    if (!out) return ET_ERR_INVALID_ARG;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device < 0 || device >= count) {
        cudaGetLastError();
        return ET_ERR_NO_DEVICE;
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return ET_ERR_NO_DEVICE;
    if (prop.major != 10) return ET_ERR_NO_DEVICE;  // kernels are built for sm_100a only
    et_ctx *ctx = new (std::nothrow) et_ctx;
    if (!ctx) return ET_ERR_OUT_OF_MEMORY;
    ctx->device = device;
    ctx->num_sms = prop.multiProcessorCount;
    bool ok = cudaSetDevice(device) == cudaSuccess;
    ok = ok && cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) == cudaSuccess;
    ok = ok && cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) == cudaSuccess;
    ok = ok && cudaStreamCreateWithFlags(&ctx->copy_stream2, cudaStreamNonBlocking) == cudaSuccess;
    for (auto &e : ctx->ev) ok = ok && cudaEventCreate(&e) == cudaSuccess;
    ok = ok && cudaMalloc(reinterpret_cast<void **>(&ctx->d_small), sizeof(SmallBlock)) == cudaSuccess;
    ok = ok && cudaHostAlloc(reinterpret_cast<void **>(&ctx->h_small), sizeof(SmallBlock), cudaHostAllocDefault) == cudaSuccess;
    ok = ok && unpack_init_device(device, &ctx->tune) == cudaSuccess;
    ok = ok && pack_init_device(ctx->tune.max_smem, &ctx->tune.pack_bits_ctas) == cudaSuccess;
    ctx->trie = new (std::nothrow) UnpackTrie;
    ok = ok && ctx->trie != nullptr;
    if (const char *v = getenv("ET_LANE_MIN_BYTES")) ctx->tune.lane_min_bytes = atoll(v);  // read once, here
    if (getenv("ET_DEBUG_LANES")) ctx->tune.debug = 1;
    if (!ok) {
        et_ctx_destroy(ctx);
        return ET_ERR_CUDA;
    }
    *out = ctx;
    return ET_OK;
}

extern "C" void et_ctx_destroy(et_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    unpack_free_device(&ctx->tune);
    delete ctx->trie;
    if (ctx->d_scratch) cudaFree(ctx->d_scratch);
    if (ctx->d_small) cudaFree(ctx->d_small);
    if (ctx->h_small) cudaFreeHost(ctx->h_small);
    if (ctx->h_batch) cudaFreeHost(ctx->h_batch);
    if (ctx->d_in) cudaFree(ctx->d_in);
    if (ctx->d_out) cudaFree(ctx->d_out);
    for (auto &e : ctx->ev)
        if (e) cudaEventDestroy(e);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->copy_stream2) cudaStreamDestroy(ctx->copy_stream2);
    delete ctx;
}

extern "C" const char *et_last_error(const et_ctx *ctx) { return ctx ? ctx->err : "no context"; }
extern "C" int et_ctx_set_output_fd(et_ctx *ctx, int fd) {
    if (!ctx) return ET_ERR_INVALID_ARG;
    ctx->out_fd = fd;
    return ET_OK;
}
extern "C" uint64_t et_ctx_kernel_launches(const et_ctx *ctx) { return ctx ? ctx->launches : 0; }
extern "C" int et_ctx_last_stage_ms(const et_ctx *ctx, float ms[4]) {
    if (!ctx || !ms) return ET_ERR_INVALID_ARG;
    std::memcpy(ms, ctx->stage_ms, sizeof ctx->stage_ms);
    return ET_OK;
}

extern "C" uint32_t et_ctx_last_decode_rounds(const et_ctx *ctx) { return ctx ? ctx->last_decode_rounds : 0; }

extern "C" int et_ctx_set_tuning(et_ctx *ctx, int key, long long value) {
    if (!ctx) return ET_ERR_INVALID_ARG;
    switch (key) {
        case ET_TUNE_LANE_MIN_BYTES: ctx->tune.lane_min_bytes = value; return ET_OK;
        case ET_TUNE_DEBUG: ctx->tune.debug = (int)value; return ET_OK;  // bit 0: lane decoder timings, bit 1: phases of the sharded calls
        case ET_TUNE_NO_TRANSFER: ctx->tune.no_transfer = value != 0; return ET_OK;
    }
    return fail(ctx, ET_ERR_INVALID_ARG, "unknown tuning key %d", key);
}

extern "C" int et_alloc_pinned(size_t bytes, void **out) {
    if (!out) return ET_ERR_INVALID_ARG;
    *out = nullptr;
    const cudaError_t e = cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return e == cudaErrorMemoryAllocation ? ET_ERR_OUT_OF_MEMORY : ET_ERR_NO_DEVICE;
    }
    return ET_OK;
}
extern "C" void et_free_pinned(void *p) {
    if (p) cudaFreeHost(p);
}

// ====================================================================== K1
extern "C" int et_histogram_dev(et_ctx *ctx, const void *d_in, size_t n, uint64_t counts[256], void *stream) {
    if (!ctx || !counts || (!d_in && n)) return ET_ERR_INVALID_ARG;
    ET_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    cudaEventRecord(ctx->ev[6], s);
    const int rc = histogram_dev(ctx, d_in, n, counts, s);  // blocks until the counts are on the host
    cudaEventRecord(ctx->ev[7], s);
    ctx->stage_ms[0] = ctx->stage_ms[1] = ctx->stage_ms[2] = ctx->stage_ms[3] = 0.f;
    if (rc == ET_OK && cudaEventSynchronize(ctx->ev[7]) == cudaSuccess) cudaEventElapsedTime(&ctx->stage_ms[0], ctx->ev[6], ctx->ev[7]);
    return rc;
}

extern "C" int et_histogram(et_ctx *ctx, const uint8_t *in, size_t n, uint64_t counts[256]) {
    if (!ctx || !counts || (!in && n)) return ET_ERR_INVALID_ARG;
    ET_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc = ensure_bulk(ctx, &ctx->d_in, &ctx->d_in_cap, n);
    if (rc != ET_OK) return rc;
    ET_CUDA(ctx, cudaMemcpyAsync(ctx->d_in, in, n, cudaMemcpyHostToDevice, ctx->stream));
    return histogram_dev(ctx, ctx->d_in, n, counts, ctx->stream);
}

// ====================================================================== encode
extern "C" int et_encode_dev(et_ctx *ctx, const void *d_in, size_t n, void *d_out, size_t cap, size_t *out_len,
                             uint32_t flags, void *stream) {
    if (!ctx || !out_len || (!d_in && n)) return ET_ERR_INVALID_ARG;
    *out_len = 0;
    if (n == 0) return fail(ctx, ET_ERR_QUEUE_EMPTY, "empty input: QueueEmpty (encode.zig:138)");
    if (n > 0xFFFFFFFFull) return fail(ctx, ET_ERR_TOO_LARGE, "n=%zu does not fit the 4-byte body length", n);
    const bool write_out = (flags & ET_FLAG_WRITE_OUTPUT) != 0;
    if (write_out && !d_out) return ET_ERR_INVALID_ARG;
    ET_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    const auto t0 = std::chrono::steady_clock::now();
    StageTimer tm{ctx, s, (flags & (ET_FLAG_DEBUG | ET_FLAG_TIMING)) != 0};

    tm.mark(0);
    uint64_t counts[256];
    int rc = histogram_dev(ctx, d_in, n, counts, s);  // E1
    if (rc != ET_OK) return rc;
    tm.mark(1);
    EncodePlan plan;
    rc = plan_encode(ctx, counts, n, cap, flags, &plan);  // E2-E4
    if (rc != ET_OK) return rc;
    if (flags & ET_FLAG_DEBUG) print_dictionary(ctx->out_fd, plan.cb);
    if (write_out) {
        rc = write_encoded_dev(ctx, d_in, n, plan, static_cast<uint8_t *>(d_out), s, &tm);
        if (rc != ET_OK) return rc;
        tm.finish(4);
    }
    *out_len = plan.total;  // returned even on a dry run (encode.zig:336)
    if (flags & ET_FLAG_DEBUG) {
        fd_printf(ctx->out_fd, "\nbits in output: %zu\n", plan.total * 8);  // encode.zig:320
        const auto us = std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t0).count();
        fd_printf(ctx->out_fd, "time taken: %lldμs\n", (long long)us);  // encode.zig:27
    }
    return ET_OK;
}

extern "C" int et_encode(et_ctx *ctx, const uint8_t *in, size_t n, uint8_t *out, size_t cap, size_t *out_len,
                         uint32_t flags) {
    if (!ctx || !out_len || (!in && n)) return ET_ERR_INVALID_ARG;
    *out_len = 0;
    if (n == 0) return fail(ctx, ET_ERR_QUEUE_EMPTY, "empty input: QueueEmpty (encode.zig:138)");
    if (n > 0xFFFFFFFFull) return fail(ctx, ET_ERR_TOO_LARGE, "n=%zu does not fit the 4-byte body length", n);
    const bool write_out = (flags & ET_FLAG_WRITE_OUTPUT) != 0;
    if (write_out && !out) return ET_ERR_INVALID_ARG;
    ET_CUDA(ctx, cudaSetDevice(ctx->device));
    const auto t0 = std::chrono::steady_clock::now();
    cudaStream_t s = ctx->stream;
    int rc = ensure_bulk(ctx, &ctx->d_in, &ctx->d_in_cap, n);
    if (rc != ET_OK) return rc;

    // E1 overlapped with the upload: the input goes up in slices on copy_stream; the
    // histogram of slice k runs on `s` while slice k+1 is still in flight.
    unsigned long long *d_counts = ctx->d_small->counts;
    ET_CUDA(ctx, cudaMemsetAsync(d_counts, 0, 2048, s));
    const size_t slice = (size_t)64 << 20;
    for (size_t off = 0; off < n; off += slice) {
        const size_t len = std::min(slice, n - off);
        ET_CUDA(ctx, cudaMemcpyAsync(ctx->d_in + off, in + off, len, cudaMemcpyHostToDevice, ctx->copy_stream));
        ET_CUDA(ctx, cudaEventRecord(ctx->ev[4], ctx->copy_stream));
        ET_CUDA(ctx, cudaStreamWaitEvent(s, ctx->ev[4], 0));
        ET_CUDA(ctx, launch_histogram(ctx->d_in + off, len, d_counts, ctx->num_sms, s));
        ctx->launches += 1;
    }
    ET_CUDA(ctx, cudaMemcpyAsync(ctx->h_small->counts, d_counts, sizeof ctx->h_small->counts, cudaMemcpyDeviceToHost, s));
    ET_CUDA(ctx, cudaStreamSynchronize(s));
    uint64_t counts[256];
    std::memcpy(counts, ctx->h_small->counts, sizeof ctx->h_small->counts);

    EncodePlan plan;
    rc = plan_encode(ctx, counts, n, cap, flags, &plan);
    if (rc != ET_OK) return rc;
    if (flags & ET_FLAG_DEBUG) print_dictionary(ctx->out_fd, plan.cb);
    if (write_out) {
        size_t hl = 0;
        rc = et_write_header(&plan.cb, n, out, cap, &hl);  // header straight into the caller's buffer
        if (rc != ET_OK) return fail(ctx, rc, "header");
        const size_t body_bytes = plan.total - hl;
        rc = ensure_bulk(ctx, &ctx->d_out, &ctx->d_out_cap, body_bytes + 16);
        if (rc != ET_OK) return rc;
        rc = pack_dev(ctx, ctx->d_in, n, plan.cb, 0, ctx->d_out, s);
        if (rc != ET_OK) return rc;
        if (body_bytes) ET_CUDA(ctx, cudaMemcpyAsync(out + hl, ctx->d_out, body_bytes, cudaMemcpyDeviceToHost, s));
        ET_CUDA(ctx, cudaStreamSynchronize(s));
    }
    *out_len = plan.total;
    if (flags & ET_FLAG_DEBUG) {
        fd_printf(ctx->out_fd, "\nbits in output: %zu\n", plan.total * 8);
        const auto us = std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t0).count();
        fd_printf(ctx->out_fd, "time taken: %lldμs\n", (long long)us);
    }
    if (!(flags & ET_FLAG_QUIET)) print_summary((double)n, (double)plan.total);
    return ET_OK;
}

extern "C" int et_pack_shard_dev(et_ctx *ctx, const void *d_in, size_t n, const et_codebook *cb, uint32_t bit_phase,
                                 uint64_t shard_bits, void *d_out, size_t cap, size_t *out_bytes, void *stream) {
    if (!ctx || !cb || !d_out || bit_phase > 7 || (!d_in && n)) return ET_ERR_INVALID_ARG;
    ET_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    const size_t bytes = (size_t)((bit_phase + shard_bits + 7) >> 3);
    if (bytes > cap) return fail(ctx, ET_ERR_NO_SPACE, "shard needs %zu bytes, capacity %zu", bytes, cap);
    StageTimer tm{ctx, s, true};
    tm.mark(0);
    tm.mark(1);
    tm.mark(2);
    if (n) {
        const int rc = pack_dev(ctx, d_in, n, *cb, bit_phase, static_cast<uint8_t *>(d_out), s);
        if (rc != ET_OK) return rc;
    }
    tm.mark(3);
    ET_CUDA(ctx, cudaStreamSynchronize(s));
    tm.finish(4);
    if (out_bytes) *out_bytes = bytes;
    return ET_OK;
}

// ====================================================================== decode
namespace {

// The dictionary's trie into ctx->trie, with ET_FLAG_VALIDATE's checks when validate.  *fixed_len (on success): the length of
// every code when they form a complete code of one length, else 0.
int make_trie(et_ctx *ctx, const et_dictionary &dict, bool validate, uint32_t *fixed_len) {
    UnpackTrie *t = ctx->trie;
    int rc = make_unpack_trie(dict, t);
    if (rc == ET_OK && validate && !t->prefix_free) rc = ET_ERR_CORRUPT;
    if (rc == ET_OK && validate && !t->complete) rc = ET_ERR_CORRUPT;
    if (rc != ET_OK) {
        const bool why_incomplete = rc == ET_ERR_CORRUPT && validate && t->prefix_free;
        return fail(ctx, rc, rc == ET_ERR_UNSUPPORTED ? "dictionary code longer than 32 bits"
                             : why_incomplete        ? "dictionary is not a complete code (Kraft sum != 1)"
                                                     : "dictionary is not a prefix code");
    }
    *fixed_len = (t->complete && t->prefix_free && dict.min_length == dict.max_length) ? dict.max_length : 0u;
    return ET_OK;
}

// The dictionary's trie goes up; the decoder's tables are derived from it on the device (launch_build_tables).
// validate: ET_FLAG_VALIDATE was passed.
int upload_unpack_tables(et_ctx *ctx, const et_dictionary &dict, cudaStream_t s, bool validate = false) {
    const int rc = make_trie(ctx, dict, validate, &ctx->fixed_len);
    if (rc != ET_OK) return rc;
    UnpackTrie *t = ctx->trie;
    std::memcpy(ctx->h_small->nodes, t->nodes, (size_t)t->n_nodes * 4);
    ET_CUDA(ctx, cudaMemcpyAsync(ctx->d_small->nodes, ctx->h_small->nodes, (size_t)t->n_nodes * 4, cudaMemcpyHostToDevice, s));
    int launches = 0;
    ET_CUDA(ctx, launch_build_tables(ctx->d_small->nodes, ctx->d_small->lut, ctx->d_small->slots, ctx->d_small->table_work, s, &launches));
    ctx->launches += (uint64_t)launches;
    return ET_OK;
}

// Bit offsets at which a chunk can be entered, for codes that synchronise slowly (lengths within 2 bits of each other); else 0.
uint32_t transfer_states_of(const et_dictionary &dict) {
    return (dict.max_length - dict.min_length <= 2 && dict.max_length <= 16) ? dict.max_length : 0u;
}

// Decode the part of a device-resident body that `g` describes: min(symbols found, max_symbols) bytes to d_out.
// *st = the status words it ended with (symbols found, entry, exit).  tables_ready: upload_unpack_tables() was
// already called for this dictionary (the pipelined host path does it before it queues the bulk uploads, which
// would otherwise delay it).
int unpack_dev(et_ctx *ctx, const UnpackGeometry &g, const et_dictionary &dict, uint8_t *d_out, uint64_t max_symbols,
               cudaStream_t s, DecodeStatus *st, StageTimer *tm = nullptr, bool tables_ready = false, bool validate = false) {
    int rc = tables_ready ? ET_OK : upload_unpack_tables(ctx, dict, s, validate);
    if (rc != ET_OK) return rc;
    if (tm) tm->mark(2);

    const uint32_t chunk_bytes = unpack_chunk_bytes(g, ctx->tune, dict.min_length, dict.max_length);
    const uint32_t transfer_states = transfer_states_of(dict);
    rc = ensure_scratch(ctx, unpack_scratch_bytes(g, chunk_bytes, transfer_states));
    if (rc != ET_OK) return rc;
    const uint32_t *d_clut = ctx->d_small->lut;
    const uint32_t *d_wlut = d_clut + kLutSize;
    int launches = 0;
    uint32_t rounds = 0;
    ET_CUDA(ctx, launch_unpack(g, chunk_bytes, d_clut, d_wlut, ctx->d_small->nodes, ctx->d_small->slots, d_out, max_symbols,
                               ctx->d_scratch, &ctx->h_small->status, s, ctx->tune, ctx->fixed_len, transfer_states, &launches, &rounds));
    ctx->launches += (uint64_t)launches;
    ctx->last_decode_rounds = rounds;
    *st = ctx->h_small->status;  // launch_unpack left the stream idle
    if (st->error_flags & kErrInvalidCode) return fail(ctx, ET_ERR_CORRUPT, "body contains a bit pattern that is not a code");
    return ET_OK;
}

// What is known about a stream before its body is touched.  Returns ET_OK with *empty = true when there is
// nothing to decode: the dictionary ended early (decode.zig:66 just runs out of bytes; the reference's own
// output for a single distinct symbol reads back like this) — the reference then returns 0 bytes.
int check_stream(et_ctx *ctx, const et_dictionary &dict, size_t n, uint32_t flags, bool *empty) {
    *empty = dict.truncated || dict.n_entries == 0;
    if (dict.body_offset > n) return fail(ctx, ET_ERR_CORRUPT, "dictionary runs past the end of the stream");
    if (!(flags & ET_FLAG_VALIDATE)) return ET_OK;
    if (*empty) {
        if (dict.n_entries == 0 && n == 5) return ET_OK;  // the 9-byte file of a single distinct symbol (encode.zig:270-275)
        return fail(ctx, ET_ERR_CORRUPT, "the stream ends inside its dictionary (%u entries read)", dict.n_entries);
    }
    const uint64_t body_bits = (uint64_t)(n - dict.body_offset) * 8;
    if ((uint64_t)dict.body_len * dict.min_length > body_bits)
        return fail(ctx, ET_ERR_CORRUPT, "body of %zu bytes cannot hold %u symbols of at least %u bits", n - (size_t)dict.body_offset,
                    dict.body_len, dict.min_length);
    return ET_OK;
}

// et_decode_dev's result for a stream in which the decoder found `total` symbols (not clipped to `cap`): *out_len, or
// NoSpaceLeft when the text, min(total, body_len) symbols, does not fit `cap`.  A text of exactly `cap` symbols fits,
// whatever body_len claims: the reference's writer only fails on a byte it cannot store.
int decode_result(et_ctx *ctx, const et_dictionary &dict, size_t cap, uint64_t total, size_t *out_len) {
    const uint64_t text = std::min<uint64_t>(total, dict.body_len);
    if (text > cap) return fail(ctx, ET_ERR_NO_SPACE, "NoSpaceLeft: %llu symbols, capacity %zu", (unsigned long long)text, cap);
    *out_len = (size_t)text;
    return ET_OK;
}

}  // namespace

extern "C" int et_decode_dev(et_ctx *ctx, const void *d_in, size_t n, void *d_out, size_t cap, size_t *out_len,
                             uint32_t flags, void *stream) {
    if (!ctx || !out_len || !d_in) return ET_ERR_INVALID_ARG;
    *out_len = 0;
    ET_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    const auto t0 = std::chrono::steady_clock::now();
    StageTimer tm{ctx, s, (flags & (ET_FLAG_DEBUG | ET_FLAG_TIMING)) != 0};
    tm.mark(0);
    // D1+D2: the dictionary is parsed on the host from the first bytes of the stream
    const size_t head = std::min(n, kMaxHeaderBytes);
    uint8_t *h_header = ctx->h_small->header;
    ET_CUDA(ctx, cudaMemcpyAsync(h_header, d_in, head, cudaMemcpyDeviceToHost, s));
    ET_CUDA(ctx, cudaStreamSynchronize(s));
    et_dictionary dict;
    int rc = et_parse_header(h_header, head, &dict);
    if (rc != ET_OK) return fail(ctx, rc, "cannot parse the .et dictionary");
    bool empty = false;
    if ((rc = check_stream(ctx, dict, n, flags, &empty)) != ET_OK) return rc;
    tm.mark(1);
    if (!(flags & ET_FLAG_WRITE_OUTPUT) || empty) return ET_OK;  // dry run: bytes_written stays 0 (decode.zig:185-188)
    if (!d_out && cap) return ET_ERR_INVALID_ARG;
    const uint64_t want = std::min<uint64_t>(dict.body_len, cap);
    DecodeStatus st;
    rc = unpack_dev(ctx, unpack_geometry(static_cast<const uint8_t *>(d_in) + dict.body_offset, n - dict.body_offset), dict,
                    static_cast<uint8_t *>(d_out), want, s, &st, &tm, false, (flags & ET_FLAG_VALIDATE) != 0);  // D3
    if (rc != ET_OK) return rc;
    tm.mark(3);
    ET_CUDA(ctx, cudaEventSynchronize(ctx->ev[3]));
    tm.finish(4);
    if ((rc = decode_result(ctx, dict, cap, st.total, out_len)) != ET_OK) return rc;
    if (flags & ET_FLAG_DEBUG) {
        const auto us = std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t0).count();
        fd_printf(ctx->out_fd, "time taken: %lldμs\n", (long long)us);  // decode.zig:16
    }
    return ET_OK;
}

extern "C" int et_decode(et_ctx *ctx, const uint8_t *in, size_t n, uint8_t *out, size_t cap, size_t *out_len,
                         uint32_t flags) {
    if (!ctx || !out_len || !in) return ET_ERR_INVALID_ARG;
    *out_len = 0;
    ET_CUDA(ctx, cudaSetDevice(ctx->device));
    const auto t0 = std::chrono::steady_clock::now();
    cudaStream_t s = ctx->stream;
    et_dictionary dict;
    int rc = et_parse_header(in, n, &dict);  // D1+D2 straight from the caller's buffer
    if (rc != ET_OK) return fail(ctx, rc, "cannot parse the .et dictionary");
    bool empty = false;
    if ((rc = check_stream(ctx, dict, n, flags, &empty)) != ET_OK) return rc;
    const bool write_out = (flags & ET_FLAG_WRITE_OUTPUT) != 0, print_out = (flags & ET_FLAG_PRINT_OUTPUT) != 0;
    const bool validate = (flags & ET_FLAG_VALIDATE) != 0;
    uint64_t produced = 0;
    if ((write_out || print_out) && !empty) {
        const size_t body_bytes = n - dict.body_offset;
        const uint64_t want = write_out ? std::min<uint64_t>(dict.body_len, cap) : dict.body_len;
        rc = ensure_bulk(ctx, &ctx->d_in, &ctx->d_in_cap, body_bytes + 16);
        if (rc != ET_OK) return rc;
        rc = ensure_bulk(ctx, &ctx->d_out, &ctx->d_out_cap, want + 16);
        if (rc != ET_OK) return rc;
        // D3, pipelined over the PCIe link: the body goes up in slices on one copy stream, each
        // slice is decoded as soon as it (and 64 bytes of the next one) has landed, and its text
        // goes back down on a second copy stream while the next slice is decoded — upload,
        // decode and download overlap (the link is full duplex).  A slice starts on the exact
        // codeword boundary at which the slice before it ended, so nothing is guessed.
        const size_t kSlice = (size_t)64 << 20;
        const size_t n_slices = body_bytes > 2 * kSlice ? (body_bytes + kSlice - 1) / kSlice : 1;
        if (n_slices == 1) {
            if (body_bytes)
                ET_CUDA(ctx, cudaMemcpyAsync(ctx->d_in, in + dict.body_offset, body_bytes, cudaMemcpyHostToDevice, s));
            DecodeStatus st;
            rc = unpack_dev(ctx, unpack_geometry(ctx->d_in, body_bytes), dict, ctx->d_out, want, s, &st, nullptr, false, validate);
            if (rc != ET_OK) return rc;
            produced = std::min<uint64_t>(st.total, want);
            if (write_out) {  // the first cap bytes go home even when the text does not fit, as from et_decode_dev
                if (produced) ET_CUDA(ctx, cudaMemcpyAsync(out, ctx->d_out, produced, cudaMemcpyDeviceToHost, s));
                ET_CUDA(ctx, cudaStreamSynchronize(s));
                size_t fits = 0;  // *out_len is set below
                if ((rc = decode_result(ctx, dict, cap, st.total, &fits)) != ET_OK) return rc;
            }
        } else {
            rc = upload_unpack_tables(ctx, dict, s, validate);  // before the bulk uploads: copies in one direction run in issue order
            if (rc != ET_OK) return rc;
            std::vector<cudaEvent_t> up(n_slices, nullptr);
            auto cleanup = [&]() {
                for (auto &e : up)
                    if (e) cudaEventDestroy(e);
            };
            const uint8_t *body = in + dict.body_offset;
            for (size_t k = 0; k < n_slices; ++k) {  // every upload is queued at once; events mark their arrival
                const size_t lo = k * kSlice, hi = std::min(body_bytes, lo + kSlice);
                cudaError_t e = cudaEventCreateWithFlags(&up[k], cudaEventDisableTiming);
                if (e == cudaSuccess) e = cudaMemcpyAsync(ctx->d_in + lo, body + lo, hi - lo, cudaMemcpyHostToDevice, ctx->copy_stream);
                if (e == cudaSuccess) e = cudaEventRecord(up[k], ctx->copy_stream);
                if (e != cudaSuccess) {
                    cleanup();
                    return fail(ctx, ET_ERR_CUDA, "upload of slice %zu: %s", k, cudaGetErrorString(e));
                }
            }
            uint64_t head_bit = 0;  // first codeword of the next slice, bits from the start of the body
            // symbols found so far; decoding stops at body_len, or once one symbol more than fits `cap` has been found
            uint64_t found = 0;
            const uint64_t enough = write_out ? std::min<uint64_t>(dict.body_len, (uint64_t)cap + 1) : dict.body_len;
            for (size_t k = 0; k < n_slices && found < enough; ++k) {
                const bool last = k + 1 == n_slices;
                // slice k owns body bytes [k*kSlice - 64, (k+1)*kSlice - 64): what it needs to look ahead is uploaded
                const size_t own_lo = k ? k * kSlice - 64 : 0, own_hi = last ? body_bytes : (k + 1) * kSlice - 64;
                const size_t avail = std::min(body_bytes, (k + 1) * kSlice);
                cudaStreamWaitEvent(s, up[k], 0);
                DecodeStatus st;
                rc = unpack_dev(ctx, unpack_geometry_shard(ctx->d_in, avail, own_lo, own_hi, (long long)head_bit), dict,
                                ctx->d_out + produced, want - produced, s, &st, nullptr, true);
                if (rc != ET_OK) {
                    cudaStreamSynchronize(ctx->copy_stream);
                    cleanup();
                    return rc;
                }
                head_bit = (uint64_t)own_hi * 8 + st.exit;
                const uint64_t got = std::min<uint64_t>(st.total, want - produced);
                if (write_out && got)  // unpack_dev returned after its kernels finished: the text is ready to go down
                    cudaMemcpyAsync(out + produced, ctx->d_out + produced, got, cudaMemcpyDeviceToHost, ctx->copy_stream2);
                produced += got;
                found += st.total;
            }
            cudaStreamSynchronize(ctx->copy_stream);
            const cudaError_t e = cudaStreamSynchronize(ctx->copy_stream2);
            cleanup();
            if (e != cudaSuccess) return fail(ctx, ET_ERR_CUDA, "download: %s", cudaGetErrorString(e));
            size_t fits = 0;
            if (write_out && (rc = decode_result(ctx, dict, cap, found, &fits)) != ET_OK) return rc;
        }
        if (print_out && produced) {  // decode.zig:189 prints every symbol to std_out
            std::vector<uint8_t> text(produced);
            ET_CUDA(ctx, cudaMemcpy(text.data(), ctx->d_out, produced, cudaMemcpyDeviceToHost));
            size_t done = 0;
            while (done < text.size()) {
                const ssize_t w = write(ctx->out_fd, text.data() + done, text.size() - done);
                if (w <= 0) break;
                done += (size_t)w;
            }
        }
    }
    *out_len = write_out ? (size_t)produced : 0;  // counted only when written (decode.zig:185-188)
    if (flags & ET_FLAG_DEBUG) {
        const auto us = std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t0).count();
        fd_printf(ctx->out_fd, "time taken: %lldμs\n", (long long)us);
    }
    if (!(flags & ET_FLAG_QUIET)) print_summary((double)n, (double)*out_len);
    return ET_OK;
}

extern "C" int et_unpack_shard_dev(et_ctx *ctx, const void *d_range, size_t range_bytes, size_t own_begin_byte,
                                   size_t own_end_byte, const et_dictionary *dict, int64_t head_bit, void *d_out, size_t cap,
                                   uint64_t *n_symbols, uint64_t *entry_bit, uint64_t *exit_bit, void *stream) {
    if (!ctx || !d_range || !dict || !n_symbols || (!d_out && cap)) return ET_ERR_INVALID_ARG;
    if ((reinterpret_cast<uintptr_t>(d_range) & 15u) || (own_begin_byte & 31u) || own_begin_byte > own_end_byte ||
        own_end_byte > range_bytes || (own_end_byte != range_bytes && ((own_end_byte & 31u) || own_end_byte + 32 > range_bytes)))
        return fail(ctx, ET_ERR_INVALID_ARG, "shard geometry: 16-byte aligned range, 32-byte aligned owned part, 32 bytes of look-ahead");
    if (head_bit >= 0 && ((uint64_t)head_bit < own_begin_byte * 8 || (uint64_t)head_bit >= own_begin_byte * 8 + 64))
        return fail(ctx, ET_ERR_INVALID_ARG, "head_bit must lie in the first 64 bits of the owned part");
    if (dict->n_entries == 0 || dict->truncated) {  // nothing can be decoded (decode.zig:66 ran out of dictionary bytes)
        *n_symbols = 0;
        if (entry_bit) *entry_bit = (uint64_t)own_begin_byte * 8;
        if (exit_bit) *exit_bit = (uint64_t)own_end_byte * 8;
        return ET_OK;
    }
    ET_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    StageTimer tm{ctx, s, true};
    tm.mark(0);
    tm.mark(1);
    const UnpackGeometry g = unpack_geometry_shard(d_range, range_bytes, own_begin_byte, own_end_byte, (long long)head_bit);
    DecodeStatus st;
    const int rc = unpack_dev(ctx, g, *dict, static_cast<uint8_t *>(d_out), cap, s, &st, &tm);
    if (rc != ET_OK) return rc;
    const uint64_t found = st.total;
    tm.mark(3);
    ET_CUDA(ctx, cudaEventSynchronize(ctx->ev[3]));
    tm.finish(4);
    *n_symbols = found;  // the caller's text offsets are sums of these: never a clipped count
    if (found > cap) return fail(ctx, ET_ERR_NO_SPACE, "NoSpaceLeft: the shard holds %llu symbols, capacity %zu", (unsigned long long)found, cap);
    // entry: bits past the first bit of the 32-byte sector grid the chunks are cut on (= own_begin: it is 32-byte aligned)
    if (entry_bit) *entry_bit = (uint64_t)own_begin_byte * 8 + st.entry;
    if (exit_bit) *exit_bit = (uint64_t)own_end_byte * 8 + st.exit;
    return ET_OK;
}

// ====================================================================== synthetic inputs
extern "C" int et_synth_dev(et_ctx *ctx, void *d_out, size_t n, uint64_t seed, uint64_t first_index,
                            const uint32_t thresholds[256], void *stream) {
    if (!ctx || (!d_out && n) || !thresholds) return ET_ERR_INVALID_ARG;
    ET_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    std::memcpy(ctx->h_small->thresholds, thresholds, sizeof ctx->h_small->thresholds);
    ET_CUDA(ctx, cudaMemcpyAsync(ctx->d_small->thresholds, ctx->h_small->thresholds, sizeof ctx->h_small->thresholds, cudaMemcpyHostToDevice, s));
    ET_CUDA(ctx, launch_synth(static_cast<uint8_t *>(d_out), n, seed, first_index,
                              ctx->d_small->thresholds, s));
    ET_CUDA(ctx, cudaStreamSynchronize(s));
    return ET_OK;
}

#include "et_shard.inc"
#include "et_batch.inc"
#include "et_batch_encode.inc"
