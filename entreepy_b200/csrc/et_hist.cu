// K1 — byte histogram (replaces encode.zig:43-47).
//
// HBM-bound: N bytes in, 2 KiB out.  The usual smem histogram serialises on hot bins
// (space is 17 % of text, one symbol is 38 % of the Fibonacci input).  Here every lane
// owns a private column of the table: counter (bin, lane) lives at word bin*32+lane, so
// the 32 addresses of one warp-wide shared atomic always fall in 32 different banks no
// matter what the data is — throughput is independent of the symbol distribution.
// Different warps of the CTA share the table, hence atomics (ATOMS, no return value).
#include "et_device.cuh"
#include "et_kernels.cuh"

namespace et {

namespace {

__device__ __forceinline__ void count_word(uint8_t *table_lane, uint32_t w) {
    // byte b -> byte offset b*128 inside the lane's view of the table
    atomicAdd(reinterpret_cast<uint32_t *>(table_lane + ((w << 7) & 0x7f80u)), 1u);
    atomicAdd(reinterpret_cast<uint32_t *>(table_lane + ((w >> 1) & 0x7f80u)), 1u);
    atomicAdd(reinterpret_cast<uint32_t *>(table_lane + ((w >> 9) & 0x7f80u)), 1u);
    atomicAdd(reinterpret_cast<uint32_t *>(table_lane + ((w >> 17) & 0x7f80u)), 1u);
}

__global__ void __launch_bounds__(kHistThreads) histogram_kernel(const uint8_t *__restrict__ in, size_t n,
                                                                 unsigned long long *__restrict__ counts) {
    __shared__ __align__(16) uint32_t table[256 * 32];  // [bin][lane], 32 KiB
    for (int i = threadIdx.x; i < 256 * 32; i += kHistThreads) table[i] = 0;
    __syncthreads();

    const uint32_t lane = threadIdx.x & 31;
    uint8_t *table_lane = reinterpret_cast<uint8_t *>(table) + lane * 4;

    // ragged head (up to the first 16-byte boundary) and tail: block 0, one byte per thread
    const size_t head = min(n, (size_t)((16 - (reinterpret_cast<uintptr_t>(in) & 15)) & 15));
    const size_t n_vec = (n - head) >> 4;
    const size_t tail_begin = head + (n_vec << 4);
    if (blockIdx.x == 0) {
        for (size_t i = threadIdx.x; i < head; i += kHistThreads) atomicAdd(&table[in[i] * 32 + lane], 1u);
        for (size_t i = tail_begin + threadIdx.x; i < n; i += kHistThreads) atomicAdd(&table[in[i] * 32 + lane], 1u);
    }

    const uint4 *vec = reinterpret_cast<const uint4 *>(in + head);
    const size_t stride = (size_t)gridDim.x * kHistThreads;
    size_t i = (size_t)blockIdx.x * kHistThreads + threadIdx.x;
    // four independent 16-byte loads in flight per thread
    for (; i + 3 * stride < n_vec; i += 4 * stride) {
        const uint4 a = ld_stream_v4(vec + i);
        const uint4 b = ld_stream_v4(vec + i + stride);
        const uint4 c = ld_stream_v4(vec + i + 2 * stride);
        const uint4 d = ld_stream_v4(vec + i + 3 * stride);
        count_word(table_lane, a.x); count_word(table_lane, a.y); count_word(table_lane, a.z); count_word(table_lane, a.w);
        count_word(table_lane, b.x); count_word(table_lane, b.y); count_word(table_lane, b.z); count_word(table_lane, b.w);
        count_word(table_lane, c.x); count_word(table_lane, c.y); count_word(table_lane, c.z); count_word(table_lane, c.w);
        count_word(table_lane, d.x); count_word(table_lane, d.y); count_word(table_lane, d.z); count_word(table_lane, d.w);
    }
    for (; i < n_vec; i += stride) {
        const uint4 a = ld_stream_v4(vec + i);
        count_word(table_lane, a.x); count_word(table_lane, a.y); count_word(table_lane, a.z); count_word(table_lane, a.w);
    }
    __syncthreads();

    // fold the 32 lane columns of each bin; the rotation keeps the 32 threads of a warp on
    // 32 different banks while they walk their rows
    if (threadIdx.x < 256) {
        const uint32_t bin = threadIdx.x;
        unsigned long long sum = 0;
#pragma unroll 8
        for (uint32_t k = 0; k < 32; ++k) sum += table[bin * 32 + ((k + lane) & 31)];
        if (sum) atomicAdd(&counts[bin], sum);
    }
}

}  // namespace

cudaError_t launch_histogram(const uint8_t *d_in, size_t n, unsigned long long *d_counts, int num_sms,
                             cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    const size_t n_vec = n >> 4;
    // 4 CTAs x 512 threads fill an SM (2048 threads, 128 KiB of tables)
    size_t blocks = (n_vec + (size_t)kHistThreads * 4 - 1) / ((size_t)kHistThreads * 4);
    const size_t cap = (size_t)num_sms * 4;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    histogram_kernel<<<(unsigned)blocks, kHistThreads, 0, stream>>>(d_in, n, d_counts);
    return cudaGetLastError();
}

// ---------------------------------------------------------------- batched histogram (et_encode_batch_dev)
namespace {
constexpr int kBatchHistThreads = 256;

// A CTA per tile of one stream: the same lane-column table as histogram_kernel, folded into the stream's counts.
__global__ void __launch_bounds__(kBatchHistThreads) batch_histogram_kernel(const EncHistTile *__restrict__ tiles,
                                                                            unsigned long long *__restrict__ counts) {
    __shared__ __align__(16) uint32_t table[256 * 32];  // [bin][lane], 32 KiB
    for (int i = threadIdx.x; i < 256 * 32; i += kBatchHistThreads) table[i] = 0;
    const EncHistTile t = tiles[blockIdx.x];
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31;
    uint8_t *table_lane = reinterpret_cast<uint8_t *>(table) + lane * 4;
    for (uint32_t b0 = threadIdx.x * 16u; b0 < t.hi; b0 += kBatchHistThreads * 16u) {
        if (b0 >= t.lo && b0 + 16u <= t.hi) {
            const uint4 a = ld_stream_v4(reinterpret_cast<const uint4 *>(t.base + b0));
            count_word(table_lane, a.x); count_word(table_lane, a.y); count_word(table_lane, a.z); count_word(table_lane, a.w);
        } else {  // the ragged ends of the stream: only its own bytes
            for (uint32_t k = max(b0, t.lo); k < min(b0 + 16u, t.hi); ++k) atomicAdd(&table[t.base[k] * 32 + lane], 1u);
        }
    }
    __syncthreads();
    const uint32_t bin = threadIdx.x;
    unsigned long long sum = 0;
#pragma unroll 8
    for (uint32_t k = 0; k < 32; ++k) sum += table[bin * 32 + ((k + lane) & 31)];
    if (sum) atomicAdd(&counts[(size_t)t.item * 256 + bin], sum);
}
static_assert(kBatchHistThreads == 256, "a thread per bin folds the table");
}  // namespace

cudaError_t launch_batch_histogram(const EncBatchLayout &L, uint32_t hist_tiles, cudaStream_t stream, int *launches) {
    if (hist_tiles == 0) return cudaSuccess;
    batch_histogram_kernel<<<hist_tiles, kBatchHistThreads, 0, stream>>>(L.hist_tiles, L.counts);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

// ---------------------------------------------------------------- synthetic input generator
namespace {
__device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}
__global__ void __launch_bounds__(256) synth_kernel(uint8_t *__restrict__ out, size_t n, uint64_t seed, uint64_t first,
                                                    const uint32_t *__restrict__ thresholds) {
    __shared__ uint32_t thr[256];
    thr[threadIdx.x] = thresholds[threadIdx.x];
    __syncthreads();
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint32_t r = (uint32_t)(splitmix64(seed + first + i) >> 32);
        // smallest s with thr[s] > r  (thr is non-decreasing, thr[255] treated as +inf)
        uint32_t lo = 0, hi = 255;
        while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            if (thr[mid] > r) hi = mid; else lo = mid + 1;
        }
        out[i] = (uint8_t)lo;
    }
}
}  // namespace

cudaError_t launch_synth(uint8_t *d_out, size_t n, uint64_t seed, uint64_t first_index, const uint32_t *d_thresholds,
                         cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    size_t blocks = (n + 255) / 256;
    if (blocks > 148 * 64) blocks = 148 * 64;
    synth_kernel<<<(unsigned)blocks, 256, 0, stream>>>(d_out, n, seed, first_index, d_thresholds);
    return cudaGetLastError();
}

}  // namespace et
