// K2 — body pack (replaces encode.zig:303-318) and the seam fix-up.
//
// Codes of at most 32 bits (every dictionary the reference emits faithfully) take the lane-run
// path: two streaming passes with warps as the unit of work, nothing waits at a block-wide
// barrier.
//   pass A  region_bits_kernel  bits of every run of 64 consecutive symbols and of every region (32 runs =
//                               2048 symbols), a warp per region;
//   scan    region_prefix_kernel + group_scan_kernel: bits before each region inside its group of 1024, bits
//                               before every group;
//   pass B  pack_runs_kernel  persistent warps, one region at a time.  A lane owns one run: its
//                             bit offset inside the region comes from a warp scan of the run
//                             totals; per symbol one conflict-free 64-bit shared load of
//                             {code, len} (table replicated for 16 lanes: entry (sym, lane & 15)
//                             at sym*128 + lane*8, a 64-bit load is served half a warp at a
//                             time); adjacent symbols are fused into pairs when they fit 32
//                             bits; everything goes through one 64-bit accumulator whose whole
//                             words are ORed straight into their place in the warp's shared bit
//                             image, which is assembled at the region's final bit position inside
//                             its 16-byte output blocks; the image is byte-swapped to stream order
//                             (big-endian bit packing) and stored as aligned 16-byte vectors.
// A single pass with a decoupled look-back over tiles of 16 regions was built and measured (r2, text-1G: 1.93 ms
// against 0.93 ms for the two passes): the CTA-wide lockstep it needs bounds it (stall_barrier 4.6 per issued
// instruction).  With the offsets known from pass A every region is independent.
// Codes longer than 32 bits (where the reference itself emits truncated paths, SURVEY §0.4) use
// the wide kernel further down (4096-symbol tiles, look-back).
//
// Regions own whole output bytes only.  The (at most two) bytes a region shares with its
// neighbours go to seam_head/seam_tail and are merged by seam_fixup_kernel, so the output needs no
// pre-zeroing and no global atomics, and regions with zero bits (the symbol the reference drops
// when all 256 byte values occur, SURVEY §0.2) are handled.
//
// Algorithmic HBM bytes per symbol: 1 read + len/8 written (text: 1.586 B/symbol); pass A reads
// the text a second time (not credited).
#include <cstring>

#include "et_device.cuh"
#include "et_kernels.cuh"

namespace et {

namespace {

constexpr int kWarps = kPackThreads / 32;

struct PackArgs {
    const uint8_t *in_aligned;
    uint32_t misalign;
    uint64_t v_end;
    uint32_t num_tiles;
    const void *tables;
    uint8_t *out;
    uint32_t bit_phase;
    unsigned long long *tile_state;
    uint8_t *seam_head;
    uint8_t *seam_tail;
    uint32_t *ticket;
    uint32_t *tile_bits;               // [num_tiles] bits of the earlier tiles of the same group (narrow path)
    unsigned long long *group_prefix;  // [n_groups] bits before each group of tiles
    uint32_t group_tiles;              // tiles per group (a power of two)
    uint32_t group_shift;              // log2(group_tiles)
    uint32_t interior_lo, interior_hi; // tiles [lo, hi) lie wholly inside the input
    uint16_t *run_bits;                // [32 * regions] lane-run pack: bits of every run of 64 symbols
    uint32_t n_regions;                // lane-run pack: regions of 2048 symbols (one warp each)
    uint32_t image_words;              // lane-run pack: words of a warp's bit image (guard included)
};

__device__ __forceinline__ uint32_t warp_inclusive_scan(uint32_t v, uint32_t lane) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t up = __shfl_up_sync(0xffffffffu, v, d);
        if (lane >= (uint32_t)d) v += up;
    }
    return v;
}

// Look back over the predecessors of `tile` and return the bit offset at which it starts.
// Called by warp 0 only.  Tile 0 publishes a prefix directly, so the walk always ends.
__device__ __forceinline__ unsigned long long lookback_exclusive(const unsigned long long *state, uint32_t tile,
                                                                uint32_t lane) {
    unsigned long long exclusive = 0;
    long long base = (long long)tile - 1;
    for (;;) {
        const long long idx = base - (long long)lane;
        unsigned long long d;
        uint32_t has_prefix, pending;
        do {  // wait only for the descriptors between this tile and the nearest published prefix
            d = idx >= 0 ? ld_relaxed_u64(state + idx) : kStatusPrefix;
            has_prefix = __ballot_sync(0xffffffffu, (d & kStatusMask) == kStatusPrefix);
            pending = __ballot_sync(0xffffffffu, (d & kStatusMask) == 0);
            if (has_prefix) pending &= (1u << (__ffs((int)has_prefix) - 1)) - 1u;
        } while (pending);
        const uint32_t first = has_prefix ? (uint32_t)__ffs((int)has_prefix) - 1u : 31u;
        unsigned long long v = lane <= first ? (d & ~kStatusMask) : 0ull;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        exclusive += v;
        if (has_prefix) return exclusive;
        base -= 32;
    }
}

// ------------------------------------------------------------------ narrow kernel (codes <= 32 bits)
constexpr int kTableLanes = 16;
constexpr int kTableBytes = 256 * kTableLanes * 8;                    // 32 KiB
constexpr int kStageGuard = 4;                                        // zero words in front of the image

// ---- scan: bits before each group (one block; groups are sized so that there are at most a few thousand).
__global__ void __launch_bounds__(1024) group_scan_kernel(const PackArgs a, uint32_t n_groups) {
    __shared__ unsigned long long part[1024];
    const uint32_t t = threadIdx.x;
    const uint32_t per = (n_groups + 1023u) / 1024u;
    const uint32_t g_lo = min(t * per, n_groups), g_hi = min(g_lo + per, n_groups);
    unsigned long long sum = 0;
    for (uint32_t g = g_lo; g < g_hi; ++g) sum += a.group_prefix[g];
    part[t] = sum;
    __syncthreads();
    for (int d = 1; d < 1024; d <<= 1) {
        const unsigned long long v = t >= (uint32_t)d ? part[t - d] : 0ull;
        __syncthreads();
        part[t] += v;
        __syncthreads();
    }
    unsigned long long run = part[t] - sum + a.bit_phase;
    for (uint32_t g = g_lo; g < g_hi; ++g) {
        const unsigned long long gs = a.group_prefix[g];
        a.group_prefix[g] = run;
        run += gs;
    }
}

// ------------------------------------------------------------------ lane-run pack (codes <= 32 bits)
// The same two passes with warps instead of CTAs as the unit, so that nothing waits at a
// block-wide barrier and the per-tile overhead (block scan, three barriers, image zeroing by the
// whole CTA) is gone:
//   pass A  region_bits_kernel: one streaming pass; bits of every RUN of 64 consecutive symbols
//           (u16), of every region of 32 runs before it inside its group, of every group;
//   scan    group_scan_kernel (one block);
//   pass B  pack_runs_kernel: persistent warps.  A lane owns one run: four 16-byte loads, its
//           bit offset inside the region from a warp scan of the run totals, then the 64
//           symbols go through one 64-bit accumulator straight to their place in the warp's
//           shared bit image, at the region's bit position in its output blocks.  The image is
//           swapped to stream order and stored as aligned 16-byte vectors; the two bytes a
//           region may share with its neighbours take the seam arrays, as above.
constexpr int kRunSyms = 64;
constexpr int kRegionSyms = 32 * kRunSyms;  // 2048
constexpr int kRunWarps = 16;

__device__ __forceinline__ bool region_is_interior(const PackArgs &a, uint32_t r) {
    return r >= a.interior_lo && r < a.interior_hi;
}

// (acc << len) | code on a 64-bit accumulator, len 0..32.  pos is the absolute BIT address of the next bit
// in shared memory (byte address x 8 + bit, MSB first inside a word); when it crosses a word boundary the
// 32 bits before the boundary are complete and are STORED under a predicate — no branch, the lanes of a warp
// stay together whatever their code lengths are.  A lane's first such word also covers the last bits of the
// lanes before it (zeros here): those lanes OR their unfinished last word in after the warp has met
// (pack_runs_kernel), so every word of the image is written exactly once and ORed at most a few times.
struct BitAcc {
    uint32_t hi, lo, pos;
    uint32_t wp;  // shared address of the word that holds bit `pos` (kept beside pos: deriving it is a shift and a mask per store)
};
__device__ __forceinline__ void open_acc(BitAcc &b, uint32_t bit_address) {
    b.hi = b.lo = 0;
    b.pos = bit_address;
    b.wp = (bit_address >> 3) & ~3u;
}
__device__ __forceinline__ void push_acc(BitAcc &b, uint32_t code, uint32_t len) {
    b.hi = __funnelshift_lc(b.lo, b.hi, len);
    b.lo = __funnelshift_lc(0u, b.lo, len) | code;
    const uint32_t p2 = b.pos + len;
    if ((b.pos ^ p2) & 32u) {
        asm volatile("st.shared.u32 [%0], %1;" ::"r"(b.wp), "r"(__funnelshift_r(b.lo, b.hi, p2)) : "memory");
        b.wp += 4u;
    }
    b.pos = p2;
}

// {code, length} of symbol k (0..3, first in the lowest byte) of text word w from the lane's column of the shared table
// (tab_lane_s: its shared address).  One byte permute and one multiply-add per symbol - symbol x 128 + column, the
// multiplier in a register (`r128`, a value the assembler cannot know, or it turns the multiply into a shift and an add) -
// where shift, mask, OR of the lane's offset and add of the base were four instructions, three of them for the ALU pipe.
template <int K>
__device__ __forceinline__ uint2 table_entry(uint32_t w, uint32_t tab_lane_s, uint32_t r128) {
    const uint32_t sym = K == 0 ? (w & 0xffu) : K == 3 ? (w >> 24) : __byte_perm(w, 0u, 0x4440u + K);
    uint32_t addr;
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(addr) : "r"(sym), "r"(r128), "r"(tab_lane_s));
    uint2 e;
    asm("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(e.x), "=r"(e.y) : "r"(addr));
    return e;
}
__device__ __forceinline__ uint32_t opaque_128(const PackArgs &a) {
    uint32_t v = a.image_words ? 128u : 129u;  // image_words is never 0
    asm volatile("" : "+r"(v));
    return v;
}

template <int K>
__device__ __forceinline__ uint32_t table_length(uint32_t w, uint32_t len_lane_s, uint32_t r128) {  // the same for pass A's [symbol][lane] table of lengths
    const uint32_t sym = K == 0 ? (w & 0xffu) : K == 3 ? (w >> 24) : __byte_perm(w, 0u, 0x4440u + K);
    uint32_t addr, len;
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(addr) : "r"(sym), "r"(r128), "r"(len_lane_s));
    asm("ld.shared.u32 %0, [%1];" : "=r"(len) : "r"(addr));
    return len;
}

// Pass A's work on one region r (a warp): the bits of its 32 runs and its total.  Interior regions take the four vectors of
// the lane, loaded coalesced (load i of lane L is vector 32 i + L of the region, a quarter of run 8 i + L / 4).
__device__ __forceinline__ void region_bits_interior(const PackArgs &a, uint32_t r, uint32_t lane, const uint4 (&v)[4], uint32_t len_lane_s,
                                                     uint32_t r128) {
    uint32_t total = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const uint32_t w[4] = {v[i].x, v[i].y, v[i].z, v[i].w};
        uint32_t bits = 0;
#pragma unroll
        for (int q = 0; q < 4; ++q)
            bits += table_length<0>(w[q], len_lane_s, r128) + table_length<1>(w[q], len_lane_s, r128) +
                    table_length<2>(w[q], len_lane_s, r128) + table_length<3>(w[q], len_lane_s, r128);
        bits += __shfl_xor_sync(0xffffffffu, bits, 1);
        bits += __shfl_xor_sync(0xffffffffu, bits, 2);  // the run's bits, in its four lanes
        if ((lane & 3u) == 0) a.run_bits[(size_t)r * 32 + 8 * i + (lane >> 2)] = (uint16_t)bits;
        total += (lane & 3u) == 0 ? bits : 0u;
    }
    total = __reduce_add_sync(0xffffffffu, total);
    if (lane == 0) a.tile_bits[r] = total;
}
__device__ __forceinline__ void region_bits_ragged(const PackArgs &a, uint32_t r, uint32_t lane, const uint32_t *len_sh) {
    uint32_t bits = 0;
    {  // ragged ends of the input: a lane takes its own run, only the symbols that exist
        const uint64_t v0 = (uint64_t)r * kRegionSyms + (uint64_t)lane * kRunSyms;
        for (uint32_t i = 0; i < (uint32_t)kRunSyms; ++i)
            if (v0 + i >= a.misalign && v0 + i < a.v_end) bits += len_sh[(uint32_t)a.in_aligned[v0 + i] * 32];
    }
    a.run_bits[(size_t)r * 32 + lane] = (uint16_t)bits;
    const uint32_t total = __reduce_add_sync(0xffffffffu, bits);
    if (lane == 0) a.tile_bits[r] = total;
}

// Pass A, a warp per region: four coalesced 16-byte loads per lane, a run's bit count is the sum over the four lanes that
// hold it (two shuffles), and nothing in the kernel waits for anything - no barrier, no running total carried by one
// thread (round 1's slab form, 4096 symbols per CTA step with the group's running total kept
// by thread 0, spent a third of its issue slots on those: 288 us per GiB against ~190 us here).  It writes the
// run totals and every region's total; region_prefix_kernel turns the totals into prefixes inside groups of 1024.
// Pass A's table of lengths, [sym][lane]: a warp-wide lookup never has a bank conflict.
__device__ __forceinline__ void load_len_table(uint32_t *len_sh, const PackArgs &a, uint32_t tid) {
    for (int i = tid; i < 256 * 32; i += kPackThreads) len_sh[i] = static_cast<const uint2 *>(a.tables)[i >> 5].y;
    __syncthreads();
}
__global__ void __launch_bounds__(kPackThreads) region_bits_kernel(const PackArgs a) {
    __shared__ uint32_t len_sh[256 * 32];
    load_len_table(len_sh, a, threadIdx.x);
    const uint32_t lane = threadIdx.x & 31;
    const uint8_t *len_lane = reinterpret_cast<const uint8_t *>(len_sh) + lane * 4;
    const uint32_t len_lane_s = (uint32_t)__cvta_generic_to_shared(len_lane), r128 = opaque_128(a);
    const uint32_t stride = gridDim.x * kWarps;
    // coalesced: load i of lane L is vector 32 i + L of the region, i.e. a quarter of run 8 i + L / 4 (a lane loading
    // its own run, 64 bytes apart from its neighbour's, fetches every 32-byte sector twice from L2: measured 2.09 GB
    // of L2 traffic per GiB and an L2-bound kernel).  The next region's vectors are requested before this one's are used.
    uint4 nv[4];
    bool have = false;
    auto request = [&](uint32_t rr) {
        have = rr < a.n_regions && region_is_interior(a, rr);
        if (have) {
            const uint4 *src = reinterpret_cast<const uint4 *>(a.in_aligned + (uint64_t)rr * kRegionSyms) + lane;
            nv[0] = ld_stream_v4(src);
            nv[1] = ld_stream_v4(src + 32);
            nv[2] = ld_stream_v4(src + 64);
            nv[3] = ld_stream_v4(src + 96);
        }
    };
    request(blockIdx.x * kWarps + (threadIdx.x >> 5));
    for (uint32_t r = blockIdx.x * kWarps + (threadIdx.x >> 5); r < a.n_regions; r += stride) {
        if (have) {
            const uint4 v[4] = {nv[0], nv[1], nv[2], nv[3]};
            request(r + stride);
            region_bits_interior(a, r, lane, v, len_lane_s, r128);
            continue;
        }
        region_bits_ragged(a, r, lane, len_sh);
        request(r + stride);
    }
}
// tile_bits[r]: the region's bits -> bits of the regions before it inside its group of kPrefixGroup; group_prefix[g]: the
// group's bits (group_scan_kernel makes prefixes of those).
constexpr uint32_t kPrefixGroup = 1024;
__global__ void __launch_bounds__(kPrefixGroup) region_prefix_kernel(const PackArgs a) {
    __shared__ uint32_t warp_sum[32];
    const uint32_t t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const uint32_t r = blockIdx.x * kPrefixGroup + t;
    const uint32_t v = r < a.n_regions ? a.tile_bits[r] : 0u;
    const uint32_t incl = warp_inclusive_scan(v, lane);
    if (lane == 31) warp_sum[warp] = incl;
    __syncthreads();
    uint32_t before = 0, total = 0;
    for (uint32_t w = 0; w < 32; ++w) {
        const uint32_t s = warp_sum[w];
        if (w < warp) before += s;
        total += s;
    }
    if (r < a.n_regions) a.tile_bits[r] = before + incl - v;
    if (t == 0) a.group_prefix[blockIdx.x] = total;
}

// Four vectors of a lane's run and which of the 64 symbols exist (ragged ends of the input only).
__device__ __forceinline__ void load_run(const PackArgs &a, uint32_t r, uint32_t lane, bool interior, uint4 (&raw)[4],
                                         unsigned long long *valid) {
    const uint64_t v0 = (uint64_t)r * kRegionSyms + (uint64_t)lane * kRunSyms;  // virtual byte index
    *valid = ~0ull;
    if (interior) {
#pragma unroll
        for (int i = 0; i < 4; ++i) raw[i] = ld_stream_v4(a.in_aligned + v0 + 16 * i);
        return;
    }
    *valid = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const long long lo = (long long)a.misalign - (long long)(v0 + 16 * i), hi = (long long)a.v_end - (long long)(v0 + 16 * i);
        const int l = (int)max(lo, 0ll), h = (int)min(hi, 16ll);
        raw[i] = make_uint4(0, 0, 0, 0);
        if (h > 0 && l < 16) {
            raw[i] = ld_partial_v4(a.in_aligned + v0 + 16 * i, l, h);
            *valid |= (unsigned long long)((0xffffu >> (16 - h)) & (0xffffu << l)) << (16 * i);
        }
    }
}

// The 64 symbols of a lane's run through the accumulator (their codes from the lane's column of the shared table).
__device__ __forceinline__ void pack_run_symbols(BitAcc &acc, const uint4 (&raw)[4], unsigned long long valid, bool interior,
                                                 const uint8_t *table_lane, uint32_t r128) {
    if (interior) {
        const uint32_t tab_lane_s = (uint32_t)__cvta_generic_to_shared(table_lane);
        uint4 v0 = raw[0], v1 = raw[1], v2 = raw[2], v3 = raw[3];
#pragma unroll 1
        for (int it = 0; it < 4; ++it) {  // one 16-byte vector per trip: the body must stay inside the instruction cache
            const uint32_t rw[4] = {v0.x, v0.y, v0.z, v0.w};
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const uint32_t w = rw[q];
                // the four symbols of a word: their codes are merged in registers and go into the accumulator
                // as ONE piece when they fit 32 bits together (text: ~19 bits), else as two pairs, else one by one
                const uint2 e0 = table_entry<0>(w, tab_lane_s, r128), e1 = table_entry<1>(w, tab_lane_s, r128);
                const uint2 e2 = table_entry<2>(w, tab_lane_s, r128), e3 = table_entry<3>(w, tab_lane_s, r128);
                const uint32_t l01 = e0.y + e1.y, l23 = e2.y + e3.y, len = l01 + l23;
                if (len <= 32u) {
                    const uint32_t c01 = __funnelshift_lc(0u, e0.x, e1.y) | e1.x, c23 = __funnelshift_lc(0u, e2.x, e3.y) | e3.x;
                    push_acc(acc, __funnelshift_lc(0u, c01, l23) | c23, len);
                } else {
                    if (l01 <= 32u) {
                        push_acc(acc, __funnelshift_lc(0u, e0.x, e1.y) | e1.x, l01);
                    } else {
                        push_acc(acc, e0.x, e0.y);
                        push_acc(acc, e1.x, e1.y);
                    }
                    if (l23 <= 32u) {
                        push_acc(acc, __funnelshift_lc(0u, e2.x, e3.y) | e3.x, l23);
                    } else {
                        push_acc(acc, e2.x, e2.y);
                        push_acc(acc, e3.x, e3.y);
                    }
                }
            }
            v0 = v1;
            v1 = v2;
            v2 = v3;
        }
    } else {
#pragma unroll
        for (int q = 0; q < 16; ++q) {  // ragged ends of the input: one symbol at a time, only those that exist
            const uint4 v = raw[q >> 2];
            uint32_t w = (q & 3) == 0 ? v.x : (q & 3) == 1 ? v.y : (q & 3) == 2 ? v.z : v.w;
            uint32_t ok = (uint32_t)(valid >> (4 * q)) & 15u;
#pragma unroll 1
            for (int k = 0; k < 4; ++k, w >>= 8, ok >>= 1) {
                const uint2 e = *reinterpret_cast<const uint2 *>(table_lane + (w & 0xffu) * (kTableLanes * 8));
                if (ok & 1u) push_acc(acc, e.x, e.y);
            }
        }
    }
}

// The finished bit image of region r goes to its place in the output: swapped to stream order, stored as aligned 16-byte
// vectors; the (at most two) bytes it shares with its neighbours go to the seam arrays.  The image is assembled at frame
// positions (frame: the 16-byte blocks of the output that the region touches; frame word f is image word kStageGuard + f,
// MSB first: pack_runs_kernel knows where the region goes before it packs), so a block of the output is four image words
// as they stand.  Frame bit of region bit 0 (< 128):
__device__ __forceinline__ uint32_t region_frame_shift(const PackArgs &a, unsigned long long bit_begin) {
    return (uint32_t)(reinterpret_cast<uintptr_t>(a.out + (bit_begin >> 3)) & 15u) * 8u + (uint32_t)(bit_begin & 7);
}
__device__ __forceinline__ void region_copy_out(const PackArgs &a, uint32_t r, const uint32_t *stage, uint8_t *edge,
                                                unsigned long long bit_begin, uint32_t region_bits, uint32_t lane) {
    const unsigned long long bit_end = bit_begin + region_bits;
    uint8_t *first_byte = a.out + (bit_begin >> 3);              // byte holding the region's first bit
    const uint32_t align = (uint32_t)(reinterpret_cast<uintptr_t>(first_byte) & 15u);
    uint8_t *gbase = first_byte - align;                         // frame byte k <-> gbase[k]
    const uint32_t shift = align * 8 + (uint32_t)(bit_begin & 7);  // frame bit of region bit 0 (< 128)
    const uint32_t used_bits = shift + region_bits;
    const uint32_t n_chunks = (used_bits + 127u) >> 7;
    const unsigned long long byte0 = bit_begin >> 3;
    const unsigned long long full_lo = (bit_begin + 7) >> 3, full_hi = bit_end >> 3;  // owned bytes [lo,hi)
    const uint32_t s_lo = (uint32_t)(full_lo - byte0) + align;                       // frame coordinates
    const uint32_t s_hi = full_hi >= full_lo ? (uint32_t)(full_hi - byte0) + align : s_lo;
    const bool has_head = (bit_begin & 7) != 0;
    const bool has_tail = (bit_end & 7) != 0 && full_hi >= full_lo;
    const uint32_t s_head = align;
    const uint32_t s_tail = (uint32_t)(full_hi - byte0) + align;  // only meaningful when has_tail
    if (lane == 0) {
        if (!has_head) a.seam_head[r] = 0;
        if (!has_tail) a.seam_tail[r] = 0;
    }
    for (uint32_t c = lane; c < n_chunks; c += 32) {
        const uint4 q = reinterpret_cast<const uint4 *>(stage + kStageGuard)[c];
        const uint4 v = make_uint4(bswap32(q.x), bswap32(q.y), bswap32(q.z), bswap32(q.w));
        const uint32_t k0 = c * 16;
        if (k0 >= s_lo && k0 + 16 <= s_hi) {
            st_stream_v4(gbase + k0, v);
        } else {
            // a block at the ragged start (slot 0) or end (slot 1) of the region: parked, the warp stores its bytes below
            *reinterpret_cast<uint4 *>(edge + (c == 0 ? 0 : 16)) = v;
        }
    }
    // The two ragged blocks, one byte per lane (lanes 0-15: the first block, 16-31: the last one): a single lane
    // walking their bytes one at a time cost the warp ~200 instructions per region with 31 lanes idle.
    __syncwarp();
    if (n_chunks) {
        const uint32_t blk = lane < 16 ? 0u : n_chunks - 1u, k0 = blk * 16u, k = k0 + (lane & 15u);
        const bool ragged = !(k0 >= s_lo && k0 + 16u <= s_hi) && (lane < 16 || n_chunks > 1);
        if (ragged) {
            const uint32_t byte = edge[(lane < 16 ? 0u : 16u) + (lane & 15u)];
            if (k >= s_lo && k < s_hi) gbase[k] = (uint8_t)byte;
            if (has_head && k == s_head) a.seam_head[r] = (uint8_t)byte;
            if (has_tail && k == s_tail) a.seam_tail[r] = (uint8_t)byte;
        }
    }
    __syncwarp();  // the slots are free again
}

// Pass B's shared memory: the table, replicated for kTableLanes lanes, and the warp's bit image cleared.
__device__ __forceinline__ void load_run_table(uint8_t *table, const PackArgs &a, uint32_t *stage, uint32_t tid) {
    const uint32_t lane = tid & 31;
    const uint2 *src = static_cast<const uint2 *>(a.tables);
    uint2 *dst = reinterpret_cast<uint2 *>(table);
    for (int i = tid; i < 256 * kTableLanes; i += kRunWarps * 32) dst[i] = src[i / kTableLanes];
    for (uint32_t i = lane; i < a.image_words; i += 32) stage[i] = 0;
    __syncthreads();
}

// Pass B's work on region r once a lane holds its run (raw, valid): the run offsets, the region's end for the seam
// fix-up, the image assembled at the positions of the output frame, and the copy-out.  bit_begin: the region's first
// bit in the stream's body.
__device__ __forceinline__ void pack_region(const PackArgs &a, uint32_t r, uint32_t lane, const uint4 (&raw)[4], unsigned long long valid,
                                            bool interior, uint32_t my_bits, unsigned long long bit_begin, uint32_t *stage, uint8_t *edge,
                                            const uint8_t *table_lane, uint32_t r128) {
    const uint32_t incl = warp_inclusive_scan(my_bits, lane);
    const uint32_t region_bits = __shfl_sync(0xffffffffu, incl, 31);
    const uint32_t my_off = incl - my_bits;
    const unsigned long long bit_end = bit_begin + region_bits;
    if (lane == 0) a.tile_state[r] = bit_end;  // for the seam fix-up

    // ---- assemble at region-relative positions (words hold stream bits MSB-first)
    {
        // the word in which the region ends is only ever ORed into (or not touched at all), and the byte in which
        // it ends may reach into the word after it: both start from zero
        // (the image is assembled at the positions of the output frame - region bit 0 at bit `shift` - so that the
        // copy-out has nothing to shift; what lies before the region's first bit in its first block is never stored)
        const uint32_t shift = region_frame_shift(a, bit_begin);
        if (lane < 2) stage[kStageGuard + ((shift + region_bits) >> 5) + lane] = 0;
        __syncwarp();
        BitAcc acc;
        open_acc(acc, (uint32_t)__cvta_generic_to_shared(stage + kStageGuard) * 8u + shift + my_off);
        pack_run_symbols(acc, raw, valid, interior, table_lane, r128);
        __syncwarp();  // every whole word is in place
        if (acc.pos & 31u) atomicOr(stage + kStageGuard + ((shift + my_off + my_bits) >> 5), acc.lo << (32u - (acc.pos & 31u)));
    }
    __syncwarp();  // image complete
    region_copy_out(a, r, stage, edge, bit_begin, region_bits, lane);
}

// Pass B.  Dynamic shared memory: table (32 KiB, 16-lane replicated) | per warp: bit image | per warp: 32 edge bytes.
__global__ void __launch_bounds__(kRunWarps * 32, 2) pack_runs_kernel(const PackArgs a) {
    extern __shared__ __align__(16) uint8_t smem[];
    uint8_t *table = smem;
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint32_t *stage = reinterpret_cast<uint32_t *>(smem + kTableBytes) + (size_t)warp * a.image_words;
    uint8_t *edge = smem + kTableBytes + (size_t)kRunWarps * a.image_words * 4 + warp * 32;
    load_run_table(table, a, stage, tid);
    const uint8_t *table_lane = table + (lane & (kTableLanes - 1)) * 8;
    const uint32_t r128 = opaque_128(a);
    const uint32_t stride = gridDim.x * kRunWarps;
    uint32_t r = blockIdx.x * kRunWarps + warp;
    if (r >= a.n_regions) return;

    const uint32_t stage_run_s = (uint32_t)__cvta_generic_to_shared(stage + kStageGuard);
    for (;;) {
        const bool interior = region_is_interior(a, r);
        uint4 raw[4];
        unsigned long long valid = ~0ull;
        if (interior) {
            // The region's 2 KiB come in with coalesced cp.async (L2 -> shared memory, no registers) into the warp's bit
            // image, which is idle until the packing starts; a lane then reads its own run - 64 bytes - from there.  (A
            // lane loading its run straight from global memory shares every 32-byte sector with its neighbour and pulls
            // it from L2 twice.)  The 16-byte pieces of a run are stored XOR-swizzled so that neither the cp.async
            // writes nor the four 16-byte reads of a lane meet in a bank.
            const uint8_t *src = a.in_aligned + (uint64_t)r * kRegionSyms;
#pragma unroll
            for (uint32_t i = 0; i < 4; ++i) {
                const uint32_t v = 32u * i + lane, chunk = (v & ~3u) | ((v & 3u) ^ ((v >> 3) & 3u));
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(stage_run_s + 16u * chunk), "l"(src + 16u * v) : "memory");
            }
            asm volatile("cp.async.wait_all;" ::: "memory");
            __syncwarp();
#pragma unroll
            for (uint32_t j = 0; j < 4; ++j) {
                const uint32_t chunk = 4u * lane + (j ^ ((lane >> 1) & 3u));
                asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];"
                             : "=r"(raw[j].x), "=r"(raw[j].y), "=r"(raw[j].z), "=r"(raw[j].w)
                             : "r"(stage_run_s + 16u * chunk)
                             : "memory");
            }
            __syncwarp();  // every lane holds its run: the image may be written
        } else {
            load_run(a, r, lane, false, raw, &valid);
        }
        const uint32_t my_bits = a.run_bits[(size_t)r * 32 + lane];
        const unsigned long long bit_begin = a.group_prefix[r >> a.group_shift] + a.tile_bits[r];
        const uint32_t r_next = r + stride;
        if (r_next < a.n_regions) {  // the next region's text and run totals on their way into L2 (no registers held)
            const uint8_t *nx = lane < 16 ? a.in_aligned + (uint64_t)r_next * kRegionSyms + lane * 128u
                                          : reinterpret_cast<const uint8_t *>(a.run_bits + (size_t)r_next * 32);
            if (lane <= 16) asm volatile("prefetch.global.L2 [%0];" ::"l"(nx));
        }
        pack_region(a, r, lane, raw, valid, interior, my_bits, bit_begin, stage, edge, table_lane, r128);
        __syncwarp();  // everyone has read the image
        if (r_next >= a.n_regions) break;
        r = r_next;
    }
}

// ------------------------------------------------------------------ wide kernel (codes of 33..64 bits)
constexpr int kWideMaxLen = 64;
constexpr int kWideTableBytes = 256 * 8 + 256;  // codes + lengths, not replicated
// worst-case tile bits + up to 127 bits of alignment slack + one spare word, in uint4 units
constexpr int kWideStageWords = (((kPackTileSyms * kWideMaxLen + 128 + 32) + 127) / 128) * 4;

__global__ void __launch_bounds__(kPackThreads) pack_wide_kernel(const PackArgs a) {
    extern __shared__ __align__(16) uint8_t smem[];
    uint32_t *stage = reinterpret_cast<uint32_t *>(smem);
    uint8_t *table = smem + kWideStageWords * 4;
    __shared__ uint32_t warp_sum[kWarps];
    __shared__ unsigned long long tile_base_sh;
    __shared__ uint32_t tile_sh;
    __shared__ __align__(16) uint8_t edge_sh[2][16];  // first / last block of a tile, for bytewise stores

    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    for (int i = tid; i < kWideStageWords; i += kPackThreads) stage[i] = 0;
    {
        const uint8_t *src = static_cast<const uint8_t *>(a.tables);
        for (int i = tid; i < kWideTableBytes; i += kPackThreads) table[i] = src[i];
    }
    const unsigned long long *wide_code = reinterpret_cast<const unsigned long long *>(table);
    const uint8_t *wide_len = table + 256 * 8;

    for (;;) {
        __syncthreads();  // staging is clean, previous tile_sh/tile_base_sh consumed
        if (tid == 0) tile_sh = atomicAdd(a.ticket, 1u);
        __syncthreads();
        const uint32_t tile = tile_sh;
        if (tile >= a.num_tiles) break;

        // ---- (1) load + lookup
        const uint64_t v0 = (uint64_t)tile * kPackTileSyms + (uint64_t)tid * kPackItems;  // virtual byte index
        const bool edge = v0 < a.misalign || v0 + kPackItems > a.v_end;
        uint4 raw;
        if (!edge) {
            raw = ld_stream_v4(a.in_aligned + v0);
        } else {
            const long long lo = (long long)a.misalign - (long long)v0, hi = (long long)a.v_end - (long long)v0;
            raw = (hi <= 0 || lo >= 16) ? make_uint4(0, 0, 0, 0)
                                        : ld_partial_v4(a.in_aligned + v0, (int)max(lo, 0ll), (int)min(hi, 16ll));
        }
        const uint32_t rw[4] = {raw.x, raw.y, raw.z, raw.w};
        uint32_t my_bits = 0;
#pragma unroll
        for (int i = 0; i < kPackItems; ++i) {
            const uint32_t w = rw[i >> 2];
            const int sh = 8 * (i & 3);
            bool valid = true;
            if (edge) valid = (v0 + i >= a.misalign) && (v0 + i < a.v_end);
            const uint32_t sym = (w >> sh) & 0xffu;
            my_bits += valid ? wide_len[sym] : 0u;
        }

        // ---- (2) block scan of bit totals, look-back for the tile's bit offset
        const uint32_t incl = warp_inclusive_scan(my_bits, lane);
        if (lane == 31) warp_sum[warp] = incl;
        __syncthreads();
        uint32_t warp_off = 0, tile_bits = 0;
#pragma unroll
        for (int wq = 0; wq < kWarps; ++wq) {
            const uint32_t s = warp_sum[wq];
            if (wq < (int)warp) warp_off += s;
            tile_bits += s;
        }
        const uint32_t my_off = warp_off + incl - my_bits;
        if (warp == 0) {
            unsigned long long start;
            if (tile == 0) {
                start = a.bit_phase;
            } else {
                if (lane == 0) st_relaxed_u64(a.tile_state + tile, kStatusAggregate | tile_bits);
                start = lookback_exclusive(a.tile_state, tile, lane);
            }
            if (lane == 0) {
                st_relaxed_u64(a.tile_state + tile, kStatusPrefix | (start + tile_bits));
                tile_base_sh = start;
            }
        }
        __syncthreads();
        const unsigned long long bit_begin = tile_base_sh;           // B_i: first bit of the tile in the output
        const unsigned long long bit_end = bit_begin + tile_bits;    // E_i
        uint8_t *first_byte = a.out + (bit_begin >> 3);              // byte holding bit B_i
        const uint32_t align = (uint32_t)(reinterpret_cast<uintptr_t>(first_byte) & 15u);
        uint8_t *gbase = first_byte - align;                         // staging byte k <-> gbase[k]
        const uint32_t stage_bit0 = align * 8 + (uint32_t)(bit_begin & 7);

        // ---- (3) assemble: words hold stream bits MSB-first; all stores are ORs because the
        // first and last word of a thread are shared with its neighbours
        {
            uint32_t pos = stage_bit0 + my_off;
            uint32_t fill = pos & 31u;  // bits pending in acc
            uint32_t *wp = stage + (pos >> 5);
            unsigned long long acc = 0;
#pragma unroll
            for (int i = 0; i < kPackItems; ++i) {
                {
                    const uint32_t w = rw[i >> 2];
                    const uint32_t sym = (w >> (8 * (i & 3))) & 0xffu;
                    bool valid = true;
                    if (edge) valid = (v0 + i >= a.misalign) && (v0 + i < a.v_end);
                    const uint32_t len = valid ? wide_len[sym] : 0u;
                    const unsigned long long code = wide_code[sym];
                    if (len > 32u) {  // high piece first: len-32 bits
                        const uint32_t hl = len - 32u;
                        acc = (acc << hl) | (code >> 32);
                        fill += hl;
                        if (fill >= 32u) {
                            fill -= 32u;
                            atomicOr(wp++, (uint32_t)(acc >> fill));
                        }
                    }
                    const uint32_t ll = len > 32u ? 32u : len;
                    if (ll) {
                        acc = (acc << ll) | (code & 0xffffffffull);
                        fill += ll;
                        if (fill >= 32u) {
                            fill -= 32u;
                            atomicOr(wp++, (uint32_t)(acc >> fill));
                        }
                    }
                }
            }
            if (fill) atomicOr(wp, (uint32_t)(acc << (32u - fill)));
        }
        __syncthreads();

        // ---- (4) copy out whole bytes the tile owns, park the shared ones in the seam arrays
        {
            const uint32_t used_bits = stage_bit0 + tile_bits;
            const uint32_t n_chunks = (used_bits + 127u) >> 7;
            const unsigned long long byte0 = bit_begin >> 3;
            const unsigned long long full_lo = (bit_begin + 7) >> 3, full_hi = bit_end >> 3;  // owned bytes [lo,hi)
            const uint32_t s_lo = (uint32_t)(full_lo - byte0) + align;                       // staging coordinates
            const uint32_t s_hi = full_hi >= full_lo ? (uint32_t)(full_hi - byte0) + align : s_lo;
            const bool has_head = (bit_begin & 7) != 0;
            const bool has_tail = (bit_end & 7) != 0 && full_hi >= full_lo;
            const uint32_t s_head = align;
            const uint32_t s_tail = (uint32_t)(full_hi - byte0) + align;  // only meaningful when has_tail
            if (tid == 0) {
                if (!has_head) a.seam_head[tile] = 0;
                if (!has_tail) a.seam_tail[tile] = 0;
            }
            uint4 *stage4 = reinterpret_cast<uint4 *>(stage);
            for (uint32_t c = tid; c < n_chunks; c += kPackThreads) {
                uint4 v = stage4[c];
                stage4[c] = make_uint4(0, 0, 0, 0);
                v.x = bswap32(v.x); v.y = bswap32(v.y); v.z = bswap32(v.z); v.w = bswap32(v.w);
                const uint32_t k0 = c * 16;
                if (k0 >= s_lo && k0 + 16 <= s_hi) {
                    st_stream_v4(gbase + k0, v);
                } else {
                    // a block at the ragged start or end of the tile: through a small per-thread buffer
                    uint4 *tmp = reinterpret_cast<uint4 *>(edge_sh[c == 0 ? 0 : 1]);
                    *tmp = v;
                    const uint8_t *tb = reinterpret_cast<const uint8_t *>(tmp);
                    const uint32_t lo_k = max(k0, s_lo), hi_k = min(k0 + 16u, s_hi);
                    for (uint32_t kk = lo_k; kk < hi_k; ++kk) gbase[kk] = tb[kk - k0];
                    if (has_head && s_head >= k0 && s_head < k0 + 16u) a.seam_head[tile] = tb[s_head - k0];
                    if (has_tail && s_tail >= k0 && s_tail < k0 + 16u) a.seam_tail[tile] = tb[s_tail - k0];
                }
            }
        }
    }
}

// One thread per tile: the byte a tile's last bits end in (when it also starts in that
// tile) is the OR of that tile's tail and the heads of every following tile that starts
// in the same byte.  Byte 0 of a shard that begins mid-byte has no owner; thread 0 adds it.
__device__ __forceinline__ void seam_fixup_tile(const unsigned long long *__restrict__ tile_state, const uint8_t *__restrict__ seam_head,
                                                const uint8_t *__restrict__ seam_tail, uint32_t num_tiles, uint32_t bit_phase,
                                                uint8_t *__restrict__ out, uint32_t i) {
    auto end_of = [&](uint32_t j) { return tile_state[j] & ~kStatusMask; };
    auto begin_of = [&](uint32_t j) { return j == 0 ? (unsigned long long)bit_phase : end_of(j - 1); };
    auto merge_from = [&](unsigned long long byte, uint32_t value, uint32_t j) {
        for (; j < num_tiles; ++j) {
            if ((begin_of(j) >> 3) != byte) break;
            value |= seam_head[j];
            if ((end_of(j) >> 3) > byte) break;
        }
        out[byte] = (uint8_t)value;
    };
    const unsigned long long b = begin_of(i), e = end_of(i);
    if ((e & 7) != 0 && ((e >> 3) << 3) >= b) merge_from(e >> 3, seam_tail[i], i + 1);
    if (i == 0 && bit_phase != 0) merge_from(0, 0, 0);
}
__global__ void __launch_bounds__(256) seam_fixup_kernel(const unsigned long long *__restrict__ tile_state,
                                                         const uint8_t *__restrict__ seam_head,
                                                         const uint8_t *__restrict__ seam_tail, uint32_t num_tiles,
                                                         uint32_t bit_phase, uint8_t *__restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= num_tiles) return;
    seam_fixup_tile(tile_state, seam_head, seam_tail, num_tiles, bit_phase, out, i);
}

// ------------------------------------------------------------------ batched pack (et_encode_batch_dev)
// The lane-run pack of many streams at once.  Stream j owns the regions [R_j, R_j + n_regions) of the group; its PackArgs
// hold its own geometry, table and output (out = its body, d_out + header_len), with run_bits, tile_bits, tile_state and the
// seam arrays moved to its first region, so that the device functions above run on it with stream-local region numbers.
// The scan runs over the regions of every stream: a region's body bit is prefix(R_j + r) - prefix(R_j).
struct BatchPackArgs {
    PackArgs a;
    uint64_t first_region;         // R_j
    const uint8_t *header;         // the stream's header in the group's scratch
    uint32_t header_len;
};
static_assert(kEncPrefixGroup == kPrefixGroup, "the batched scan uses region_prefix_kernel's groups");

__device__ __forceinline__ unsigned long long batch_region_prefix(const BatchPackArgs &b, uint32_t r) {
    return b.a.group_prefix[(b.first_region + r) / kPrefixGroup] + b.a.tile_bits[r];
}

// Pass A over tiles of kEncTileRegions regions of one stream: the stream's table of lengths, then a warp per region.
__global__ void __launch_bounds__(kPackThreads) batch_region_bits_kernel(const BatchPackArgs *__restrict__ args,
                                                                         const BatchTile *__restrict__ tiles) {
    __shared__ uint32_t len_sh[256 * 32];
    const BatchTile tile = tiles[blockIdx.x];
    const PackArgs &a = args[tile.item].a;
    load_len_table(len_sh, a, threadIdx.x);
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t len_lane_s = (uint32_t)__cvta_generic_to_shared(reinterpret_cast<const uint8_t *>(len_sh) + lane * 4);
    const uint32_t r128 = opaque_128(a);
    for (uint32_t r = tile.first + (threadIdx.x >> 5); r < min(tile.first + kEncTileRegions, a.n_regions); r += kWarps) {
        if (region_is_interior(a, r)) {
            const uint4 *src = reinterpret_cast<const uint4 *>(a.in_aligned + (uint64_t)r * kRegionSyms) + lane;
            const uint4 v[4] = {ld_stream_v4(src), ld_stream_v4(src + 32), ld_stream_v4(src + 64), ld_stream_v4(src + 96)};
            region_bits_interior(a, r, lane, v, len_lane_s, r128);
        } else {
            region_bits_ragged(a, r, lane, len_sh);
        }
    }
}

// Pass B over tiles of up to kEncTileRegions regions of one stream, a warp per region.  Dynamic shared memory as
// pack_runs_kernel's: table | per warp: bit image | per warp: 32 edge bytes (every stream of the group has the group's
// image_words).
__global__ void __launch_bounds__(kRunWarps * 32, 2) batch_pack_runs_kernel(const BatchPackArgs *__restrict__ args,
                                                                            const BatchTile *__restrict__ tiles) {
    extern __shared__ __align__(16) uint8_t smem[];
    uint8_t *table = smem;
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const BatchTile tile = tiles[blockIdx.x];
    const BatchPackArgs &b = args[tile.item];
    const PackArgs &a = b.a;
    uint32_t *stage = reinterpret_cast<uint32_t *>(smem + kTableBytes) + (size_t)warp * a.image_words;
    uint8_t *edge = smem + kTableBytes + (size_t)kRunWarps * a.image_words * 4 + warp * 32;
    load_run_table(table, a, stage, tid);
    const uint32_t r = tile.first + warp;
    if (r >= a.n_regions) return;
    const uint8_t *table_lane = table + (lane & (kTableLanes - 1)) * 8;
    const uint32_t r128 = opaque_128(a);
    const bool interior = region_is_interior(a, r);
    uint4 raw[4];
    unsigned long long valid = ~0ull;
    load_run(a, r, lane, interior, raw, &valid);
    const uint32_t my_bits = a.run_bits[(size_t)r * 32 + lane];
    const unsigned long long bit_begin = batch_region_prefix(b, r) - batch_region_prefix(b, 0);
    pack_region(a, r, lane, raw, valid, interior, my_bits, bit_begin, stage, edge, table_lane, r128);
}

// The seam fix-up over the same tiles (a thread per region; the merge stops at the end of the stream), and the header of
// every stream by the CTA of its first tile.  The body starts on a byte boundary and the regions store only the bytes they
// own, so no byte holds both header and body.
constexpr int kBatchSeamThreads = 64;
__global__ void __launch_bounds__(kBatchSeamThreads) batch_seam_fixup_kernel(const BatchPackArgs *__restrict__ args,
                                                                             const BatchTile *__restrict__ tiles) {
    const BatchTile tile = tiles[blockIdx.x];
    const BatchPackArgs &b = args[tile.item];
    const PackArgs &a = b.a;
    const uint32_t r = tile.first + threadIdx.x;
    if (threadIdx.x < kEncTileRegions && r < a.n_regions)
        seam_fixup_tile(a.tile_state, a.seam_head, a.seam_tail, a.n_regions, 0, a.out, r);
    if (tile.first == 0)
        for (uint32_t k = threadIdx.x; k < b.header_len; k += kBatchSeamThreads) a.out[(int64_t)k - (int64_t)b.header_len] = b.header[k];
}
static_assert(kEncTileRegions <= kBatchSeamThreads && kEncTileRegions == kRunWarps, "a tile is a region per warp of pass B");

}  // namespace

PackGeometry pack_geometry(const void *d_in, size_t n) {
    PackGeometry g;
    const uintptr_t p = reinterpret_cast<uintptr_t>(d_in);
    g.misalign = (uint32_t)(p & 15u);
    g.in_aligned = reinterpret_cast<const uint8_t *>(p - g.misalign);
    g.v_end = (uint64_t)g.misalign + n;
    g.num_tiles = (uint32_t)((g.v_end + kPackTileSyms - 1) / kPackTileSyms);
    return g;
}

size_t pack_scratch_bytes(const PackGeometry &g) { return pack_layout(nullptr, g.num_tiles).bytes; }

cudaError_t pack_init_device(int max_smem, int *bits_ctas_per_sm) {
    cudaError_t err = cudaFuncSetAttribute(pack_runs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem);
    if (err != cudaSuccess) return err;
    err = cudaFuncSetAttribute(batch_pack_runs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem);
    if (err != cudaSuccess) return err;
    int per_sm = 0;
    err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, region_bits_kernel, kPackThreads, 0);
    if (err != cudaSuccess) return err;
    *bits_ctas_per_sm = per_sm < 1 ? 1 : per_sm;
    return cudaSuccess;
}

// Words of a warp's bit image in pass B: a region at max_len bits a symbol, the frame's slack and the guard, in whole
// 16-byte blocks.
static uint32_t run_image_words(uint32_t max_len) { return (uint32_t)(kStageGuard + (kRegionSyms * max_len + 31) / 32 + 16 + 3) & ~3u; }

// The lane-run fields of a stream's PackArgs: its interior regions, the groups of the region scan and the bit image.
static void set_lane_runs(PackArgs &a, const PackGeometry &g, uint32_t max_len) {
    a.interior_lo = g.misalign ? 1u : 0u;
    a.interior_hi = (uint32_t)(g.v_end / kRegionSyms);
    if (a.interior_hi < a.interior_lo) a.interior_hi = a.interior_lo;
    a.image_words = run_image_words(max_len);
    // (a region holds at most 2048 x 32 bits, a group 2^26: the prefix inside a group fits 32 bits)
    a.group_tiles = kPrefixGroup;
    a.group_shift = 10;
}

cudaError_t launch_pack(const PackGeometry &g, const void *d_tables, bool wide, uint32_t max_len, uint8_t *d_out, uint32_t bit_phase,
                        void *scratch_base, int num_sms, cudaStream_t stream, int *launches, int bits_ctas_per_sm) {
    if (g.num_tiles == 0) return cudaSuccess;
    const PackLayout s = pack_layout(scratch_base, g.num_tiles);
    cudaError_t err = cudaSuccess;
    PackArgs a;
    a.in_aligned = g.in_aligned;
    a.misalign = g.misalign;
    a.v_end = g.v_end;
    a.num_tiles = g.num_tiles;
    a.tables = d_tables;
    a.out = d_out;
    a.bit_phase = bit_phase;
    a.tile_state = s.tile_state;
    a.seam_head = s.seam_head;
    a.seam_tail = s.seam_tail;
    a.ticket = s.ticket;
    a.tile_bits = s.tile_bits;
    a.group_prefix = s.group_prefix;
    a.group_tiles = 1;
    a.group_shift = 0;
    a.interior_lo = g.misalign ? 1u : 0u;
    a.interior_hi = (uint32_t)(g.v_end / kPackTileSyms);
    if (a.interior_hi < a.interior_lo) a.interior_hi = a.interior_lo;

    if (wide) {
        // look-back descriptors and the ticket start from zero
        err = cudaMemsetAsync(s.ticket, 0, reinterpret_cast<uint8_t *>(s.tile_state + g.num_tiles) - reinterpret_cast<uint8_t *>(s.ticket), stream);
        if (err != cudaSuccess) return err;
        const int smem = kWideStageWords * 4 + kWideTableBytes;
        err = cudaFuncSetAttribute(pack_wide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (err != cudaSuccess) return err;
        int per_sm = (227 * 1024) / (smem + 1024);
        if (per_sm > 2048 / kPackThreads) per_sm = 2048 / kPackThreads;
        if (per_sm < 1) per_sm = 1;
        unsigned grid = (unsigned)num_sms * (unsigned)per_sm;
        if (grid > g.num_tiles) grid = g.num_tiles;
        pack_wide_kernel<<<grid, kPackThreads, smem, stream>>>(a);
        if (launches) *launches += 1;
    } else {
        // lane-run path: regions of 2048 symbols, in the slots of the same layout
        const uint32_t n_regions = (uint32_t)((g.v_end + kRegionSyms - 1) / kRegionSyms);
        a.run_bits = s.run_bits;
        a.n_regions = n_regions;
        a.num_tiles = n_regions;
        set_lane_runs(a, g, max_len);
        if (a.image_words < kStageGuard + kRegionSyms / 4) a.image_words = kStageGuard + kRegionSyms / 4;  // the image also stages the region's text
        // pass A: run and region totals (a warp per region), prefixes inside groups of 1024 regions, prefixes of the groups
        const uint32_t groups = (n_regions + kPrefixGroup - 1) / kPrefixGroup;
        {
            int per_sm = bits_ctas_per_sm;  // CTAs of 8 warps that fit an SM (32 KB table each, 48 registers per thread: five)
            if (per_sm < 1 && (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, region_bits_kernel, kPackThreads, 0) != cudaSuccess || per_sm < 1))
                per_sm = 4;
            unsigned pa_grid = (unsigned)num_sms * (unsigned)per_sm;
            const unsigned need = (n_regions + kWarps - 1) / kWarps;
            if (pa_grid > need) pa_grid = need;
            region_bits_kernel<<<pa_grid, kPackThreads, 0, stream>>>(a);
        }
        region_prefix_kernel<<<groups, kPrefixGroup, 0, stream>>>(a);
        group_scan_kernel<<<1, 1024, 0, stream>>>(a, groups);
        const int smem = kTableBytes + kRunWarps * (int)a.image_words * 4 + kRunWarps * 32;
        if (bits_ctas_per_sm < 1) {  // no pack_init_device() for this context
            err = cudaFuncSetAttribute(pack_runs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
            if (err != cudaSuccess) return err;
        }
        int per_sm = (227 * 1024) / (smem + 1024);
        if (per_sm > 2) per_sm = 2;  // __launch_bounds__(.., 2)
        if (per_sm < 1) per_sm = 1;
        unsigned grid = (unsigned)num_sms * (unsigned)per_sm;  // persistent warps: the table is loaded once per CTA
        const unsigned need = (n_regions + kRunWarps - 1) / kRunWarps;
        if (grid > need) grid = need;
        pack_runs_kernel<<<grid, kRunWarps * 32, smem, stream>>>(a);
        if (launches) *launches += 4;
        err = cudaGetLastError();
        if (err != cudaSuccess) return err;
        seam_fixup_kernel<<<(n_regions + 255) / 256, 256, 0, stream>>>(a.tile_state, a.seam_head, a.seam_tail, n_regions,
                                                                     bit_phase, d_out);
        if (launches) *launches += 1;
        return cudaGetLastError();
    }
    err = cudaGetLastError();
    if (err != cudaSuccess) return err;
    seam_fixup_kernel<<<(g.num_tiles + 255) / 256, 256, 0, stream>>>(s.tile_state, s.seam_head, s.seam_tail,
                                                                    g.num_tiles, bit_phase, d_out);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

// ------------------------------------------------------------------ batched pack (et_batch_encode.inc)
size_t batch_pack_args_bytes() { return sizeof(BatchPackArgs); }

void batch_fill_pack_args(void *dst, const EncBatchLayout &L, const BatchPackStream &s, uint32_t max_len) {
    BatchPackArgs b{};
    PackArgs &a = b.a;
    const PackGeometry &g = s.g;
    a.in_aligned = g.in_aligned;
    a.misalign = g.misalign;
    a.v_end = g.v_end;
    a.num_tiles = s.n_regions;
    a.n_regions = s.n_regions;
    a.tables = L.tables + (size_t)s.table * 512;
    a.out = s.d_out + s.header_len;
    a.bit_phase = 0;
    a.tile_state = L.region_end + s.first_region;
    a.seam_head = L.seam_head + s.first_region;
    a.seam_tail = L.seam_tail + s.first_region;
    a.tile_bits = L.region_bits + s.first_region;
    a.run_bits = L.run_bits + s.first_region * 32;
    a.group_prefix = L.group_prefix;  // indexed by the group's region numbers (batch_region_prefix)
    set_lane_runs(a, g, max_len);
    b.first_region = s.first_region;
    b.header = L.headers + s.header_off;
    b.header_len = s.header_len;
    std::memcpy(dst, &b, sizeof b);
}

cudaError_t launch_pack_batch(const EncBatchLayout &L, uint32_t n_tiles, uint64_t n_regions, uint32_t max_len, cudaStream_t stream,
                              int *launches) {
    if (n_tiles == 0) return cudaSuccess;
    const BatchPackArgs *args = reinterpret_cast<const BatchPackArgs *>(L.args);
    // the scan over every region of the group, with the single-stream kernels
    PackArgs s{};
    s.tile_bits = L.region_bits;
    s.group_prefix = L.group_prefix;
    s.n_regions = (uint32_t)n_regions;
    s.bit_phase = 0;
    const uint32_t groups = (uint32_t)((n_regions + kPrefixGroup - 1) / kPrefixGroup);
    batch_region_bits_kernel<<<n_tiles, kPackThreads, 0, stream>>>(args, L.tiles);
    region_prefix_kernel<<<groups, kPrefixGroup, 0, stream>>>(s);
    group_scan_kernel<<<1, 1024, 0, stream>>>(s, groups);
    // the warps' images are sized by the group's longest code, as launch_pack sizes them by the stream's
    const int smem = kTableBytes + kRunWarps * (int)run_image_words(max_len) * 4 + kRunWarps * 32;
    batch_pack_runs_kernel<<<n_tiles, kRunWarps * 32, smem, stream>>>(args, L.tiles);
    batch_seam_fixup_kernel<<<n_tiles, kBatchSeamThreads, 0, stream>>>(args, L.tiles);
    if (launches) *launches += 5;
    return cudaGetLastError();
}

}  // namespace et
