// K3-K5 — parallel Huffman decode of an .et body (replaces decode.zig:143-203).
//
// The stream carries no block index, so nobody knows where a codeword starts.  The body is
// cut into chunks and the codeword boundary at which each chunk starts is found by
// self-synchronisation plus a fixpoint check:
//   sync 0   every chunk starts decoding a few words BEFORE its first bit, from a guess.
//            Huffman codes re-synchronise after a few symbols, so by the time the walk
//            enters the chunk it is almost always on a true boundary.  It records where it
//            entered, how many symbols begin in the chunk and where its last codeword ends.
//   sync r   a chunk whose recorded entry differs from its left neighbour's recorded end
//            decodes again from there.  A pass in which nothing differed proves, by
//            induction from chunk 0 (true start), that every entry is the true one.  Text
//            needs one repair round; codes with nearly equal lengths (uniform bytes:
//            7/8-bit codes) need tens; the worst case is one round per chunk and still ends.
//   scan     exclusive scan of the symbol counts (64-bit);
//   write    every chunk decodes once more from its proven entry.
// Nothing here bets on luck: the guess only decides how many chunks the repair rounds redo.
//
// Two implementations of that protocol live in this file:
//   * the LANE-INTERLEAVED decoder (second half of the file) for long streams of codes that
//     re-synchronise quickly — the path the benchmarks run: chunks of 33 words, a warp per
//     region of 32 chunks staged in shared memory, flat two-lookup walks, the text of a
//     region assembled in shared memory and stored as whole 16-byte vectors;
//   * the per-THREAD chunk kernels (first half) for short streams and for codes whose lengths
//     differ by at most 2 bits: one thread per chunk of 32..4096 bytes, stream words in
//     registers 16 bytes at a time, bit position and symbol count (or output address) in ONE
//     register, table entries that are pre-packed adds for it.  Anything unusual there (ragged
//     ends of the stream, output clipped by body_len) takes the generic walker, one symbol at
//     a time with every check.
// All of them are bound by instruction issue and the integer pipe, not by HBM (ncu: profiles/),
// so the walkers are written for instruction count.
#include <cstdio>
#include <cstdlib>

#include "et_device.cuh"
#include "et_kernels.cuh"

namespace et {

namespace {

constexpr uint32_t kPosMask = 0x1ffu;  // position field of a packed walk state (bit 8 = marker)

struct DecArgs {
    const uint8_t *body_aligned;
    uint64_t grid_bit;            // first bit of chunk 0 (own_begin rounded down to a 32-byte sector)
    uint64_t own_end_bit;         // symbols that begin before this bit are decoded
    uint64_t end_bit;             // no code may extend past this bit
    uint64_t byte_lo, byte_hi;    // readable bytes
    uint32_t head_off;            // first codeword of chunk 0, bits past grid_bit (when head_known)
    uint32_t head_known;
    uint32_t n_chunks;
    uint32_t chunk_bytes;         // multiple of 16
    uint32_t fixed_len;           // > 0: every code has this length (complete code): entries in closed form, no run-up
    const uint32_t *clut;
    const uint32_t *wlut;
    const uint32_t *nodes;
    const uint16_t *slots;        // slot of every marker window (kLutSize), then the second-level tables
    const uint16_t *t_count;      // lane-interleaved decoder: device-built tables (lane_tables_kernel)
    const uint32_t *t_write;
    const uint8_t *t_single;
    uint16_t *start_off;          // [n] first codeword of the chunk, bits past the chunk's first bit
    uint16_t *exit_off;           // [n] first codeword boundary at or after the chunk's end, bits past that end
    uint32_t *count;              // [n] symbols that begin inside the chunk
    mid_t *mid;                   // [n] lane-interleaved decoder: where the parts of the chunk begin (lane_count<true>)
    unsigned long long *block_prefix;  // [ceil(n / kChunkThreads)] exclusive scan of per-block symbol counts
    uint32_t *changed;            // [1]
    uint32_t *max_sum;            // [1] symbols of the largest region
    unsigned long long *group_prefix;  // [ceil(regions / 1024)] lane-interleaved decoder: scan of the group sums
    uint32_t *work;               // [regions] lane-interleaved decoder: regions in which an entry has to be repaired
    uint32_t *work_count;         // [1]
    uint32_t *edge;               // [regions] lane-interleaved decoder: entry of the region's first chunk | exit of its last << 16
    uint8_t *self_listed;         // [regions] ... the count walk put the region on the repair list itself
    uint32_t *rsum;               // [regions] ... symbols of the region
    uint32_t *error_flags;
    unsigned long long *total;
    uint32_t *entry_exit;
    uint8_t *tr_exit;             // [n << s_log2] transfer functions of the chunks: exit for every possible entry (slowly synchronising codes)
    uint16_t *tr_cnt;             // [n << s_log2] ... and the symbols
    unsigned long long *dbg;      // ET_TUNE_DEBUG: per CTA {smid, start ns, end ns} of the two big lane kernels (or null)
    uint8_t *out;
    uint64_t max_symbols;
};

// ------------------------------------------------------------------ shared-window accessors
__device__ __forceinline__ uint32_t smem_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
// Makes a value opaque to the compiler, which otherwise recomputes shared-window addresses inside the hot loops.
__device__ __forceinline__ uint32_t pinned(uint32_t x) {
    asm volatile("" : "+r"(x));
    return x;
}
__device__ __forceinline__ uint32_t lds_u16(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint32_t lds_u8(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
// Loads from the decode tables: filled once per CTA before the walks, read-only afterwards, so the
// compiler may schedule these freely among the (volatile) stores of the text.
__device__ __forceinline__ uint32_t lds_tab_u16(uint32_t addr) {
    uint32_t v;
    asm("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts_u32(uint32_t addr, uint32_t v) {
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

// ------------------------------------------------------------------ long codes
// A code longer than the first-level window: walk the trie with the remaining window bits.
// Returns the code length (symbol in *sym) or 0 when no code matches.
__device__ __noinline__ uint32_t long_code(uint32_t win, uint32_t node, const uint32_t *__restrict__ nodes,
                                           uint32_t *sym) {
    if (node == kChildNone) return 0;
    for (int b = kLutBits; b < 32; ++b) {
        const uint32_t bit = (win >> (31 - b)) & 1u;
        const uint32_t child = (__ldg(nodes + node) >> (16 * bit)) & 0xFFFFu;
        if (child == kChildNone) return 0;
        if (child & kChildLeaf) {
            *sym = child & 0xFFu;
            return (uint32_t)b + 1u;
        }
        node = child;
    }
    return 0;
}

// Table index of the 12-bit window at the current position, as a byte offset into a u32 table.
__device__ __forceinline__ uint32_t window_offset(uint32_t hi, uint32_t lo, uint32_t c) {
    return (__funnelshift_l(lo, hi, c) >> (32 - kLutBits - 2)) & ((kLutSize - 1) << 2);
}

// The fast loops stopped on a marker: the code at the current position is longer than the
// window.  Returns the add for that one code (len | 1 << 9); bits that are no code at all
// (incomplete dictionary) are skipped one at a time and flagged.
__device__ __forceinline__ uint32_t long_code_add(uint32_t hi, uint32_t lo, uint32_t c, const uint32_t *__restrict__ wlut,
                                                  const uint32_t *__restrict__ nodes, uint32_t *sym, uint32_t *bad) {
    const uint32_t win = __funnelshift_l(lo, hi, c);
    const uint32_t len = long_code(win, __ldg(wlut + (win >> (32 - kLutBits))) & 0xffffu, nodes, sym);
    if (len) return len | (1u << 9);
    *bad = 1u;
    return 1u;
}

// ------------------------------------------------------------------ fast walkers (per-thread chunk kernels)
// Packed state c: bits 0-8 position relative to the 32-bit word being decoded (bit 8 set =
// marker entry hit), bits 9+ symbol count (count walk) or staging address (write walk).
//
// One 16-byte piece (w0..w3, w4 = first word of the next piece).  LAST: the piece ends the
// chunk, so only symbols that BEGIN before its last bit may be consumed: in the last word a
// multi-symbol window is used only while it cannot cross that bit, then single symbols.
// Returns c relative to the first word of the next piece.
// (`last` is a run-time flag so that the body exists once: eight inlined copies of these loops
// did not fit the instruction cache.)
// t16_s != 0: shared address of the table of 16-bit windows (u16: bits consumed | whole codes << 9, kLutMarker when not
// even one code begins the window) - twice the symbols per lookup for codes of about a byte; the last word of a chunk
// still goes through the 12-bit table, which knows where to stop.
template <bool T16 = false>
__device__ __forceinline__ uint32_t count_piece(const uint32_t (&w)[5], uint32_t c, bool last, uint32_t clut_s,
                                                const uint32_t *__restrict__ wlut, const uint32_t *__restrict__ nodes, uint32_t t16_s = 0) {
#pragma unroll
    for (int wi = 0; wi < 4; ++wi) {
        const uint32_t hi = w[wi], lo = w[wi + 1];
        for (;;) {
            if (wi < 3 || !last) {
                if (T16)
                    while (!(c & 0x1e0u)) c += lds_u16(t16_s + ((__funnelshift_l(lo, hi, c) >> 15) & 0x1fffeu));
                else
                    while (!(c & 0x1e0u)) c += lds_u16(clut_s + window_offset(hi, lo, c));
            } else {
                while ((c & kPosMask) <= (uint32_t)(32 - kLutBits)) c += lds_u16(clut_s + window_offset(hi, lo, c));
                while (!(c & 0x1e0u)) c += lds_u16(clut_s + window_offset(hi, lo, c) + 2);
            }
            if (!(c & kLutMarker)) break;
            uint32_t sym, bad;
            c += long_code_add(hi, lo, c, wlut, nodes, &sym, &bad) - kLutMarker;
        }
        c -= 32u;
    }
    return c;
}

// Output side of the write walk.  Decoded symbols are shifted into a 64-bit register (newest
// byte on top).  Every fourth symbol the finished 32-bit word is stored, under a predicate (no
// branch, so the lanes of a warp stay together), into the thread's ring of 16 words in shared
// memory: word m of lane L sits at ring + ((m + 1) & 15) * 128 + L * 4, so a lane only ever
// touches its own bank and neither these stores nor the loads of the flush can conflict.
// Where the lanes of a warp meet again anyway (the end of each 32-bit stream word) whole 32-byte
// sectors leave for global memory (whole sectors: the text in flight on the GPU is larger than
// L2, a half-written sector would go to DRAM twice).
// The symbol count n in the walk state doubles as the byte index from the sector grid of the
// destination: it starts at head_skip, the bytes of the first sector that belong to the chunk
// before.  Ring capacity: after a flush fewer than 32 bytes are pending and one stream word
// yields at most 33 symbols (32 one-bit codes plus the second symbol of the last window), so
// at most 64 bytes = 16 words are ever pending.
struct OutRing {
    uint32_t ring_s;   // shared address of this lane's slot 0
    uint8_t *gsector;  // global address of the sector being assembled (32-byte aligned)
    uint32_t head_skip;
    uint32_t lo, hi;   // the last 8 symbols, newest in the top byte of hi
    uint32_t stored;   // sectors that have left for global memory
};

// shared address of word m of the ring, given (m + 1) in bits 11+ of a walk state
__device__ __forceinline__ uint32_t ring_slot_after(const OutRing &r, uint32_t c) { return ((c >> 4) & 0x780u) + r.ring_s; }
__device__ __forceinline__ uint32_t ring_slot(const OutRing &r, uint32_t m) { return (((m + 1u) & 15u) << 7) + r.ring_s; }

// Append `syms` (1 or 2 symbols in its low bytes; shift = 8 or 16; shift 0 appends nothing) and
// advance the walk state by `add` (bits | symbols << 9).
__device__ __forceinline__ uint32_t emit(uint32_t c, OutRing &r, uint32_t syms, uint32_t shift, uint32_t add) {
    r.lo = __funnelshift_r(r.lo, r.hi, shift);
    r.hi = __funnelshift_r(r.hi, syms, shift);
    const uint32_t before = c;
    c += add;
    // the symbol count crossed a multiple of 4: a word is complete (one symbol of the next word may sit on top of it)
    const uint32_t crossed = (before ^ c) & (4u << 9);
    const uint32_t w = (c & (1u << 9)) ? __funnelshift_r(r.lo, r.hi, 24) : r.hi;
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %0, 0;\n\t@p st.shared.u32 [%1], %2;\n\t}" ::"r"(crossed),
        "r"(ring_slot_after(r, c)), "r"(w)
        : "memory");
    return c;
}

// End of a stream word: finished sectors leave together.
__device__ __forceinline__ void flush_sectors(uint32_t c, OutRing &r) {
    while (((c >> 14) & 0x3ffffu) > r.stored) {
        const uint32_t m0 = r.stored * 8u;  // first word of the sector; 8 consecutive slots, wrapping at 16
        if (r.head_skip) {  // first sector of the chunk: its leading bytes belong to the chunk before
            for (uint32_t k = r.head_skip; k < 32u; ++k) r.gsector[k] = (uint8_t)lds_u8(ring_slot(r, m0 + (k >> 2)) + (k & 3u));
            r.head_skip = 0;
        } else {
            uint32_t v[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = lds_u32(ring_slot(r, m0 + i));
            *reinterpret_cast<uint4 *>(r.gsector) = make_uint4(v[0], v[1], v[2], v[3]);
            *reinterpret_cast<uint4 *>(r.gsector + 16) = make_uint4(v[4], v[5], v[6], v[7]);
        }
        r.gsector += 32;
        r.stored += 1;
    }
}

__device__ __forceinline__ uint32_t write_piece(const uint32_t (&w)[5], uint32_t c, bool last, uint32_t wlut_s, OutRing &r,
                                                const uint32_t *__restrict__ clut, const uint32_t *__restrict__ wlut,
                                                const uint32_t *__restrict__ nodes, uint32_t *bad) {
#pragma unroll
    for (int wi = 0; wi < 4; ++wi) {
        const uint32_t hi = w[wi], lo = w[wi + 1];
        for (;;) {
            if (wi < 3 || !last) {
                while (!(c & 0x1e0u)) {
                    const uint32_t e = lds_u32(wlut_s + window_offset(hi, lo, c));
                    c = emit(c, r, e, (e >> 22) & 0x18u, e >> 16);  // a marker entry appends nothing and sets bit 8
                }
            } else {
                while ((c & kPosMask) <= (uint32_t)(32 - kLutBits)) {
                    const uint32_t e = lds_u32(wlut_s + window_offset(hi, lo, c));
                    c = emit(c, r, e, (e >> 22) & 0x18u, e >> 16);
                }
                while (!(c & 0x1e0u)) {  // one symbol at a time up to the chunk's last bit
                    const uint32_t off = window_offset(hi, lo, c);
                    const uint32_t a = __ldg(clut + (off >> 2)) >> 16;
                    if (a & kLutMarker) {
                        c |= kLutMarker;
                        break;
                    }
                    c = emit(c, r, lds_u32(wlut_s + off), 8u, a);
                }
            }
            if (!(c & kLutMarker)) break;
            uint32_t sym = 0;
            const uint32_t add = long_code_add(hi, lo, c, wlut, nodes, &sym, bad);
            c -= kLutMarker;
            c = (add != 1u) ? emit(c, r, sym, 8u, add) : c + 1u;
        }
        c -= 32u;
        flush_sectors(c, r);
    }
    return c;
}

// ------------------------------------------------------------------ stream access
__device__ __forceinline__ uint4 load_piece(const DecArgs &a, uint64_t piece) {
    // 16 aligned bytes as four big-endian words; bytes outside the readable range read as 0
    const uint64_t byte = piece * 16;
    uint4 raw;
    if (byte >= a.byte_lo && byte + 16 <= a.byte_hi) {
        raw = __ldg(reinterpret_cast<const uint4 *>(a.body_aligned + byte));
    } else {
        const long long lo = (long long)a.byte_lo - (long long)byte, hi = (long long)a.byte_hi - (long long)byte;
        raw = (hi <= 0 || lo >= 16) ? make_uint4(0, 0, 0, 0)
                                    : ld_partial_v4(a.body_aligned + byte, (int)max(lo, 0ll), (int)min(hi, 16ll));
    }
    return make_uint4(bswap32(raw.x), bswap32(raw.y), bswap32(raw.z), bswap32(raw.w));
}
__device__ __forceinline__ uint4 load_piece_fast(const DecArgs &a, uint64_t piece) {
    const uint4 raw = __ldg(reinterpret_cast<const uint4 *>(a.body_aligned) + piece);
    return make_uint4(bswap32(raw.x), bswap32(raw.y), bswap32(raw.z), bswap32(raw.w));
}

// ------------------------------------------------------------------ generic walker
// Sequential big-endian word reader over guarded 16-byte loads.
struct WordReader {
    uint4 q;
    uint64_t qi;
    __device__ __forceinline__ void seek(const DecArgs &a, uint64_t wi) {
        qi = wi >> 2;
        q = load_piece(a, qi);
    }
    __device__ __forceinline__ uint32_t word(const DecArgs &a, uint64_t wi) {
        if ((wi >> 2) != qi) seek(a, wi);
        const uint32_t k = (uint32_t)wi & 3u;
        return k == 0 ? q.x : k == 1 ? q.y : k == 2 ? q.z : q.w;
    }
};

// Decode from absolute bit `pos` every symbol that begins before `own_end`; nothing may end
// after `hard_end` (the end of the stream).  Returns the position reached.  WRITE stores the
// symbols at out[o..) while o < max_symbols.
// clut / wlut: the first-level tables to read - the global ones (a.clut, a.wlut) or a copy in shared memory where the
// caller has one (a walk through L2-resident tables costs ~10x the latency per symbol).
template <bool WRITE>
__device__ __noinline__ uint64_t walk_generic(const DecArgs &a, uint64_t pos, uint64_t own_end, uint64_t hard_end,
                                              uint32_t *count, uint64_t o, uint32_t *bad, const uint32_t *clut = nullptr,
                                              const uint32_t *wlut = nullptr) {
    if (!clut) clut = a.clut;
    if (!wlut) wlut = a.wlut;
    uint32_t n = 0;
    uint64_t wi = pos >> 5;
    WordReader rd;
    rd.seek(a, wi);
    uint32_t hi = rd.word(a, wi), lo = rd.word(a, wi + 1);
    while (pos < own_end) {
        const uint64_t need = pos >> 5;
        if (need != wi) {  // a step never consumes more than 32 bits
            wi = need;
            hi = lo;
            lo = rd.word(a, wi + 1);
        }
        const uint32_t win = __funnelshift_l(lo, hi, (uint32_t)pos & 31u);
        const uint32_t idx = win >> (32 - kLutBits);
        const uint32_t c = clut[idx];
        uint32_t len = (c >> 16) & 0xffu, sym = WRITE ? (wlut[idx] & 0xffu) : 0u;
        if (c & kLutMarker) {
            len = long_code(win, __ldg(a.wlut + idx) & 0xffffu, a.nodes, &sym);
            if (len == 0) {  // no code here (incomplete dictionary): skip one bit, like the fast walkers
                *bad = 1u;
                pos += 1;
                continue;
            }
        }
        if (pos + len > hard_end) break;  // final pad bits look like the start of a longer code
        if (WRITE) {
            if (o < a.max_symbols) a.out[o] = (uint8_t)sym;
            ++o;
        }
        pos += len;
        n += 1;
    }
    *count = n;
    return pos;
}

// ------------------------------------------------------------------ chunk geometry
struct Chunk {
    uint64_t begin, end;  // bits; end is clipped to own_end_bit
    bool interior;        // every piece, the piece before and the piece after are plain readable stream
    bool walkable;        // every piece and the piece after can be loaded whole: the fast walkers may run from a KNOWN start
};
__device__ __forceinline__ Chunk chunk_of(const DecArgs &a, uint32_t c) {
    Chunk k;
    const uint64_t bits = (uint64_t)a.chunk_bytes * 8;
    k.begin = a.grid_bit + (uint64_t)c * bits;
    const uint64_t e = k.begin + bits;
    k.end = e < a.own_end_bit ? e : a.own_end_bit;
    k.walkable = e <= a.own_end_bit && e + 128 <= a.end_bit && (e >> 3) + 16 <= a.byte_hi;
    k.interior = k.walkable && (k.begin >> 3) >= a.byte_lo + 16 && k.begin >= a.grid_bit + 256;
    // (a stream that starts inside the first 16-byte piece of chunk 0 - byte_lo < 16 - shares that piece with whatever
    // precedes it in the caller's buffer: the same aligned 16 bytes, so loading it whole cannot fault, and a walk from
    // the known start never looks at the bits before it)
    return k;
}

// 32 aligned bytes (one DRAM sector) as two pieces of big-endian words.
struct Pair {
    uint4 a, b;
};
// The raw load and the byte swap are kept apart on purpose: the next sector is requested a
// whole sector of decoding before its first use, and nothing touches the loaded registers
// (not even the swap) until then, so the load never stalls the walk.
__device__ __forceinline__ Pair load_pair_raw(const DecArgs &a, uint64_t pair) {
    Pair p;
    p.a = __ldg(reinterpret_cast<const uint4 *>(a.body_aligned) + 2 * pair);
    p.b = __ldg(reinterpret_cast<const uint4 *>(a.body_aligned) + 2 * pair + 1);
    return p;
}
__device__ __forceinline__ uint4 swap4(uint4 v) { return make_uint4(bswap32(v.x), bswap32(v.y), bswap32(v.z), bswap32(v.w)); }
__device__ __forceinline__ Pair swap_pair(const Pair &p) {
    Pair q;
    q.a = swap4(p.a);
    q.b = swap4(p.b);
    return q;
}
__device__ __forceinline__ void prefetch_chunk_l2(const DecArgs &a, const Chunk &k) {
    const uint8_t *p = a.body_aligned + (k.begin >> 3);
    for (uint32_t off = 0; off < a.chunk_bytes + 32u; off += 128u) asm volatile("prefetch.global.L2 [%0];" ::"l"(p + off));
}

// Count walk of an interior chunk.  warm: start one piece early from a guess and report where
// the walk entered the chunk; else start at `start` (bits past the chunk's first bit).
// Chunks are whole 32-byte sectors; the stream is read a sector at a time, one sector ahead.
// Returns the packed state relative to the chunk's end.
template <bool T16 = false>
__device__ __forceinline__ uint32_t count_chunk_fast(const DecArgs &a, const Chunk &k, uint32_t start, bool warm,
                                                     uint32_t clut_s, uint32_t *entry, uint32_t t16_s = 0) {
    const uint64_t pair0 = k.begin >> 8;
    const uint32_t n_pairs = a.chunk_bytes >> 5;
    prefetch_chunk_l2(a, k);
    uint32_t w[5];
    uint32_t c = start;
    const uint32_t n_pieces = a.chunk_bytes >> 4;
    (void)n_pairs;
    Pair raw = load_pair_raw(a, pair0);
    if (warm) {  // only the position survives the run-up; it stops on the first boundary inside the chunk
        const uint4 pre = load_piece_fast(a, 2 * pair0 - 1);
        w[0] = pre.x; w[1] = pre.y; w[2] = pre.z; w[3] = pre.w; w[4] = bswap32(raw.a.x);
        c = count_piece(w, 0u, true, clut_s, a.wlut, a.nodes) & kPosMask;
    }
    *entry = c;
    Pair cur = raw;
#pragma unroll 1
    for (uint32_t p = 0; p < n_pieces; ++p) {
        if (!(p & 1u)) {  // a new sector: swap the one that has arrived, request the next (the piece after the chunk at the end)
            cur = swap_pair(raw);
            if (p + 2 < n_pieces)
                raw = load_pair_raw(a, pair0 + (p >> 1) + 1);
            else
                raw.a = __ldg(reinterpret_cast<const uint4 *>(a.body_aligned) + 2 * (pair0 + (p >> 1) + 1));
            w[0] = cur.a.x; w[1] = cur.a.y; w[2] = cur.a.z; w[3] = cur.a.w; w[4] = cur.b.x;
        } else {
            w[0] = cur.b.x; w[1] = cur.b.y; w[2] = cur.b.z; w[3] = cur.b.w; w[4] = bswap32(raw.a.x);
        }
        c = count_piece<T16>(w, c, p + 1 == n_pieces, clut_s, a.wlut, a.nodes, t16_s);
    }
    return c;
}

// The count walk of chunk c from `start` (known: a proven boundary; else a guess, and the walk begins 128 bits early).
__device__ __forceinline__ void sync_chunk(const DecArgs &a, uint32_t c, uint32_t start, bool known, const uint32_t *clut_sh) {
    const Chunk k = chunk_of(a, c);
    uint32_t cnt = 0, entry = start, exit_bits = 0;
    if (k.interior || (known && k.walkable && start < 256u)) {
        const uint32_t s = count_chunk_fast(a, k, start, !known, smem_addr(clut_sh), &entry);
        cnt = s >> 9;
        exit_bits = s & kPosMask;
    } else {
        uint64_t pos = k.begin + start;
        uint32_t bad = 0, dummy = 0;
        if (!known && k.begin >= a.byte_lo * 8 + 128) {  // same run-up as the fast path
            pos = walk_generic<false>(a, k.begin - 128, k.begin, a.end_bit, &dummy, 0, &bad, clut_sh);
            if (pos < k.begin) pos = k.begin;
        }
        entry = (uint32_t)(pos - k.begin);
        if (pos < k.end) pos = walk_generic<false>(a, pos, k.end, a.end_bit, &cnt, 0, &bad, clut_sh);
        exit_bits = pos > k.end ? (uint32_t)(pos - k.end) : 0u;
    }
    a.start_off[c] = (uint16_t)entry;
    a.exit_off[c] = (uint16_t)exit_bits;
    a.count[c] = cnt;
}

__global__ void __launch_bounds__(kChunkThreads, 6) chunk_sync_kernel(const DecArgs a, int round) {
    __shared__ __align__(16) uint32_t clut_sh[kLutSize];
    const uint32_t c = blockIdx.x * kChunkThreads + threadIdx.x;
    uint32_t start = 0;
    bool work = c < a.n_chunks;
    if (work && round != 0) {
        if (c == 0) {
            work = false;
        } else {
            start = a.exit_off[c - 1];
            work = start != a.start_off[c];
        }
    }
    if (!__syncthreads_or(work)) return;  // later rounds touch only the chunks whose entry moved
    for (int i = threadIdx.x; i < kLutSize; i += kChunkThreads) clut_sh[i] = a.clut[i];
    __syncthreads();
    if (!work) return;
    if (round != 0) *a.changed = 1u;
    if (c == 0 && a.head_known) start = a.head_off;
    bool known = round != 0 || (c == 0 && a.head_known);
    if (a.fixed_len && round == 0) {
        // Codes of one length never re-synchronise (a wrong phase stays wrong for ever), but they need not: every
        // boundary is a whole number of codes past the first one.  Without a known head the first entry is a guess
        // (bit 0 of the owned part); the others are consistent with it, and the caller repairs the guess.
        const uint64_t begin = chunk_of(a, c).begin, base = a.grid_bit + (a.head_known ? a.head_off : 0u);
        if (begin > base) start = (uint32_t)((a.fixed_len - (begin - base) % a.fixed_len) % a.fixed_len);
        known = true;
    }
    sync_chunk(a, c, start, known, clut_sh);
}

// ------------------------------------------------------------------ transfer functions (slowly synchronising codes)
// Codes whose lengths are nearly equal (uniform bytes: 7 and 8 bits) re-synchronise after kilobytes, sometimes after
// a hundred: the repair rounds above then walk the longest unsynchronised stretch one chunk per round, a sequential
// dependency no amount of parallel hardware shortens.  But a chunk can only be ENTERED at max_len different bit
// offsets (the first codeword boundary at or after its first bit lies less than one code past it), so its effect is a
// function from at most max_len entries to (exit, symbols).  One thread per (chunk, entry) tabulates it; composing the
// functions left to right is associative, so the true entry of every chunk comes out of a scan - no rounds, no luck.
// The cost is max_len count walks instead of one (8 for byte-uniform data), all of them parallel.
__global__ void __launch_bounds__(kChunkThreads, 6) chunk_transfer_kernel(const DecArgs a, uint32_t s_log2, uint32_t n_states) {
    __shared__ __align__(16) uint32_t clut_sh[kLutSize];
    for (int i = threadIdx.x; i < kLutSize; i += kChunkThreads) clut_sh[i] = a.clut[i];
    __syncthreads();
    const uint32_t idx = (gridDim.x - 1u - blockIdx.x) * kChunkThreads + threadIdx.x;  // last chunks first: the stream's ragged end is the slow one
    const uint32_t c = idx >> s_log2, e = idx & ((1u << s_log2) - 1u);
    if (c >= a.n_chunks || e >= n_states) return;
    if (c == 0) {  // chunk 0 is entered at the head of the stream (or at its guess, for a shard): one walk, what the scan starts from
        if (e == 0) sync_chunk(a, 0, a.head_known ? a.head_off : 0u, a.head_known != 0, clut_sh);
        return;
    }
    const Chunk k = chunk_of(a, c);
    uint32_t cnt = 0, exit_bits = 0;
    if (k.walkable) {
        uint32_t entry;
        const uint32_t s = count_chunk_fast(a, k, e, false, smem_addr(clut_sh), &entry);
        cnt = s >> 9;
        exit_bits = s & kPosMask;
    } else {
        uint64_t pos = k.begin + e;
        uint32_t bad = 0;
        if (pos < k.end) pos = walk_generic<false>(a, pos, k.end, a.end_bit, &cnt, 0, &bad, clut_sh);
        exit_bits = pos > k.end ? (uint32_t)(pos - k.end) : 0u;
    }
    a.tr_exit[idx] = (uint8_t)(exit_bits < n_states ? exit_bits : 0xFFu);  // 0xFF cannot be composed: the final check then fails and the rounds take over
    a.tr_cnt[idx] = (uint16_t)cnt;
}

// Maps are 16 nibbles in a 64-bit word (entry e -> nibble e).  The scan of the chunks' functions, three kernels:
//   compose_segments  every thread composes the functions of kSegChunks consecutive chunks, a block-wide scan composes
//                     the segments of the block (exclusive prefix per thread, total per block);
//   compose_blocks    one block scans the block totals;
//   compose_apply     every thread enters its segment with the true entry in hand and writes what the repair rounds
//                     would have settled on: start_off, exit_off, count.
constexpr unsigned long long kIdentMap = 0xFEDCBA9876543210ull;
__device__ __forceinline__ unsigned long long map_then(unsigned long long first, unsigned long long second, uint32_t n_states) {
    unsigned long long out = 0;
    for (uint32_t e = 0; e < n_states; ++e) {
        const uint32_t x = (uint32_t)(first >> (4 * e)) & 15u;
        out |= ((second >> (4 * x)) & 15ull) << (4 * e);
    }
    return out;
}
// The chunk's function as a nibble map (an exit that is no state maps to 0: caught by the final check).
__device__ __forceinline__ unsigned long long row_map(const DecArgs &a, uint32_t c, uint32_t s_log2, uint32_t n_states) {
    unsigned long long m = 0;
    const uint8_t *row = a.tr_exit + ((size_t)c << s_log2);
    if (s_log2 >= 3) {  // rows of 8 or 16 bytes: one or two 8-byte loads
        for (uint32_t h = 0; h < (1u << (s_log2 - 3)); ++h) {
            const unsigned long long v = *reinterpret_cast<const unsigned long long *>(row + 8 * h);
            for (uint32_t e = 0; e < 8 && 8 * h + e < n_states; ++e) m |= ((v >> (8 * e)) & 15ull) << (4 * (8 * h + e));
        }
    } else {
        for (uint32_t e = 0; e < n_states; ++e) m |= (unsigned long long)(row[e] & 15u) << (4 * e);
    }
    return m;
}
// seg_prefix[t]: composition of the segments before thread t inside its block; block_map[b]: the whole block.
__global__ void __launch_bounds__(kSegThreads) compose_segments_kernel(const DecArgs a, uint32_t s_log2, uint32_t n_states,
                                                                       unsigned long long *seg_prefix, unsigned long long *block_map) {
    __shared__ unsigned long long maps[kSegThreads];
    const uint32_t t = threadIdx.x, g = blockIdx.x * kSegThreads + t;
    const uint32_t lo = max(min(g * kSegChunks, a.n_chunks), 1u), hi = max(min(g * kSegChunks + kSegChunks, a.n_chunks), 1u);  // chunk 0 is entered at the head
    unsigned long long m = kIdentMap;
    for (uint32_t c = lo; c < hi; ++c) m = map_then(m, row_map(a, c, s_log2, n_states), n_states);
    maps[t] = m;
    __syncthreads();
    for (int d = 1; d < (int)kSegThreads; d <<= 1) {  // inclusive scan: maps[t] = segments 0..t of the block, left to right
        const unsigned long long left = t >= (uint32_t)d ? maps[t - d] : kIdentMap;
        __syncthreads();
        maps[t] = map_then(left, maps[t], n_states);
        __syncthreads();
    }
    seg_prefix[g] = t ? maps[t - 1] : kIdentMap;
    if (t == kSegThreads - 1) block_map[blockIdx.x] = maps[t];
}
__global__ void __launch_bounds__(1024) compose_blocks_kernel(uint32_t n_blocks, uint32_t n_states, unsigned long long *block_map) {
    // exclusive scan of the block maps, in place: thread t composes a run of them, a block-wide scan composes the runs
    __shared__ unsigned long long maps[1024];
    const uint32_t t = threadIdx.x, per = (n_blocks + 1023u) / 1024u;
    const uint32_t lo = min(t * per, n_blocks), hi = min(lo + per, n_blocks);
    unsigned long long m = kIdentMap;
    for (uint32_t b = lo; b < hi; ++b) m = map_then(m, block_map[b], n_states);
    maps[t] = m;
    __syncthreads();
    for (int d = 1; d < 1024; d <<= 1) {
        const unsigned long long left = t >= (uint32_t)d ? maps[t - d] : kIdentMap;
        __syncthreads();
        maps[t] = map_then(left, maps[t], n_states);
        __syncthreads();
    }
    unsigned long long run = t ? maps[t - 1] : kIdentMap;
    for (uint32_t b = lo; b < hi; ++b) {
        const unsigned long long mb = block_map[b];
        block_map[b] = run;
        run = map_then(run, mb, n_states);
    }
}
__global__ void __launch_bounds__(kSegThreads) compose_apply_kernel(const DecArgs a, uint32_t s_log2, uint32_t n_states,
                                                                    const unsigned long long *seg_prefix, const unsigned long long *block_map) {
    const uint32_t g = blockIdx.x * kSegThreads + threadIdx.x;
    const uint32_t lo = max(min(g * kSegChunks, a.n_chunks), 1u), hi = max(min(g * kSegChunks + kSegChunks, a.n_chunks), 1u);
    if (lo >= hi) return;
    uint32_t e = a.exit_off[0];  // where chunk 0 (walked from the head) leaves the stream
    if (e >= n_states) e = 0;
    e = (uint32_t)(block_map[blockIdx.x] >> (4 * e)) & 15u;
    e = (uint32_t)(seg_prefix[g] >> (4 * e)) & 15u;
    for (uint32_t c = lo; c < hi; ++c) {
        const size_t i = ((size_t)c << s_log2) + e;
        const uint32_t x = a.tr_exit[i];
        a.start_off[c] = (uint16_t)e;
        a.exit_off[c] = (uint16_t)(x < n_states ? x : 0u);
        a.count[c] = a.tr_cnt[i];
        e = x < n_states ? x : 0u;
    }
}

// ------------------------------------------------------------------ scan
__global__ void __launch_bounds__(kChunkThreads) chunk_sum_kernel(const DecArgs a) {
    __shared__ uint32_t warp_sum[kChunkThreads / 32];
    const uint32_t c = blockIdx.x * kChunkThreads + threadIdx.x;
    uint32_t v = c < a.n_chunks ? a.count[c] : 0u;
    // the check of the guessed entries rides along: does every chunk start where its left neighbour ended?
    if (c > 0 && c < a.n_chunks && a.start_off[c] != a.exit_off[c - 1]) *a.changed = 1u;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) warp_sum[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long s = 0;
        for (int i = 0; i < kChunkThreads / 32; ++i) s += warp_sum[i];
        a.block_prefix[blockIdx.x] = s;
    }
}

// One block: in-place exclusive scan of `arr` (block sums, or the sums of groups of 1024 regions); total and the
// shard's entry/exit.
__global__ void __launch_bounds__(1024) chunk_scan_kernel(const DecArgs a, unsigned long long *arr, uint32_t n_blocks) {
    __shared__ unsigned long long part[1024];
    const uint32_t t = threadIdx.x;
    const uint32_t per = (n_blocks + 1023u) / 1024u;
    const uint32_t lo = min(t * per, n_blocks), hi = min(lo + per, n_blocks);
    unsigned long long sum = 0;
    for (uint32_t i = lo; i < hi; ++i) sum += arr[i];
    part[t] = sum;
    __syncthreads();
    for (int d = 1; d < 1024; d <<= 1) {
        const unsigned long long v = t >= (uint32_t)d ? part[t - d] : 0ull;
        __syncthreads();
        part[t] += v;
        __syncthreads();
    }
    unsigned long long run = part[t] - sum;
    for (uint32_t i = lo; i < hi; ++i) {
        const unsigned long long v = arr[i];
        arr[i] = run;
        run += v;
    }
    if (t == 1023) {
        *a.total = part[1023];
        a.entry_exit[0] = a.start_off[0];
        a.entry_exit[1] = a.exit_off[a.n_chunks - 1];
    }
}

// ------------------------------------------------------------------ write
__global__ void __launch_bounds__(kChunkThreads, 5) chunk_write_kernel(const DecArgs a) {
    __shared__ __align__(16) uint32_t wlut_sh[kLutSize];
    __shared__ __align__(16) uint32_t rings[(kChunkThreads / 32) * 16 * 32];  // per warp: 16 words x 32 lanes
    __shared__ uint32_t warp_sum[kChunkThreads / 32];
    for (int i = threadIdx.x; i < kLutSize; i += kChunkThreads) wlut_sh[i] = a.wlut[i];

    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t bid = gridDim.x - 1u - blockIdx.x;  // last chunks first: the stream's ragged end (walked with every check) is the slow one
    const uint32_t c = bid * kChunkThreads + tid;
    const bool live = c < a.n_chunks;
    const uint32_t cnt = live ? a.count[c] : 0u;
    // where this chunk's text goes: block prefix + exclusive scan inside the block
    uint32_t incl = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t up = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= (uint32_t)d) incl += up;
    }
    if (lane == 31) warp_sum[warp] = incl;
    __syncthreads();
    uint32_t before = 0;
    for (uint32_t q = 0; q < warp; ++q) before += warp_sum[q];
    const unsigned long long o = a.block_prefix[bid] + before + (incl - cnt);
    if (!live || cnt == 0 || o >= a.max_symbols) return;

    const Chunk k = chunk_of(a, c);
    const uint32_t start = a.start_off[c];
    uint32_t bad = 0;
    if ((k.interior || (k.walkable && start < 256u)) && o + cnt <= a.max_symbols) {
        uint8_t *dst = a.out + o;
        OutRing r;
        r.ring_s = smem_addr(rings) + warp * 2048u + lane * 4u;
        r.head_skip = (uint32_t)(reinterpret_cast<uintptr_t>(dst) & 31u);
        r.gsector = dst - r.head_skip;
        r.lo = r.hi = 0;
        r.stored = 0;
        const uint32_t head = r.head_skip;
        uint32_t s = start | (head << 9);
        const uint64_t pair0 = k.begin >> 8;
        const uint32_t n_pairs = a.chunk_bytes >> 5;
        const uint32_t wlut_s = smem_addr(wlut_sh);
        // (no L2 prefetch of the whole chunk here: with the text also streaming out, lines fetched that early are evicted before use)
        uint32_t w[5];
        const uint32_t n_pieces = a.chunk_bytes >> 4;
        (void)n_pairs;
        Pair raw = load_pair_raw(a, pair0);
        Pair cur = raw;
#pragma unroll 1
        for (uint32_t p = 0; p < n_pieces; ++p) {
            if (!(p & 1u)) {  // a new sector: swap the one that has arrived, request the next (the piece after the chunk at the end)
                cur = swap_pair(raw);
                if (p + 2 < n_pieces)
                    raw = load_pair_raw(a, pair0 + (p >> 1) + 1);
                else
                    raw.a = __ldg(reinterpret_cast<const uint4 *>(a.body_aligned) + 2 * (pair0 + (p >> 1) + 1));
                w[0] = cur.a.x; w[1] = cur.a.y; w[2] = cur.a.z; w[3] = cur.a.w; w[4] = cur.b.x;
            } else {
                w[0] = cur.b.x; w[1] = cur.b.y; w[2] = cur.b.z; w[3] = cur.b.w; w[4] = bswap32(raw.a.x);
            }
            s = write_piece(w, s, p + 1 == n_pieces, wlut_s, r, a.clut, a.wlut, a.nodes, &bad);
        }
        // the unfinished word goes to the ring, then what is left of the last sector leaves bytewise
        const uint32_t n_end = s >> 9;  // bytes from the sector grid, head included
        if (n_end & 3u) sts_u32(ring_slot(r, n_end >> 2), r.hi >> (8u * (4u - (n_end & 3u))));
        for (uint32_t kk = r.head_skip ? head : (n_end & ~31u); kk < n_end; ++kk)
            r.gsector[kk & 31u] = (uint8_t)lds_u8(ring_slot(r, kk >> 2) + (kk & 3u));
    } else {
        uint32_t n = 0;
        if (k.begin + start < k.end) walk_generic<true>(a, k.begin + start, k.end, a.end_bit, &n, o, &bad, nullptr, wlut_sh);
    }
    if (bad) atomicOr(a.error_flags, kErrInvalidCode);
}

// ------------------------------------------------------------------ first-level tables from the trie, on the device
// The host parses the dictionary into a trie (a few hundred nodes, microseconds) and uploads only that; the lookup tables
// every decoder kernel reads (clut, wlut, marker slots, second-level tables: layouts in et_internal.h) are derived from
// it here, one thread per 12-bit window - without 80 KB of host table building and upload in front of every decode.
__global__ void __launch_bounds__(256) build_tables_kernel(const uint32_t *__restrict__ nodes, uint32_t *__restrict__ clut,
                                                           uint32_t *__restrict__ wlut, uint16_t *__restrict__ slots,
                                                           uint32_t *__restrict__ slot_count, uint32_t *__restrict__ slot_window) {
    const uint32_t w = blockIdx.x * 256 + threadIdx.x;
    if (w >= (uint32_t)kLutSize) return;
    uint32_t node = 0, pos = 0, cnt = 0, len0 = 0, len01 = 0, sym0 = 0, sym1 = 0;
    bool dead = false;  // ran into a bit pattern that is no code
    for (uint32_t b = 0; b < (uint32_t)kLutBits; ++b) {
        const uint32_t child = (__ldg(nodes + node) >> (16 * ((w >> (kLutBits - 1 - b)) & 1u))) & 0xFFFFu;
        if (child == kChildNone) {
            dead = true;
            break;
        }
        if (child & kChildLeaf) {
            if (cnt == 0) sym0 = child & 0xFFu, len0 = b + 1;
            if (cnt == 1) sym1 = child & 0xFFu, len01 = b + 1;
            ++cnt;
            pos = b + 1;
            node = 0;
        } else {
            node = child;
        }
    }
    uint16_t slot = kNoSlot;
    if (cnt == 0) {
        const uint32_t stuck = dead ? kChildNone : node;  // the trie node the window's bits lead to: the code is longer
        clut[w] = kLutMarker | (kLutMarker << 16);
        wlut[w] = (stuck & 0xFFFFu) | (kLutMarker << 16);
        if (stuck != kChildNone) {  // second level: the next 8 bits (the first kMaxSubTables marker windows to ask get one)
            const uint32_t k = atomicAdd(slot_count, 1u);
            if (k < kMaxSubTables) {
                slot = (uint16_t)k;
                slot_window[k] = w | (stuck << 16);
            }
        }
    } else {
        const uint32_t all = pos | (cnt << 9), one = len0 | (1u << 9);
        const uint32_t two = cnt >= 2 ? (len01 | (2u << 9)) : one;
        clut[w] = all | (one << 16);
        wlut[w] = sym0 | (sym1 << 8) | (two << 16);
    }
    slots[w] = slot;
}
// sub[slot][next 8 bits] = symbol | length << 8 for codes of 13..20 bits behind a marker window, 0 otherwise.
__global__ void __launch_bounds__(256) build_sub_tables_kernel(const uint32_t *__restrict__ nodes, uint16_t *__restrict__ slots,
                                                               const uint32_t *__restrict__ slot_count, const uint32_t *__restrict__ slot_window) {
    const uint32_t slot = blockIdx.x, x = threadIdx.x;  // one block per slot, one thread per 8-bit continuation
    uint16_t entry = 0;
    if (slot < min(*slot_count, kMaxSubTables)) {
        uint32_t node = slot_window[slot] >> 16;
        for (uint32_t b = 0; b < kSubBits; ++b) {
            const uint32_t child = (__ldg(nodes + node) >> (16 * ((x >> (kSubBits - 1 - b)) & 1u))) & 0xFFFFu;
            if (child == kChildNone) break;
            if (child & kChildLeaf) {
                entry = (uint16_t)((child & 0xFFu) | ((kLutBits + b + 1) << 8));
                break;
            }
            node = child;
        }
    }
    slots[kLutSize + (slot << kSubBits) + x] = entry;
}

#include "et_lanes.inc"

// The transfer-function walks with two tables in shared memory: the 16-bit windows (128 KiB: two codes of a byte per
// lookup where the 12-bit table of chunk_transfer_kernel gives one) and the 12-bit table for the last word of a chunk.
// One persistent CTA of 1024 threads per SM (the tables are loaded once), a thread per (chunk, entry), last chunks first.
constexpr uint32_t kCount16TableBytes = (1u << 16) * 2;
constexpr uint32_t kTransfer16Threads = 1024;
__global__ void __launch_bounds__(kTransfer16Threads, 1) chunk_transfer16_kernel(const DecArgs a, uint32_t s_log2, uint32_t n_states,
                                                                                const uint16_t *__restrict__ t16) {
    extern __shared__ __align__(128) uint8_t dyn[];
    uint32_t *clut_sh = reinterpret_cast<uint32_t *>(dyn + kCount16TableBytes);
    table_to_shared(dyn, t16, kCount16TableBytes);
    for (int i = threadIdx.x; i < kLutSize; i += kTransfer16Threads) clut_sh[i] = a.clut[i];
    __syncthreads();
    const uint32_t t16_s = smem_addr(dyn), clut_s = smem_addr(clut_sh);
    const uint64_t total = (uint64_t)a.n_chunks << s_log2;
    for (uint64_t item = (uint64_t)blockIdx.x * kTransfer16Threads + threadIdx.x; item < total; item += (uint64_t)gridDim.x * kTransfer16Threads) {
        const uint32_t idx = (uint32_t)(total - 1u - item);
        const uint32_t c = idx >> s_log2, e = idx & ((1u << s_log2) - 1u);
        if (e >= n_states) continue;
        if (c == 0) {  // chunk 0 is entered at the head of the stream (or at its guess, for a shard): one walk, what the scan starts from
            if (e == 0) sync_chunk(a, 0, a.head_known ? a.head_off : 0u, a.head_known != 0, clut_sh);
            continue;
        }
        const Chunk k = chunk_of(a, c);
        uint32_t cnt = 0, exit_bits = 0;
        if (k.walkable) {
            uint32_t entry;
            const uint32_t s = count_chunk_fast<true>(a, k, e, false, clut_s, &entry, t16_s);
            cnt = s >> 9;
            exit_bits = s & kPosMask;
        } else {
            uint64_t pos = k.begin + e;
            uint32_t bad = 0;
            if (pos < k.end) pos = walk_generic<false>(a, pos, k.end, a.end_bit, &cnt, 0, &bad, clut_sh);
            exit_bits = pos > k.end ? (uint32_t)(pos - k.end) : 0u;
        }
        a.tr_exit[idx] = (uint8_t)(exit_bits < n_states ? exit_bits : 0xFFu);
        a.tr_cnt[idx] = (uint16_t)cnt;
    }
}

uint64_t chunk_count(const UnpackGeometry &g, uint32_t chunk_bytes) {
    const uint64_t grid_bit = g.own_begin_bit / 256 * 256;
    const uint64_t bits = (uint64_t)chunk_bytes * 8;
    return g.own_end_bit > grid_bit ? (g.own_end_bit - grid_bit + bits - 1) / bits : 0;
}

}  // namespace

// Once per context (the shared-memory opt-in of the two big kernels is a property of the function on the
// context's device): what the device offers, and the attributes the launches rely on.
cudaError_t unpack_init_device(int device, UnpackTuning *tune) {
    cudaError_t err;
    if ((err = cudaDeviceGetAttribute(&tune->num_sms, cudaDevAttrMultiProcessorCount, device)) != cudaSuccess) return err;
    if ((err = cudaDeviceGetAttribute(&tune->max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, device)) != cudaSuccess) return err;
    if ((err = cudaFuncSetAttribute(region_write_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, tune->max_smem)) != cudaSuccess)
        return err;
    if ((err = cudaFuncSetAttribute(chunk_transfer16_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, tune->max_smem)) != cudaSuccess)
        return err;
    if ((err = cudaFuncSetAttribute(region_sync_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, tune->max_smem)) != cudaSuccess)
        return err;
    // the lane-interleaved decoder's tables, built on the device for every stream (lane_tables_kernel)
    return cudaMalloc(&tune->d_lane_tables, kCountTableBytes + kWriteTableBytes + kSingleTableBytes + kCount16TableBytes);
}
void unpack_free_device(UnpackTuning *tune) {
    if (tune->d_lane_tables) cudaFree(tune->d_lane_tables);
    tune->d_lane_tables = nullptr;
}

// d_nodes holds the trie (uploaded); builds clut | wlut (contiguous: d_clut, d_clut + kLutSize) and the slot / second-level
// tables.  d_work: 2 + kMaxSubTables words of device scratch.
cudaError_t launch_build_tables(const uint32_t *d_nodes, uint32_t *d_clut, uint16_t *d_slots, uint32_t *d_work, cudaStream_t stream,
                                int *launches) {
    cudaError_t err = cudaMemsetAsync(d_work, 0, 4, stream);
    if (err != cudaSuccess) return err;
    build_tables_kernel<<<kLutSize / 256, 256, 0, stream>>>(d_nodes, d_clut, d_clut + kLutSize, d_slots, d_work, d_work + 2);
    build_sub_tables_kernel<<<kMaxSubTables, 1u << kSubBits, 0, stream>>>(d_nodes, d_slots, d_work, d_work + 2);
    if (launches) *launches += 2;
    return cudaGetLastError();
}

UnpackGeometry unpack_geometry(const void *d_body, size_t body_bytes) {
    UnpackGeometry g;
    const uintptr_t p = reinterpret_cast<uintptr_t>(d_body);
    const uint32_t mis = (uint32_t)(p & 15u);
    g.body_aligned = reinterpret_cast<const uint8_t *>(p - mis);
    g.byte_lo = mis;
    g.byte_hi = (uint64_t)mis + body_bytes;
    g.own_begin_bit = (uint64_t)mis * 8;
    g.own_end_bit = g.byte_hi * 8;
    g.end_bit = g.byte_hi * 8;
    g.head_known = true;
    g.head_bit = g.own_begin_bit;
    return g;
}

UnpackGeometry unpack_geometry_shard(const void *d_range, size_t range_bytes, size_t own_begin_byte, size_t own_end_byte,
                                     long long head_bit) {
    UnpackGeometry g;
    g.body_aligned = static_cast<const uint8_t *>(d_range);  // caller guarantees 16-byte alignment
    g.byte_lo = 0;
    g.byte_hi = range_bytes;
    g.own_begin_bit = (uint64_t)own_begin_byte * 8;
    g.own_end_bit = (uint64_t)own_end_byte * 8;
    g.end_bit = (uint64_t)range_bytes * 8;
    g.head_known = head_bit >= 0;
    g.head_bit = head_bit >= 0 ? (uint64_t)head_bit : g.own_begin_bit;
    return g;
}

// Streams of at least this many bytes take the lane-interleaved decoder (enough regions to give every
// SM a full set of warps).  ET_TUNE_LANE_MIN_BYTES overrides it (tests run the path on small inputs).
static uint64_t lane_path_min_bytes(const UnpackTuning &tune) {
    if (tune.lane_min_bytes >= 0)
        return (uint64_t)tune.lane_min_bytes > 2 * kRegionBytes ? (uint64_t)tune.lane_min_bytes : 2 * kRegionBytes;
    // MEASURED (r2, text): below ~2 MB of stream the per-thread kernels are as fast or faster (fewer launches, smaller tables
    // to load); 1.2 MB: 0.135 ms against 0.144, 2.5 MB: 0.148 against 0.132, 4.9 MB: 0.171 against 0.119
    return (uint64_t)tune.num_sms * 3 * kRegionBytes;
}

// Chunk size.  256 B suits codes that re-synchronise within a few symbols.  When all code
// lengths are (nearly) equal a wrong parse survives for kilobytes (uniform bytes: 7/8-bit
// codes, ~2 KB on average), and every fixpoint round repairs only one chunk's worth of it, so
// such codes get chunks longer than their synchronisation distance.  Short streams get
// shorter chunks so that the GPU is not left mostly idle.
uint32_t unpack_chunk_bytes(const UnpackGeometry &g, const UnpackTuning &tune, uint32_t min_length, uint32_t max_length) {
    const int num_sms = tune.num_sms;
    const uint64_t bytes = (g.own_end_bit - g.own_begin_bit + 7) / 8;
    const uint32_t spread = max_length - min_length;
    if (spread > 2 && bytes >= lane_path_min_bytes(tune)) return kLaneBytes;  // lane-interleaved decoder
    if (spread <= 2 && max_length <= kMaxStates) {
        // slowly synchronising codes go through transfer functions (max_length walks per chunk, all parallel); the write
        // walk is one thread per chunk, so short chunks keep the GPU full
        uint32_t cb = 512u;
        while (cb > 256u && bytes / cb * max_length < (uint64_t)num_sms * 4096) cb >>= 1;
        return cb;
    }
    uint32_t cb = spread <= 1 ? 4096u : spread == 2 ? 1024u : 256u;
    const uint32_t floor_cb = cb > 256u ? 256u : 32u;
    while (cb > floor_cb && bytes / cb < (uint64_t)num_sms * 2048) cb >>= 1;
    return cb;
}

size_t unpack_scratch_bytes(const UnpackGeometry &g, uint32_t chunk_bytes, uint32_t transfer_states) {
    return decode_layout(nullptr, chunk_count(g, chunk_bytes), chunk_bytes == kLaneBytes, transfer_states).bytes;
}

// Lane-interleaved decoder: the same protocol as below with regions of 32 chunks per warp.  One extra
// look at the scratch header after the scan: the largest region sizes the text stage of a warp.
static cudaError_t launch_unpack_lanes(const DecArgs &a, uint32_t n_regions, const DecodeStatus *d_status, DecodeStatus *h_status, cudaStream_t stream,
                                       const UnpackTuning &tune, int *launches, uint32_t *rounds_out) {
    cudaError_t err;
    const int max_smem = tune.max_smem, num_sms = tune.num_sms;
    // count walk: one CTA per SM, as many warps as images fit beside the tables
    uint32_t sync_warps = ((uint32_t)max_smem - kSyncTableBytes) / kImgBytes;
    if (sync_warps > kMaxLaneWarps) sync_warps = kMaxLaneWarps;
    if (tune.sync_warps > 0 && (uint32_t)tune.sync_warps < sync_warps) sync_warps = (uint32_t)tune.sync_warps;
    if (sync_warps > 4) sync_warps &= ~3u;  // the same number of warps on each of the SM's four schedulers: they share the regions evenly
    // a stream with fewer regions than the GPU has warps for: a few warps on every SM rather than full CTAs on a few SMs
    auto spread = [&](uint32_t warps_max) {
        uint32_t w = ((n_regions + (uint32_t)num_sms - 1) / (uint32_t)num_sms + 3u) & ~3u;
        return w < 4u ? 4u : w > warps_max ? warps_max : w;
    };
    if (sync_warps > 4) sync_warps = spread(sync_warps);
    const uint32_t sync_smem = kSyncTableBytes + sync_warps * kImgBytes;
    const uint32_t sync_blocks = (n_regions + sync_warps - 1) / sync_warps;
    const uint32_t sync_grid = sync_blocks < (uint32_t)num_sms ? sync_blocks : (uint32_t)num_sms;
    DecArgs &am = const_cast<DecArgs &>(a);
    unsigned long long *d_dbg = nullptr;
    if (tune.debug & 1) {
        if (cudaMalloc(&d_dbg, 2 * 256 * 35 * 8) == cudaSuccess) cudaMemsetAsync(d_dbg, 0, 2 * 256 * 35 * 8, stream);
    }
    am.dbg = d_dbg;
    lane_tables_kernel<<<(1u << 16) / 256, 256, 0, stream>>>(a.nodes, const_cast<uint16_t *>(a.t_count), const_cast<uint32_t *>(a.t_write),
                                                            const_cast<uint8_t *>(a.t_single), nullptr);
    if (launches) *launches += 1;
    const uint32_t check_grid = (n_regions + 31u) / 32u;  // 8 warps x 4 regions per CTA
    // one repair round: list the regions with a wrong entry, walk those again from their neighbours' exits
    auto repair = [&](int round) -> cudaError_t {
        cudaError_t e = cudaMemsetAsync(a.work_count, 0, 4, stream);
        if (e != cudaSuccess) return e;
        region_check_kernel<<<check_grid, 256, 0, stream>>>(a, n_regions);
        region_sync_kernel<<<sync_grid, sync_warps * 32, sync_smem, stream>>>(a, n_regions, round, sync_warps);
        if (launches) *launches += 2;
        return cudaSuccess;
    };
    if ((err = cudaMemsetAsync(a.work_count, 0, 4, stream)) != cudaSuccess) return err;
    region_sync_kernel<<<sync_grid, sync_warps * 32, sync_smem, stream>>>(a, n_regions, 0, sync_warps);
    // first repair round: the count walk listed the regions whose chunks disagree, edge_check adds those whose first
    // chunk does not start where the region before ended
    edge_check_kernel<<<(n_regions + 255) / 256, 256, 0, stream>>>(a, n_regions);
    region_sync_kernel<<<sync_grid, sync_warps * 32, sync_smem, stream>>>(a, n_regions, 1, sync_warps);
    if (launches) *launches += 3;
    if ((err = cudaMemsetAsync(a.changed, 0, 2 * sizeof(uint32_t), stream)) != cudaSuccess) return err;  // changed and max_sum
    uint32_t rounds = 2;
    for (;;) {
        const uint32_t n_groups = (n_regions + kGroupRegions - 1) / kGroupRegions;
        region_sum_kernel<<<n_groups, 1024, 0, stream>>>(a, n_regions);
        chunk_scan_kernel<<<1, 1024, 0, stream>>>(a, a.group_prefix, n_groups);
        region_apply_kernel<<<n_groups, 1024, 0, stream>>>(a, n_regions);
        const uint32_t write_warps = spread(tune.write_warps > 0 ? (uint32_t)tune.write_warps : 16u);
        const uint32_t write_blocks = (n_regions + write_warps - 1) / write_warps;
        region_write_kernel<<<write_blocks < (uint32_t)num_sms ? write_blocks : (uint32_t)num_sms, 512, max_smem, stream>>>(
            a, n_regions, (uint32_t)max_smem, write_warps);
        if (launches) *launches += 4;
        // one look at the scratch header: error flags, symbols found, "an entry was wrong", entry and exit of the shard
        if ((err = cudaMemcpyAsync(h_status, d_status, kDecodeStatusReadBack, cudaMemcpyDeviceToHost, stream)) != cudaSuccess) return err;
        if ((err = cudaStreamSynchronize(stream)) != cudaSuccess) return err;
        if ((tune.debug & 1) && d_dbg) {
            static unsigned long long h[2 * 256 * 35];
            cudaMemcpy(h, d_dbg, sizeof h, cudaMemcpyDeviceToHost);
            for (int k = 0; k < 2; ++k) {
                unsigned long long t0 = ~0ull, t1 = 0;
                for (int i = 0; i < 256; ++i)
                    if (h[(k * 256 + i) * 3 + 2]) {
                        t0 = h[(k * 256 + i) * 3 + 1] < t0 ? h[(k * 256 + i) * 3 + 1] : t0;
                        t1 = h[(k * 256 + i) * 3 + 2] > t1 ? h[(k * 256 + i) * 3 + 2] : t1;
                    }
                fprintf(stderr, "[lanes] %s kernel: %.1f us; per CTA (smid:start..end us):", k ? "write" : "sync", (t1 - t0) / 1e3);
                for (int i = 0; i < 256; ++i)
                    if (h[(k * 256 + i) * 3 + 2])
                        fprintf(stderr, " %llu:%.0f..%.0f", h[(k * 256 + i) * 3], (h[(k * 256 + i) * 3 + 1] - t0) / 1e3, (h[(k * 256 + i) * 3 + 2] - t0) / 1e3);
                fprintf(stderr, "\n");
                int slow = 0;
                for (int i = 0; i < 256; ++i)
                    if (h[(k * 256 + i) * 3 + 2] > h[(k * 256 + slow) * 3 + 2]) slow = i;
                fprintf(stderr, "[lanes] slowest block %d, its warps end at (us):", slow);
                for (int w = 0; w < 32; ++w)
                    if (h[2 * 256 * 3 + (k * 256 + slow) * 32 + w]) fprintf(stderr, " %d:%.0f", w, (h[2 * 256 * 3 + (k * 256 + slow) * 32 + w] - t0) / 1e3);
                fprintf(stderr, "\n");
            }
        }
        if (tune.debug & 1)
            fprintf(stderr, "[lanes] regions=%u chunks=%u max_sum=%u rounds=%u changed=%u\n", n_regions, a.n_chunks,
                    h_status->max_sum, rounds, h_status->changed);
        if (h_status->changed == 0) break;  // every entry was the true one: what the write walk produced stands
        // entries still moving: fixpoint rounds, four per host visit; a check that lists nothing is the proof
        for (;;) {
            for (int i = 0; i < 4; ++i)
                if ((err = repair((int)rounds + i)) != cudaSuccess) return err;
            rounds += 4;
            if ((err = cudaMemsetAsync(a.changed, 0, 2 * sizeof(uint32_t), stream)) != cudaSuccess) return err;
            if ((err = cudaMemsetAsync(a.work_count, 0, 4, stream)) != cudaSuccess) return err;
            region_check_kernel<<<check_grid, 256, 0, stream>>>(a, n_regions);
            if (launches) *launches += 1;
            if ((err = cudaMemcpyAsync(h_status, d_status, kDecodeStatusReadBack, cudaMemcpyDeviceToHost, stream)) != cudaSuccess) return err;
            if ((err = cudaStreamSynchronize(stream)) != cudaSuccess) return err;
            if (tune.debug & 1) fprintf(stderr, "[lanes] repair rounds=%u changed=%u\n", rounds, h_status->changed);
            if (h_status->changed == 0) break;
            if (rounds > a.n_chunks + 8u) return cudaErrorUnknown;  // cannot happen: each round settles one more chunk
        }
        if ((err = cudaMemsetAsync(a.error_flags, 0, 4, stream)) != cudaSuccess) return err;  // raised by a wrong parse
    }
    if (rounds_out) *rounds_out = rounds;
    if (d_dbg) cudaFree(d_dbg);
    return cudaGetLastError();
}

cudaError_t launch_unpack(const UnpackGeometry &g, uint32_t chunk_bytes, const uint32_t *d_clut, const uint32_t *d_wlut,
                          const uint32_t *d_nodes, const uint16_t *d_slots, uint8_t *d_out, uint64_t max_symbols, void *scratch_base,
                          DecodeStatus *h_status, cudaStream_t stream, const UnpackTuning &tune, uint32_t fixed_len, uint32_t transfer_states,
                          int *launches, uint32_t *rounds_out) {
    const uint64_t n64 = chunk_count(g, chunk_bytes);
    const bool lanes = chunk_bytes == kLaneBytes;
    const DecodeLayout L = decode_layout(scratch_base, n64, lanes, transfer_states);
    cudaError_t err = cudaMemsetAsync(L.status, 0, sizeof(DecodeStatus), stream);
    if (err != cudaSuccess) return err;
    if (rounds_out) *rounds_out = 0;
    if (n64 == 0) {  // nothing to decode: all-zero status
        *h_status = DecodeStatus{};
        return cudaStreamSynchronize(stream);
    }
    const uint32_t n = (uint32_t)n64;
    const uint32_t nb = (uint32_t)L.n_blocks;
    DecArgs a;
    a.body_aligned = g.body_aligned;
    a.grid_bit = g.own_begin_bit / 256 * 256;  // chunks are whole 32-byte sectors
    a.own_end_bit = g.own_end_bit;
    a.end_bit = g.end_bit;
    a.byte_lo = g.byte_lo;
    a.byte_hi = g.byte_hi;
    a.head_known = g.head_known ? 1u : 0u;
    a.head_off = (uint32_t)(g.head_bit - a.grid_bit);
    a.n_chunks = n;
    a.chunk_bytes = chunk_bytes;
    a.fixed_len = fixed_len;
    a.clut = d_clut;
    a.wlut = d_wlut;
    a.nodes = d_nodes;
    a.slots = d_slots;
    a.t_count = reinterpret_cast<const uint16_t *>(tune.d_lane_tables);
    a.t_write = reinterpret_cast<const uint32_t *>(static_cast<const uint8_t *>(tune.d_lane_tables) + kCountTableBytes);
    a.t_single = static_cast<const uint8_t *>(tune.d_lane_tables) + kCountTableBytes + kWriteTableBytes;
    a.error_flags = &L.status->error_flags;
    a.total = &L.status->total;
    a.changed = &L.status->changed;
    a.max_sum = &L.status->max_sum;
    a.entry_exit = &L.status->entry;
    a.work_count = &L.status->work_count;
    a.block_prefix = L.block_prefix;
    a.count = L.count;
    a.start_off = L.start_off;
    a.exit_off = L.exit_off;
    a.mid = L.mid;
    a.group_prefix = L.group_prefix;
    a.work = L.work;
    a.edge = L.edge;
    a.rsum = L.rsum;
    a.self_listed = L.self_listed;
    a.tr_exit = L.tr_exit;
    a.tr_cnt = L.tr_cnt;
    a.out = d_out;
    a.max_symbols = max_symbols;
    a.dbg = nullptr;

    if (lanes) return launch_unpack_lanes(a, nb, L.status, h_status, stream, tune, launches, rounds_out);

    // Common case (codes that re-synchronise quickly): one walk from the guesses, one repair
    // round for the few chunks whose run-up was too short (text: 0.1 % of them; their exits do
    // not move, because a walk that missed 128 bits of run-up still locks on inside 2048 bits of
    // chunk), the final check fused into the block sums, the write walk — and a single look at
    // the flag at the very end.  Only when that check failed (slowly synchronising codes) do
    // the fixpoint rounds run, and the sums and the write walk are repeated.
    const bool transfer = L.tr_log2 != 0 && !fixed_len && n > 1 && !tune.no_transfer;
    uint32_t rounds = 2;
    if (transfer) {
        // slowly synchronising codes: the chunks' transfer functions and a scan instead of repair rounds
        const uint32_t s_log2 = L.tr_log2;
        const uint64_t threads = (uint64_t)n << s_log2;
        if (tune.d_lane_tables && threads >= (uint64_t)tune.num_sms * kTransfer16Threads * 4 &&
            (size_t)tune.max_smem >= kCount16TableBytes + kLutSize * 4u) {
            uint16_t *t16 = reinterpret_cast<uint16_t *>(static_cast<uint8_t *>(tune.d_lane_tables) + kCountTableBytes + kWriteTableBytes + kSingleTableBytes);
            lane_tables_kernel<<<(1u << 16) / 256, 256, 0, stream>>>(a.nodes, nullptr, nullptr, nullptr, t16);
            chunk_transfer16_kernel<<<tune.num_sms, kTransfer16Threads, kCount16TableBytes + kLutSize * 4u, stream>>>(a, s_log2, transfer_states, t16);
            if (launches) *launches += 1;
        } else
            chunk_transfer_kernel<<<(unsigned)((threads + kChunkThreads - 1) / kChunkThreads), kChunkThreads, 0, stream>>>(a, s_log2, transfer_states);
        const uint32_t seg_blocks = (uint32_t)L.seg_blocks;
        compose_segments_kernel<<<seg_blocks, kSegThreads, 0, stream>>>(a, s_log2, transfer_states, L.seg_prefix, L.block_map);
        compose_blocks_kernel<<<1, 1024, 0, stream>>>(seg_blocks, transfer_states, L.block_map);
        compose_apply_kernel<<<seg_blocks, kSegThreads, 0, stream>>>(a, s_log2, transfer_states, L.seg_prefix, L.block_map);
        if (launches) *launches += 4;
        rounds = 1;
    } else {
        chunk_sync_kernel<<<nb, kChunkThreads, 0, stream>>>(a, 0);
        chunk_sync_kernel<<<nb, kChunkThreads, 0, stream>>>(a, 1);
        if (launches) *launches += 2;
    }
    err = cudaMemsetAsync(a.changed, 0, 4, stream);
    if (err != cudaSuccess) return err;
    // Fixpoint rounds, four per host visit (the flag is cleared before the last of them: a round
    // that changed nothing is the proof).
    auto settle = [&]() -> cudaError_t {
        for (;;) {
            for (int i = 0; i < 3; ++i) chunk_sync_kernel<<<nb, kChunkThreads, 0, stream>>>(a, (int)rounds + i);
            cudaError_t e = cudaMemsetAsync(a.changed, 0, 4, stream);
            if (e != cudaSuccess) return e;
            chunk_sync_kernel<<<nb, kChunkThreads, 0, stream>>>(a, (int)rounds + 3);
            rounds += 4;
            if (launches) *launches += 4;
            e = cudaMemcpyAsync(&h_status->changed, a.changed, 4, cudaMemcpyDeviceToHost, stream);
            if (e != cudaSuccess) return e;
            e = cudaStreamSynchronize(stream);
            if (e != cudaSuccess) return e;
            if (h_status->changed == 0) return cudaSuccess;
            if (rounds > n + 8u) return cudaErrorUnknown;  // cannot happen: each round settles one more chunk
        }
    };
    // Long chunks were chosen because this code synchronises slowly: the guesses are known to be
    // poor, so settle the entries before spending a write walk on them.
    if (chunk_bytes > 256u && !fixed_len && !transfer) {
        err = settle();
        if (err != cudaSuccess) return err;
    }
    for (;;) {
        chunk_sum_kernel<<<nb, kChunkThreads, 0, stream>>>(a);
        chunk_scan_kernel<<<1, 1024, 0, stream>>>(a, a.block_prefix, nb);
        chunk_write_kernel<<<nb, kChunkThreads, 0, stream>>>(a);
        if (launches) *launches += 3;
        err = cudaMemcpyAsync(h_status, L.status, kDecodeStatusReadBack, cudaMemcpyDeviceToHost, stream);  // for the caller as well
        if (err != cudaSuccess) return err;
        err = cudaStreamSynchronize(stream);
        if (err != cudaSuccess) return err;
        if (h_status->changed == 0) break;  // every entry was the true one: what the write walk produced stands
        err = settle();
        if (err != cudaSuccess) return err;
        // the error flags the first write walk may have raised came from a wrong parse
        err = cudaMemsetAsync(a.error_flags, 0, 4, stream);
        if (err != cudaSuccess) return err;
    }
    if (rounds_out) *rounds_out = rounds;
    return cudaGetLastError();
}

}  // namespace et
