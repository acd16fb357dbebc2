"""Device scratch layouts (entreepy_b200/csrc/et_scratch.h), checked on the CPU with one g++ driver:
- the decoder's and the pack's scratch: every array lies inside the block, meets its alignment, overlaps no other array
  and holds the elements the kernels index; the block is no larger than the sizing formulas the layouts replaced, plus
  alignment padding;
- the batched decoder's group scratch (batch_layout): every array lies inside the block, is aligned and overlaps no
  other, for item counts up to a whole group and chunk counts up to the chunks of a group's bytes; the runs the host
  clears, uploads and reads back hold exactly their arrays; and the layout the head gather uses places its arrays where
  the full layout does;
- the batched encoder's group scratch (enc_batch_layout): the same, for region and tile counts up to those of a group's
  bytes and header bytes up to a full header per text; the layout the histogram uses places its arrays where the full
  layout does.
Also: the built library exports the batch entry point."""
import ctypes
import os
import shutil
import subprocess

import pytest

from conftest import ROOT
from entreepy_b200 import _abi

CSRC = os.path.join(ROOT, "entreepy_b200", "csrc")

DRIVER = r"""
#include <algorithm>
#include <cstdio>
#include <string>
#include <vector>

#include "et_scratch.h"

using namespace et;

static_assert(offsetof(DecodeStatus, error_flags) == 4 && offsetof(DecodeStatus, total) == 8, "status layout");
static_assert(offsetof(DecodeStatus, changed) == 16 && offsetof(DecodeStatus, max_sum) == 20, "status layout");
static_assert(offsetof(DecodeStatus, entry) == 24 && offsetof(DecodeStatus, exit) == 28, "status layout");
static_assert(offsetof(DecodeStatus, work_count) == 32 && kDecodeStatusReadBack == 32, "status layout");

struct Arr {
    const char *name;
    const void *p;
    size_t bytes;  // what the kernels may touch: element count x element size
    size_t align = kScratchAlign;
};

static uint8_t *const kBase = reinterpret_cast<uint8_t *>(uintptr_t(1) << 40);
static int failures = 0;
static long layouts = 0;

static size_t off(const void *p) { return (size_t)(static_cast<const uint8_t *>(p) - kBase); }

#define CHECK(cond, ...)                                   \
    do {                                                   \
        if (!(cond) && ++failures <= 20) {                 \
            fprintf(stderr, __VA_ARGS__);                  \
            fprintf(stderr, "  [%s]\n", #cond);            \
        }                                                  \
    } while (0)

static void check(const char *what, std::vector<Arr> arrs, size_t bytes, size_t limit) {
    ++layouts;
    for (const Arr &a : arrs) {
        CHECK(a.p != nullptr, "%s: %s missing", what, a.name);
        if (!a.p) return;
        const size_t off = (size_t)(static_cast<const uint8_t *>(a.p) - kBase);
        CHECK(off % a.align == 0, "%s: %s at %zu is not %zu-byte aligned", what, a.name, off, a.align);
        CHECK(off + a.bytes <= bytes, "%s: %s [%zu, %zu) ends past the block of %zu bytes", what, a.name, off, off + a.bytes, bytes);
    }
    for (size_t i = 0; i < arrs.size(); ++i)
        for (size_t j = i + 1; j < arrs.size(); ++j) {
            const uint8_t *a = static_cast<const uint8_t *>(arrs[i].p), *b = static_cast<const uint8_t *>(arrs[j].p);
            const bool overlap = a < b + arrs[j].bytes && b < a + arrs[i].bytes;
            CHECK(!overlap, "%s: %s and %s overlap", what, arrs[i].name, arrs[j].name);
        }
    CHECK(bytes <= limit + 4096, "%s: %zu bytes, the old formula gave %zu", what, bytes, limit);
}

static uint64_t cdiv(uint64_t a, uint64_t b) { return (a + b - 1) / b; }

// The decoder's scratch before the layout was declared once (unpack_scratch_bytes).
static size_t old_decode_bytes(uint64_t n, bool lanes) {
    const uint64_t nb = cdiv(n, lanes ? 32 : kChunkThreads);
    const uint64_t ng = cdiv(nb, kGroupRegions);
    const size_t transfer = lanes ? 0 : (size_t)n * kMaxStates * 3 + 64 + ((size_t)n / kSegChunks + 2 * kSegThreads + 64) * 8;
    return 64 + (size_t)nb * 8 + (size_t)n * (4 + 2 + 2 + sizeof(mid_t)) + 64 + (size_t)ng * 8 + 64 + (size_t)nb * (4 + 4 + 4 + 1) + 320 + transfer;
}

static void check_decode(uint64_t n, bool lanes, uint32_t states) {
    char what[128];
    snprintf(what, sizeof what, "decode n=%llu lanes=%d states=%u", (unsigned long long)n, (int)lanes, states);
    const DecodeLayout L = decode_layout(kBase, n, lanes, states);
    const DecodeLayout S = decode_layout(nullptr, n, lanes, states);
    CHECK(S.bytes == L.bytes && S.status == nullptr && S.count == nullptr, "%s: sizing differs from carving", what);
    const uint64_t nb = cdiv(n, lanes ? 32 : kChunkThreads);
    CHECK(L.n_blocks == nb, "%s: %llu blocks", what, (unsigned long long)L.n_blocks);
    std::vector<Arr> arrs = {
        {"status", L.status, sizeof(DecodeStatus)},
        {"block_prefix", L.block_prefix, nb * 8},
        {"count", L.count, n * 4},
        {"start_off", L.start_off, n * 2},
        {"exit_off", L.exit_off, n * 2},
    };
    if (lanes) {
        arrs.push_back({"mid", L.mid, n * sizeof(mid_t)});
        arrs.push_back({"group_prefix", L.group_prefix, (cdiv(nb, 1024) + 1) * 8});
        arrs.push_back({"work", L.work, (nb + 8) * 4});
        arrs.push_back({"edge", L.edge, (nb + 8) * 4});
        arrs.push_back({"rsum", L.rsum, (nb + 8) * 4});
        arrs.push_back({"self_listed", L.self_listed, nb});
    }
    const bool transfer = !lanes && states >= 2 && states <= kMaxStates;
    CHECK((L.tr_exit != nullptr) == transfer && (L.seg_prefix != nullptr) == transfer, "%s: transfer arrays", what);
    if (transfer) {
        uint32_t s_log2 = 1;
        while ((1u << s_log2) < states) ++s_log2;
        CHECK(L.tr_log2 == s_log2, "%s: tr_log2 %u", what, L.tr_log2);
        const uint64_t seg_blocks = cdiv(n, kSegChunks * kSegThreads);
        CHECK(L.seg_blocks == seg_blocks, "%s: %llu segment blocks", what, (unsigned long long)L.seg_blocks);
        arrs.push_back({"tr_exit", L.tr_exit, (n << s_log2)});
        arrs.push_back({"tr_cnt", L.tr_cnt, (n << s_log2) * 2});
        arrs.push_back({"seg_prefix", L.seg_prefix, seg_blocks * kSegThreads * 8});
        arrs.push_back({"block_map", L.block_map, seg_blocks * 8});
    }
    check(what, arrs, L.bytes, old_decode_bytes(n, lanes));
}

// The pack's scratch before (pack_scratch_bytes).
static size_t old_pack_bytes(uint32_t num_tiles) {
    const size_t t = (size_t)num_tiles * 2 + 2;
    const size_t groups = (t + 7) / 8;
    return 16 + t * 14 + groups * 8 + 16 + t * 64 + 64;
}

static void check_pack(uint64_t n, uint32_t misalign) {
    char what[128];
    snprintf(what, sizeof what, "pack n=%llu misalign=%u", (unsigned long long)n, misalign);
    const uint64_t v_end = n + misalign;
    const uint32_t num_tiles = (uint32_t)cdiv(v_end, 4096);
    const PackLayout L = pack_layout(kBase, num_tiles);
    CHECK(pack_layout(nullptr, num_tiles).bytes == L.bytes, "%s: sizing differs from carving", what);
    const uint64_t slots = 2ull * num_tiles + 2;
    const uint64_t regions = cdiv(v_end, 2048);
    CHECK(num_tiles <= slots && regions <= slots && cdiv(regions, 1024) <= (slots + 7) / 8, "%s: slots", what);
    check(what,
          {{"ticket", L.ticket, 16, 16},
           {"tile_state", L.tile_state, slots * 8, 16},
           {"group_prefix", L.group_prefix, (slots + 7) / 8 * 8, 8},
           {"tile_bits", L.tile_bits, slots * 4, 4},
           {"seam_head", L.seam_head, slots, 1},
           {"seam_tail", L.seam_tail, slots, 1},
           {"run_bits", L.run_bits, slots * 64, 16}},
          L.bytes, old_pack_bytes(num_tiles));
}

static void scratch_layouts() {
    const uint64_t counts[] = {0, 1, 31, 32, 33, 255, 256, 257, 1023, 1024, 1025, 1ull << 20};
    std::vector<uint32_t> states = {0};
    for (uint32_t s = 2; s <= kMaxStates; ++s) states.push_back(s);
    // the lane decoder's chunks of 33 words, and the per-thread chunk sizes
    const uint32_t chunk_sizes[] = {132, 32, 64, 128, 256, 512, 1024, 2048, 4096};
    for (uint32_t cb : chunk_sizes) {
        std::vector<uint64_t> ns(std::begin(counts), std::end(counts));
        ns.push_back(cdiv(4ull << 30, cb));  // a 4 GiB body
        for (uint64_t n : ns)
            for (uint32_t s : states) check_decode(n, cb == 132, s);
    }
    std::vector<uint64_t> lengths = {1ull << 30, (1ull << 32) - 16};
    for (uint64_t b : {2048ull, 4096ull, 8192ull, 3ull * 4096})
        for (uint64_t d = 0; d <= 17; ++d) {
            lengths.push_back(b + d);
            if (d <= b) lengths.push_back(b - d);
        }
    for (uint64_t n : lengths)
        for (uint32_t m : {0u, 1u, 15u}) check_pack(n, m);
}

// ---- the batched decoder's group scratch
static void check_batch(uint32_t items, size_t args_bytes, uint64_t tiles, uint64_t node_words, uint64_t chunks) {
    char what[160];
    snprintf(what, sizeof what, "items=%u args=%zu tiles=%llu nodes=%llu chunks=%llu", items, args_bytes, (unsigned long long)tiles,
             (unsigned long long)node_words, (unsigned long long)chunks);
    ++layouts;
    const BatchLayout L = batch_layout(kBase, items, args_bytes, tiles, node_words, chunks);
    const BatchLayout S = batch_layout(nullptr, items, args_bytes, tiles, node_words, chunks);
    CHECK(S.bytes == L.bytes && S.host_bytes == L.host_bytes && S.status == nullptr, "%s: sizing differs from carving", what);
    const std::vector<Arr> arrs = {
        {"status", L.status, sizeof(BatchStatus)},
        {"item_status", L.item_status, items * sizeof(BatchItemStatus)},
        {"work", L.work, (size_t)items * kBatchWorkWords * 4},
        {"sources", L.sources, items * sizeof(BatchSource)},
        {"heads", L.heads, (size_t)items * kBatchHeadBytes},
        {"args", L.args, (size_t)items * args_bytes},
        {"tiles", L.tiles, tiles * sizeof(BatchTile)},
        {"nodes", L.nodes, node_words * 4},
        {"lut", L.lut, (size_t)items * 2 * kLutSize * 4},
        {"slots", L.slots, (size_t)items * kBatchSlots * 2},
        {"tile_sums", L.tile_sums, (tiles + 1) * 8},
        {"count", L.count, chunks * 4},
        {"start_off", L.start_off, chunks * 2},
        {"exit_off", L.exit_off, chunks * 2},
    };
    for (const Arr &a : arrs) {
        CHECK(a.p != nullptr, "%s: %s missing", what, a.name);
        if (!a.p) return;
        CHECK(off(a.p) % kScratchAlign == 0, "%s: %s at %zu is not aligned", what, a.name, off(a.p));
        CHECK(off(a.p) + a.bytes <= L.bytes, "%s: %s ends past the block", what, a.name);
    }
    for (size_t i = 0; i < arrs.size(); ++i)
        for (size_t j = i + 1; j < arrs.size(); ++j) {
            const size_t a = off(arrs[i].p), b = off(arrs[j].p);
            CHECK(!(a < b + arrs[j].bytes && b < a + arrs[i].bytes), "%s: %s and %s overlap", what, arrs[i].name, arrs[j].name);
        }
    // the runs: cleared [0, clear_bytes) = status .. work; read back [0, status_bytes) = status, item_status;
    // uploaded [upload_begin, upload_end) = args .. nodes; the pinned mirror [0, host_bytes) = everything up to nodes
    CHECK(off(L.status) == 0 && off(L.work) + arrs[2].bytes == L.clear_bytes && L.clear_bytes <= off(L.sources), "%s: cleared run", what);
    CHECK(off(L.item_status) + arrs[1].bytes == L.status_bytes && L.status_bytes <= off(L.work), "%s: status run", what);
    CHECK(L.upload_begin == off(L.args) && L.upload_end == off(L.nodes) + arrs[7].bytes, "%s: upload run", what);
    CHECK(L.host_bytes == L.upload_end && L.host_bytes <= off(L.lut), "%s: host mirror", what);
    // the head gather sizes the block without tiles, tries or chunks: its arrays must sit where the full layout has them
    const BatchLayout H = batch_layout(kBase, items, args_bytes, 0, 0, 0);
    CHECK(H.sources == L.sources && H.heads == L.heads && H.args == L.args && H.status == L.status && H.work == L.work,
          "%s: head layout differs", what);
    // a group's tables: at most kBatchGroupItems x 48 KB and change
    CHECK(items > kBatchGroupItems || L.bytes - (tiles + 1) * 8 - chunks * 8 - node_words * 4 - tiles * 8 <=
          (size_t)items * (49152 + 4096 + 512 + 16 + args_bytes) + 64 * kScratchAlign, "%s: %zu bytes", what, L.bytes);
}

static void batch_decode_layouts() {
    const uint32_t item_counts[] = {1, 2, 3, 255, 256, kBatchGroupItems - 1, kBatchGroupItems};
    for (uint32_t items : item_counts)
        for (size_t args_bytes : {(size_t)8, (size_t)296, (size_t)304})
            for (uint64_t chunks : std::vector<uint64_t>{0, 1, 255, 256, 257, 1ull << 20, kBatchGroupBytes / 32 + 2ull * kBatchGroupItems}) {
                const uint64_t tiles = (chunks + 255) / 256 + (chunks ? items : 0);
                for (uint64_t nodes : std::vector<uint64_t>{0, items, items * 255ull, items * (uint64_t)kMaxTrieNodes})
                    check_batch(items, args_bytes, tiles, nodes, chunks);
            }
}

// ---- the batched encoder's group scratch
static void check_enc_batch(uint32_t items, uint64_t hist, uint32_t packed, size_t args_bytes, uint64_t header_bytes, uint64_t tiles,
                  uint64_t regions) {
    char what[200];
    snprintf(what, sizeof what, "items=%u hist=%llu packed=%u args=%zu headers=%llu tiles=%llu regions=%llu", items,
             (unsigned long long)hist, packed, args_bytes, (unsigned long long)header_bytes, (unsigned long long)tiles,
             (unsigned long long)regions);
    ++layouts;
    const EncBatchLayout L = enc_batch_layout(kBase, items, hist, packed, args_bytes, header_bytes, tiles, regions);
    const EncBatchLayout S = enc_batch_layout(nullptr, items, hist, packed, args_bytes, header_bytes, tiles, regions);
    CHECK(S.bytes == L.bytes && S.host_bytes == L.host_bytes && S.counts == nullptr, "%s: sizing differs from carving", what);
    const std::vector<Arr> arrs = {
        {"counts", L.counts, (size_t)items * 256 * 8},
        {"hist_tiles", L.hist_tiles, hist * sizeof(EncHistTile)},
        {"args", L.args, (size_t)packed * args_bytes},
        {"tables", L.tables, (size_t)packed * 2048},
        {"headers", L.headers, header_bytes},
        {"tiles", L.tiles, tiles * sizeof(BatchTile)},
        {"run_bits", L.run_bits, regions * 64},
        {"region_bits", L.region_bits, regions * 4},
        {"group_prefix", L.group_prefix, (regions + kEncPrefixGroup - 1) / kEncPrefixGroup * 8},
        {"region_end", L.region_end, regions * 8},
        {"seam_head", L.seam_head, regions},
        {"seam_tail", L.seam_tail, regions},
    };
    for (const Arr &a : arrs) {
        CHECK(a.p != nullptr, "%s: %s missing", what, a.name);
        if (!a.p) return;
        CHECK(off(a.p) % kScratchAlign == 0, "%s: %s at %zu is not aligned", what, a.name, off(a.p));
        CHECK(off(a.p) + a.bytes <= L.bytes, "%s: %s ends past the block", what, a.name);
    }
    for (size_t i = 0; i < arrs.size(); ++i)
        for (size_t j = i + 1; j < arrs.size(); ++j) {
            const size_t a = off(arrs[i].p), b = off(arrs[j].p);
            CHECK(!(a < b + arrs[j].bytes && b < a + arrs[i].bytes), "%s: %s and %s overlap", what, arrs[i].name, arrs[j].name);
        }
    // the runs: cleared and read back [0, counts_bytes) = counts; uploaded [hist_begin, hist_end) = hist_tiles and
    // [upload_begin, upload_end) = args .. tiles; the pinned mirror [0, host_bytes) = everything up to tiles
    CHECK(off(L.counts) == 0 && L.counts_bytes == arrs[0].bytes && L.counts_bytes <= off(L.hist_tiles), "%s: counts run", what);
    CHECK(L.hist_begin == off(L.hist_tiles) && L.hist_end == L.hist_begin + arrs[1].bytes && L.hist_end <= off(L.args), "%s: histogram run", what);
    CHECK(L.upload_begin == off(L.args) && L.upload_end == off(L.tiles) + arrs[5].bytes, "%s: upload run", what);
    CHECK(L.host_bytes == L.upload_end && L.host_bytes <= off(L.run_bits), "%s: host mirror", what);
    // the histogram sizes the block before anything is packed: its arrays must sit where the full layout has them
    const EncBatchLayout H = enc_batch_layout(kBase, items, hist, 0, args_bytes, 0, 0, 0);
    CHECK(H.counts == L.counts && H.hist_tiles == L.hist_tiles && H.args == L.args && H.hist_end == L.hist_end,
          "%s: histogram layout differs", what);
}

static void batch_encode_layouts() {
    const uint32_t item_counts[] = {1, 2, 3, 255, 256, kBatchGroupItems - 1, kBatchGroupItems};
    const uint64_t group_regions = kBatchGroupBytes / 2048;
    for (uint32_t items : item_counts)
        for (size_t args_bytes : {(size_t)8, (size_t)168, (size_t)176})
            for (uint64_t regions : std::vector<uint64_t>{0, 1, 15, 16, 17, 1023, 1024, 1025, group_regions + 2ull * kBatchGroupItems}) {
                const uint64_t hist = regions ? regions / 8 + items : 0;
                for (uint32_t packed : {0u, 1u, items}) {
                    if (packed > regions || (regions && !packed)) continue;
                    const uint64_t tiles = (regions + kEncTileRegions - 1) / kEncTileRegions + packed;
                    for (uint64_t header_bytes : std::vector<uint64_t>{0, 9, packed * 300ull + 1, packed * 4096ull})
                        check_enc_batch(items, hist, packed, args_bytes, header_bytes, tiles, regions);
                }
            }
}

// argv[1]: the layouts to check - scratch (the decoder's and the pack's), batch_decode (batch_layout) or batch_encode
// (enc_batch_layout)
int main(int argc, char **argv) {
    const std::string which = argc > 1 ? argv[1] : "";
    if (which == "scratch")
        scratch_layouts();
    else if (which == "batch_decode")
        batch_decode_layouts();
    else if (which == "batch_encode")
        batch_encode_layouts();
    else
        return 2;
    printf("%ld layouts, %d failures\n", layouts, failures);
    return failures ? 1 : 0;
}
"""


@pytest.fixture(scope="module")
def layout_driver(tmp_path_factory):
    cxx = shutil.which("g++")
    assert cxx, "g++ is needed to compile the layout driver"
    d = tmp_path_factory.mktemp("scratch_layout")
    src, exe = d / "driver.cpp", d / "driver"
    src.write_text(DRIVER)
    r = subprocess.run([cxx, "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I", CSRC, "-o", str(exe), str(src)],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    return str(exe)


def _check_layouts(layout_driver, which):
    r = subprocess.run([layout_driver, which], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert " 0 failures" in r.stdout and not r.stdout.startswith("0 layouts"), r.stdout


def test_scratch_layouts_hold_every_array(layout_driver):
    _check_layouts(layout_driver, "scratch")


def test_batch_layout_holds_every_array(layout_driver):
    _check_layouts(layout_driver, "batch_decode")


def test_batch_encode_layout_holds_every_array(layout_driver):
    _check_layouts(layout_driver, "batch_encode")


def test_library_exports_the_batch_entry_point():
    L = ctypes.CDLL(_abi.LIB_PATH)
    assert hasattr(L, "et_decode_batch_dev")
    assert "et_decode_batch_dev" in _abi.SYMBOLS
