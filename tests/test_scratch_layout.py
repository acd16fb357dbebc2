"""Device scratch layouts (entreepy_b200/csrc/et_scratch.h), checked on the CPU: every array of the decoder's and the
pack's scratch lies inside the block, meets its alignment, overlaps no other array and holds the elements the kernels
index; the block is no larger than the sizing formulas the layouts replaced, plus alignment padding."""
import os
import shutil
import subprocess

import pytest

from conftest import ROOT

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

#define CHECK(cond, ...)                                   \
    do {                                                   \
        if (!(cond) && ++failures <= 20) {                 \
            fprintf(stderr, __VA_ARGS__);                  \
            fprintf(stderr, "  [%s]\n", #cond);            \
        }                                                  \
    } while (0)

// pairs of arrays that may share bytes (a path that uses one never uses the other)
static bool exempt(const std::vector<std::pair<std::string, std::string>> &ok, const char *a, const char *b) {
    for (auto &e : ok)
        if ((e.first == a && e.second == b) || (e.first == b && e.second == a)) return true;
    return false;
}

static void check(const char *what, std::vector<Arr> arrs, size_t bytes, size_t limit,
                  const std::vector<std::pair<std::string, std::string>> &ok = {}) {
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
            CHECK(!overlap || exempt(ok, arrs[i].name, arrs[j].name), "%s: %s and %s overlap", what, arrs[i].name, arrs[j].name);
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
           {"run_bits", L.run_bits, slots * 64, 16},
           {"tile_desc", L.tile_desc, slots * 8, 16}},
          L.bytes, old_pack_bytes(num_tiles), {{"tile_desc", "run_bits"}});
}

int main() {
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
    printf("%ld layouts, %d failures\n", layouts, failures);
    return failures ? 1 : 0;
}
"""


# ET_WRITE_CHAINS=4 (four parts per chunk in the lane write walk) doubles the lane decoder's `mid` records.
@pytest.fixture(scope="module", params=[[], ["-DET_WRITE_CHAINS=4"]], ids=["chains2", "chains4"])
def layout_driver(request, tmp_path_factory):
    cxx = shutil.which("g++")
    assert cxx, "g++ is needed to compile the layout driver"
    d = tmp_path_factory.mktemp("scratch_layout")
    src, exe = d / "driver.cpp", d / "driver"
    src.write_text(DRIVER)
    r = subprocess.run([cxx, "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", *request.param, "-I", CSRC, "-o", str(exe), str(src)],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    return str(exe)


def test_scratch_layouts_hold_every_array(layout_driver):
    r = subprocess.run([layout_driver], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert " 0 failures" in r.stdout and not r.stdout.startswith("0 layouts"), r.stdout
