"""The batched encoder's scratch layout (enc_batch_layout, entreepy_b200/csrc/et_scratch.h), checked on the CPU: every array
lies inside the block, is aligned and overlaps no other, for item counts up to a whole group, region and tile counts up
to those of a group's bytes and header bytes up to a full header per text; the runs the host clears, uploads and reads
back hold exactly their arrays; and the layout the histogram uses places its arrays where the full layout does."""
import os
import shutil
import subprocess

import pytest

from conftest import ROOT

CSRC = os.path.join(ROOT, "entreepy_b200", "csrc")

DRIVER = r"""
#include <cstdio>
#include <vector>

#include "et_scratch.h"

using namespace et;

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

struct Arr {
    const char *name;
    const void *p;
    size_t bytes;
};

static size_t off(const void *p) { return (size_t)(static_cast<const uint8_t *>(p) - kBase); }

static void check(uint32_t items, uint64_t hist, uint32_t packed, size_t args_bytes, uint64_t header_bytes, uint64_t tiles,
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

int main() {
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
                        check(items, hist, packed, args_bytes, header_bytes, tiles, regions);
                }
            }
    printf("%ld layouts, %d failures\n", layouts, failures);
    return failures ? 1 : 0;
}
"""


@pytest.fixture(scope="module")
def layout_driver(tmp_path_factory):
    cxx = shutil.which("g++")
    assert cxx, "g++ is needed to compile the layout driver"
    d = tmp_path_factory.mktemp("batch_encode_layout")
    src, exe = d / "driver.cpp", d / "driver"
    src.write_text(DRIVER)
    r = subprocess.run([cxx, "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I", CSRC, "-o", str(exe), str(src)],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    return str(exe)


def test_batch_encode_layout_holds_every_array(layout_driver):
    r = subprocess.run([layout_driver], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert " 0 failures" in r.stdout and not r.stdout.startswith("0 layouts"), r.stdout
