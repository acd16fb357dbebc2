"""The batched decoder's scratch layout (batch_layout, entreepy_b200/csrc/et_scratch.h), checked on the CPU: every array
lies inside the block, is aligned and overlaps no other, for item counts up to a whole group and chunk counts up to the
chunks of a group's bytes; the runs the host clears, uploads and reads back hold exactly their arrays; and the layout the
head gather uses places its arrays where the full layout does.  Also: the built library exports the batch entry point."""
import ctypes
import os
import shutil
import subprocess

import pytest

from conftest import ROOT
from entreepy_b200 import _abi

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

static void check(uint32_t items, size_t args_bytes, uint64_t tiles, uint64_t node_words, uint64_t chunks) {
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

int main() {
    const uint32_t item_counts[] = {1, 2, 3, 255, 256, kBatchGroupItems - 1, kBatchGroupItems};
    for (uint32_t items : item_counts)
        for (size_t args_bytes : {(size_t)8, (size_t)296, (size_t)304})
            for (uint64_t chunks : std::vector<uint64_t>{0, 1, 255, 256, 257, 1ull << 20, kBatchGroupBytes / 32 + 2ull * kBatchGroupItems}) {
                const uint64_t tiles = (chunks + 255) / 256 + (chunks ? items : 0);
                for (uint64_t nodes : std::vector<uint64_t>{0, items, items * 255ull, items * (uint64_t)kMaxTrieNodes})
                    check(items, args_bytes, tiles, nodes, chunks);
            }
    printf("%ld layouts, %d failures\n", layouts, failures);
    return failures ? 1 : 0;
}
"""


@pytest.fixture(scope="module")
def layout_driver(tmp_path_factory):
    cxx = shutil.which("g++")
    assert cxx, "g++ is needed to compile the layout driver"
    d = tmp_path_factory.mktemp("batch_layout")
    src, exe = d / "driver.cpp", d / "driver"
    src.write_text(DRIVER)
    r = subprocess.run([cxx, "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I", CSRC, "-o", str(exe), str(src)],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    return str(exe)


def test_batch_layout_holds_every_array(layout_driver):
    r = subprocess.run([layout_driver], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert " 0 failures" in r.stdout and not r.stdout.startswith("0 layouts"), r.stdout


def test_library_exports_the_batch_entry_point():
    L = ctypes.CDLL(_abi.LIB_PATH)
    assert hasattr(L, "et_decode_batch_dev")
    assert "et_decode_batch_dev" in _abi.SYMBOLS
