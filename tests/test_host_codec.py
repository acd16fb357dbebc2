"""Host half of the product (tree/codes/header/dictionary) and the C-ABI surface — no GPU needed."""
import ctypes
import os
import re

import numpy as np
import pytest

import entreepy_b200 as et
from conftest import FIXTURES, ROOT, make_cases
from entreepy_b200 import _abi
from oracle import oracle


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "entreepy_b200.h")).read()
    declared = set(re.findall(r"ET_API[^;(]*?\b(et_[a-z0-9_]+)\(", header))
    assert declared == set(_abi.SYMBOLS)
    L = ctypes.CDLL(_abi.LIB_PATH)
    for name in declared:
        assert hasattr(L, name), name
    assert _abi.load().et_abi_version() == 1


def _same_codes(cb, occ):
    data, length = oracle.build_dictionary(occ)
    return all(cb.code[s].length == length[s] and cb.code[s].data == data[s] for s in range(256))


def test_codebook_matches_oracle_on_fixtures(fixtures, manifest):
    for name in FIXTURES:
        occ = oracle.histogram(fixtures[name])
        cb = et.build_codebook(occ)
        assert _same_codes(cb, occ)
        assert (cb.min_length, cb.max_length) == (manifest[name]["min_len"], manifest[name]["max_len"])
        assert cb.body_bits == manifest[name]["body_bits"]


def test_codebook_tie_breaking_random_histograms():
    rng = np.random.default_rng(11)
    for trial in range(300):
        k = int(rng.integers(1, 257))
        occ = np.zeros(256, dtype=np.uint64)
        syms = rng.choice(256, k, replace=False)
        hi = int(rng.choice([2, 3, 8, 100, 10**6, 2**40]))  # small ranges force many ties
        occ[syms] = rng.integers(1, hi + 1, k).astype(np.uint64)
        assert _same_codes(et.build_codebook(occ), occ), trial


def test_codebook_deep_tree_truncates_like_the_reference():
    fib = [1, 1]
    while len(fib) < 40:
        fib.append(fib[-1] + fib[-2])
    occ = np.zeros(256, dtype=np.uint64)
    occ[10 : 10 + len(fib)] = fib
    cb = et.build_codebook(occ)
    assert cb.max_length == 39 and _same_codes(cb, occ)


def test_empty_histogram_is_queue_empty():
    with pytest.raises(et.EntreepyError) as e:
        et.build_codebook(np.zeros(256, dtype=np.uint64))
    assert e.value.name == "QueueEmpty"


def test_header_bytes_match_golden(fixtures, golden_et, manifest):
    for name in FIXTURES:
        cb = et.build_codebook(oracle.histogram(fixtures[name]))
        hdr = et.write_header(cb, len(fixtures[name]))
        assert len(hdr) == manifest[name]["et_header_bytes"]
        assert golden_et[name].startswith(hdr)


def test_header_matches_oracle_on_cases():
    for name, data in make_cases().items():
        cb = et.build_codebook(oracle.histogram(data))
        hdr = et.write_header(cb, data.size)
        full = oracle.encode(data, cap=9000 + 5 * data.size).tobytes()
        assert full.startswith(hdr), name
        assert len(full) == len(hdr) + (cb.body_bits + 7) // 8, name


def test_header_matches_oracle_for_codes_over_32_bits():
    # exact Fibonacci counts at the chain's minimum size: the longest code has `depth` bits, and the header writes its
    # bits as the reference does past 32 (encode.zig:311 shifts by a u5: emitted_bit); the text order does not matter
    from entreepy_b200 import synth

    for depth, n in ((33, 14_930_351), (34, 24_157_816), (36, 63_245_985)):
        counts = np.array(synth.fibonacci_counts(n, depth), dtype=np.uint64)
        assert int(counts.sum()) == n and int(oracle.build_dictionary(counts)[1].max()) == depth
        cb = et.build_codebook(counts)
        assert cb.max_length == depth
        hdr = et.write_header(cb, n)
        full = oracle.encode(np.repeat(np.arange(256, dtype=np.uint8), counts.astype(np.int64))).tobytes()
        assert full.startswith(hdr), depth
        assert len(full) == len(hdr) + (cb.body_bits + 7) // 8, depth


def test_body_length_field_wraps_at_32_bits():
    cb = et.build_codebook(oracle.histogram(b"ab"))
    assert et.write_header(cb, 2**32 + 5)[5:9] == (5).to_bytes(4, "big")  # encode.zig:279


def test_parse_header_round_trips_the_dictionary(golden_et, fixtures):
    for name in FIXTURES:
        d = et.parse_header(golden_et[name][4:])
        cb = et.build_codebook(oracle.histogram(fixtures[name]))
        assert d.n_entries == cb.n_entries and d.body_len == len(fixtures[name])
        for e in range(d.n_entries):
            c = cb.code[d.symbol[e]]
            assert (d.length[e], d.code[e]) == (c.length, c.data)
        assert [d.symbol[e] for e in range(d.n_entries)] == sorted(d.symbol[e] for e in range(d.n_entries))


def test_parse_header_on_truncated_streams_follows_the_reference(golden_et):
    et_file = golden_et["nice.shakespeare.txt"][4:]
    for cut in (0, 3):  # decode.zig:36-42 reads compressed_text[1..4]: out of bounds
        with pytest.raises(et.EntreepyError):
            et.parse_header(et_file[:cut])
    whole = et.parse_header(et_file)
    assert not whole.truncated
    # the dictionary state machine stops when the bytes run out (decode.zig:66): what was read stands, the body is empty
    for cut in (5, 20, 60):
        d = et.parse_header(et_file[:cut])
        assert d.truncated and d.n_entries < whole.n_entries and d.body_offset == cut and d.body_len == whole.body_len
        for e in range(d.n_entries):
            assert (d.symbol[e], d.length[e], d.code[e]) == (whole.symbol[e], whole.length[e], whole.code[e])


def test_single_symbol_file_parses_to_an_empty_dictionary():
    enc = oracle.encode(np.full(1000, 7, dtype=np.uint8)).tobytes()
    assert len(enc) == 9  # encode.zig:270-275: zero entries
    d = et.parse_header(enc[4:])
    assert d.n_entries == 0 and d.truncated and d.body_len == 1000 and d.body_offset == 5


def test_no_cpu_fallback_without_a_device():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present; the failure path is for CPU-only hosts")
    with pytest.raises(et.EntreepyError) as e:
        et.Codec(0)
    assert e.value.name == "NoDevice"
    with pytest.raises(et.EntreepyError):
        et.encode(b"hello")  # the drop-in entry point must not quietly compute on the CPU


def test_product_does_not_import_the_oracle():
    pkg = os.path.join(ROOT, "entreepy_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cpp", ".h", ".cuh")):
                text = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "liboracle" not in text and "import oracle" not in text and "from oracle" not in text, f


def test_synth_generator_is_deterministic(manifest):
    from entreepy_b200 import synth

    thr = synth.thresholds_from_weights(synth.text_weights(manifest["midsummer_histogram"]))
    a = synth.generate(100000, thr)
    b = np.concatenate([synth.generate(40000, thr), synth.generate(60000, thr, first_index=40000)])
    assert np.array_equal(a, b)
    assert set(np.unique(a)) <= {s for s, c in enumerate(manifest["midsummer_histogram"]) if c}
    assert synth.splitmix64(np.uint64(0)) == np.uint64(0xE220A8397B1DCDAF)  # published splitmix64 vector


def test_fibonacci_counts_give_the_deepest_faithful_tree():
    # SURVEY §0.4: exact Fibonacci counts scaled to 256 MiB make a chain of depth 32 — the deepest codes the
    # reference represents faithfully; the host codebook and the oracle agree on every code of it
    from entreepy_b200 import synth

    counts = np.array(synth.fibonacci_counts(1 << 28, 32), dtype=np.uint64)
    assert int(counts.sum()) == 1 << 28 and int((counts > 0).sum()) == 33
    o_code, o_len = oracle.build_dictionary(counts)
    assert int(o_len.max()) == 32 and sorted(int(x) for x in o_len[o_len > 0]) == [1] + list(range(2, 33)) + [32]
    cb = et.build_codebook(counts)
    assert [cb.code[s].length for s in range(256)] == [int(x) for x in o_len]
    assert [cb.code[s].data for s in range(256)] == [int(x) for x in o_code]
    # i.i.d. sampling from the same weights does not reach that depth (why the bench uses exact counts)
    sample = synth.generate(1 << 20, synth.thresholds_from_weights(synth.fibonacci_weights(32)))
    assert int(oracle.build_dictionary(oracle.histogram(sample))[1].max()) < 32
