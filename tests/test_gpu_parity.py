"""Parity of the CUDA path (through the C ABI) with the CPU oracle.  Run with -m gpu on a B200.

Bar: bit-exact.  Encode: .et bytes identical to the oracle's for the same input.  Decode: the
original bytes (north_star), identical to the oracle's decode of the same stream.
"""
import hashlib

import numpy as np
import pytest

import entreepy_b200 as et
from conftest import FIXTURES, make_cases
from entreepy_b200 import _abi, synth
from oracle import oracle

pytestmark = pytest.mark.gpu


def _oracle_et(data):
    return oracle.encode(data, cap=9000 + 5 * int(np.asarray(data).size)).tobytes()


def _flags(**kw):
    return et.EncodeFlags(write_output=True, no_scratch_limit=True, **kw)


# ---------------------------------------------------------------- K1
def test_histogram_matches_oracle(codec, fixtures):
    for name in FIXTURES:
        assert np.array_equal(codec.histogram(fixtures[name]), oracle.histogram(fixtures[name])), name
    for name, data in make_cases().items():
        assert np.array_equal(codec.histogram(data), oracle.histogram(data)), name


def test_histogram_unaligned_device_pointers(codec):
    import torch

    rng = np.random.default_rng(5)
    host = rng.integers(0, 256, 1 << 20, dtype=np.uint8)
    dev = torch.from_numpy(host).cuda()
    for off, n in [(0, 1 << 20), (1, 1000), (3, 65536 + 7), (15, 17), (16, 16), (7, 1), (9, 0), (5, (1 << 20) - 5)]:
        got = codec.histogram_dev(dev.data_ptr() + off, n)
        assert np.array_equal(got, oracle.histogram(host[off : off + n])), (off, n)


# ---------------------------------------------------------------- encode
def test_encode_golden_files(codec, fixtures, golden_et, manifest):
    for name in FIXTURES:
        n, out = codec.encode(fixtures[name])
        assert n == manifest[name]["et_bytes"]
        assert hashlib.sha256(out.tobytes()).hexdigest() == manifest[name]["et_sha256"]
        assert out.tobytes() == golden_et[name]


def test_encode_matches_oracle_on_cases(codec, manifest):
    thr = synth.thresholds_from_weights(synth.text_weights(manifest["midsummer_histogram"]))
    cases = dict(make_cases())
    cases["text_3M"] = synth.generate((3 << 20) + 77, thr)  # 1537 regions of the lane-run pack, the last one ragged
    for name, data in cases.items():
        n, out = codec.encode(data, _flags())
        assert out.tobytes() == _oracle_et(data), name


def test_encode_dry_run_returns_size_only(codec, fixtures, manifest):
    n, out = codec.encode(fixtures["nice.shakespeare.txt"], et.EncodeFlags(write_output=False))
    assert n == 374 and out is None  # encode.zig:319,336; README.md:51


def test_encode_empty_input_is_queue_empty(codec):
    with pytest.raises(et.EntreepyError) as e:
        codec.encode(b"")
    assert e.value.name == "QueueEmpty"


def test_encode_respects_capacity_and_reference_scratch(codec):
    rng = np.random.default_rng(2)
    data = rng.integers(0, 256, 50000, dtype=np.uint8)
    with pytest.raises(et.EntreepyError) as e:
        codec.encode(data, et.EncodeFlags(write_output=True), cap=1000)
    assert e.value.name == "NoSpaceLeft"


def test_encode_text_sizes_and_alignments(codec, manifest):
    import torch

    thr = synth.thresholds_from_weights(synth.text_weights(manifest["midsummer_histogram"]))
    host = synth.generate((1 << 21) + 77, thr)
    dev = torch.from_numpy(host).cuda()
    out = torch.empty(host.size + 16384, dtype=torch.uint8, device="cuda")
    for off, n, out_off in [(0, host.size, 0), (1, 100000, 3), (13, 4096 * 3 - 13, 1), (16, 4096, 15), (5, 4090, 7),
                            (0, 1 << 20, 9)]:
        got = codec.encode_dev(dev.data_ptr() + off, n, out.data_ptr() + out_off, out.numel() - out_off,
                               _abi.FLAG_WRITE_OUTPUT | _abi.FLAG_NO_SCRATCH_LIMIT)
        want = _oracle_et(host[off : off + n])
        assert got == len(want), (off, n)
        assert out[out_off : out_off + got].cpu().numpy().tobytes() == want, (off, n, out_off)


def _chain_bytes(depth):
    """Smallest text whose exact Fibonacci counts (synth.fibonacci_counts) make a chain of `depth`: one copy of each of
    the two rarest symbols."""
    f = [1, 1]
    while len(f) < depth + 1:
        f.append(f[-1] + f[-2])
    return sum(f)


def _encode_dev_counted(codec, d_in, n, d_out, cap):
    """encode_dev -> (size, kernel launches it took)."""
    before = codec.kernel_launches
    size = codec.encode_dev(d_in, n, d_out, cap, _abi.FLAG_WRITE_OUTPUT | _abi.FLAG_NO_SCRATCH_LIMIT)
    return size, codec.kernel_launches - before


def _first_difference(got, want):
    """None when the byte strings are equal, else (first differing index, len(got), len(want))."""
    a, b = np.frombuffer(got, np.uint8), np.frombuffer(want, np.uint8)
    if a.size == b.size and np.array_equal(a, b):
        return None
    m = min(a.size, b.size)
    diff = np.flatnonzero(a[:m] != b[:m])
    return (int(diff[0]) if diff.size else m, a.size, b.size)


def _expected_size(counts, n):
    cb = et.build_codebook(np.asarray(counts, dtype=np.uint64))
    return len(et.write_header(cb, n)) + (cb.body_bits + 7) // 8


def test_encode_wide_codes_fibonacci_depth_32_and_beyond(codec):
    # Exact Fibonacci counts make a chain whose longest code has `depth` bits (i.i.d. sampling from the same weights stops
    # near 20 bits).  Depth 32 is the deepest code the narrow pack takes and the reference represents faithfully
    # (SURVEY §0.4).  Past it pack_wide_kernel emits the reference's truncated codes (encode.zig:311 shifts by a u5),
    # which must still match bit for bit.  Depth 38 is 166 MB: about 40 K tiles of look-back.
    import torch

    for depth in (32, 33, 34, 36, 38):
        n = _chain_bytes(depth)
        counts = synth.fibonacci_counts(n, depth)
        assert int(oracle.build_dictionary(np.array(counts, dtype=np.uint64))[1].max()) == depth
        dev = synth.shuffled_dev(counts, seed=depth)
        size_want = _expected_size(counts, n)
        out = torch.empty(size_want + 64, dtype=torch.uint8, device="cuda")
        size, launches = _encode_dev_counted(codec, dev.data_ptr(), n, out.data_ptr(), out.numel())
        # from launch_pack: histogram, pack_wide_kernel, seam_fixup_kernel | histogram, four narrow pack kernels, seam fix-up
        assert launches == (3 if depth > 32 else 6), (depth, launches)
        want = _oracle_et(dev.cpu().numpy())
        assert size == size_want == len(want), (depth, size, size_want, len(want))
        assert _first_difference(out[:size].cpu().numpy().tobytes(), want) is None, depth


def test_encode_wide_codes_sizes_and_alignments(codec):
    # Depth 33 on the wide path: the input at every 16-byte phase, last tiles of 1, 15, 16, 4095 and 4096 symbols, odd
    # output offsets, guard bytes on both sides (zero, or stale bytes that must stay); then the host-buffer entry point,
    # and the decoder, which refuses codes over 32 bits without writing anything.
    import torch

    n0 = _chain_bytes(33)
    rng = np.random.default_rng(33)
    core = np.repeat(np.arange(256, dtype=np.uint8), np.array(synth.fibonacci_counts(n0, 33), dtype=np.int64))
    rng.shuffle(core)
    # the pads only add copies of the two most frequent symbols (1- and 2-bit codes): a slice that holds the core keeps the chain
    pad = 8192 + 32
    top2 = np.array([32, 33], dtype=np.uint8)
    host = np.concatenate([rng.choice(top2, pad), core, rng.choice(top2, pad)])
    dev = torch.from_numpy(host).cuda()
    assert dev.data_ptr() % 16 == 0
    lasts, out_offs = (1, 15, 16, 4095, 4096), (0, 1, 3, 7, 9, 15, 16, 33)
    for off in range(16):
        last = lasts[off % len(lasts)]
        n = pad + n0 + (last - off - (pad + n0)) % 4096  # the tiles cover bytes [0, off + n) of dev: the last holds `last`
        assert (off + n - 1) % 4096 + 1 == last and off + n <= host.size
        data = host[off : off + n]
        occ = oracle.histogram(data)
        assert int(oracle.build_dictionary(occ)[1].max()) == 33, off
        want = _oracle_et(data)
        assert len(want) == _expected_size(occ, n)
        out_off, fill = out_offs[off % len(out_offs)], 0xA5 if off % 2 else 0
        out = torch.full((out_off + len(want) + 64,), fill, dtype=torch.uint8, device="cuda")
        size, launches = _encode_dev_counted(codec, dev.data_ptr() + off, n, out.data_ptr() + out_off, out.numel() - out_off)
        assert size == len(want) and launches == 3, (off, n, size, launches)
        got = out.cpu().numpy()
        assert (got[:out_off] == fill).all() and (got[out_off + size :] == fill).all(), (off, n, out_off)
        assert _first_difference(got[out_off : out_off + size].tobytes(), want) is None, (off, n, out_off)
    # et_encode: host buffers, the input uploaded in slices
    data = host[5 : 5 + pad + n0 + 4095]
    assert int(oracle.build_dictionary(oracle.histogram(data))[1].max()) == 33
    n_out, enc = codec.encode(data, _flags())
    assert _first_difference(enc.tobytes(), _oracle_et(data)) is None
    # et_decode_dev: the dictionary holds codes of 33 bits, which the reference's decoder cannot hold
    src = torch.from_numpy(enc.copy()).cuda()
    out = torch.full((data.size + 64,), 0xA5, dtype=torch.uint8, device="cuda")
    with pytest.raises(et.EntreepyError) as e:
        codec.decode_dev(src.data_ptr() + 4, n_out - 4, out.data_ptr(), data.size)
    assert e.value.name == "Unsupported"
    assert bool((out == 0xA5).all())


def test_encode_wide_codes_dropped_symbol_zero_bit_tiles(codec):
    # All 256 byte values: the most frequent one (symbol 33 of a depth-33 chain) gets no code (encode.zig:70).  A run of
    # it longer than three tiles, starting inside an output byte, gives whole tiles of zero bits that begin and end in
    # the same byte: seam_fixup_kernel merges the heads of a chain of tiles from the wide kernel's tile states.
    import torch

    counts = synth.fibonacci_counts(_chain_bytes(33), 33)[:34] + [200_000] * 222
    assert sum(counts) == 59_330_351
    base = synth.shuffled_dev(counts, seed=34).cpu().numpy()
    _, length = oracle.build_dictionary(np.array(counts, dtype=np.uint64))
    assert int(length.max()) == 33 and length[33] == 0
    run, at = 20_000, 30_000_001
    bit = int(length[base[:at]].sum(dtype=np.int64))
    while at % 2 == 0 or bit % 8 == 0:  # an odd offset, and the run begins inside a byte of the body
        bit += int(length[base[at]])
        at += 1
    host = np.concatenate([base[:at], np.full(run, 33, np.uint8), base[at:]])
    occ = oracle.histogram(host)
    _, length = oracle.build_dictionary(occ)
    assert int((occ > 0).sum()) == 256 and int(length.max()) == 33 and length[33] == 0
    in_off = 3
    assert (in_off + at + run) // 4096 - (in_off + at + 4095) // 4096 >= 3  # whole tiles inside the run
    buf = torch.zeros(host.size + 16, dtype=torch.uint8, device="cuda")
    buf[in_off : in_off + host.size] = torch.from_numpy(host).cuda()
    want = _oracle_et(host)
    assert len(want) == _expected_size(occ, host.size)
    out = torch.full((len(want) + 64,), 0xA5, dtype=torch.uint8, device="cuda")
    size, launches = _encode_dev_counted(codec, buf.data_ptr() + in_off, host.size, out.data_ptr() + 1, out.numel() - 1)
    assert size == len(want) and launches == 3, (size, launches)
    got = out.cpu().numpy()
    assert got[0] == 0xA5 and (got[1 + size :] == 0xA5).all()
    assert _first_difference(got[1 : 1 + size].tobytes(), want) is None


# ---------------------------------------------------------------- decode
def test_decode_golden_files(codec, fixtures, golden_et):
    for name in FIXTURES:
        n, out = codec.decode(golden_et[name][4:])  # file[4..] as main.zig:204
        assert n == len(fixtures[name]) and out.tobytes() == fixtures[name], name


def test_round_trip_like_the_reference_tests(codec, fixtures):
    # test.zig:7-33: encode into a buffer, decode encoded[4..len], compare strings
    for name in FIXTURES:
        n, enc = codec.encode(fixtures[name])
        m, dec = codec.decode(enc[4:n])
        assert dec.tobytes() == fixtures[name]


def test_decode_matches_oracle_on_cases(codec):
    for name, data in make_cases().items():
        stream = _oracle_et(data)[4:]
        if name in ("one_byte", "single_symbol_run"):
            # zero dictionary entries: the reference reads back 0 bytes without an error (decode.zig:66, empty body)
            n, out = codec.decode(stream)
            assert n == 0 and out.size == 0, name
            continue
        want = oracle.decode(stream, data.size).tobytes()
        n, out = codec.decode(stream)
        assert out.tobytes() == want, name
        if name not in ("all_256_once", "all_256_uniform", "dropped_symbol_dominates"):
            assert want == data.tobytes(), name  # lossless wherever the reference encoder is


def test_decode_dry_run_writes_nothing(codec, golden_et):
    n, out = codec.decode(golden_et["test.txt"][4:], et.DecodeFlags(write_output=False))
    assert n == 0 and out is None  # decode.zig:185-188,219


def test_decode_rejects_garbage(codec):
    with pytest.raises(et.EntreepyError):
        codec.decode(b"\x01\x00\x00")  # the reference indexes compressed_text[1..4] out of bounds (decode.zig:36-42)
    # second entry truncated: the reference's dictionary state machine runs out of bytes (decode.zig:66), the body is
    # empty and nothing is decoded - no error.  ET_FLAG_VALIDATE (reference TODO, main.zig:199) makes it one.
    cut = bytes([1, 0, 0, 0, 9, 65, 1, 0b10100001, 0b00000000])  # a = "1", then b with length 1 and no code bit
    n, out = codec.decode(cut)
    assert n == 0 and out.size == 0
    with pytest.raises(et.EntreepyError) as e:
        codec.decode(cut, et.DecodeFlags(write_output=True, validate=True))
    assert e.value.name == "Corrupt"


def test_single_symbol_round_trip_is_the_reference_s(codec):
    # one distinct symbol: the root is a leaf, the code has length 0, the dictionary is empty (encode.zig:204-212,
    # 270-275) and the file is 9 bytes; the reference decoder reads back 0 bytes without an error (decode.zig:66)
    data = np.full(1000, 97, dtype=np.uint8)
    n, enc = codec.encode(data)
    assert n == 9 and enc.tobytes() == oracle.encode(data).tobytes()
    m, out = codec.decode(enc[4:n])
    assert m == 0 and out.size == 0
    assert codec.decode(enc[4:n], et.DecodeFlags(write_output=True, validate=True))[0] == 0


def _dict_stream(entries, body_len, body):
    """file[4..] for a hand-made dictionary: entries = [(symbol, length, code)]."""
    bits = []
    for sym, length, code in entries:
        bits += [(sym >> (7 - k)) & 1 for k in range(8)] + [(length >> (7 - k)) & 1 for k in range(8)]
        bits += [(code >> (length - 1 - k)) & 1 for k in range(length)]
    bits += [0] * (-len(bits) % 8)
    d = np.packbits(np.array(bits, dtype=np.uint8)).tobytes()
    return bytes([len(entries) - 1]) + int(body_len).to_bytes(4, "big") + d + bytes(body)


def test_validate_flag_and_reference_acceptance(codec):
    strict = et.DecodeFlags(write_output=True, validate=True)
    # a = 0, b = 01 (a is a prefix of b): the reference tries lengths from the shortest up (decode.zig:175-181), so
    # b can never match; body 0 1 0 0 ... decodes as a, then "1" is no code
    stream = _dict_stream([(97, 1, 0b0), (98, 2, 0b01)], 3, [0b00000000])
    n, out = codec.decode(stream)
    assert out.tobytes() == b"aaa"
    with pytest.raises(et.EntreepyError) as e:
        codec.decode(stream, strict)
    assert e.value.name == "Corrupt"
    # a repeated (length, code): the later entry overwrites the earlier one (decode.zig:123-125)
    stream = _dict_stream([(97, 1, 0b0), (98, 1, 0b1), (99, 1, 0b1)], 4, [0b01010000])
    assert codec.decode(stream)[1].tobytes() == b"acac"
    with pytest.raises(et.EntreepyError):
        codec.decode(stream, strict)
    # incomplete code (Kraft sum 3/4): accepted as long as the body only uses what exists; rejected when validated
    stream = _dict_stream([(97, 1, 0b0), (98, 2, 0b10)], 3, [0b01000000])
    assert codec.decode(stream)[1].tobytes() == b"aba"
    with pytest.raises(et.EntreepyError):
        codec.decode(stream, strict)
    # body too short for body_len symbols
    good = oracle.encode(np.frombuffer(b"abracadabra" * 30, dtype=np.uint8)).tobytes()[4:]
    assert codec.decode(good, strict)[1].tobytes() == b"abracadabra" * 30
    with pytest.raises(et.EntreepyError):
        codec.decode(good[:-70], strict)


def test_fixed_length_codes_take_closed_form_entries(codec):
    # 2^k equiprobable symbols: every code has k bits, a wrong parse never re-synchronises (k = 3, 5, 6, 7 do not
    # divide the 128-bit run-up).  The entries follow from the first one in closed form: no repair rounds.
    import torch

    rng = np.random.default_rng(31)
    for k, n in ((7, (64 << 20) + 5), (3, (64 << 20) + 1), (5, 3_000_001), (6, 70001), (1, 100003), (2, 1 << 20)):
        syms = torch.from_numpy(rng.permutation(256)[: 1 << k].astype(np.uint8)).cuda()
        g = torch.Generator(device="cuda")
        g.manual_seed(k)
        text = syms[torch.randint(0, 1 << k, (n,), generator=g, device="cuda")].contiguous()  # near-equal counts: a full tree
        torch.cuda.synchronize()
        enc = torch.empty(n + 8192, dtype=torch.uint8, device="cuda")
        size = codec.encode_dev(text.data_ptr(), n, enc.data_ptr(), enc.numel(), et._abi.FLAG_WRITE_OUTPUT | et._abi.FLAG_NO_SCRATCH_LIMIT)
        d = et.parse_header(enc[4:4 + 2048].cpu().numpy())
        assert d.min_length == d.max_length == k
        dec = torch.zeros(n, dtype=torch.uint8, device="cuda")
        got = codec.decode_dev(enc.data_ptr() + 4, size - 4, dec.data_ptr(), n)
        assert got == n and torch.equal(dec, text), k
        assert codec.last_decode_rounds <= 2, (k, codec.last_decode_rounds)


def test_round_trip_text_16m_property(codec, manifest):
    import torch

    thr = synth.thresholds_from_weights(synth.text_weights(manifest["midsummer_histogram"]))
    n = (1 << 24) + 3
    dev = torch.empty(n, dtype=torch.uint8, device="cuda")
    codec.synth_dev(dev.data_ptr(), n, synth.SEED, 0, thr)
    assert np.array_equal(dev[: 1 << 16].cpu().numpy(), synth.generate(1 << 16, thr))  # CPU twin agrees
    enc = torch.empty(n + 8192, dtype=torch.uint8, device="cuda")
    size = codec.encode_dev(dev.data_ptr(), n, enc.data_ptr(), enc.numel())
    host = dev.cpu().numpy()
    want = _oracle_et(host)
    assert size == len(want)
    assert hashlib.sha256(enc[:size].cpu().numpy().tobytes()).hexdigest() == hashlib.sha256(want).hexdigest()
    dec = torch.zeros(n, dtype=torch.uint8, device="cuda")
    got = codec.decode_dev(enc.data_ptr() + 4, size - 4, dec.data_ptr(), n)
    assert got == n and torch.equal(dec, dev)


# ---------------------------------------------------------------- check rounds (streams that do not re-synchronise quickly)
def test_slow_synchronising_streams_need_no_rounds_with_transfer_functions(codec):
    # 255 equiprobable symbols: 7- and 8-bit codes only; a wrong start survives for kilobytes, so guessed chunk entries are
    # wrong (SURVEY §0.2, config 4b).  The decoder tabulates every chunk's transfer function (exit and symbols for each
    # of the <= max_len possible entries) and scans them: no repair rounds.  The rounds (round 1's way, still the fallback
    # when the final check fails) stay selectable and must agree.
    rng = np.random.default_rng(3)
    for n in (70000, (1 << 22) + 11, (1 << 25) + 3):
        data = rng.integers(1, 256, n, dtype=np.uint8)
        stream = _oracle_et(data)[4:]
        m, out = codec.decode(stream)
        assert m == n and out.tobytes() == data.tobytes()
        assert codec.last_decode_rounds <= 2
        if n < (1 << 25):
            codec.set_tuning(_abi.TUNE_NO_TRANSFER, 1)
            try:
                m, out = codec.decode(stream)
                assert m == n and out.tobytes() == data.tobytes()
                assert codec.last_decode_rounds > 2
            finally:
                codec.set_tuning(_abi.TUNE_NO_TRANSFER, 0)
    # lengths 5..7 (spread 2) and a body that does not start on a 16-byte boundary
    data = rng.choice(np.arange(40, dtype=np.uint8), 3_000_017, p=np.r_[np.full(24, 2.0), np.full(16, 1.0)] / 64.0)
    stream = _oracle_et(data)[4:]
    d = et.parse_header(stream)
    assert d.max_length - d.min_length <= 2
    m, out = codec.decode(stream)
    assert m == data.size and out.tobytes() == data.tobytes() and codec.last_decode_rounds <= 2
    # text re-synchronises within a few symbols: the first check round finds nothing to repair
    text = rng.choice(np.frombuffer(b"etaoin shrdlu\n,.", dtype=np.uint8), 1 << 22)
    m, out = codec.decode(_oracle_et(text)[4:])
    assert out.tobytes() == text.tobytes() and codec.last_decode_rounds == 2


def test_decode_every_length_up_to_two_chunks_and_all_alignments(codec):
    # ragged ends: streams shorter than a piece, a chunk, and a few chunks; body at every 16-byte phase
    import torch

    rng = np.random.default_rng(21)
    alphabet = np.frombuffer(b"etaoin shrdlu\n,.", dtype=np.uint8)
    for n in list(range(1, 70)) + [127, 128, 129, 255, 256, 257, 700, 1023, 1025, 5000]:
        data = rng.choice(alphabet, n)
        if np.unique(data).size < 2:
            continue
        stream = _oracle_et(data)[4:]
        m, out = codec.decode(stream)
        assert m == n and out.tobytes() == data.tobytes(), n
    data = rng.choice(alphabet, 100000)
    et_file = _oracle_et(data)
    dev = torch.zeros(len(et_file) + 64, dtype=torch.uint8, device="cuda")
    out = torch.zeros(data.size + 64, dtype=torch.uint8, device="cuda")
    for phase in range(16):
        dev[phase : phase + len(et_file)] = torch.from_numpy(np.frombuffer(et_file, dtype=np.uint8).copy()).cuda()
        got = codec.decode_dev(dev.data_ptr() + phase + 4, len(et_file) - 4, out.data_ptr() + (phase * 7) % 16, data.size)
        o = (phase * 7) % 16
        assert got == data.size and out[o : o + got].cpu().numpy().tobytes() == data.tobytes(), phase


def test_host_decode_pipelined_in_slices(codec, manifest):
    # bodies above 128 MiB are uploaded, decoded and downloaded in overlapping 64 MiB slices (et_decode);
    # every slice must start exactly where the one before it ended
    import torch

    thr = synth.thresholds_from_weights(synth.text_weights(manifest["midsummer_histogram"]))
    n = (3 << 26) * 4 // 3 + 12345  # ~256 MiB of text -> ~150 MiB of body: three slices
    dev = torch.empty(n, dtype=torch.uint8, device="cuda")
    codec.synth_dev(dev.data_ptr(), n, synth.SEED, 0, thr)
    h_in, h_et, h_out = codec.pinned(n), codec.pinned(n + 16384), codec.pinned(n)
    torch.from_numpy(h_in)[:] = dev.cpu()
    size = codec.encode_into(h_in, h_et)
    assert size - 400 > (128 << 20)
    got = codec.decode_into(h_et[4:size], h_out)
    assert got == n and np.array_equal(h_out, h_in)
