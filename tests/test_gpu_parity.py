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


def test_encode_wide_codes_fibonacci_depth_32_and_beyond(codec):
    # depth 32 = deepest the reference represents faithfully (SURVEY §0.4); depth 34 exercises the
    # truncated-code emission (encode.zig:311 shift is u5) which must still match bit for bit
    rng = np.random.default_rng(9)
    for depth in (27, 32, 34):
        w = synth.fibonacci_weights(depth)
        n = 1 << 22
        data = synth.generate(n, synth.thresholds_from_weights(w), seed=depth)
        # make sure every symbol occurs, rarest ones at least once, so the tree has full depth
        data[: depth + 1] = np.arange(depth + 1, dtype=np.uint8)
        occ = oracle.histogram(data)
        _, length = oracle.build_dictionary(occ)
        n_out, out = codec.encode(data, _flags())
        assert out.tobytes() == _oracle_et(data), (depth, int(length.max()))


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
