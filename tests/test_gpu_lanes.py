"""The lane-interleaved decoder (regions of 32 chunks per warp) on inputs of every shape.

Long streams take it by default; et_ctx_set_tuning(ET_TUNE_LANE_MIN_BYTES, 0) sends short ones through it as well, so the
oracle can check it at sizes it finishes in seconds.  Bar: bit-exact (the original text).
"""
import numpy as np
import pytest

import entreepy_b200 as et
from conftest import make_cases
from entreepy_b200 import synth
from oracle import oracle

pytestmark = pytest.mark.gpu
FILL = 0xA5  # what an output holds before a call: a decoder that writes zeros, or skips a zero byte, shows


def _oracle_et(data):
    return oracle.encode(data, cap=9000 + 5 * int(np.asarray(data).size)).tobytes()


@pytest.fixture()
def lanes(codec):
    codec.set_tuning(et._abi.TUNE_LANE_MIN_BYTES, 0)
    yield
    codec.set_tuning(et._abi.TUNE_LANE_MIN_BYTES, -1)


def test_lane_decoder_on_the_oracle_cases(codec, lanes):
    for name, data in make_cases().items():
        if name in ("one_byte", "single_symbol_run"):
            continue
        stream = _oracle_et(data)[4:]
        want = oracle.decode(stream, data.size).tobytes()
        n, out = codec.decode(stream)
        assert out.tobytes() == want, name


def test_lane_decoder_text_sizes(codec, lanes, manifest):
    thr = synth.thresholds_from_weights(synth.text_weights(manifest["midsummer_histogram"]))
    host = synth.generate((3 << 20) + 321, thr)
    # region = 4224 body bytes ~ 7200 symbols: streams of 2..3 regions, ragged ends, a few hundred regions
    for n in (14000, 14500, 15000, 21599, 21600, 21700, 30011, 100003, 1 << 20, host.size):
        data = host[:n]
        m, out = codec.decode(_oracle_et(data)[4:])
        assert m == n and out.tobytes() == data.tobytes(), n
        assert codec.last_decode_rounds == 2


def test_lane_decoder_alignments_and_capacity(codec, lanes, manifest):
    import torch

    thr = synth.thresholds_from_weights(synth.text_weights(manifest["midsummer_histogram"]))
    data = synth.generate(300007, thr, seed=11)
    et_file = _oracle_et(data)
    src = torch.from_numpy(np.frombuffer(et_file, dtype=np.uint8).copy()).cuda()
    dev = torch.zeros(len(et_file) + 64, dtype=torch.uint8, device="cuda")
    out = torch.empty(data.size + 64, dtype=torch.uint8, device="cuda")
    for phase in range(16):
        dev[phase : phase + len(et_file)] = src
        o = (phase * 7) % 16
        out.fill_(FILL)
        torch.cuda.synchronize()  # the library works on its own stream
        got = codec.decode_dev(dev.data_ptr() + phase + 4, len(et_file) - 4, out.data_ptr() + o, data.size)
        assert got == data.size and out[o : o + got].cpu().numpy().tobytes() == data.tobytes(), phase
        assert bool((out[o + got :] == FILL).all()) and bool((out[:o] == FILL).all())  # nothing outside the text
    # output clipped by the caller's capacity: exactly cap bytes are written, NoSpaceLeft reported
    for cap in (1, 4223, 7200, 100000, data.size - 1):
        out.fill_(FILL)
        torch.cuda.synchronize()
        with pytest.raises(et.EntreepyError) as e:
            codec.decode_dev(dev.data_ptr() + 15 + 4, len(et_file) - 4, out.data_ptr(), cap)
        assert e.value.name == "NoSpaceLeft"
        assert out[:cap].cpu().numpy().tobytes() == data[:cap].tobytes() and bool((out[cap:] == FILL).all()), cap


def test_lane_decoder_long_codes_and_skew(codec, lanes):
    # Fibonacci weights: one-bit codes next to codes of 27 and 32 bits (the trie path inside the flat loop);
    # the text of a region is up to 8x its stream bytes, so the stage of a warp is sized per stream
    for depth in (19, 27, 32):
        w = synth.fibonacci_weights(depth)
        data = synth.generate(1 << 21, synth.thresholds_from_weights(w), seed=depth)
        data[: depth + 1] = np.arange(depth + 1, dtype=np.uint8)
        m, out = codec.decode(_oracle_et(data)[4:])
        assert m == data.size and out.tobytes() == data.tobytes(), depth
    rng = np.random.default_rng(17)
    w = rng.random(256) ** 8
    data = rng.choice(256, 1 << 21, p=w / w.sum()).astype(np.uint8)
    data[:256] = np.arange(256, dtype=np.uint8)
    stream = _oracle_et(data)[4:]
    m, out = codec.decode(stream)
    assert out.tobytes() == oracle.decode(stream, data.size).tobytes()
    # two symbols, one bit each: eight symbols per stream byte
    data = rng.integers(0, 2, 1 << 20, dtype=np.uint8)
    m, out = codec.decode(_oracle_et(data)[4:])
    assert m == data.size and out.tobytes() == data.tobytes()


def _handmade_stream(lengths, codes, text):
    """file[4..] of an .et whose dictionary is given outright: lengths[s] (0 = absent), codes[s] (first bit on top)."""
    bits = []

    def put(v, n):
        bits.extend((int(v) >> (n - 1 - i)) & 1 for i in range(n))

    live = [s for s in range(256) if lengths[s]]
    put(len(live) - 1, 8)
    put(text.size, 32)
    for s in live:
        put(s, 8)
        put(lengths[s], 8)
        put(codes[s], int(lengths[s]))
    bits.extend([0] * (-(len(bits) + 32) % 8))  # the four bytes before are whole
    head = np.packbits(np.array(bits, dtype=np.uint8))
    ln = np.asarray(lengths, dtype=np.int64)[text]
    cd = np.asarray(codes, dtype=np.uint64)[text]
    start = np.cumsum(ln) - ln
    within = np.arange(int(ln.sum()), dtype=np.int64) - np.repeat(start, ln)
    body = (np.repeat(cd, ln) >> (np.repeat(ln, ln) - 1 - within).astype(np.uint64)) & np.uint64(1)
    return head.tobytes() + np.packbits(body.astype(np.uint8)).tobytes()


def test_lane_decoder_deepest_codes_anywhere(codec, lanes):
    # A chain written out by hand: symbol k is k ones and a zero, the last one all ones - codes of up to 32 bits, which a
    # text would need 2^32 symbols to produce, here one symbol in a hundred, so that chunks in the middle of the stream
    # (the fast walkers, both of them) meet them at every position of their windows.  The oracle reads the stream
    # back; the library must read the same.  Beyond 32 bits the library refuses the dictionary (the reference's
    # decoder cannot hold such a code: DESIGN.md), whatever the oracle makes of it.
    rng = np.random.default_rng(40)
    for depth in (20, 27, 32, 34):
        lengths = [0] * 256
        codes = [0] * 256
        for k in range(depth + 1):
            lengths[k] = min(k + 1, depth)
            codes[k] = ((1 << k) - 1) << 1 if k < depth else (1 << depth) - 1
        text = np.minimum(rng.geometric(0.5, 1 << 21) - 1, depth).astype(np.uint8)
        deep = rng.random(text.size) < 0.01
        text[deep] = rng.integers(depth - 18, depth + 1, int(deep.sum()))
        stream = _handmade_stream(lengths, codes, text)
        want = oracle.decode(stream, text.size)
        assert want.tobytes() == text.tobytes(), depth  # the oracle reads it back
        if depth > 32:
            with pytest.raises(et.EntreepyError) as e:
                codec.decode(stream)
            assert e.value.name == "Unsupported"
            continue
        m, out = codec.decode(stream)
        assert m == text.size and out.tobytes() == text.tobytes(), depth


def _marker_windows(lengths, codes):
    """12-bit windows that are proper prefixes of longer codes.  The first kMaxSubTables (16) of them to ask get a
    second-level table (build_table_entry); lookups behind the others walk the trie (code_slow, code_at_global)."""
    return len({int(codes[s]) >> (int(lengths[s]) - 12) for s in range(256) if int(lengths[s]) > 12})


def _many_windows_handmade(rng):
    """A complete code of 252 symbols with 20 marker windows, behind which chains run to 21..32 bits: the prefixes 1, 01,
    .., 0000001 (1..7 bits), then the 32 windows under 0000000: 12 of them are codes, 20 are markers."""
    entries = [(k + 1, 1) for k in range(7)] + [(12, w) for w in range(20, 32)]
    for w, depth in zip(range(20), [9] * 12 + [10, 10, 11, 12, 13, 14, 15, 20]):
        entries += [(13 + j, (w << (j + 1)) | (((1 << j) - 1) << 1)) for j in range(depth)]  # j ones and a zero
        entries.append((12 + depth, (w << depth) | ((1 << depth) - 1)))
    assert sum(2.0 ** -length for length, _ in entries) == 1.0
    lengths, codes = [0] * 256, [0] * 256
    symbols = rng.permutation(256)[: len(entries)]
    for s, (length, code) in zip(symbols, entries):
        lengths[s], codes[s] = length, code
    short = symbols[:7]
    text = np.where(rng.random(1 << 21) < 0.8, short[np.minimum(rng.geometric(0.5, 1 << 21) - 1, 6)],
                    rng.choice(symbols, 1 << 21)).astype(np.uint8)
    return lengths, codes, text


def test_lane_decoder_over_sixteen_marker_windows(codec, lanes):
    # More marker windows than second-level tables: which windows get one follows atomicAdd order and may change from run
    # to run; lookups behind the rest walk the trie, deep into it for the hand-made chains.  Every run, every path
    # (lanes, default tuning, the batch call, shards) must read the oracle's text back.
    import torch

    from test_gpu_shards import _unpack_in_shards

    rng = np.random.default_rng(16)
    streams = []
    for frequent, count in ((64, 16384), (16, 131072)):  # codes of 6..15 bits, 32 windows; 4..13 bits, 111 windows
        counts = np.zeros(256, dtype=np.int64)
        counts[:frequent], counts[frequent:255] = count, 16
        data = np.repeat(np.arange(256, dtype=np.uint8), counts)
        rng.shuffle(data)
        codes, lengths = oracle.build_dictionary(counts.astype(np.uint64))
        streams.append((_oracle_et(data)[4:], data, _marker_windows(lengths, codes)))
    lengths, codes, text = _many_windows_handmade(rng)
    stream = _handmade_stream(lengths, codes, text)
    assert oracle.decode(stream, text.size).tobytes() == text.tobytes()
    assert max(lengths) == 32 and min(length for length in lengths if length > 12) == 13
    streams.append((stream, text, _marker_windows(lengths, codes)))
    assert [(s[1].size, s[2]) for s in streams] == [(1_051_632, 32), (2_100_976, 111), (1 << 21, 20)]

    for stream, data, _ in streams:
        for run in range(3):
            m, out = codec.decode(stream)
            assert m == data.size and out.tobytes() == data.tobytes(), (data.size, run)
    _unpack_in_shards(codec, streams[1][1], 3, expect_guess_right=False)
    codec.set_tuning(et._abi.TUNE_LANE_MIN_BYTES, -1)
    for stream, data, _ in streams:
        m, out = codec.decode(stream)
        assert m == data.size and out.tobytes() == data.tobytes(), data.size
    ins = [torch.from_numpy(np.frombuffer(s, dtype=np.uint8).copy()).cuda() for s, _, _ in streams]
    outs = [torch.full((d.size + 64,), FILL, dtype=torch.uint8, device="cuda") for _, d, _ in streams]
    torch.cuda.synchronize()
    res = codec.decode_batch_dev([(i.data_ptr(), i.numel(), o.data_ptr(), d.size) for i, o, (_, d, _) in zip(ins, outs, streams)])
    for (_, data, _), o, r in zip(streams, outs, res):
        assert r == (et._abi.OK, data.size), (data.size, r)
        assert o[: data.size].cpu().numpy().tobytes() == data.tobytes() and bool((o[data.size :] == FILL).all()), data.size


def test_lane_decoder_repairs_wrong_guesses(codec, lanes):
    # 40 of 48 symbols equiprobable: most codes have 6 or 7 bits and a wrong parse survives for a long time, so
    # the run-up guesses are often wrong and the repair rounds have to settle the entries
    rng = np.random.default_rng(5)
    w = np.ones(48)
    w[:8] = 9.0  # lengths 3..7: a spread wide enough for the lane path, still slow to synchronise
    data = rng.choice(48, 1 << 20, p=w / w.sum()).astype(np.uint8)
    lengths = oracle.build_dictionary(oracle.histogram(data))[1]
    assert int(lengths.max()) - int(lengths[lengths > 0].min()) > 2
    m, out = codec.decode(_oracle_et(data)[4:])
    assert m == data.size and out.tobytes() == data.tobytes()


def test_lane_decoder_survives_random_bodies(codec, lanes):
    # Random bytes behind a dictionary: with a complete code every bit pattern decodes to something (compare with the
    # oracle); with an incomplete one the walkers meet patterns that are no code at all, everywhere in their windows.
    # The call must come back (an answer or Corrupt) and the context must still decode a good stream afterwards - a
    # walk that leaves its shared memory would poison the CUDA context for good.
    rng = np.random.default_rng(77)
    good = rng.choice(64, 1 << 20, p=(lambda w: w / w.sum())(rng.random(64) ** 3)).astype(np.uint8)
    good[:64] = np.arange(64, dtype=np.uint8)
    good_stream = _oracle_et(good)[4:]
    for trial in range(6):
        n_syms = int(rng.integers(3, 31))  # codes of up to 30 bits
        lengths = [0] * 256
        codes = [0] * 256
        # a chain code (prefix-free); dropping the all-ones leaf makes it incomplete
        for k in range(n_syms):
            lengths[k] = min(k + 1, n_syms - 1) if trial % 2 == 0 else k + 1
            codes[k] = ((1 << k) - 1) << 1 if (k < n_syms - 1 or trial % 2) else (1 << (n_syms - 1)) - 1
        body = rng.integers(0, 256, int(rng.integers(200_000, 900_000)), dtype=np.uint8)
        if trial % 2:  # incomplete: long runs of ones are no code
            body[rng.integers(0, body.size, body.size // 50)] = 0xFF
        head = _handmade_stream(lengths, codes, np.zeros(1, dtype=np.uint8))
        n_claim = body.size * 3
        stream = bytes([head[0]]) + int(n_claim).to_bytes(4, "big") + head[5:-1] + body.tobytes()
        try:
            m, out = codec.decode(stream)
            if trial % 2 == 0:
                want = oracle.decode(stream, n_claim)
                assert m == want.size and out.tobytes() == want.tobytes(), trial
        except et.EntreepyError as e:
            assert e.name in ("Corrupt", "NoSpaceLeft"), (trial, e.name)
        m, out = codec.decode(good_stream)
        assert m == good.size and out.tobytes() == good.tobytes(), trial
