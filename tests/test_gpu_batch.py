"""et_decode_batch_dev against et_decode_dev and the oracle: every item of a batch must end with the status, the
out_len and the d_out bytes the single call gives it, whatever its neighbours are.  Run with -m gpu on a B200."""
import ctypes
import json
import os

import numpy as np
import pytest

import entreepy_b200 as et
from conftest import GOLDEN, make_cases
from entreepy_b200 import _abi, synth
from oracle import oracle

pytestmark = pytest.mark.gpu

WRITE = _abi.FLAG_WRITE_OUTPUT
GUARD = 64  # bytes on both sides of every output, which must keep the fill
FILL = 0xA5  # what every output holds before a call: a decoder that writes zeros, or skips a zero byte, shows


def _stream(data):
    """file[4..] of the oracle's .et for data."""
    return oracle.encode(data, cap=9000 + 5 * int(np.asarray(data).size)).tobytes()[4:]


def _fuzz_input(rng):
    """Like test_gpu_fuzz: random alphabet of 2..256 symbols, random skew, 1 B .. 3 MB."""
    m = int(rng.integers(2, 257))
    skew = float(rng.choice([0.0, 0.5, 1.0, 2.0, 4.0, 8.0]))
    w = rng.random(m) ** skew if skew else np.ones(m)
    syms = rng.permutation(256)[:m].astype(np.uint8)
    n = int(rng.choice([rng.integers(1, 5000), rng.integers(5000, 70000), rng.integers(70000, 600000),
                        rng.integers(600000, 3000000)]))
    return syms[rng.choice(m, n, p=w / w.sum())]


def _dict_stream(entries, body_len, body):
    """file[4..] for a hand-made dictionary: entries = [(symbol, length, code)]."""
    bits = []
    for sym, length, code in entries:
        bits += [(sym >> (7 - k)) & 1 for k in range(8)] + [(length >> (7 - k)) & 1 for k in range(8)]
        bits += [(code >> (length - 1 - k)) & 1 for k in range(length)]
    bits += [0] * (-len(bits) % 8)
    d = np.packbits(np.array(bits, dtype=np.uint8)).tobytes()
    return bytes([len(entries) - 1]) + int(body_len).to_bytes(4, "big") + d + bytes(body)


_TEXT_THRESHOLDS = []


def _text(n, seed):
    """n bytes with the letter frequencies of the Midsummer fixture (a code that synchronises within a few symbols)."""
    if not _TEXT_THRESHOLDS:
        man = json.load(open(os.path.join(GOLDEN, "manifest.json")))
        _TEXT_THRESHOLDS.append(synth.thresholds_from_weights(synth.text_weights(man["midsummer_histogram"])))
    return synth.generate(n, _TEXT_THRESHOLDS[0], seed=seed)


def _single(codec, d_in, n, d_out, cap, flags):
    got = ctypes.c_size_t(0)
    rc = codec._lib.et_decode_dev(codec._ctx, d_in, n, d_out, cap, ctypes.byref(got), flags, None)
    return rc, got.value


class Items:
    """Device copies of the streams at the given offsets, and outputs filled with FILL with guard bytes around them."""

    def __init__(self, streams, caps, in_offs=None, out_offs=None):
        import torch

        k = len(streams)
        self.streams, self.caps = streams, caps
        self.in_offs = in_offs or [0] * k
        self.out_offs = out_offs or [0] * k
        self.ins = []
        for s, off in zip(streams, self.in_offs):
            t = torch.zeros(len(s) + off + 16, dtype=torch.uint8)
            t[off:off + len(s)] = torch.frombuffer(bytearray(s), dtype=torch.uint8)
            self.ins.append(t.cuda())

    def outputs(self):
        import torch

        outs = [torch.full((GUARD + off + cap + GUARD,), FILL, dtype=torch.uint8, device="cuda") for off, cap in zip(self.out_offs, self.caps)]
        torch.cuda.synchronize()  # the library works on its own stream
        return outs

    def args(self, outs):
        return [(self.ins[k].data_ptr() + self.in_offs[k], len(self.streams[k]), outs[k].data_ptr() + GUARD + self.out_offs[k], self.caps[k])
                for k in range(len(self.streams))]

    def text(self, outs, k, n):
        off = GUARD + self.out_offs[k]
        return outs[k][off:off + n].cpu().numpy().tobytes()


def _batch_matches_single(codec, items, flags=WRITE):
    """Runs the batch and the single call on every item; asserts they agree byte for byte (guards included)."""
    import torch

    single_out, batch_out = items.outputs(), items.outputs()
    single = [_single(codec, *a, flags) for a in items.args(single_out)]
    batch = codec.decode_batch_dev(items.args(batch_out), flags)
    torch.cuda.synchronize()
    for k in range(len(items.streams)):
        assert batch[k] == single[k], (k, batch[k], single[k])
        assert torch.equal(batch_out[k], single_out[k]), (k, batch[k])
        off, cap = GUARD + items.out_offs[k], items.caps[k]
        assert bool((batch_out[k][:off] == FILL).all()) and bool((batch_out[k][off + cap:] == FILL).all()), k
        if batch[k][0] == _abi.OK:  # nothing past out_len either
            assert bool((batch_out[k][off + batch[k][1]:] == FILL).all()), k
    return batch, batch_out


def test_batch_matches_single_calls_and_oracle(codec, golden_et):
    rng = np.random.default_rng(20261020)
    inputs = list(make_cases().values()) + [np.frombuffer(golden_et[n][4:], dtype=np.uint8) for n in sorted(golden_et)]
    n_cases = len(make_cases())
    while len(inputs) < n_cases + len(golden_et) + 40:
        data = _fuzz_input(rng)
        if np.unique(data).size >= 2:
            inputs.append(data)
    # routed for certain: a body long enough for the lane decoder, uniform bytes (transfer functions)
    inputs += [_text(4_500_000, 11), rng.integers(0, 256, 1_000_000, dtype=np.uint8)]
    streams, caps, texts = [], [], []
    for k, data in enumerate(inputs):
        if n_cases <= k < n_cases + len(golden_et):  # a golden file: already a stream
            s = data.tobytes()
            body_len = int(et.parse_header(s).body_len)
        else:
            s, body_len = _stream(data), data.size
        streams.append(s)
        caps.append(body_len)
        texts.append(oracle.decode(s, body_len).tobytes() if et.parse_header(s).n_entries else b"")  # no entries: nothing to decode
    items = Items(streams, caps, [int(x) for x in rng.integers(0, 16, len(streams))], [int(x) for x in rng.integers(0, 16, len(streams))])
    res, outs = _batch_matches_single(codec, items)
    for k, (status, n) in enumerate(res):
        assert status == _abi.OK and n == len(texts[k]), (k, status, n, len(texts[k]))
        assert items.text(outs, k, n) == texts[k], k


@pytest.mark.parametrize("validate", [False, True])
def test_failing_items_do_not_affect_their_neighbours(codec, golden_et, validate):
    flags = WRITE | (_abi.FLAG_VALIDATE if validate else 0)
    text = np.frombuffer(b"abracadabra, the quick brown fox " * 200, dtype=np.uint8)
    good = _stream(text)
    streams = [
        golden_et["a_midsummer_nights_dream.txt"][4:],
        b"\x01\x00\x00",                                                # garbage: the dictionary cannot be parsed
        good,
        bytes([1, 0, 0, 0, 9, 65, 1, 0b10100001, 0b00000000]),          # dictionary truncated mid-way
        golden_et["test.txt"][4:],
        good,                                                           # capacity one byte short
        _dict_stream([(97, 1, 0b0), (98, 2, 0b01)], 3, [0b00000000]),   # not a prefix code: ET_FLAG_VALIDATE rejects it
        _dict_stream([(97, 1, 0b0), (98, 2, 0b10)], 3, [0b11000000]),   # body holds a bit pattern that is no code
        golden_et["nice.shakespeare.txt"][4:],
    ]
    caps = [int(et.parse_header(s).body_len) if len(s) > 5 else 16 for s in streams]
    caps[5] -= 1
    items = Items(streams, caps, [3, 0, 5, 1, 7, 0, 2, 9, 15], [1, 0, 2, 0, 15, 4, 0, 3, 8])
    res, outs = _batch_matches_single(codec, items, flags)
    assert res[1][0] == _abi.ERR_CORRUPT
    assert res[3] == ((_abi.ERR_CORRUPT, 0) if validate else (_abi.OK, 0))
    assert res[5] == (_abi.ERR_NO_SPACE, 0)
    assert res[6] == ((_abi.ERR_CORRUPT, 0) if validate else (_abi.OK, 3))
    assert res[7][0] == _abi.ERR_CORRUPT
    for k in (0, 2, 4, 8):
        want = oracle.decode(streams[k], caps[k]).tobytes()
        assert res[k] == (_abi.OK, len(want)) and items.text(outs, k, len(want)) == want, k


def test_dry_run_writes_nothing(codec, golden_et):
    import torch

    streams = [golden_et[n][4:] for n in sorted(golden_et)] + [_stream(_text(5000, 3))]
    caps = [int(et.parse_header(s).body_len) for s in streams]
    items = Items(streams, caps, [0, 1, 2, 3], [4, 5, 6, 7])
    res, outs = _batch_matches_single(codec, items, flags=0)
    assert all(r == (_abi.OK, 0) for r in res), res
    assert all(bool((o == FILL).all()) for o in outs)
    torch.cuda.synchronize()


def test_call_level_arguments(codec, golden_et):
    L = codec._lib
    assert L.et_decode_batch_dev(codec._ctx, None, 0, WRITE, None) == _abi.OK
    assert L.et_decode_batch_dev(codec._ctx, None, 3, WRITE, None) == _abi.ERR_INVALID_ARG
    assert codec.decode_batch_dev([]) == []
    # the same d_in twice, into two outputs
    s = golden_et["a_midsummer_nights_dream.txt"][4:]
    cap = int(et.parse_header(s).body_len)
    items = Items([s], [cap])
    outs = items.outputs() + items.outputs()
    a = items.args(outs[:1])[0]
    b = (a[0], a[1], outs[1].data_ptr() + GUARD, cap)
    res = codec.decode_batch_dev([a, b])
    want = oracle.decode(s, cap).tobytes()
    assert res == [(_abi.OK, len(want))] * 2
    assert items.text(outs, 0, len(want)) == want and outs[1][GUARD:GUARD + len(want)].cpu().numpy().tobytes() == want


def test_more_streams_than_one_group(codec):
    rng = np.random.default_rng(5)
    texts = [_text(int(rng.integers(2, 600)), seed=1000 + k) for k in range(3000)]
    streams = [_stream(t) for t in texts]
    items = Items(streams, [t.size for t in texts], [int(x) for x in rng.integers(0, 16, 3000)], [int(x) for x in rng.integers(0, 16, 3000)])
    outs = items.outputs()
    res = codec.decode_batch_dev(items.args(outs))
    for k, t in enumerate(texts):
        want = oracle.decode(streams[k], t.size).tobytes() if et.parse_header(streams[k]).n_entries else b""
        assert res[k] == (_abi.OK, len(want)), (k, res[k])
        assert items.text(outs, k, len(want)) == want, k


def test_launches_do_not_grow_with_the_batch(codec):
    streams = [_stream(_text(4096, seed=k)) for k in range(512)]
    counts = []
    for b in (16, 512):
        items = Items(streams[:b], [4096] * b)
        outs = items.outputs()
        before = codec.kernel_launches
        res = codec.decode_batch_dev(items.args(outs))
        counts.append(codec.kernel_launches - before)
        assert all(r == (_abi.OK, 4096) for r in res)
        assert codec.last_decode_rounds == 2
    # one group: 1 head gather, 2 table builds, sync 0 and 1, sum, scan, write
    assert counts == [8, 8], counts


def _codes_3_to_7(rng, n):
    """40 of 48 symbols equiprobable, 8 of them more frequent: code lengths 3..7, a spread too wide for transfer functions,
    and still slow to synchronise (test_lane_decoder_repairs_wrong_guesses)."""
    w = np.ones(48)
    w[:8] = 9.0
    return rng.choice(48, n, p=w / w.sum()).astype(np.uint8)


def _batch_with_oracle(codec, inputs, rng):
    """The oracle's streams of `inputs` at random offsets, none long enough for the lane decoder: the batch against single
    calls, then every item against the oracle.  -> (streams, kernel launches of one more batch call, its rounds)."""
    import torch

    streams = [_stream(d) for d in inputs]
    lane_min = torch.cuda.get_device_properties(0).multi_processor_count * 3 * 4224  # lane_path_min_bytes
    for s in streams:
        d = et.parse_header(s)
        assert d.max_length - d.min_length <= 2 or len(s) - d.body_offset < lane_min
    items = Items(streams, [d.size for d in inputs], [int(x) for x in rng.integers(0, 16, len(streams))],
                  [int(x) for x in rng.integers(0, 16, len(streams))])
    res, outs = _batch_matches_single(codec, items)
    for k, data in enumerate(inputs):
        assert res[k] == (_abi.OK, data.size) and items.text(outs, k, data.size) == data.tobytes(), k
    again = items.outputs()
    before = codec.kernel_launches
    assert codec.decode_batch_dev(items.args(again)) == res
    launches, rounds = codec.kernel_launches - before, codec.last_decode_rounds
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip(again, outs))
    return streams, launches, rounds


def test_batch_repair_rounds_of_slowly_synchronising_streams(codec):
    # Streams whose guessed chunk entries are wrong and that stay in the batch: launch_unpack_batch runs its fixpoint
    # rounds (settle) and a second write walk, and clears the item status before it.  With ET_TUNE_NO_TRANSFER, codes
    # whose lengths are within 2 bits of each other (uniform bytes: 7 and 8 bits) are such streams; so may be a stream of
    # 3..7-bit codes under any tuning.  A body long enough for 512-byte chunks settles before its first write walk
    # (settle_first).  Launches per group: 8 (test_launches_do_not_grow_with_the_batch), 4 per host visit of the rounds,
    # 3 for a second write walk.
    import torch

    rng = np.random.default_rng(41)
    fixed = rng.permutation(np.repeat(rng.permutation(256)[:32].astype(np.uint8), 20_000))  # 5-bit codes: closed-form entries
    d = et.parse_header(_stream(fixed))
    assert d.min_length == d.max_length == 5
    mixed = [_text(200_003, 7), _codes_3_to_7(rng, 1 << 20), _text(1_000_003, 8), fixed]
    uniform = [rng.integers(1, 256, n, dtype=np.uint8) for n in (70_001, 300_007, 1_000_003, 4_000_037)]
    big = rng.integers(1, 256, 48_000_017, dtype=np.uint8)
    codec.set_tuning(_abi.TUNE_NO_TRANSFER, 1)
    try:
        # chunks of 256 bytes: a write walk, the rounds, a second write walk
        _, launches, rounds = _batch_with_oracle(codec, uniform + mixed, rng)
        assert rounds > 2 and launches > 11 and (launches - 11) % 4 == 0, (rounds, launches)
        # unpack_chunk_bytes keeps 512-byte chunks once body / 512 x max_length >= SMs x 4096: the rounds, one write walk
        streams, launches, rounds = _batch_with_oracle(codec, [big] + uniform[:2] + mixed, rng)
        d = et.parse_header(streams[0])
        assert (len(streams[0]) - d.body_offset) // 512 * d.max_length >= torch.cuda.get_device_properties(0).multi_processor_count * 4096
        assert rounds > 2 and launches > 8 and (launches - 8) % 4 == 0, (rounds, launches)
    finally:
        codec.set_tuning(_abi.TUNE_NO_TRANSFER, 0)
    # default tuning: the codes of 3..7 bits among streams that synchronise at once still need the rounds
    _, launches, rounds = _batch_with_oracle(codec, mixed, rng)
    assert rounds > 2 and launches > 11 and (launches - 11) % 4 == 0, (rounds, launches)
