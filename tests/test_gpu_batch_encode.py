"""et_encode_batch_dev against et_encode_dev and the oracle: every item of a batch must end with the status, the out_len
and the d_out bytes the single call gives it, whatever its neighbours are.  Run with -m gpu on a B200."""
import ctypes
import json
import os

import numpy as np
import pytest

from conftest import FIXTURES, GOLDEN, make_cases
from entreepy_b200 import _abi, synth
from oracle import oracle

pytestmark = pytest.mark.gpu

WRITE = _abi.FLAG_WRITE_OUTPUT
GUARD = 64  # bytes on both sides of every output, which must keep the fill
FILL = 0xA5  # what every output holds before a call: an encoder that writes zeros, or skips a zero byte, shows


def _oracle_et(data):
    """The oracle's whole .et file (magic included) for data."""
    return oracle.encode(data, cap=9000 + 5 * int(np.asarray(data).size)).tobytes()


def _fuzz_input(rng):
    """Like test_gpu_fuzz: random alphabet of 2..256 symbols, random skew, 1 B .. 3 MB."""
    m = int(rng.integers(2, 257))
    skew = float(rng.choice([0.0, 0.5, 1.0, 2.0, 4.0, 8.0]))
    w = rng.random(m) ** skew if skew else np.ones(m)
    syms = rng.permutation(256)[:m].astype(np.uint8)
    n = int(rng.choice([rng.integers(1, 5000), rng.integers(5000, 70000), rng.integers(70000, 600000),
                        rng.integers(600000, 3000000)]))
    return syms[rng.choice(m, n, p=w / w.sum())]


_TEXT_THRESHOLDS = []


def _thresholds():
    if not _TEXT_THRESHOLDS:
        man = json.load(open(os.path.join(GOLDEN, "manifest.json")))
        _TEXT_THRESHOLDS.append(synth.thresholds_from_weights(synth.text_weights(man["midsummer_histogram"])))
    return _TEXT_THRESHOLDS[0]


def _text(n, seed):
    """n bytes with the letter frequencies of the Midsummer fixture."""
    return synth.generate(n, _thresholds(), seed=seed)


def _cap(n):
    return 9000 + 2 * n


def _single(codec, d_in, n, d_out, cap, flags):
    got = ctypes.c_size_t(0)
    rc = codec._lib.et_encode_dev(codec._ctx, d_in, n, d_out, cap, ctypes.byref(got), flags, None)
    return rc, got.value


class Texts:
    """Device copies of the texts at the given offsets, and zeroed outputs with guard bytes around them."""

    def __init__(self, texts, caps=None, in_offs=None, out_offs=None):
        import torch

        k = len(texts)
        self.texts = [np.asarray(t, dtype=np.uint8) for t in texts]
        self.caps = caps or [_cap(t.size) for t in self.texts]
        self.in_offs = in_offs or [0] * k
        self.out_offs = out_offs or [0] * k
        self.ins = []
        for t, off in zip(self.texts, self.in_offs):
            d = torch.zeros(t.size + off + 16, dtype=torch.uint8)
            d[off:off + t.size] = torch.from_numpy(t.copy())
            self.ins.append(d.cuda())
        torch.cuda.synchronize()

    def outputs(self):
        import torch

        outs = [torch.full((GUARD + off + cap + GUARD,), FILL, dtype=torch.uint8, device="cuda") for off, cap in zip(self.out_offs, self.caps)]
        torch.cuda.synchronize()  # the library's stream does not wait for torch's: the fill is in place before it writes
        return outs

    def args(self, outs):
        return [(self.ins[k].data_ptr() + self.in_offs[k], self.texts[k].size, outs[k].data_ptr() + GUARD + self.out_offs[k], self.caps[k])
                for k in range(len(self.texts))]

    def file(self, outs, k, n):
        off = GUARD + self.out_offs[k]
        return outs[k][off:off + n].cpu().numpy().tobytes()


def _random_offsets(rng, k):
    return [int(x) for x in rng.integers(0, 16, k)], [int(x) for x in rng.integers(0, 16, k)]


def _batch_matches_single(codec, texts, flags=WRITE, patch=None):
    """Runs the batch and the single call on every item; asserts they agree byte for byte (guards included).
    patch(args): changes the argument tuples of some items in place (both runs see the same ones).  -> (results, outputs)"""
    import torch

    single_out, batch_out = texts.outputs(), texts.outputs()
    sa, ba = texts.args(single_out), texts.args(batch_out)
    if patch:
        patch(sa, single_out)
        patch(ba, batch_out)
    single = [_single(codec, *a, flags) for a in sa]
    batch = codec.encode_batch_dev(ba, flags)
    torch.cuda.synchronize()
    for k in range(len(texts.texts)):
        assert batch[k] == single[k], (k, batch[k], single[k])
        assert torch.equal(batch_out[k], single_out[k]), (k, batch[k])
        off, cap = GUARD + texts.out_offs[k], texts.caps[k]
        assert bool((batch_out[k][:off] == FILL).all()) and bool((batch_out[k][off + cap:] == FILL).all()), k
        if batch[k][0] == _abi.OK and flags & WRITE:  # nothing past out_len either
            assert bool((batch_out[k][off + batch[k][1]:] == FILL).all()), k
    return batch, batch_out


def _assert_oracle(texts, res, outs, ks=None):
    for k in ks if ks is not None else range(len(texts.texts)):
        want = _oracle_et(texts.texts[k])
        assert res[k] == (_abi.OK, len(want)), (k, res[k], len(want))
        assert texts.file(outs, k, len(want)) == want, k


def _launches(codec, fn):
    before = codec.kernel_launches
    r = fn()
    return r, codec.kernel_launches - before


def test_batch_matches_single_calls_and_oracle(codec, fixtures):
    rng = np.random.default_rng(20261021)
    inputs = list(make_cases().values()) + [np.frombuffer(fixtures[n], dtype=np.uint8) for n in FIXTURES]
    # lengths around multiples of the pack's regions (2048) and tiles (4096), and of the histogram tiles (16384)
    for n in (2047, 2048, 2049, 4095, 4096, 4097, 6143, 6145, 16383, 16384, 16385, 32768 + 2047, 32768 * 3 + 1):
        inputs.append(_text(n, seed=n))
    n_fixed = len(inputs)
    while len(inputs) < n_fixed + 40:
        data = _fuzz_input(rng)
        if np.unique(data).size >= 2:
            inputs.append(data)
    texts = Texts(inputs, None, *_random_offsets(rng, len(inputs)))
    res, outs = _batch_matches_single(codec, texts)
    _assert_oracle(texts, res, outs)


def test_failing_items_do_not_affect_their_neighbours(codec, fixtures):
    import torch

    good = np.frombuffer(b"abracadabra, the quick brown fox " * 200, dtype=np.uint8)
    mid = np.frombuffer(fixtures["a_midsummer_nights_dream.txt"], dtype=np.uint8)
    inputs = [mid, good, good, good, good, good, _text(70_001, 5), good, mid, mid]  # item 8 reads item 0's d_in
    caps = [_cap(t.size) for t in inputs]
    caps[5] = len(_oracle_et(good)) - 1  # capacity one byte short
    texts = Texts(inputs, caps, [3, 0, 5, 1, 7, 9, 2, 11, 4, 15], [1, 0, 2, 0, 15, 4, 0, 3, 8, 6])
    huge = torch.zeros(1 << 32, dtype=torch.uint8, device="cuda")  # a real 2^32-byte text: a wrong implementation reads it
    torch.cuda.synchronize()

    def patch(args, outs):
        args[1] = (args[1][0], 0, args[1][2], args[1][3])                     # n == 0
        args[2] = (None, args[2][1], args[2][2], args[2][3])                  # d_in == NULL
        args[3] = (args[3][0], args[3][1], None, args[3][3])                  # WRITE with d_out == NULL
        args[7] = (huge.data_ptr(), 1 << 32, args[7][2], args[7][3])          # n = 2^32
        args[8] = (args[0][0], args[0][1], args[8][2], args[8][3])            # the same d_in as item 0

    res, outs = _batch_matches_single(codec, texts, patch=patch)
    assert res[1] == (_abi.ERR_QUEUE_EMPTY, 0)
    assert res[2] == (_abi.ERR_INVALID_ARG, 0)
    assert res[3] == (_abi.ERR_INVALID_ARG, 0)
    assert res[5] == (_abi.ERR_NO_SPACE, 0)
    assert res[7] == (_abi.ERR_TOO_LARGE, 0)
    _assert_oracle(texts, res, outs, (0, 4, 6, 9))
    want = _oracle_et(mid)
    assert res[8] == (_abi.OK, len(want)) and texts.file(outs, 8, len(want)) == want
    del huge


def test_dry_run_writes_nothing(codec, fixtures):
    inputs = [np.frombuffer(fixtures[n], dtype=np.uint8) for n in FIXTURES] + [_text(5000, 3), np.full(100, 9, np.uint8)]
    texts = Texts(inputs, None, [0, 1, 2, 3, 4], [4, 5, 6, 7, 8])
    res, outs = _batch_matches_single(codec, texts, flags=0)
    assert res == [(_abi.OK, len(_oracle_et(t))) for t in inputs], res
    assert all(bool((o == FILL).all()) for o in outs)


def test_zero_bit_regions_and_single_symbol_texts(codec):
    rng = np.random.default_rng(3)
    cases = make_cases()
    # every byte value occurs: the most frequent symbol gets no code, and a long run of it makes regions of zero bits
    # (one of them begins inside a byte of the body)
    base = rng.integers(0, 256, 60_001, dtype=np.uint8)
    base[rng.random(base.size) < 0.3] = 200
    runs = np.concatenate([base[:30_001], np.full(20_000, 200, np.uint8), base[30_001:], np.full(5000, 200, np.uint8)])
    dropped = [cases["all_256_uniform"], cases["dropped_symbol_dominates"], cases["all_256_once"], runs]
    for d in dropped:
        _, length = oracle.build_dictionary(oracle.histogram(d))
        assert np.unique(d).size == 256 and (length == 0).sum() == 1, "a dropped symbol"
    single = [np.full(n, s, np.uint8) for n, s in ((1, 65), (1000, 7), (2048, 0), (4097, 255), (70_000, 33))]
    inputs = dropped + single
    texts = Texts(inputs, None, *_random_offsets(rng, len(inputs)))
    res, outs = _batch_matches_single(codec, texts)
    _assert_oracle(texts, res, outs)
    assert all(r == (_abi.OK, 9) for r in res[len(dropped):]), res


def test_codes_longer_than_32_bits_take_the_wide_route(codec):
    import torch

    rng = np.random.default_rng(33)
    f = [1, 1]
    while len(f) < 34:
        f.append(f[-1] + f[-2])
    n = sum(f)  # the smallest text whose exact Fibonacci counts make a chain of 33
    counts = synth.fibonacci_counts(n, 33)
    fib = synth.shuffled_dev(counts, seed=33).cpu().numpy()
    assert int(oracle.build_dictionary(np.array(counts, dtype=np.uint64))[1].max()) == 33
    inputs = [_text(5000, 1), fib, _text(100_003, 2), _text(4096, 4)]
    texts = Texts(inputs, None, *_random_offsets(rng, len(inputs)))
    flags = WRITE | _abi.FLAG_NO_SCRATCH_LIMIT
    res, outs = _batch_matches_single(codec, texts, flags)
    _assert_oracle(texts, res, outs)
    # one group: the histogram and the five batched pack launches for the narrow texts, pack_wide_kernel and its seam fix-up
    again = texts.outputs()
    r, launches = _launches(codec, lambda: codec.encode_batch_dev(texts.args(again), flags))
    torch.cuda.synchronize()
    assert r == res and launches == 8, launches
    assert all(torch.equal(a, b) for a, b in zip(again, outs))


def test_a_text_of_a_whole_group_takes_the_single_stream_route(codec):
    import torch

    rng = np.random.default_rng(256)
    big_n = 256 << 20
    big = torch.empty(big_n, dtype=torch.uint8, device="cuda")
    codec.synth_dev(big.data_ptr(), big_n, 77, 0, _thresholds())
    big_host = big.cpu().numpy()
    small = [_text(int(rng.integers(1, 9000)), seed=k) for k in range(5)]
    inputs = small[:3] + [big_host] + small[3:]
    texts = Texts(inputs, None, *_random_offsets(rng, len(inputs)))
    del big
    flags = WRITE | _abi.FLAG_NO_SCRATCH_LIMIT
    outs = texts.outputs()
    res, launches = _launches(codec, lambda: codec.encode_batch_dev(texts.args(outs), flags))
    # groups: the three texts before it (6 launches), the big text alone through et_encode_dev (its histogram, four pack
    # kernels, the seam fix-up: 6), the two after it (6)
    assert launches == 18, launches
    _assert_oracle(texts, res, outs)
    single = texts.outputs()
    for k, a in enumerate(texts.args(single)):
        assert _single(codec, *a, flags) == res[k], k
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip(single, outs))


def test_more_texts_than_one_group(codec):
    rng = np.random.default_rng(5)
    inputs = [_text(int(rng.integers(2, 600)), seed=1000 + k) for k in range(3000)]
    texts = Texts(inputs, None, *_random_offsets(rng, len(inputs)))
    res, outs = _batch_matches_single(codec, texts)
    _assert_oracle(texts, res, outs)


def test_launches_do_not_grow_with_the_batch(codec):
    inputs = [_text(4096, seed=k) for k in range(512)]
    counts = []
    for b in (16, 512):
        texts = Texts(inputs[:b])
        outs = texts.outputs()
        res, launches = _launches(codec, lambda: codec.encode_batch_dev(texts.args(outs)))
        counts.append(launches)
        assert all(r[0] == _abi.OK for r in res)
        if b == 16:
            _assert_oracle(texts, res, outs)
    # one group: the histogram, pass A, the region scan, the group scan, pass B, the seam fix-up with the headers
    assert counts == [6, 6], counts


def test_device_round_trip(codec, fixtures):
    import torch

    rng = np.random.default_rng(8)
    # every text of 2..255 distinct symbols comes back (when all 256 occur, the format drops the most frequent one)
    inputs = [t for t in make_cases().values() if 2 <= np.unique(t).size < 256]
    inputs += [np.frombuffer(fixtures[n], dtype=np.uint8) for n in FIXTURES] + [_text(int(rng.integers(1, 300_000)), k) for k in range(20)]
    texts = Texts(inputs, None, *_random_offsets(rng, len(inputs)))
    outs = texts.outputs()
    args = texts.args(outs)
    res = codec.encode_batch_dev(args)
    assert all(r[0] == _abi.OK for r in res), res
    back = [torch.zeros(t.size + 16, dtype=torch.uint8, device="cuda") for t in texts.texts]
    dec = codec.decode_batch_dev([(a[2] + 4, r[1] - 4, b.data_ptr() + 3, t.size) for a, r, b, t in zip(args, res, back, texts.texts)])
    for k, t in enumerate(texts.texts):
        assert dec[k] == (_abi.OK, t.size), (k, dec[k])
        assert back[k][3:3 + t.size].cpu().numpy().tobytes() == t.tobytes(), k


def test_call_level_arguments_and_stage_times(codec):
    L = codec._lib
    assert L.et_encode_batch_dev(codec._ctx, None, 0, WRITE, None) == _abi.OK
    assert L.et_encode_batch_dev(codec._ctx, None, 3, WRITE, None) == _abi.ERR_INVALID_ARG
    assert codec.encode_batch_dev([]) == []
    texts = Texts([_text(3000, k) for k in range(4)])
    outs = texts.outputs()
    res = codec.encode_batch_dev(texts.args(outs), WRITE | _abi.FLAG_TIMING)
    _assert_oracle(texts, res, outs)
    ms = (ctypes.c_float * 4)()
    assert L.et_ctx_last_stage_ms(codec._ctx, ctypes.byref(ms)) == _abi.OK
    assert ms[0] > 0 and ms[2] > 0 and ms[3] == 0, list(ms)
