"""The multi-GPU kernel entry points against the oracle, on ONE device (SURVEY §8e).

et_pack_shard_dev / et_unpack_shard_dev are what every rank of the sharded path calls.  Here the ranks are
emulated on cuda:0 so that the oracle can check their bytes:
  * direct calls: a text cut into k shards, every shard packed at its final bit offset (all eight bit phases,
    cuts at every residue mod 16, shards shorter than a byte of output, a dropped 256th symbol at a seam,
    codes of 32 bits), header + OR of the shards' bytes == oracle.encode(text), byte for byte;
    et_unpack_shard_dev with head_bit = -1 on 32-byte cuts of an oracle body: symbols, entry and exit
    against the true codeword boundaries, concatenated text == original;
  * the whole protocol (entreepy_b200.sharded.ShardedCodec with the real GpuBackend) for world 2, 3 and 8:
    one thread and one et_ctx per rank, exchanges through an in-process stand-in for the NCCL collectives.
Bar: bit-exact.  (test.zig:7-33 is the reference's round trip; the reference itself has nothing sharded.)
"""
import threading

import numpy as np
import pytest

import entreepy_b200 as et
from conftest import make_cases
from entreepy_b200 import _abi, sharded, synth
from oracle import oracle

pytestmark = pytest.mark.gpu


def _oracle_et(data):
    return oracle.encode(data, cap=9000 + 5 * int(np.asarray(data).size)).tobytes()


def _text(n, seed=5):
    """English-frequency text (code lengths 3..17: shard bit offsets take every phase)."""
    import json
    import os

    from conftest import GOLDEN

    man = json.load(open(os.path.join(GOLDEN, "manifest.json")))
    thr = synth.thresholds_from_weights(synth.text_weights(man["midsummer_histogram"]))
    return synth.generate(n, thr, seed=synth.SEED + seed)


def _fib32():
    """Exact Fibonacci counts: the Huffman tree is a chain, the longest code has 32 bits (SURVEY §0.4)."""
    counts = synth.fibonacci_counts(9_300_000, 32)
    data = np.repeat(np.arange(256, dtype=np.uint8), counts)
    np.random.default_rng(8).shuffle(data)
    return data


def _chain33():
    """Exact Fibonacci counts at the smallest size for a chain of depth 33: two symbols with 33-bit codes, one copy each
    (pack_wide_kernel)."""
    counts = synth.fibonacci_counts(14_930_351, 33)
    data = np.repeat(np.arange(256, dtype=np.uint8), counts)
    np.random.default_rng(9).shuffle(data)
    return data


def _chain33_at_cuts(world):
    """_chain33 with its 33-bit codes moved to the starts of ranks 1 and 2 of the sharded encoder: their heads cannot
    price their first output byte (first_output_byte), so the ranks exchange the real bytes after the pack."""
    data = _chain33()
    _, length = oracle.build_dictionary(oracle.histogram(data))
    starts = sharded.ShardPlan(data.size, world, 0).bounds[1:3]
    for at, deep in zip(starts, np.flatnonzero(length[data] == 33)):
        data[[at, deep]] = data[[deep, at]]
    assert all(length[data[at]] == 33 for at in starts)
    assert any(_boundaries(data)[at] % 8 for at in starts)  # a rank that starts inside a byte
    return data


def _dropped_run_at_cut(world):
    """All 256 byte values, the most frequent (255) gets no code; a run of it crosses the start of rank 1, which falls
    inside a byte of the body: rank 1's first eight symbols give no bits, so the ranks exchange the real first bytes
    after the pack."""
    text = np.random.default_rng(300 + world).integers(0, 256, 143_000, dtype=np.uint8)
    at = sharded.ShardPlan(text.size, world, 0).bounds[1]
    for lead in range(1000, 1008):  # the run's first bit, and so rank 1's, moves with the code before it
        data = text.copy()
        data[at - lead : at + 2000] = 255
        if _boundaries(data)[at] % 8:
            break
    assert et.build_codebook(oracle.histogram(data)).code[255].length == 0
    assert _boundaries(data)[at] % 8
    return data


def _pack_in_shards(codec, data, cuts):
    """Pack data[cuts[i]:cuts[i+1]] at its final bit offset with et_pack_shard_dev; -> (header, body, phases)."""
    import torch

    cb = et.build_codebook(oracle.histogram(data))
    header = et.write_header(cb, data.size)
    dev = torch.from_numpy(np.ascontiguousarray(data)).cuda()
    bits = [codec.shard_bits(oracle.histogram(data[lo:hi]), cb) for lo, hi in zip(cuts[:-1], cuts[1:])]
    offs = np.concatenate([[0], np.cumsum(bits)]).astype(np.int64)
    body = np.zeros(int((offs[-1] + 7) // 8), dtype=np.uint8)
    phases = []
    for i, (lo, hi) in enumerate(zip(cuts[:-1], cuts[1:])):
        out = torch.full(((hi - lo) * 4 + 64,), 0xAA, dtype=torch.uint8, device="cuda")  # stale bytes must not leak
        phase = int(offs[i] & 7)
        nbytes = codec.pack_shard_dev(dev.data_ptr() + lo, hi - lo, cb, phase, bits[i], out.data_ptr(), out.numel())
        assert nbytes == (phase + bits[i] + 7) // 8
        got = out[:nbytes].cpu().numpy()
        if nbytes and phase:
            assert got[0] >> (8 - phase) == 0, "bits before bit_phase must be zero"
        first = int(offs[i] >> 3)
        body[first : first + nbytes] |= got
        if bits[i]:
            phases.append(phase)
    return header, body.tobytes(), phases


def test_pack_shards_at_every_bit_phase_match_the_oracle(codec):
    data = _text(200_003)
    want = _oracle_et(data)
    seen = set()
    for world in (2, 3, 8):
        for shift in range(16):  # cuts at every residue mod 16: the kernels' 16-byte loads start anywhere
            per = data.size // world
            cuts = [0] + [r * per + shift + 3 * r for r in range(1, world)] + [data.size]
            header, body, phases = _pack_in_shards(codec, data, cuts)
            assert header + body == want, (world, shift)
            seen.update(phases)
    assert seen == set(range(8)), seen


def test_pack_shards_tiny_dropped_and_deep(codec):
    rng = np.random.default_rng(12)
    # shards shorter than one byte of output (1..3 symbols of 3-4 bits), several of them inside one byte
    data = _text(5000, seed=2)
    cuts = [0, 1, 2, 4, 5, 7, 2000, 2001, 2003, 4999, 5000]
    header, body, _ = _pack_in_shards(codec, data, cuts)
    assert header + body == _oracle_et(data)
    # all 256 byte values: the most frequent one gets no code (encode.zig:70) - shards that start or end with runs of it,
    # and one shard that consists of nothing else (zero bits)
    data = np.concatenate([rng.integers(0, 256, 30000, dtype=np.uint8), np.full(5000, 255, np.uint8),
                           rng.integers(0, 255, 30000, dtype=np.uint8), np.full(64, 255, np.uint8)])
    assert et.build_codebook(oracle.histogram(data)).code[255].length == 0
    want = _oracle_et(data)
    for cuts in ([0, 30000, 35000, 65000, data.size], [0, 29990, 30010, 34990, 35003, data.size], [0, 31000, 33000, data.size]):
        header, body, _ = _pack_in_shards(codec, data, cuts)
        assert header + body == want, cuts
    # every case of the single-GPU suite, cut in three
    for name, case in make_cases().items():
        if np.unique(case).size < 2:
            continue
        cuts = [0, case.size // 3, (2 * case.size) // 3 + 1, case.size]
        header, body, _ = _pack_in_shards(codec, case, cuts)
        assert header + body == _oracle_et(case), name
    # codes of 32 bits straddling shard seams
    data = _fib32()
    assert et.build_codebook(oracle.histogram(data)).max_length == 32
    cuts = [0, 1_000_001, 1_000_002, 4_000_013, 9_000_000, data.size]
    header, body, _ = _pack_in_shards(codec, data, cuts)
    assert header + body == _oracle_et(data)
    # codes of 33 bits (the wide kernel): shards at every bit phase, shards that begin or end with a 33-bit code, and one
    # that holds nothing else
    data = _chain33()
    _, length = oracle.build_dictionary(oracle.histogram(data))
    assert int(length.max()) == 33
    bounds = _boundaries(data)
    at_phase = [t + int(np.flatnonzero(bounds[t : t + 256] % 8 == ph)[0]) for ph, t in zip(range(8), range(1_000_003, 14_000_000, 1_600_000))]
    d0, d1 = (int(x) for x in np.flatnonzero(length[data] == 33))
    want = _oracle_et(data)
    seen = set()
    for cuts in ([0] + at_phase + [data.size], sorted({0, d0, d0 + 1, d1 - 5, d1 + 1, data.size})):
        header, body, phases = _pack_in_shards(codec, data, cuts)
        assert header + body == want, cuts
        seen.update(phases)
    assert seen == set(range(8)), seen


def _boundaries(data):
    """Bit position of every codeword boundary of the oracle's body for `data` (len = symbols + 1)."""
    _, length = oracle.build_dictionary(oracle.histogram(data))
    return np.concatenate([[0], np.cumsum(length[data].astype(np.int64))])


def _unpack_in_shards(codec, data, world, expect_guess_right):
    import torch

    stream = _oracle_et(data)[4:]
    d = et.parse_header(stream)
    body = np.frombuffer(stream, dtype=np.uint8)[d.body_offset :]
    bounds = _boundaries(data)
    assert (bounds[-1] + 7) // 8 == body.size
    cuts = sharded.body_cuts(body.size, world)
    text, redone = [], 0
    for r in range(world):
        if cuts[r] == cuts[r + 1]:
            continue
        s = max(cuts[r] - sharded.LEAD_IN, 0) if r else 0
        t = min(cuts[r + 1] + sharded.LOOK_AHEAD, body.size) if r + 1 < world else body.size
        rng_dev = torch.from_numpy(body[s:t].copy()).cuda()
        out = torch.zeros(8 * (t - s) + 64, dtype=torch.uint8, device="cuda")
        own_lo, own_hi = cuts[r] - s, cuts[r + 1] - s
        # the truth: first boundary at or after each cut, symbols that begin in between
        i_lo = int(np.searchsorted(bounds, cuts[r] * 8, side="left"))
        i_hi = int(np.searchsorted(bounds, cuts[r + 1] * 8, side="left")) if r + 1 < world else data.size
        true_entry = int(bounds[i_lo]) - s * 8
        true_exit = (int(bounds[i_hi]) - s * 8) if r + 1 < world else None
        n, entry, exit_ = codec.unpack_shard_dev(rng_dev.data_ptr(), t - s, own_lo, own_hi, d, 0 if r == 0 else -1, out.data_ptr(), out.numel())
        if entry != true_entry:  # the run-up had not locked on (slowly synchronising codes): again from the true boundary
            assert not expect_guess_right, (r, entry, true_entry)
            redone += 1
            n, entry, exit_ = codec.unpack_shard_dev(rng_dev.data_ptr(), t - s, own_lo, own_hi, d, true_entry, out.data_ptr(), out.numel())
        assert entry == true_entry, (r, entry, true_entry)
        if true_exit is not None:
            assert n == i_hi - i_lo and exit_ == true_exit, (r, n, i_hi - i_lo, exit_, true_exit)
        else:  # the last shard does not know body_len: the final pad bits may read as a few more (short) codes
            assert i_hi - i_lo <= n <= i_hi - i_lo + 7, (r, n, i_hi - i_lo)
        text.append(out[: i_hi - i_lo].cpu().numpy())
    assert np.array_equal(np.concatenate(text), data)
    return redone


def test_unpack_shards_entry_exit_and_text(codec):
    thr_text = _text(1_500_007)
    for world in (2, 3, 8):
        assert _unpack_in_shards(codec, thr_text, world, expect_guess_right=True) == 0
    # 7/8-bit codes: a wrong parse survives for kilobytes, so 64 bytes of lead-in are not enough for most shards
    uni = np.random.default_rng(4).integers(1, 256, 600_011, dtype=np.uint8)
    redone = sum(_unpack_in_shards(codec, uni, world, expect_guess_right=False) for world in (3, 8))
    assert redone > 0
    # the lane-interleaved decoder on the same shards (it is what long streams take)
    codec.set_tuning(_abi.TUNE_LANE_MIN_BYTES, 0)
    try:
        for world in (2, 8):
            assert _unpack_in_shards(codec, thr_text, world, expect_guess_right=True) == 0
        deep = _fib32()
        assert _unpack_in_shards(codec, deep, 3, expect_guess_right=True) == 0
    finally:
        codec.set_tuning(_abi.TUNE_LANE_MIN_BYTES, -1)


def test_unpack_shard_reports_no_space(codec):
    import torch

    data = _text(100_000)
    stream = _oracle_et(data)[4:]
    d = et.parse_header(stream)
    body = torch.from_numpy(np.frombuffer(stream, dtype=np.uint8)[d.body_offset :].copy()).cuda()
    out = torch.zeros(data.size, dtype=torch.uint8, device="cuda")
    with pytest.raises(et.EntreepyError) as e:
        codec.unpack_shard_dev(body.data_ptr(), body.numel(), 0, body.numel(), d, 0, out.data_ptr(), 1000)
    assert e.value.name == "NoSpaceLeft"


# ---------------------------------------------------------------- the whole protocol, ranks as threads on one GPU
class ThreadComm:
    """sharded.Comm's three exchanges between threads of one process (what NCCL does between ranks)."""

    def __init__(self, world, rank, shared):
        self.world, self.rank, self.s = world, rank, shared

    def _exchange(self, value):
        self.s["slots"][self.rank] = value
        self.s["barrier"].wait()
        got = list(self.s["slots"])
        self.s["barrier"].wait()
        return got

    def allgather_array(self, values):
        return np.stack(self._exchange(np.asarray(values, dtype=np.int64).copy()))

    def allgather_ints(self, values):
        return [list(v) for v in self._exchange(list(values))]

    def all_to_all_bytes(self, send, send_splits, recv_splits):
        import torch

        parts, so = [], 0
        for q in range(self.world):
            parts.append(send[so : so + int(send_splits[q])].clone())
            so += int(send_splits[q])
        torch.cuda.synchronize()
        everyone = self._exchange(parts)
        mine = [everyone[q][self.rank] for q in range(self.world)]
        assert [int(m.numel()) for m in mine] == [int(x) for x in recv_splits]
        return torch.cat(mine) if mine else torch.empty(0, dtype=torch.uint8, device=send.device)


def _run_ranks(world, data, results, native=False, decode=True):
    """results[rank] = (header, the rank's own body bytes, total bytes, all-gathers of the native encode (None when not
    native)) + with decode: (text offset, text, rounds).  decode=False stops after the encode (codes over 32 bits)."""
    import torch

    shared = {"slots": [None] * world, "barrier": threading.Barrier(world)}
    errors = []

    def rank_main(rank):
        try:
            torch.cuda.set_device(0)
            with et.Codec(0) as codec:
                plan = sharded.ShardPlan(data.size, world, rank)
                tcomm = ThreadComm(world, rank, shared)
                gathers = [0]

                def allgather(send):
                    gathers[0] += 1
                    return b"".join(tcomm._exchange(send))

                if native:  # the protocol inside the library; its all-gathers come back to this process through a callback
                    ncomm = codec.comm_callback(rank, world, allgather)
                    coder = sharded.NativeShardedCodec(codec, plan, ncomm, tcomm)
                else:
                    coder = sharded.ShardedCodec(sharded.GpuBackend(codec), plan, tcomm)
                t_in = torch.from_numpy(data[plan.lo : plan.hi].copy()).cuda()
                t_body = torch.zeros(plan.n_local * 4 + 4096, dtype=torch.uint8, device="cuda")
                torch.cuda.synchronize()
                res = coder.encode(t_in, t_body)
                mine = t_body[res.own_lo - res.first_byte : res.own_hi - res.first_byte].cpu().numpy().tobytes()
                encoded = (res.header, mine, res.total_bytes, gathers[0] if native else None)
                if not decode:
                    results[rank] = encoded
                    if native:
                        codec.comm_destroy(ncomm)
                    return
                t_range = coder.scatter_body(res, t_body)
                cuts, ranges = coder.decode_ranges(res.body_bytes)
                s, t = ranges[rank]
                t_out = torch.zeros(8 * max(t - s, 1) + 64, dtype=torch.uint8, device="cuda")
                torch.cuda.synchronize()
                dres = coder.decode(res.header[4:], res.body_bytes, t_range, t_out)
                results[rank] = encoded + (dres.offset, t_out[: dres.n_local].cpu().numpy().tobytes(), dres.rounds)
                if native:
                    codec.comm_destroy(ncomm)
        except BaseException as exc:  # noqa: BLE001 - reported by the test thread
            errors.append((rank, exc))
            shared["barrier"].abort()

    threads = [threading.Thread(target=rank_main, args=(r,)) for r in range(world)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    if errors:
        raise errors[0][1]


def _check_protocol(world, name, data, native=False, decode=True, encode_gathers=None):
    """The sharded .et against the oracle's, then (decode) the text.  encode_gathers: the all-gathers every rank's native
    encode must make.  -> the largest decode rounds count."""
    results = [None] * world
    _run_ranks(world, data, results, native, decode)
    want = _oracle_et(data)
    header = results[0][0]
    assert header + b"".join(r[1] for r in results) == want, f"{name}: sharded .et differs from the oracle's (world {world})"
    assert all(r[2] == len(want) for r in results)
    if encode_gathers is not None:
        assert [r[3] for r in results] == [encode_gathers] * world, (name, world, [r[3] for r in results])
    if not decode:
        return None
    lossless = np.unique(data).size < 256  # the reference drops a symbol when all 256 occur (SURVEY §0.2)
    expect = data.tobytes() if lossless else oracle.decode(np.frombuffer(want, np.uint8)[4:], data.size).tobytes()
    full = bytearray(len(expect))
    for *_, off, chunk, _ in results:
        full[off : off + len(chunk)] = chunk
    assert sum(len(r[5]) for r in results) == len(expect), name
    assert bytes(full) == expect, f"{name}: sharded decode differs (world {world})"
    return max(r[6] for r in results)


@pytest.mark.parametrize("world", [2, 3, 8])
def test_sharded_protocol_on_real_kernels(world):
    rng = np.random.default_rng(100 + world)
    assert _check_protocol(world, "text", _text(2_000_003, seed=world)) == 1
    rounds = _check_protocol(world, "uniform255", rng.integers(1, 256, 700_001, dtype=np.uint8))
    assert world == 2 or rounds >= 2  # 7/8-bit codes: 64 bytes of lead-in rarely lock on, the repeat loop runs
    _check_protocol(world, "all256", np.concatenate([rng.integers(0, 256, 90_000, dtype=np.uint8), np.full(3000, 255, np.uint8),
                                                     rng.integers(0, 256, 50_000, dtype=np.uint8)]))
    _check_protocol(world, "tiny", _text(50 + world))
    for name, case in make_cases().items():
        if np.unique(case).size >= 2 and case.size >= 16 * world:
            _check_protocol(world, name, case)
    if world == 3:
        _check_protocol(world, "fib32", _fib32())


@pytest.mark.parametrize("world", [2, 3, 8])
def test_sharded_protocol_inside_the_library(world):
    """et_encode_sharded_dev / et_decode_sharded_dev (exchanges through an et_comm) against the oracle."""
    rng = np.random.default_rng(200 + world)
    assert _check_protocol(world, "text", _text(2_000_003, seed=10 + world), native=True, encode_gathers=1) == 1
    rounds = _check_protocol(world, "uniform255", rng.integers(1, 256, 700_001, dtype=np.uint8), native=True)
    assert world == 2 or rounds >= 2
    _check_protocol(world, "all256", np.concatenate([rng.integers(0, 256, 90_000, dtype=np.uint8), np.full(3000, 255, np.uint8),
                                                     rng.integers(0, 256, 50_000, dtype=np.uint8)]), native=True)
    # the second exchange of the encoder: rank 1 starts inside a byte with a run of the symbol that has no code
    _check_protocol(world, "all256_run_at_cut", _dropped_run_at_cut(world), native=True, encode_gathers=2)
    if world > 2:  # ... or with a code of 33 bits; the decoder refuses such codes (the reference's cannot hold them)
        _check_protocol(world, "chain33", _chain33_at_cuts(world), native=True, decode=False, encode_gathers=2)
    _check_protocol(world, "tiny", _text(50 + world), native=True)
    for name, case in make_cases().items():
        if np.unique(case).size >= 2 and case.size >= 16 * world:
            _check_protocol(world, name, case, native=True)
    if world == 3:
        _check_protocol(world, "fib32", _fib32(), native=True)
