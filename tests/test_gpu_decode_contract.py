"""Every decode route at the edges of its output, against the oracle.  Run with -m gpu on a B200.

For a stream s and a capacity cap, the oracle's text is full = oracle.decode(s, body_len): body_len symbols, or as many
as the bits of the body hold when that is fewer (symbols made of the zero padding of the last byte included).  Every
route must return NoSpaceLeft when len(full) > cap and otherwise OK with out_len = len(full), and it must write exactly
full[:cap] into the caller's buffer: no byte before it, no byte after it, whatever the buffer held.  The routes are the
decoders et_decode_dev picks from (per-thread chunks, the fixed_len closed form, transfer functions, repair rounds, the
lane-interleaved decoder), et_decode_batch_dev (its own kernels, and the streams it hands to unpack_dev) and the host
et_decode in one slice or several.  Each test first shows that its streams take the route it is named after: a change
of routing changes the kernel launches or the rounds of a call.
"""
import ctypes
import json
import os

import numpy as np
import pytest

import entreepy_b200 as et
from conftest import GOLDEN
from entreepy_b200 import _abi, synth
from oracle import oracle

pytestmark = pytest.mark.gpu

WRITE = _abi.FLAG_WRITE_OUTPUT
OK, NO_SPACE = _abi.OK, _abi.ERR_NO_SPACE
GUARD = 64                  # bytes on both sides of every output that must keep the fill
FILLS = (0xA5, 0x00)        # alternate from case to case: a kernel that writes zeros, or skips a zero, fails one of them
LANE_BYTES, REGION_CHUNKS, TILE_CHUNKS = 132, 32, 256  # lane decoder chunks and regions; chunks of a batch tile

# Kernel launches of one et_decode_dev call (a B200, 148 SMs), and the rounds it reports.  Every call builds the tables
# first (build_tables_kernel, build_sub_tables_kernel).  Then
#   chunks    sync 0 and sync 1, sum, scan and write: 2 + 5, the guesses plus one repair round;
#   fixed     the same launches; the entries follow in closed form;
#   transfer  the chunks' transfer functions, three compose kernels, sum, scan and write: 2 + 4 + 3, no rounds; chunks
#             of 512 bytes have enough transfer threads for the shared-memory kernel, which needs its table first: one more;
#   lanes     the lane tables, sync 0, the edge check and sync 1, the region sums, scan and apply, the write walk
#             (launch_unpack_lanes): 2 + 8.
REACH = {
    "chunks": (7, 2),
    "fixed": (7, 2),
    "transfer256": (9, 1),
    "transfer512": (10, 1),
    "lanes": (10, 2),
}


def _pin(what, got, want):
    assert got == want, (what, got, want)


def _reach(route, launches, rounds):
    _pin(route, (launches, rounds), REACH[route])


def _repair_reach(launches, rounds, write_walks):
    # the fixpoint rounds, four per host visit (one launch each), around write_walks of sum, scan and write
    assert rounds > 2, rounds
    _pin(("repair", rounds, write_walks), launches, 4 + (rounds - 2) + 3 * write_walks)


# ---------------------------------------------------------------- streams and what the oracle reads from them
def _encode(data):
    return oracle.encode(data, cap=9000 + 5 * int(np.asarray(data).size)).tobytes()[4:]


def _with_body_len(s, body_len):
    return s[:1] + int(body_len).to_bytes(4, "big") + s[5:]


class Stream:
    """file[4..] of an .et, every symbol its body holds (the oracle, as if body_len were unbounded), and the body bit at
    which each of them ends."""

    def __init__(self, s):
        self.s = bytes(s)
        d = et.parse_header(self.s)
        self.body_len, self.off = int(d.body_len), int(d.body_offset)
        self.min_len, self.max_len = int(d.min_length), int(d.max_length)
        self.body_bytes = len(self.s) - self.off
        lengths = np.zeros(256, dtype=np.uint8)
        zero = []
        for i in range(d.n_entries):
            lengths[d.symbol[i]] = d.length[i]
            if int(d.code[i]) == 0:
                zero.append(int(d.length[i]))
        self.zero_code = min(zero, default=0)  # length of the all-zero code: padding bits decode to it
        self.all = oracle.decode(_with_body_len(self.s, 0xFFFFFFFF), self.body_bytes * 8 // self.min_len + 8)
        self.ends = np.cumsum(lengths[self.all], dtype=np.int64)
        self.held = int(self.all.size)

    def held_in(self, body_bytes):
        """Symbols whose code ends inside the first body_bytes bytes of the body."""
        return int(np.searchsorted(self.ends, body_bytes * 8, side="right"))

    def first_at(self, bit):
        """Index of the first symbol that begins at or after body bit `bit`."""
        return 0 if bit <= 0 else min(int(np.searchsorted(self.ends, bit, side="left")) + 1, self.held)

    def expect(self, body_len, body_bytes, cap):
        """-> (status, bytes written, out_len) by the oracle's rule."""
        text = min(body_len, self.held if body_bytes == self.body_bytes else self.held_in(body_bytes))
        return (NO_SPACE, cap, 0) if text > cap else (OK, text, text)


def _sms():
    import torch

    return torch.cuda.get_device_properties(0).multi_processor_count


def _chunk_bytes(st, lane_min=None):
    """unpack_chunk_bytes for st's body: the chunk grid every decoder walks (132 bytes: the lane decoder)."""
    sms, spread, n = _sms(), st.max_len - st.min_len, st.body_bytes
    lane_min = sms * 3 * 4224 if lane_min is None else max(lane_min, 2 * 4224)
    if spread > 2 and n >= lane_min:
        return LANE_BYTES
    if spread <= 2 and st.max_len <= 16:
        cb = 512
        while cb > 256 and n // cb * st.max_len < sms * 4096:
            cb >>= 1
        return cb
    cb = 4096 if spread <= 1 else 1024 if spread == 2 else 256
    floor = 256 if cb > 256 else 32
    while cb > floor and n // cb < sms * 2048:
        cb >>= 1
    return cb


def _grid(st, cb, mis, every=1):
    """Symbol indices at the chunk boundaries a decoder cuts st's body at (the body's first byte at mis past a 16-byte
    boundary; chunk k begins at bit k * cb * 8 of that boundary): the first symbol that begins in chunk k and its two
    neighbours, for the second, a middle and the last of every `every`-th chunk."""
    last = (mis + st.body_bytes - 1) // cb
    ks = sorted({k // every * every for k in (every, last // 2, last)} - {0})
    cuts = []
    for k in ks:
        i = st.first_at(k * cb * 8 - mis * 8)
        cuts += [i - 1, i, i + 1]
    return [c for c in cuts if 0 < c <= st.body_len], ks


def _cases(st, cb, mis, every=1):
    """(body_len, body bytes, cap) for st whose body sits mis bytes past a 16-byte boundary.  The first case is the whole
    text into a buffer of its size (the one the route's launches are pinned on)."""
    B, N, n = st.body_len, st.held, st.body_bytes
    cuts, ks = _grid(st, cb, mis, every)
    if every > 1:  # the chunk boundaries as well
        cuts += _grid(st, cb, mis)[0]
    out = [(B, n, cap) for cap in (B, 0, 1, B - 1, B + 4096)]
    out += [(B, n, cap) for cap in cuts]
    for bl in (N + 1, N + 7, N + 10**6):  # the body holds fewer symbols than body_len claims; cap == N fits
        out += [(bl, n, cap) for cap in (N - 1, N, N + 1)]
    last_start = (mis + n - 1) // cb * cb - mis  # the body cut at byte phases inside its last chunk
    for t in sorted({n - 1, n - 3, n - 6, (last_start + n) // 2, last_start + 1}):
        if last_start < t < n:
            h = st.held_in(t)
            out += [(B, t, cap) for cap in (h - 1, h, B)]
    mid = st.first_at(ks[len(ks) // 2] * cb * 8 - mis * 8) + 5  # the body holds more: body_len ends inside a chunk
    for bl in (N - 1, mid):
        out += [(bl, n, cap) for cap in (bl - 1, bl, bl + 4096)]
    out += [(0, n, 0), (0, n, B)]
    return [(bl, t, cap) for bl, t, cap in out if cap >= 0]


def _dev_call(codec, d_in, n, d_out, cap):
    got = ctypes.c_size_t(0)
    rc = codec._lib.et_decode_dev(codec._ctx, d_in, n, d_out, cap, ctypes.byref(got), WRITE, None)
    return rc, got.value


def _first_wrong(got, fill, at, want, m):
    """None when got holds fill outside [at, at + m) and want[:m] inside, else the first index that does not."""
    exp = np.full(got.size, fill, dtype=np.uint8)
    exp[at:at + m] = want[:m]
    bad = np.flatnonzero(got != exp)
    return None if bad.size == 0 else (int(bad[0]), int(got[bad[0]]), int(exp[bad[0]]), int(bad.size))


def _check_dev(out, fill, at, want_dev, m, what):
    import torch

    ok = bool((out[:at] == fill).all()) and bool((out[at + m:] == fill).all()) and torch.equal(out[at:at + m], want_dev[:m])
    if not ok:
        raise AssertionError((what, _first_wrong(out.cpu().numpy(), fill, at, want_dev[:m].cpu().numpy(), m)))


def _run_dev(codec, st, phase, cases, reach):
    """et_decode_dev on every case: st at byte `phase` of a fresh device buffer, body_len rewritten in place, one
    poisoned output buffer at output offsets 0..15.  reach(launches, rounds) checks the first case."""
    import torch

    src = torch.zeros(phase + len(st.s) + 16, dtype=torch.uint8, device="cuda")
    src[phase:phase + len(st.s)] = torch.from_numpy(np.frombuffer(st.s, dtype=np.uint8).copy()).cuda()
    want = torch.from_numpy(st.all).cuda()
    out = torch.empty(GUARD + 16 + max(c for _, _, c in cases) + GUARD, dtype=torch.uint8, device="cuda")
    body_len = st.body_len
    for i, (bl, t, cap) in enumerate(cases):
        if bl != body_len:
            src[phase + 1:phase + 5] = torch.tensor(list(int(bl).to_bytes(4, "big")), dtype=torch.uint8)
            body_len = bl
        fill, at = FILLS[i % 2], GUARD + i % 16
        out.fill_(fill)
        torch.cuda.synchronize()  # the library works on its own stream
        before = codec.kernel_launches
        rc, got = _dev_call(codec, src.data_ptr() + phase, st.off + t, out.data_ptr() + at if cap else None, cap)
        if i == 0:
            reach(codec.kernel_launches - before, codec.last_decode_rounds)
        status, m, out_len = st.expect(bl, t, cap)
        what = (i, st.body_len, st.held, bl, t, cap)
        assert (rc, got) == (status, out_len), (what, rc, got)
        _check_dev(out, fill, at, want, m, what)


def _text_thresholds(space_factor=1):
    man = json.load(open(os.path.join(GOLDEN, "manifest.json")))
    w = list(synth.text_weights(man["midsummer_histogram"]))
    w[32] *= space_factor
    return synth.thresholds_from_weights(w)


def _zero_code_text(n, seed):
    """Text whose dictionary gives the all-zero pattern a short code (space three times as frequent as in the fixture:
    its code is 0), cut to the longest prefix of at most n bytes whose last byte ends in zero padding of at least that
    code's length, so that the body holds more symbols than body_len: the padding decodes to spaces."""
    data = synth.generate(n, _text_thresholds(3), seed=seed)
    for m in range(n, n - 64, -1):
        st = Stream(_encode(data[:m]))
        if st.held > st.body_len:
            assert 1 <= st.zero_code <= 3 and st.all[:m].tobytes() == data[:m].tobytes(), (m, st.zero_code)
            return st
    raise AssertionError("no prefix ends in padding that decodes")


def _fixed(k, n, seed):
    """2^k equiprobable symbols (a complete code of k bits; 0..0 is one of them), cut so that the padding decodes."""
    rng = np.random.default_rng(seed)
    syms = rng.permutation(256)[: 1 << k].astype(np.uint8)
    data = syms[rng.permutation(np.arange(n) % (1 << k))]  # equal counts: every code has k bits
    for m in range(n, n - 64, -1):
        st = Stream(_encode(data[:m]))
        assert st.min_len == st.max_len == k, k
        if st.held > st.body_len:
            return st
    raise AssertionError(k)


def _uniform255(n, seed):
    return Stream(_encode(np.random.default_rng(seed).integers(1, 256, n, dtype=np.uint8)))


def _codes_3_to_7(n, seed):
    """Code lengths 3..7: too wide a spread for transfer functions, slow to synchronise (test_gpu_batch)."""
    rng = np.random.default_rng(seed)
    w = np.ones(48)
    w[:8] = 9.0
    return Stream(_encode(rng.choice(48, n, p=w / w.sum()).astype(np.uint8)))


@pytest.fixture(scope="module")
def texts():
    return {"10k": _zero_code_text(10_007, 1), "300k": _zero_code_text(300_007, 2), "2m": _zero_code_text(2_000_003, 3)}


@pytest.fixture(scope="module")
def uniform():
    # 1 MB of body: 256-byte chunks; about 40 MB: 512-byte chunks (body / 512 x max_len >= SMs x 4096)
    return {"1m": _uniform255(1_000_003, 4), "40m": _uniform255(40_000_037, 5)}


@pytest.fixture(scope="module")
def lane_text():
    st = _zero_code_text(6_000_011, 6)
    assert _chunk_bytes(st) == LANE_BYTES  # a body above SMs x 3 x 4224 bytes
    return st


def _route(codec, st, reach, phase, lane_min=None, every=1):
    cb = _chunk_bytes(st, lane_min)
    _run_dev(codec, st, phase, _cases(st, cb, (phase + st.off) % 16, every), reach)
    return cb


# ---------------------------------------------------------------- et_decode_dev
def test_per_thread_chunks_short_text(codec, texts):
    for phase, st in zip((0, 5, 11), texts.values()):
        assert st.max_len - st.min_len > 2 and _chunk_bytes(st) != LANE_BYTES
        _route(codec, st, lambda n, r: _reach("chunks", n, r), phase)


def test_fixed_len_closed_form(codec):
    for k, phase in ((3, 7), (5, 0), (7, 13)):
        st = _fixed(k, 1_000_000 + 1024 * k, k)
        _route(codec, st, lambda n, r: _reach("fixed", n, r), phase)


def test_transfer_functions(codec, uniform):
    for (name, st), phase, cb in zip(uniform.items(), (3, 9), (256, 512)):
        assert st.max_len - st.min_len <= 2 and _chunk_bytes(st) == cb, name
        _route(codec, st, lambda n, r: _reach(f"transfer{cb}", n, r), phase)


def test_repair_rounds(codec, uniform):
    rng = np.random.default_rng(8)
    codec.set_tuning(_abi.TUNE_NO_TRANSFER, 1)
    try:
        # 256-byte chunks: a write walk, the rounds, a second one; 512-byte chunks settle before their only write walk
        for (name, st), walks in zip(uniform.items(), (2, 1)):
            _route(codec, st, lambda n, r: _repair_reach(n, r, walks), int(rng.integers(0, 16)))
    finally:
        codec.set_tuning(_abi.TUNE_NO_TRANSFER, 0)
    st = _codes_3_to_7(1 << 20, 9)
    assert _chunk_bytes(st) == 32
    _route(codec, st, lambda n, r: _repair_reach(n, r, 2), 6)


def test_lane_decoder(codec, texts, lane_text):
    codec.set_tuning(_abi.TUNE_LANE_MIN_BYTES, 0)
    try:
        assert _route(codec, texts["300k"], lambda n, r: _reach("lanes", n, r), 2, lane_min=0, every=REGION_CHUNKS) == LANE_BYTES
    finally:
        codec.set_tuning(_abi.TUNE_LANE_MIN_BYTES, -1)
    assert _route(codec, lane_text, lambda n, r: _reach("lanes", n, r), 14, every=REGION_CHUNKS) == LANE_BYTES


# ---------------------------------------------------------------- et_decode_batch_dev
def _run_batch(codec, streams, every):
    """Every case of every stream as one item of a single batch call, each into its own stretch of one poisoned buffer.
    -> kernel launches of the call, its rounds, and items per stream."""
    import torch

    items, checks, per_stream = [], [], []
    srcs = []
    for j, st in enumerate(streams):
        phase = (3 * j + 1) % 16
        cases = _cases(st, _chunk_bytes(st), (phase + st.off) % 16, every)
        per_stream.append(len(cases))
        copies = {}
        for bl, t, cap in cases:
            if bl not in copies:
                src = torch.zeros(phase + len(st.s) + 16, dtype=torch.uint8)
                src[phase:phase + len(st.s)] = torch.frombuffer(bytearray(_with_body_len(st.s, bl)), dtype=torch.uint8)
                copies[bl] = src.cuda()
                srcs.append(copies[bl])
            items.append((copies[bl].data_ptr() + phase, st.off + t, cap))
            checks.append((st, bl, t, cap))
    spans = [GUARD + k % 16 + cap + GUARD for k, (_, _, cap) in enumerate(items)]
    base = np.concatenate([[0], np.cumsum(spans)])
    for fill in FILLS:
        out = torch.full((int(base[-1]),), fill, dtype=torch.uint8, device="cuda")
        exp = np.full(int(base[-1]), fill, dtype=np.uint8)
        want = []
        for k, (st, bl, t, cap) in enumerate(checks):
            status, m, out_len = st.expect(bl, t, cap)
            at = int(base[k]) + GUARD + k % 16
            exp[at:at + m] = st.all[:m]
            want.append((status, out_len))
        torch.cuda.synchronize()
        before = codec.kernel_launches
        res = codec.decode_batch_dev([(d_in, n, out.data_ptr() + int(base[k]) + GUARD + k % 16 if cap else None, cap)
                                      for k, (d_in, n, cap) in enumerate(items)])
        launches, rounds = codec.kernel_launches - before, codec.last_decode_rounds
        for k, (st, bl, t, cap) in enumerate(checks):
            assert res[k] == want[k], (k, st.body_len, st.held, bl, t, cap, res[k], want[k])
        got = out.cpu().numpy()
        bad = np.flatnonzero(got != exp)
        if bad.size:
            k = int(np.searchsorted(base, bad[0], side="right")) - 1
            raise AssertionError(("item", k, checks[k][1:], "byte", int(bad[0] - base[k]), int(bad.size)))
    return launches, rounds, per_stream


def test_batch_kernels(codec, texts):
    # Every item is decoded by the batch kernels in one group: text (32-byte chunks), the closed form, and codes of 3..7
    # bits whose guessed entries are wrong, so the group runs its fixpoint rounds and a second write walk.  Launches:
    # head gather, two table builds, sync 0 and 1, sum, scan and write (8), four per host visit of the rounds, and
    # three for the second write walk.  Cuts at the tiles (256 chunks) of every stream.
    streams = [texts["10k"], texts["300k"], _fixed(5, 300_000, 5), _codes_3_to_7(1 << 20, 10)]
    launches, rounds, _ = _run_batch(codec, streams, TILE_CHUNKS)
    assert rounds > 2, rounds
    _pin(("batch", rounds), launches, 11 + (rounds - 2))


def test_batch_hands_long_and_slow_streams_to_unpack_dev(codec, texts, lane_text, uniform):
    # A lane-length body and one that takes transfer functions go through unpack_dev, one item at a time, after the
    # group's kernels have decoded the text: 8 launches for the group, then each handed-off item's own.
    streams = [texts["10k"], lane_text, uniform["1m"]]
    launches, rounds, per = _run_batch(codec, streams, 1)
    _pin(("batch hand-off", per), launches, 8 + per[1] * REACH["lanes"][0] + per[2] * REACH["transfer256"][0])


# ---------------------------------------------------------------- et_decode (host buffers)
def _run_host(codec, st, cases, want_of, reach=None):
    """et_decode through Codec.decode_into on every case into one poisoned pinned buffer."""
    src = st.s
    if not isinstance(src, np.ndarray):
        src = codec.pinned(len(st.s))
        src[:] = np.frombuffer(st.s, dtype=np.uint8)
    out = codec.pinned(GUARD + 16 + max(c for _, _, c in cases) + GUARD)
    for i, (bl, t, cap) in enumerate(cases):
        src[1:5] = np.frombuffer(int(bl).to_bytes(4, "big"), dtype=np.uint8)
        fill, at = FILLS[i % 2], GUARD + i % 16
        out[:] = fill
        before = codec.kernel_launches
        try:
            rc, got = OK, codec.decode_into(src[:st.off + t], out[at:at + cap])
        except et.EntreepyError as e:
            rc, got = e.status, 0
        if i == 0 and reach:
            reach(codec.kernel_launches - before, codec.last_decode_rounds)
        status, m, out_len = st.expect(bl, t, cap)
        what = (i, st.body_len, st.held, bl, t, cap)
        assert (rc, got) == (status, out_len), (what, rc, got)
        assert (out[:at] == fill).all() and (out[at + m:] == fill).all(), (what, _first_wrong(out, fill, at, want_of(m), m))
        assert np.array_equal(out[at:at + m], want_of(m)), (what, _first_wrong(out, fill, at, want_of(m), m))


def test_host_decode_one_slice(codec, texts):
    st = texts["2m"]
    cases = _cases(st, _chunk_bytes(st), 0)  # the body is uploaded to the start of a device buffer
    _run_host(codec, st, cases, lambda m: st.all[:m], lambda n, r: _reach("chunks", n, r))


def test_host_decode_in_slices(codec):
    # A body over 128 MiB goes up, is decoded and comes down in 64 MiB slices: cuts inside slice 1 and slice 2, and a
    # body_len one past the symbols the body holds, with room for exactly those.
    import torch

    n = (3 << 26) * 4 // 3 + 12345
    dev = torch.empty(n, dtype=torch.uint8, device="cuda")
    codec.synth_dev(dev.data_ptr(), n, synth.SEED, 0, _text_thresholds())
    text = dev.cpu().numpy()
    h_in, h_et = codec.pinned(n), codec.pinned(n + 16384)
    h_in[:] = text
    size = codec.encode_into(h_in, h_et)
    s = h_et[4:size]
    d = et.parse_header(s)
    lengths = np.zeros(256, dtype=np.int64)
    zero = 0
    for i in range(d.n_entries):
        lengths[d.symbol[i]] = d.length[i]
        zero = int(d.length[i]) if int(d.code[i]) == 0 else zero
    bits = int(np.bincount(text, minlength=256) @ lengths)
    assert d.body_len == n and (bits + 7) // 8 == size - 4 - d.body_offset > (128 << 20)
    held = n + ((-bits) % 8) // zero  # the padding decodes to the all-zero code wherever it fits

    class Big:  # what the oracle reads from s: the text, then the padding symbols (Stream without the oracle's pass)
        body_len, off, body_bytes = n, int(d.body_offset), size - 4 - int(d.body_offset)

        def expect(self, body_len, body_bytes, cap):
            t = min(body_len, held)
            return (NO_SPACE, cap, 0) if t > cap else (OK, t, t)

    Big.s, Big.held = s, held
    cuts = []
    for frac, lo, hi in ((0.6, 64 << 20, 128 << 20), (0.95, 128 << 20, Big.body_bytes)):
        m = int(n * frac)
        at_bit = int(np.bincount(text[:m], minlength=256) @ lengths)
        assert lo * 8 + 512 < at_bit < hi * 8 - 512, (frac, at_bit)  # well inside the slice
        cuts += [m, m + 1]
    B, t = n, Big.body_bytes
    cases = [(B, t, cap) for cap in [B, 0, 1, B - 1, B + 4096] + cuts]
    cases += [(held + 1, t, cap) for cap in (held - 1, held)] + [(B - 1, t, B - 2), (B - 1, t, B - 1)]
    tail = np.zeros(held - n, dtype=np.uint8)
    for i in range(d.n_entries):
        if int(d.code[i]) == 0:
            tail[:] = d.symbol[i]

    def want_of(m):
        return text[:m] if m <= n else np.concatenate([text, tail[: m - n]])

    # the tables once, then each of the three slices through the lane decoder
    _run_host(codec, Big(), cases, want_of, lambda k, r: _pin("slices", (k, r), (2 + 3 * (REACH["lanes"][0] - 2), 2)))
