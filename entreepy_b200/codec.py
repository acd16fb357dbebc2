"""Host mirror of encode()/decode() (src/encode.zig:25, src/decode.zig:13) over the C ABI."""
import ctypes
from dataclasses import dataclass

import numpy as np

from . import _abi


class EntreepyError(Exception):
    """Zig error-union analogue: .name carries the reference's error name where one exists."""

    NAMES = {
        _abi.ERR_QUEUE_EMPTY: "QueueEmpty",      # queue.zig:5, raised from encode.zig:138
        _abi.ERR_NO_SPACE: "NoSpaceLeft",        # fixedBufferStream writer
        _abi.ERR_OUT_OF_MEMORY: "OutOfMemory",
        _abi.ERR_CUDA: "CudaError",
        _abi.ERR_NO_DEVICE: "NoDevice",
        _abi.ERR_CORRUPT: "Corrupt",
        _abi.ERR_TOO_LARGE: "TooLarge",
        _abi.ERR_UNSUPPORTED: "Unsupported",
        _abi.ERR_INVALID_ARG: "InvalidArgument",
    }

    def __init__(self, status, detail=""):
        self.status = status
        self.name = self.NAMES.get(status, f"Status{status}")
        super().__init__(f"{self.name}: {detail}" if detail else self.name)


@dataclass
class EncodeFlags:  # encode.zig:9-14
    write_output: bool = False
    print_output: bool = False
    debug: bool = False
    quiet: bool = True              # extension: the "X => Y" stderr line is off unless asked for
    no_scratch_limit: bool = False  # extension: lift the 7200+n bound of encode.zig:253

    def bits(self):
        return ((_abi.FLAG_WRITE_OUTPUT if self.write_output else 0) | (_abi.FLAG_PRINT_OUTPUT if self.print_output else 0)
                | (_abi.FLAG_DEBUG if self.debug else 0) | (_abi.FLAG_QUIET if self.quiet else 0)
                | (_abi.FLAG_NO_SCRATCH_LIMIT if self.no_scratch_limit else 0))


@dataclass
class DecodeFlags:  # decode.zig:7-11
    write_output: bool = False
    print_output: bool = False
    debug: bool = False
    quiet: bool = True
    validate: bool = False  # extension: the input validation main.zig:199 leaves as a TODO

    def bits(self):
        return ((_abi.FLAG_WRITE_OUTPUT if self.write_output else 0) | (_abi.FLAG_PRINT_OUTPUT if self.print_output else 0)
                | (_abi.FLAG_DEBUG if self.debug else 0) | (_abi.FLAG_QUIET if self.quiet else 0)
                | (_abi.FLAG_VALIDATE if self.validate else 0))


def _u8(data):
    if isinstance(data, np.ndarray):
        return np.ascontiguousarray(data, dtype=np.uint8)
    return np.frombuffer(bytes(data) if not isinstance(data, (bytes, bytearray, memoryview)) else data, dtype=np.uint8)


# ---------------------------------------------------------------- host-only steps (no GPU needed)
def build_codebook(counts):
    """E2-E4.  counts[256] -> _abi.Codebook; raises QueueEmpty when all counts are zero."""
    c = np.ascontiguousarray(counts, dtype=np.uint64)
    assert c.size == 256
    cb = _abi.Codebook()
    rc = _abi.load().et_build_codebook(c.ctypes.data, ctypes.byref(cb))
    if rc:
        raise EntreepyError(rc)
    return cb


def write_header(cb, n):
    """E5.  Header bytes (magic .. dictionary pad) for a text of n bytes."""
    L = _abi.load()
    size = L.et_header_size(ctypes.byref(cb))
    out = np.empty(size, dtype=np.uint8)
    got = ctypes.c_size_t(0)
    rc = L.et_write_header(ctypes.byref(cb), n, out.ctypes.data, size, ctypes.byref(got))
    if rc:
        raise EntreepyError(rc)
    return out[: got.value].tobytes()


def parse_header(et_after_magic):
    """D1+D2.  file[4..] -> _abi.Dictionary."""
    a = _u8(et_after_magic)
    d = _abi.Dictionary()
    rc = _abi.load().et_parse_header(a.ctypes.data, a.size, ctypes.byref(d))
    if rc:
        raise EntreepyError(rc)
    return d


# ---------------------------------------------------------------- device context
class Codec:
    """One et_ctx: a CUDA device, its streams and scratch.  Not thread-safe (one caller at a time)."""

    def __init__(self, device=0):
        self._lib = _abi.load()
        self._ctx = ctypes.c_void_p()
        rc = self._lib.et_ctx_create(device, ctypes.byref(self._ctx))
        if rc:
            self._ctx = None
            raise EntreepyError(rc, "et_ctx_create failed — a B200 (sm_100) is required, there is no CPU fallback")
        self.device = device
        self._pinned = []

    def close(self):
        for p in getattr(self, "_pinned", []):
            self._lib.et_free_pinned(p)
        self._pinned = []
        if getattr(self, "_ctx", None):
            self._lib.et_ctx_destroy(self._ctx)
            self._ctx = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _check(self, rc):
        if rc:
            raise EntreepyError(rc, (self._lib.et_last_error(self._ctx) or b"").decode("utf-8", "replace"))

    @property
    def kernel_launches(self):
        return int(self._lib.et_ctx_kernel_launches(self._ctx))

    @property
    def last_decode_rounds(self):
        """Passes over the chunk entries in the last decode (2: the guesses plus one repair round sufficed; more: fixpoint rounds were needed)."""
        return int(self._lib.et_ctx_last_decode_rounds(self._ctx))

    def last_stage_ms(self):
        ms = (ctypes.c_float * 4)()
        self._lib.et_ctx_last_stage_ms(self._ctx, ctypes.byref(ms))
        return list(ms)

    def set_tuning(self, key, value):
        """et_ctx_set_tuning: _abi.TUNE_LANE_MIN_BYTES (0 sends every stream through the lane-interleaved
        decoder, -1 restores the default), _abi.TUNE_DEBUG."""
        self._check(self._lib.et_ctx_set_tuning(self._ctx, key, int(value)))

    def set_output_fd(self, fd):
        self._check(self._lib.et_ctx_set_output_fd(self._ctx, fd))

    # ---- host buffers (the drop-in entry points)
    def histogram(self, data):
        a = _u8(data)
        counts = np.zeros(256, dtype=np.uint64)
        self._check(self._lib.et_histogram(self._ctx, a.ctypes.data, a.size, counts.ctypes.data))
        return counts

    def encode(self, text, flags=None, cap=None):
        """-> (n_bytes, et_file_bytes or None).  n_bytes is returned even on a dry run (encode.zig:336)."""
        flags = flags or EncodeFlags(write_output=True)
        a = _u8(text)
        if cap is None:
            cap = self._lib.et_encode_bound(a.size) if not flags.no_scratch_limit else 9 + 2560 + 8 * a.size + 8
        out = np.empty(cap if flags.write_output else 1, dtype=np.uint8)
        n = ctypes.c_size_t(0)
        self._check(self._lib.et_encode(self._ctx, a.ctypes.data, a.size, out.ctypes.data, cap, ctypes.byref(n), flags.bits()))
        return n.value, (out[: n.value] if flags.write_output else None)

    def decode(self, et_after_magic, flags=None, cap=None):
        """file[4..] -> (bytes_written, text or None)."""
        flags = flags or DecodeFlags(write_output=True)
        a = _u8(et_after_magic)
        if cap is None:
            cap = int(parse_header(a).body_len)
        out = np.empty(max(cap, 1), dtype=np.uint8)
        n = ctypes.c_size_t(0)
        self._check(self._lib.et_decode(self._ctx, a.ctypes.data, a.size, out.ctypes.data, cap, ctypes.byref(n), flags.bits()))
        return n.value, (out[: n.value] if flags.write_output else None)

    def pinned(self, nbytes):
        """uint8[nbytes] view of page-locked host memory (et_alloc_pinned); freed with the Codec."""
        p = ctypes.c_void_p()
        rc = self._lib.et_alloc_pinned(max(int(nbytes), 1), ctypes.byref(p))
        if rc:
            raise EntreepyError(rc, "et_alloc_pinned")
        self._pinned.append(p)
        return np.ctypeslib.as_array(ctypes.cast(p, ctypes.POINTER(ctypes.c_uint8)), shape=(max(int(nbytes), 1),))[:nbytes]

    def encode_into(self, text, out, flags=None):
        """et_encode with caller-owned host buffers (numpy uint8, ideally from .pinned()) -> file size."""
        flags = flags or EncodeFlags(write_output=True)
        n = ctypes.c_size_t(0)
        self._check(self._lib.et_encode(self._ctx, text.ctypes.data, text.size, out.ctypes.data, out.size, ctypes.byref(n), flags.bits()))
        return n.value

    def decode_into(self, et_after_magic, out, flags=None):
        """et_decode with caller-owned host buffers -> bytes written."""
        flags = flags or DecodeFlags(write_output=True)
        n = ctypes.c_size_t(0)
        self._check(self._lib.et_decode(self._ctx, et_after_magic.ctypes.data, et_after_magic.size, out.ctypes.data, out.size,
                                        ctypes.byref(n), flags.bits()))
        return n.value

    # ---- device-resident buffers (raw pointers: torch tensors' data_ptr(), cudaMalloc, ...)
    def histogram_dev(self, d_in, n, stream=None):
        counts = np.zeros(256, dtype=np.uint64)
        self._check(self._lib.et_histogram_dev(self._ctx, d_in, n, counts.ctypes.data, stream))
        return counts

    def encode_dev(self, d_in, n, d_out, cap, flags=_abi.FLAG_WRITE_OUTPUT, stream=None):
        got = ctypes.c_size_t(0)
        self._check(self._lib.et_encode_dev(self._ctx, d_in, n, d_out, cap, ctypes.byref(got), flags, stream))
        return got.value

    def decode_dev(self, d_in_after_magic, n, d_out, cap, flags=_abi.FLAG_WRITE_OUTPUT, stream=None):
        got = ctypes.c_size_t(0)
        self._check(self._lib.et_decode_dev(self._ctx, d_in_after_magic, n, d_out, cap, ctypes.byref(got), flags, stream))
        return got.value

    def decode_batch_dev(self, items, flags=_abi.FLAG_WRITE_OUTPUT, stream=None):
        """et_decode_batch_dev: items = [(d_in_after_magic, n, d_out, cap)] -> [(status, out_len)], one per item, each what
        decode_dev would have given that item (a failing item carries its status and does not raise).  Raises only when
        the call itself fails (a CUDA error or allocation failure)."""
        return self._batch(self._lib.et_decode_batch_dev, items, flags, stream)

    def encode_batch_dev(self, items, flags=_abi.FLAG_WRITE_OUTPUT, stream=None):
        """et_encode_batch_dev: items = [(d_in, n, d_out, cap)] -> [(status, out_len)], one per item, each what encode_dev
        would have given that item (a failing item carries its status and does not raise; out_len is the file size, also
        on a dry run).  Raises only when the call itself fails (a CUDA error or allocation failure)."""
        return self._batch(self._lib.et_encode_batch_dev, items, flags, stream)

    def _batch(self, entry, items, flags, stream):
        arr = (_abi.BatchItem * max(len(items), 1))()
        for k, (d_in, n, d_out, cap) in enumerate(items):
            arr[k] = _abi.BatchItem(d_in, n, d_out, cap, 0, 0)
        self._check(entry(self._ctx, arr, len(items), flags, stream))
        return [(int(arr[k].status), int(arr[k].out_len)) for k in range(len(items))]

    def shard_bits(self, counts, cb):
        c = np.ascontiguousarray(counts, dtype=np.uint64)
        return int(self._lib.et_shard_bits(c.ctypes.data, ctypes.byref(cb)))

    def pack_shard_dev(self, d_in, n, cb, bit_phase, shard_bits, d_out, cap, stream=None):
        """-> bytes touched by one shard packed at bit `bit_phase` of d_out[0]."""
        nbytes = ctypes.c_size_t(0)
        self._check(self._lib.et_pack_shard_dev(self._ctx, d_in, n, ctypes.byref(cb), bit_phase, shard_bits, d_out, cap,
                                                ctypes.byref(nbytes), stream))
        return nbytes.value

    def unpack_shard_dev(self, d_range, range_bytes, own_begin, own_end, dictionary, head_bit, d_out, cap, stream=None):
        """-> (symbols, entry_bit, exit_bit) of one shard of the body (see et_unpack_shard_dev)."""
        n, ent, ext = ctypes.c_uint64(0), ctypes.c_uint64(0), ctypes.c_uint64(0)
        self._check(self._lib.et_unpack_shard_dev(self._ctx, d_range, range_bytes, own_begin, own_end, ctypes.byref(dictionary),
                                                  head_bit, d_out, cap, ctypes.byref(n), ctypes.byref(ent), ctypes.byref(ext),
                                                  stream))
        return n.value, ent.value, ext.value

    # ---- the sharded path with its exchanges inside the library (et_encode_sharded_dev / et_decode_sharded_dev)
    @staticmethod
    def comm_unique_id():
        """128 bytes made by rank 0 (ncclGetUniqueId) for et_comm_create_nccl on every rank."""
        buf = (ctypes.c_uint8 * _abi.COMM_ID_BYTES)()
        rc = _abi.load().et_comm_unique_id(buf)
        if rc:
            raise EntreepyError(rc, "libnccl.so.2 is not available")
        return bytes(buf)

    def comm_nccl(self, unique_id, rank, world):
        """et_comm over NCCL (all ranks call this together: ncclCommInitRank)."""
        comm = ctypes.c_void_p()
        buf = (ctypes.c_uint8 * _abi.COMM_ID_BYTES).from_buffer_copy(unique_id)
        self._check(self._lib.et_comm_create_nccl(self._ctx, buf, rank, world, ctypes.byref(comm)))
        return comm

    def comm_callback(self, rank, world, allgather):
        """et_comm over a host transport: allgather(send: bytes) -> bytes of every rank's block in rank order."""
        def tramp(_user, send, recv, nbytes):
            try:
                got = allgather(ctypes.string_at(send, nbytes))
                assert len(got) == nbytes * world
                ctypes.memmove(recv, got, len(got))
                return 0
            except Exception:  # noqa: BLE001 - reported as a failed exchange
                return 1

        fn = _abi.ALLGATHER_FN(tramp)
        comm = ctypes.c_void_p()
        self._check(self._lib.et_comm_create_callback(self._ctx, rank, world, fn, None, ctypes.byref(comm)))
        self._keep = getattr(self, "_keep", []) + [fn]  # the C side holds the pointer
        return comm

    def comm_destroy(self, comm):
        self._lib.et_comm_destroy(comm)

    def encode_sharded_dev(self, comm, d_in, n_local, d_out, cap, flags=0, stream=None):
        """One rank of the sharded encoder -> _abi.ShardEncoded."""
        res = _abi.ShardEncoded()
        self._check(self._lib.et_encode_sharded_dev(self._ctx, comm, d_in, n_local, d_out, cap, ctypes.byref(res), flags, stream))
        return res

    def decode_sharded_dev(self, comm, header_after_magic, d_range, range_bytes, own_begin, own_end, starts_body, d_out, cap,
                           flags=0, stream=None):
        """One rank of the sharded decoder -> _abi.ShardDecoded."""
        h = _u8(header_after_magic)
        res = _abi.ShardDecoded()
        self._check(self._lib.et_decode_sharded_dev(self._ctx, comm, h.ctypes.data, h.size, d_range, range_bytes, own_begin, own_end,
                                                    1 if starts_body else 0, d_out, cap, ctypes.byref(res), flags, stream))
        return res

    def synth_dev(self, d_out, n, seed, first_index, thresholds, stream=None):
        t = np.ascontiguousarray(thresholds, dtype=np.uint32)
        assert t.size == 256
        self._check(self._lib.et_synth_dev(self._ctx, d_out, n, seed, first_index, t.ctypes.data, stream))


_default = None


def _codec():
    global _default
    if _default is None:
        _default = Codec(0)
    return _default


def encode(text, out_writer=None, flags=None):
    """encode(text, out_writer, flags) -> usize, as src/encode.zig:25 (allocator and std_out are implicit).

    out_writer is anything with .write(bytes) (the reference takes `anytype` with writeAll);
    it receives the whole .et file in one call (encode.zig:319) when flags.write_output."""
    flags = flags or EncodeFlags(write_output=out_writer is not None)
    n, data = _codec().encode(text, flags)
    if flags.write_output and out_writer is not None:
        out_writer.write(data.tobytes())
    return n


def decode(compressed_text, out_writer=None, flags=None):
    """decode(compressed_text, out_writer, flags) -> usize, as src/decode.zig:13.

    compressed_text is file[4..] (main.zig:204, test.zig:26)."""
    flags = flags or DecodeFlags(write_output=out_writer is not None)
    n, data = _codec().decode(compressed_text, flags)
    if flags.write_output and out_writer is not None:
        out_writer.write(data.tobytes())
    return n
