"""ctypes binding of libentreepy_b200.so (include/entreepy_b200.h).  Loads the in-tree library
and fails loudly when it is missing: there is no CPU implementation behind this package."""
import ctypes
import os

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ET_LIB") or os.path.join(PKG, "lib", "libentreepy_b200.so")  # ET_LIB: another build of the library, to compare two builds run for run

OK = 0
ERR_QUEUE_EMPTY, ERR_NO_SPACE, ERR_OUT_OF_MEMORY, ERR_CUDA, ERR_NO_DEVICE = 1, 2, 3, 4, 5
ERR_CORRUPT, ERR_TOO_LARGE, ERR_UNSUPPORTED, ERR_INVALID_ARG = 6, 7, 8, 9

FLAG_WRITE_OUTPUT, FLAG_PRINT_OUTPUT, FLAG_DEBUG = 0x1, 0x2, 0x4
FLAG_QUIET, FLAG_NO_SCRATCH_LIMIT, FLAG_VALIDATE, FLAG_TIMING = 0x100, 0x200, 0x400, 0x800
TUNE_LANE_MIN_BYTES, TUNE_DEBUG, TUNE_NO_TRANSFER = 1, 2, 5  # 3, 4 and 6 are retired

# every symbol include/entreepy_b200.h declares
SYMBOLS = [
    "et_abi_version", "et_strerror", "et_ctx_create", "et_ctx_destroy", "et_last_error", "et_ctx_set_output_fd",
    "et_ctx_kernel_launches", "et_ctx_last_stage_ms", "et_ctx_last_decode_rounds", "et_ctx_set_tuning", "et_alloc_pinned", "et_free_pinned", "et_build_codebook",
    "et_header_size", "et_write_header", "et_encode_bound", "et_parse_header", "et_histogram", "et_histogram_dev",
    "et_encode", "et_decode", "et_encode_dev", "et_decode_dev", "et_decode_batch_dev", "et_encode_batch_dev", "et_pack_shard_dev", "et_shard_bits",
    "et_unpack_shard_dev", "et_synth_dev", "et_comm_unique_id", "et_comm_create_nccl", "et_comm_create_callback", "et_comm_destroy",
    "et_encode_sharded_dev", "et_decode_sharded_dev",
]
COMM_ID_BYTES = 128
ALLGATHER_FN = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t)


class ShardEncoded(ctypes.Structure):
    _fields_ = [
        ("n_total", ctypes.c_uint64), ("total_bytes", ctypes.c_uint64), ("body_bytes", ctypes.c_uint64), ("bit_offset", ctypes.c_uint64),
        ("first_byte", ctypes.c_uint64), ("local_bytes", ctypes.c_uint64), ("own_lo", ctypes.c_uint64), ("own_hi", ctypes.c_uint64),
        ("header_len", ctypes.c_uint32), ("header", ctypes.c_uint8 * 4096),
    ]


class ShardDecoded(ctypes.Structure):
    _fields_ = [("n_local", ctypes.c_uint64), ("offset", ctypes.c_uint64), ("body_len", ctypes.c_uint64), ("rounds", ctypes.c_uint32)]


class BatchItem(ctypes.Structure):
    """et_batch_item: one stream of et_decode_batch_dev or one text of et_encode_batch_dev (device pointers; out_len and status
    are written by the call)."""
    _fields_ = [("d_in", ctypes.c_void_p), ("n", ctypes.c_size_t), ("d_out", ctypes.c_void_p), ("cap", ctypes.c_size_t),
                ("out_len", ctypes.c_size_t), ("status", ctypes.c_int)]


class Code(ctypes.Structure):
    _fields_ = [("data", ctypes.c_uint32), ("length", ctypes.c_uint8)]


class Codebook(ctypes.Structure):
    _fields_ = [
        ("code", Code * 256),
        ("n_symbols", ctypes.c_uint32),
        ("n_entries", ctypes.c_uint32),
        ("min_length", ctypes.c_uint32),
        ("max_length", ctypes.c_uint32),
        ("body_bits", ctypes.c_uint64),
    ]


class Dictionary(ctypes.Structure):
    _fields_ = [
        ("n_entries", ctypes.c_uint32),
        ("body_len", ctypes.c_uint32),
        ("body_offset", ctypes.c_uint64),
        ("symbol", ctypes.c_uint8 * 256),
        ("length", ctypes.c_uint8 * 256),
        ("code", ctypes.c_uint64 * 256),
        ("min_length", ctypes.c_uint32),
        ("max_length", ctypes.c_uint32),
        ("truncated", ctypes.c_uint32),
    ]


_lib = None


def load():
    """The shared library, loaded once.  Raises if it has not been built (python -m entreepy_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m entreepy_b200.build` "
            "(nvcc, sm_100a). entreepy_b200 has no CPU fallback."
        )
    L = ctypes.CDLL(LIB_PATH)
    vp, sz, u32, u64, i = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_uint32, ctypes.c_uint64, ctypes.c_int
    szp = ctypes.POINTER(ctypes.c_size_t)
    sig = {
        "et_abi_version": (i, []),
        "et_strerror": (ctypes.c_char_p, [i]),
        "et_ctx_create": (i, [i, ctypes.POINTER(vp)]),
        "et_ctx_destroy": (None, [vp]),
        "et_last_error": (ctypes.c_char_p, [vp]),
        "et_ctx_set_output_fd": (i, [vp, i]),
        "et_ctx_kernel_launches": (u64, [vp]),
        "et_ctx_last_stage_ms": (i, [vp, ctypes.POINTER(ctypes.c_float * 4)]),
        "et_ctx_last_decode_rounds": (u32, [vp]),
        "et_ctx_set_tuning": (i, [vp, i, ctypes.c_longlong]),
        "et_alloc_pinned": (i, [sz, ctypes.POINTER(vp)]),
        "et_free_pinned": (None, [vp]),
        "et_build_codebook": (i, [vp, ctypes.POINTER(Codebook)]),
        "et_header_size": (sz, [ctypes.POINTER(Codebook)]),
        "et_write_header": (i, [ctypes.POINTER(Codebook), u64, vp, sz, szp]),
        "et_encode_bound": (sz, [sz]),
        "et_parse_header": (i, [vp, sz, ctypes.POINTER(Dictionary)]),
        "et_histogram": (i, [vp, vp, sz, vp]),
        "et_histogram_dev": (i, [vp, vp, sz, vp, vp]),
        "et_encode": (i, [vp, vp, sz, vp, sz, szp, u32]),
        "et_decode": (i, [vp, vp, sz, vp, sz, szp, u32]),
        "et_encode_dev": (i, [vp, vp, sz, vp, sz, szp, u32, vp]),
        "et_decode_dev": (i, [vp, vp, sz, vp, sz, szp, u32, vp]),
        "et_decode_batch_dev": (i, [vp, ctypes.POINTER(BatchItem), sz, u32, vp]),
        "et_encode_batch_dev": (i, [vp, ctypes.POINTER(BatchItem), sz, u32, vp]),
        "et_pack_shard_dev": (i, [vp, vp, sz, ctypes.POINTER(Codebook), u32, u64, vp, sz, szp, vp]),
        "et_shard_bits": (u64, [vp, ctypes.POINTER(Codebook)]),
        "et_unpack_shard_dev": (i, [vp, vp, sz, sz, sz, ctypes.POINTER(Dictionary), ctypes.c_int64, vp, sz,
                                    ctypes.POINTER(u64), ctypes.POINTER(u64), ctypes.POINTER(u64), vp]),
        "et_synth_dev": (i, [vp, vp, sz, u64, u64, vp, vp]),
        "et_comm_unique_id": (i, [vp]),
        "et_comm_create_nccl": (i, [vp, vp, i, i, ctypes.POINTER(vp)]),
        "et_comm_create_callback": (i, [vp, i, i, ALLGATHER_FN, vp, ctypes.POINTER(vp)]),
        "et_comm_destroy": (None, [vp]),
        "et_encode_sharded_dev": (i, [vp, vp, vp, sz, vp, sz, ctypes.POINTER(ShardEncoded), u32, vp]),
        "et_decode_sharded_dev": (i, [vp, vp, vp, sz, vp, sz, sz, sz, i, vp, sz, ctypes.POINTER(ShardDecoded), u32, vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L
