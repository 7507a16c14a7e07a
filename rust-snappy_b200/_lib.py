"""ctypes binding of libsnapb200.so (the C ABI in include/snapb200.h).

There is no fallback: if the shared library is missing this module raises, and
if no B200 is visible every compute call returns SB_E_NO_DEVICE which surfaces as
`NoDevice`.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("SNAPB200_LIB") or os.path.join(_HERE, "libsnapb200.so")


class SbError(C.Structure):
    _fields_ = [("code", C.c_uint32), ("_pad", C.c_uint32),
                ("a", C.c_uint64), ("b", C.c_uint64), ("c", C.c_uint64)]


class SbFrameResult(C.Structure):
    _fields_ = [("status", SbError), ("bytes", C.c_uint64), ("nchunks", C.c_uint32), ("_pad", C.c_uint32)]


class SbBatch(C.Structure):
    _fields_ = [
        ("in_ptrs", C.c_void_p), ("in_base", C.c_void_p), ("in_stride", C.c_uint64),
        ("in_lens", C.c_void_p), ("in_len_uniform", C.c_uint32),
        ("out_ptrs", C.c_void_p), ("out_base", C.c_void_p), ("out_stride", C.c_uint64),
        ("out_caps", C.c_void_p), ("out_cap_uniform", C.c_uint32),
        ("out_lens", C.c_void_p), ("statuses", C.c_void_p), ("count", C.c_uint32),
    ]


# every symbol include/snapb200.h declares
SYMBOLS = [
    "sb_max_compress_len", "sb_compress", "sb_decompress_len", "sb_decompress", "sb_crc32c_masked",
    "sb_compress_batch_host", "sb_decompress_batch_host", "sb_compress_batch_host_packed",
    "sb_compress_batch_device", "sb_decompress_batch_device", "sb_crc32c_masked_batch_device",
    "sb_frame_max_len", "sb_frame_encode", "sb_frame_encode_ex", "sb_frame_decode", "sb_frame_encode_device",
    "sb_frame_encode_scratch_bytes", "sb_frame_encode_device_ws", "sb_frame_decode_scratch_bytes",
    "sb_frame_decode_device_ws", "sb_frame_decode_device", "sb_reserve", "sb_alloc_count",
    "sb_compress_streams_scratch_bytes", "sb_compress_streams_device_ws", "sb_compress_streams_host_packed",
    "sb_decompress_streams_scratch_bytes", "sb_decompress_streams_device_ws",
    "sb_bind_host_thread_to_device_numa",
    "sb_launch_count", "sb_generate_blocks_device", "sb_version",
    "snappy_compress", "snappy_uncompress", "snappy_max_compressed_length", "snappy_uncompressed_length",
]

_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise ImportError(
            "libsnapb200.so is not built (run `python -c 'import __graft_entry__ as g; g.build()'`); "
            "this package has no CPU fallback")
    L = C.CDLL(SO_PATH)
    vp, sz, szp, ep = C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t), C.POINTER(SbError)
    u64p, u32p = C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)
    L.sb_version.restype = C.c_char_p
    L.sb_launch_count.restype = C.c_uint64
    L.sb_max_compress_len.restype = sz
    L.sb_max_compress_len.argtypes = [sz]
    L.sb_frame_max_len.restype = sz
    L.sb_frame_max_len.argtypes = [sz]
    L.sb_compress.argtypes = [vp, sz, vp, sz, szp, ep]
    L.sb_decompress_len.argtypes = [vp, sz, szp, ep]
    L.sb_decompress.argtypes = [vp, sz, vp, sz, szp, ep]
    L.sb_crc32c_masked.argtypes = [vp, sz, u32p, ep]
    L.sb_compress_batch_host.argtypes = [vp, vp, vp, vp, vp, vp, vp, sz, ep]
    L.sb_decompress_batch_host.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, sz, ep]
    L.sb_compress_batch_device.argtypes = [C.POINTER(SbBatch), vp, ep]
    L.sb_decompress_batch_device.argtypes = [C.POINTER(SbBatch), vp, ep]
    L.sb_crc32c_masked_batch_device.argtypes = [C.POINTER(SbBatch), vp, ep]
    L.sb_frame_encode.argtypes = [vp, sz, vp, sz, szp, ep]
    L.sb_frame_encode_ex.argtypes = [vp, sz, vp, sz, szp, C.c_int, ep]
    L.sb_frame_decode.argtypes = [vp, sz, vp, sz, szp, ep]
    L.sb_frame_encode_device.argtypes = [vp, C.c_uint64, vp, C.c_uint64, C.c_int, u64p, vp, ep]
    L.sb_compress_batch_host_packed.argtypes = [vp, vp, vp, vp, C.c_uint64, vp, vp, sz, ep]
    L.sb_frame_encode_scratch_bytes.restype = C.c_uint64
    L.sb_frame_encode_scratch_bytes.argtypes = [C.c_uint64]
    L.sb_frame_decode_scratch_bytes.restype = C.c_uint64
    L.sb_frame_decode_scratch_bytes.argtypes = [C.c_uint32]
    L.sb_frame_encode_device_ws.argtypes = [vp, C.c_uint64, vp, C.c_uint64, C.c_int, vp, vp, vp, C.c_uint64, vp, ep]
    L.sb_frame_decode_device_ws.argtypes = [vp, C.c_uint64, vp, C.c_uint64, vp, C.c_uint32, C.c_uint32, vp, vp, C.c_uint64,
                                            C.c_uint32, vp, ep]
    L.sb_frame_decode_device.argtypes = [vp, C.c_uint64, vp, C.c_uint64, vp, C.c_uint32, C.c_uint32,
                                         C.POINTER(SbFrameResult), vp, ep]
    L.sb_compress_streams_scratch_bytes.restype = C.c_uint64
    L.sb_compress_streams_scratch_bytes.argtypes = [C.c_uint32, C.c_uint64]
    L.sb_compress_streams_device_ws.argtypes = [vp, vp, C.c_uint32, C.c_uint64, vp, C.c_uint64, vp, vp, vp, vp, C.c_uint64,
                                                vp, ep]
    L.sb_compress_streams_host_packed.argtypes = [vp, vp, vp, sz, vp, C.c_uint64, vp, ep]
    L.sb_decompress_streams_scratch_bytes.restype = C.c_uint64
    L.sb_decompress_streams_scratch_bytes.argtypes = [C.c_uint32]
    L.sb_decompress_streams_device_ws.argtypes = [vp, vp, C.c_uint32, vp, C.c_uint64, vp, vp, vp, vp, C.c_uint64, vp, ep]
    L.sb_reserve.argtypes = [sz, sz, sz, ep]
    L.sb_alloc_count.restype = C.c_uint64
    L.sb_bind_host_thread_to_device_numa.argtypes = [C.c_int]
    L.sb_generate_blocks_device.argtypes = [vp, C.c_uint64, vp, C.c_uint64, C.c_uint32, C.c_uint64,
                                            C.c_uint64, C.c_uint64, vp, ep]
    L.snappy_max_compressed_length.restype = sz
    L.snappy_max_compressed_length.argtypes = [sz]
    L.snappy_compress.argtypes = [vp, sz, vp, szp]
    L.snappy_uncompress.argtypes = [vp, sz, vp, szp]
    L.snappy_uncompressed_length.argtypes = [vp, sz, szp]
    _lib = L
    return L
