"""`snap::raw` mirrored over the C ABI (reference src/raw.rs:13-14).

`Encoder.compress/compress_vec`, `Decoder.decompress/decompress_vec`,
`max_compress_len`, `decompress_len` keep the reference's argument meaning and
error behaviour (src/compress.rs:42-169, src/decompress.rs:30-110); the work is
done by the CUDA kernels behind `sb_compress` / `sb_decompress`.
`Encoder.compress_batch` / `Decoder.decompress_batch` do many independent
buffers of any size in one call each.
"""
import ctypes as C

from . import _lib
from .error import Error, from_c


def _ptr(buf):
    """address of a bytes-like object without copying (bytes, bytearray, memoryview, numpy)."""
    if isinstance(buf, bytes):
        return C.cast(C.c_char_p(buf), C.c_void_p).value, buf
    mv = memoryview(buf)
    if mv.readonly:
        b = bytes(mv)
        return C.cast(C.c_char_p(b), C.c_void_p).value, b
    arr = (C.c_char * mv.nbytes).from_buffer(mv)
    return C.addressof(arr), arr


def max_compress_len(input_len: int) -> int:
    return _lib.lib().sb_max_compress_len(input_len)


def decompress_len(data) -> int:
    p, keep = _ptr(data)
    n, e = C.c_size_t(0), _lib.SbError()
    if _lib.lib().sb_decompress_len(p, len(data), C.byref(n), C.byref(e)):
        raise from_c(e)
    return n.value


class Encoder:
    """snap::raw::Encoder (src/compress.rs:67-170)."""

    def compress(self, input, output) -> int:
        ip, k1 = _ptr(input)
        op, k2 = _ptr(output)
        n, e = C.c_size_t(0), _lib.SbError()
        if _lib.lib().sb_compress(ip, len(input), op, len(output), C.byref(n), C.byref(e)):
            raise from_c(e)
        return n.value

    def compress_vec(self, input) -> bytes:
        buf = bytearray(max(max_compress_len(len(input)), 1))
        n = self.compress(input, buf)
        return bytes(buf[:n])

    def compress_batch(self, inputs) -> list:
        """[compress_vec(x) for x in inputs] in one call (sb_compress_streams_host_packed); raises what the first
        failing input would raise in that loop."""
        data = [bytes(x) for x in inputs]
        n = len(data)
        if n == 0:
            return []
        lens = (C.c_uint64 * n)(*[len(d) for d in data])
        offs = (C.c_uint64 * n)()
        at = 0
        for i, d in enumerate(data):
            offs[i] = at
            at += len(d)
        inbuf = b"".join(data) + b"\0"
        cap = sum(max_compress_len(len(d)) for d in data)
        out = bytearray(max(cap, 1))
        out_offs = (C.c_uint64 * (n + 1))()
        ip, k1 = _ptr(inbuf)
        op, k2 = _ptr(out)
        e = _lib.SbError()
        if _lib.lib().sb_compress_streams_host_packed(ip, C.addressof(offs), C.addressof(lens), n, op, len(out),
                                                      C.addressof(out_offs), C.byref(e)):
            raise from_c(e)
        return [bytes(out[out_offs[i]:out_offs[i + 1]]) for i in range(n)]


class Decoder:
    """snap::raw::Decoder (src/decompress.rs:45-111)."""

    def decompress(self, input, output) -> int:
        ip, k1 = _ptr(input)
        op, k2 = _ptr(output) if len(output) else (None, None)
        n, e = C.c_size_t(0), _lib.SbError()
        if _lib.lib().sb_decompress(ip, len(input), op, len(output), C.byref(n), C.byref(e)):
            raise from_c(e)
        return n.value

    def decompress_vec(self, input) -> bytes:
        buf = bytearray(decompress_len(input))
        n = self.decompress(input, buf)
        return bytes(buf[:n])

    def decompress_batch(self, streams) -> list:
        """[decompress_vec(s) for s in streams] in one call (sb_decompress_batch_host, capacities from
        decompress_len); raises what the first failing stream would raise in that loop."""
        data = [bytes(x) for x in streams]
        n = len(data)
        if n == 0:
            return []
        caps = []
        for d in data:
            try:
                caps.append(decompress_len(d))
            except Error:
                caps.append(0)           # the kernel reports the same header error for this stream
        # like sb_decompress, a stream longer than 2^32-1 bytes is refused (SB_E_INVALID); it is not sent down
        too_long = [len(d) > 0xFFFFFFFF for d in data]
        data = [b"" if t else d for d, t in zip(data, too_long)]
        lens = (C.c_uint32 * n)(*[len(d) for d in data])
        in_offs, out_offs = (C.c_uint64 * n)(), (C.c_uint64 * n)()
        at = oat = 0
        for i, d in enumerate(data):
            in_offs[i], out_offs[i] = at, oat
            at += len(d)
            oat += caps[i]
        inbuf = b"".join(data) + b"\0"
        out = bytearray(oat + 1)
        out_caps = (C.c_uint32 * n)(*caps)
        out_lens = (C.c_uint32 * n)()
        st = (_lib.SbError * n)()
        ip, k1 = _ptr(inbuf)
        op, k2 = _ptr(out)
        e = _lib.SbError()
        if _lib.lib().sb_decompress_batch_host(ip, C.addressof(in_offs), C.addressof(lens), op, C.addressof(out_offs),
                                               C.addressof(out_caps), C.addressof(out_lens), C.addressof(st), n, C.byref(e)):
            raise from_c(e)
        for i in range(n):
            if too_long[i]:
                raise from_c(_lib.SbError(202, 0, 0, 0, 0))
            if st[i].code:
                raise from_c(st[i])
        return [bytes(out[out_offs[i]:out_offs[i] + out_lens[i]]) for i in range(n)]


def crc32c_masked(data) -> int:
    """crc32::CheckSummer::crc32c_masked (src/crc32.rs:35-38), computed on the GPU."""
    p, keep = _ptr(data) if len(data) else (None, None)
    out, e = C.c_uint32(0), _lib.SbError()
    if _lib.lib().sb_crc32c_masked(p, len(data), C.byref(out), C.byref(e)):
        raise from_c(e)
    return out.value
