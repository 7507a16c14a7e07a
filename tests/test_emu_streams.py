"""Kernel LOGIC checks on CPU for the raw-stream batches (K7 around K1 / K2): the same kernel sequence as
sb_compress_streams_device_ws / sb_decompress_streams_device_ws, run by the warp emulator and compared with
the oracle."""
import ctypes as C
import os
import random
import subprocess

import numpy as np
import pytest

import emu_helpers as emu
from conftest import corpus
from kats import DECODE_ERRORS

MAX = 0xFFFFFFFF
EMU = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu")
SO = os.path.join(EMU, "_build", "libemu_streams.so")
_lib = None


def lib():
    """The kernel sequences of tests/emu/emu_streams.cpp built against the warp emulator (rebuilt when stale)."""
    global _lib
    if _lib is None:
        csrc = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "rust-snappy_b200", "csrc")
        srcs = [os.path.join(EMU, f) for f in ("emu_streams.cpp", "simt_emu.cpp", "simt_emu.h")]
        srcs += [os.path.join(csrc, f) for f in os.listdir(csrc)]
        if not os.path.exists(SO) or os.path.getmtime(SO) < max(os.path.getmtime(f) for f in srcs):
            os.makedirs(os.path.dirname(SO), exist_ok=True)
            # -Bsymbolic: the emulator runtime inside this library binds to itself, not to libemu_kernels.so's copy
            subprocess.check_call(["g++", "-O2", "-g", "-std=c++17", "-fPIC", "-shared", "-Wall", "-Wno-unused-function",
                                   "-Wno-unknown-pragmas", "-Wl,-Bsymbolic", "-o", SO, "emu_streams.cpp", "simt_emu.cpp"],
                                  cwd=EMU)
        _lib = C.CDLL(SO)
    return _lib


def _units_in_memory(units):
    """Units at odd offsets of one buffer; returns (keep-alive, pointer array, length array)."""
    at, offs = 1, []
    for u in units:
        offs.append(at)
        at += len(u) + 3
    buf = np.zeros(at + 16, dtype=np.uint8)
    for o, u in zip(offs, units):
        buf[o:o + len(u)] = np.frombuffer(u, dtype=np.uint8)
    ptrs = np.array([buf.ctypes.data + o for o in offs] or [0], dtype=np.uint64)
    lens = np.array([len(u) for u in units] or [0], dtype=np.uint64)
    return buf, ptrs, lens


def streams_compress(units, cap=None, total_in=None, lens=None):
    """Returns (streams or None, offsets, statuses, result, out guard ok). `lens` overrides the lengths the kernels see
    (for refused units, which are never read)."""
    buf, ptrs, ln = _units_in_memory(units)
    if lens is not None:
        ln = np.array(lens, dtype=np.uint64)
    n = len(units)
    total_in = int(ln[:n].sum()) if total_in is None else total_in
    if cap is None:
        cap = sum(32 + int(x) + int(x) // 6 for x in ln[:n] if 32 + int(x) + int(x) // 6 <= MAX)
    out = np.full(cap + 16, 0xEE, dtype=np.uint8)
    offs = np.full(n + 1, 0xAB, dtype=np.uint64)
    st = (emu.SbError * max(n, 1))()
    res = emu.SbFrameResult()
    lib().emu_streams_compress(C.c_void_p(ptrs.ctypes.data), C.c_void_p(ln.ctypes.data), C.c_uint32(n), C.c_uint64(total_in),
                                   C.c_void_p(out.ctypes.data), C.c_uint64(cap), C.c_void_p(offs.ctypes.data), C.c_void_p(C.addressof(st)),
                                   C.byref(res))
    offs = [int(x) for x in offs]
    streams = [bytes(out[offs[i]:offs[i + 1]]) for i in range(n)] if res.bytes or n == 0 else None
    status = [(emu.ERR.get(e.code, str(e.code)), e.a, e.b) for e in st][:n]
    written = res.bytes
    return streams, offs, status, res, bytes(out[written:]) == b"\xee" * (cap + 16 - written)


def streams_decompress(streams, cap=None):
    buf, ptrs, ln = _units_in_memory(streams)
    n = len(streams)
    if cap is None:
        cap = 1 << 22
    out = np.full(cap + 16, 0xEE, dtype=np.uint8)
    offs = np.zeros(n + 1, dtype=np.uint64)
    st = (emu.SbError * max(n, 1))()
    res = emu.SbFrameResult()
    lib().emu_streams_decompress(C.c_void_p(ptrs.ctypes.data), C.c_void_p(ln.ctypes.data), C.c_uint32(n),
                                     C.c_void_p(out.ctypes.data), C.c_uint64(cap), C.c_void_p(offs.ctypes.data),
                                     C.c_void_p(C.addressof(st)), C.byref(res))
    offs = [int(x) for x in offs]
    status = [(emu.ERR.get(e.code, {202: "Invalid"}.get(e.code, str(e.code))), e.a, e.b, e.c) for e in st][:n]
    outs = [bytes(out[offs[i]:offs[i + 1]]) for i in range(n)]
    return outs, offs, status, res, bytes(out[cap:]) == b"\xee" * 16


EDGE_LENS = [0, 1, 16, 17, 65535, 65536, 65537, 131072, 131073, 300000]


def _edge_units():
    text = corpus("lcet10.txt") * 2
    return [text[7 * k:7 * k + n] for k, n in enumerate(EDGE_LENS)]


def test_streams_compress_edge_lengths(oracle):
    units = _edge_units()
    streams, offs, st, res, guard = streams_compress(units)
    assert res.status.code == 0 and guard
    assert streams == [oracle.compress(u) for u in units]
    assert all(s == ("Ok", 0, 0) for s in st)
    assert offs[0] == 0 and offs[-1] == res.bytes == sum(len(s) for s in streams)       # dense, back to back
    assert res.nchunks == sum(max(1, (len(u) + 65535) // 65536) for u in units)


def test_streams_compress_corpus_slices(oracle):
    rng = random.Random(5)
    names = ["html", "urls.10K", "fireworks.jpeg", "paper-100k.pdf", "alice29.txt", "geo.protodata", "kppkn.gtb"]
    units = []
    for _ in range(12):
        d = corpus(rng.choice(names))
        a = rng.randrange(len(d))
        units.append(d[a:a + rng.choice([1, 100, 5000, 65536, 70000, 140000])])
    streams, offs, st, res, guard = streams_compress(units, total_in=sum(map(len, units)) + 3 * 65536)   # loose bound
    assert res.status.code == 0 and guard
    assert streams == [oracle.compress(u) for u in units]


def test_streams_compress_cap_too_small_writes_nothing(oracle):
    units = _edge_units()[3:7]
    total = sum(len(oracle.compress(u)) for u in units)
    streams, offs, st, res, guard = streams_compress(units, cap=total - 1)
    assert (res.status.code, res.status.a, res.status.b, res.bytes) == (2, total - 1, total, 0)
    assert guard and streams is None                                                   # nothing written
    assert offs[-1] == total and all(s == ("BufferTooSmall", total - 1, total) for s in st)
    streams, offs, st, res, guard = streams_compress(units, cap=total)                  # the reported size is enough
    assert res.status.code == 0 and streams == [oracle.compress(u) for u in units]


def test_streams_compress_total_in_below_sum_is_invalid():
    units = _edge_units()[5:9]
    s = sum(map(len, units))
    streams, offs, st, res, guard = streams_compress(units, total_in=s - 1)
    assert (res.status.code, res.status.a, res.status.b, res.bytes) == (202, s, s - 1, 0)
    assert guard and all(x[0] == "202" for x in st)


def test_streams_compress_refused_unit_and_neighbours(oracle):
    """A unit whose max_compress_len is 0 gets TooBig{n, 2^32-1} and an empty stream; its neighbours compress.
    (The refused length is only planned with, never read, so a short buffer stands in for it here.)"""
    a, b = corpus("alice29.txt")[:70000], corpus("html")[:300]
    big = 3681400512
    streams, offs, st, res, guard = streams_compress([a, b"x", b], lens=[len(a), big, len(b)], total_in=len(a) + big + len(b))
    assert (res.status.code, res.status.a, res.status.b) == (1, big, MAX)
    assert st == [("Ok", 0, 0), ("TooBig", big, MAX), ("Ok", 0, 0)]
    assert streams == [oracle.compress(a), b"", oracle.compress(b)]


def test_streams_decompress_round_trip_and_offsets(oracle):
    units = _edge_units()
    outs, offs, st, res, guard = streams_decompress([oracle.compress(u) for u in units])
    assert guard and res.status.code == 0 and res.bytes == sum(map(len, units))
    assert outs == units
    assert offs == [int(x) for x in np.concatenate([[0], np.cumsum([len(u) for u in units])])]
    assert all(s[0] == "Ok" for s in st)


def test_streams_decompress_error_kats(oracle):
    """Each KAT stream gives the oracle's error (K2 produces it); good neighbours still decode."""
    from oracle.oracle import OracleError
    good = oracle.compress(corpus("alice29.txt")[:100000])
    streams = []
    for k in DECODE_ERRORS:
        streams += [k[1], good]
    outs, offs, st, res, guard = streams_decompress(streams)
    assert guard
    for i, k in enumerate(DECODE_ERRORS):
        with pytest.raises(OracleError) as ei:
            oracle.decompress(k[1], cap=1 << 20)
        assert st[2 * i] == tuple(ei.value.err) == k[2], k[0]
        assert st[2 * i + 1][0] == "Ok" and outs[2 * i + 1] == corpus("alice29.txt")[:100000]
    assert res.status.code == 3                                   # the first failing unit: err_empty


def test_streams_decompress_cap_too_small():
    from oracle import oracle as o
    units = _edge_units()[4:8]
    total = sum(map(len, units))
    outs, offs, st, res, guard = streams_decompress([o.compress(u) for u in units], cap=total - 1)
    assert (res.status.code, res.status.a, res.status.b, res.bytes) == (2, total - 1, total, 0)
    assert all(s == ("BufferTooSmall", total - 1, total, 0) for s in st) and offs[-1] == total


def test_streams_empty_batch():
    streams, offs, st, res, guard = streams_compress([])
    assert res.status.code == 0 and offs[0] == 0 and res.bytes == 0
    outs, offs, st, res, guard = streams_decompress([])
    assert res.status.code == 0 and offs[0] == 0
