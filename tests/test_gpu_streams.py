"""Batches of raw streams of any size on the B200: sb_compress_streams_device_ws / _host_packed,
sb_decompress_streams_device_ws and the Python Encoder.compress_batch / Decoder.decompress_batch, against the
oracle. Input tensors end exactly at the last unit byte (run with PYTORCH_NO_CUDA_MEMORY_CACHING=1 under
compute-sanitizer to check that no kernel reads past a unit)."""
import ctypes as C
import math
import random

import numpy as np
import pytest

import gpu_helpers as gh
from conftest import CORPUS, corpus
from kats import DECODE_ERRORS, adversarial_blocks

pytestmark = pytest.mark.gpu

MAX = 0xFFFFFFFF


@pytest.fixture(scope="module")
def torch():
    import torch
    torch.cuda.set_device(0)
    return torch


def _blob(size):
    b = b"".join(corpus(n) for n in CORPUS)
    return (b * (size // len(b) + 1))[:size]


def dev_units(torch, units, lens=None):
    """Units at odd offsets of one device tensor that ends exactly at the last unit byte: (tensor, ptrs, lens)."""
    offs, at = [], 1
    for u in units:
        offs.append(at)
        at += len(u) + 3
    end = offs[-1] + len(units[-1]) if units else 1
    host = np.zeros(end, dtype=np.uint8)
    for o, u in zip(offs, units):
        host[o:o + len(u)] = np.frombuffer(u, dtype=np.uint8)
    t = torch.from_numpy(host).cuda()
    ptrs = torch.tensor([t.data_ptr() + o for o in offs] or [0], dtype=torch.int64, device="cuda")
    lens = torch.tensor(lens if lens is not None else [len(u) for u in units] or [0], dtype=torch.int64, device="cuda")
    return t, ptrs, lens


def _varint(n):
    out = bytearray()
    while n >= 0x80:
        out.append((n & 0x7F) | 0x80)
        n >>= 7
    out.append(n)
    return bytes(out)


def _result(res_t):
    return gh.snap()._lib.SbFrameResult.from_buffer_copy(res_t.cpu().numpy().tobytes())


def _statuses(st_t, n):
    s = gh.snap()
    raw = st_t.cpu().numpy().tobytes()
    out = []
    for i in range(n):
        e = s._lib.SbError.from_buffer_copy(raw[32 * i:32 * i + 32])
        out.append(("Ok", 0, 0, 0) if e.code == 0 else
                    ("Invalid", e.a, e.b, e.c) if e.code == 202 else gh.err_tuple(s.error.from_c(e)))
    return out


def compress_ws(torch, ptrs, lens, count, total_in, cap, stream=None):
    """sb_compress_streams_device_ws; returns (out tensor, offsets tensor, status tensor, result tensor)."""
    L = gh.lib()
    out = torch.empty(max(cap, 1), dtype=torch.uint8, device="cuda")
    offs = torch.empty(count + 1, dtype=torch.int64, device="cuda")
    st = torch.zeros((max(count, 1), 4), dtype=torch.int64, device="cuda")
    res = torch.zeros(6, dtype=torch.int64, device="cuda")
    sb = L.sb_compress_streams_scratch_bytes(count, total_in)
    scr = torch.empty(sb, dtype=torch.uint8, device="cuda")
    e = gh.snap()._lib.SbError()
    s = stream if stream is not None else torch.cuda.current_stream()
    rc = L.sb_compress_streams_device_ws(ptrs.data_ptr(), lens.data_ptr(), count, total_in, out.data_ptr(), cap, offs.data_ptr(),
                                         st.data_ptr(), res.data_ptr(), scr.data_ptr(), sb, s.cuda_stream, C.byref(e))
    assert rc == 0, (rc, e.code, e.a, e.b)
    return out, offs, st, res, scr


def decompress_ws(torch, ptrs, lens, count, cap, stream=None):
    L = gh.lib()
    out = torch.empty(max(cap, 1), dtype=torch.uint8, device="cuda")
    offs = torch.empty(count + 1, dtype=torch.int64, device="cuda")
    st = torch.zeros((max(count, 1), 4), dtype=torch.int64, device="cuda")
    res = torch.zeros(6, dtype=torch.int64, device="cuda")
    sb = L.sb_decompress_streams_scratch_bytes(count)
    scr = torch.empty(sb, dtype=torch.uint8, device="cuda")
    e = gh.snap()._lib.SbError()
    s = stream if stream is not None else torch.cuda.current_stream()
    rc = L.sb_decompress_streams_device_ws(ptrs.data_ptr(), lens.data_ptr(), count, out.data_ptr(), cap, offs.data_ptr(),
                                           st.data_ptr(), res.data_ptr(), scr.data_ptr(), sb, s.cuda_stream, C.byref(e))
    assert rc == 0, (rc, e.code, e.a, e.b)
    return out, offs, st, res, scr


def streams_of(out, offs):
    o = offs.cpu().numpy()
    h = out.cpu().numpy()
    return [bytes(h[o[i]:o[i + 1]]) for i in range(len(o) - 1)]


@pytest.fixture(scope="module")
def parity_units():
    """~200 log-uniform sizes from 1 B to 8 MiB cut from the corpus, the adversarial blocks and a 24 MB unit."""
    rng = random.Random(7)
    blob = _blob(32 << 20)
    units = []
    for _ in range(200):
        n = int(math.exp(rng.uniform(0, math.log(8 << 20))))
        a = rng.randrange(len(blob) - n)
        units.append(blob[a:a + n])
    units += adversarial_blocks()
    units.append(_blob(24 << 20)[::-1])
    rng.shuffle(units)
    return units


def test_streams_parity_device_and_host(torch, oracle, parity_units):
    units = parity_units
    want = [oracle.compress(u) for u in units]
    n, total = len(units), sum(map(len, units))
    cap = sum(gh.lib().sb_max_compress_len(len(u)) for u in units)
    t, ptrs, lens = dev_units(torch, units)
    out, offs, st, res, _ = compress_ws(torch, ptrs, lens, n, total, cap)
    torch.cuda.synchronize()
    r = _result(res)
    assert r.status.code == 0 and r.bytes == sum(map(len, want))
    assert r.nchunks == sum(max(1, (len(u) + 65535) // 65536) for u in units)
    got = streams_of(out, offs)
    assert [i for i in range(n) if got[i] != want[i]] == []
    assert all(s[0] == "Ok" for s in _statuses(st, n))
    # the host form and the Python wrapper produce the same bytes
    assert gh.snap().raw.Encoder().compress_batch(units) == want


def test_streams_device_round_trip(torch, oracle, parity_units):
    """Compress output fed straight back: the decompress call sizes and places every output on the device."""
    units = parity_units
    n, total = len(units), sum(map(len, units))
    cap = sum(gh.lib().sb_max_compress_len(len(u)) for u in units)
    t, ptrs, lens = dev_units(torch, units)
    cout, coffs, _, _, _ = compress_ws(torch, ptrs, lens, n, total, cap)
    dptrs = cout.data_ptr() + coffs[:-1]                       # device arithmetic only: no size reaches the host
    dlens = coffs[1:] - coffs[:-1]
    out, offs, st, res, _ = decompress_ws(torch, dptrs, dlens, n, total)
    torch.cuda.synchronize()
    r = _result(res)
    assert r.status.code == 0 and r.bytes == total
    assert [int(x) for x in offs.cpu()] == [0] + list(np.cumsum([len(u) for u in units]))
    got = streams_of(out, offs)
    assert [i for i in range(n) if got[i] != units[i]] == []
    assert gh.snap().raw.Decoder().decompress_batch([oracle.compress(u) for u in units[:40]]) == units[:40]


def test_streams_corrupt_units_and_neighbours(torch, oracle):
    """KAT streams and bit-flipped streams give the oracle's error per unit; the good neighbours still decode."""
    from oracle.oracle import OracleError
    rng = random.Random(3)
    good_in = _blob(300000)
    good = oracle.compress(good_in)
    bad = [k[1] for k in DECODE_ERRORS]
    for _ in range(40):
        s = bytearray(good)
        for _ in range(rng.randrange(1, 4)):
            s[rng.randrange(len(s))] ^= 1 << rng.randrange(8)
        bad.append(bytes(s))
    streams = []
    for b in bad:
        streams += [b, good]
    want = []
    for s in streams:
        try:
            d = oracle.decompress(s, cap=oracle.decompress_len(s))
            want.append((("Ok", 0, 0, 0), d))
        except OracleError as e:
            want.append((tuple(e.err), None))
    cap_total = 0
    for s in streams:
        try:
            v = oracle.decompress_len(s)
            cap_total += v if v <= MAX else 0
        except OracleError:
            pass
    t, ptrs, lens = dev_units(torch, streams)
    out, offs, st, res, _ = decompress_ws(torch, ptrs, lens, len(streams), cap_total)
    torch.cuda.synchronize()
    got_st = _statuses(st, len(streams))
    got = streams_of(out, offs)
    for i, (w, g, s) in enumerate(zip(want, got, got_st)):
        assert s == w[0], (i, s, w[0])
        if w[1] is not None:
            assert g == w[1]
    first_bad = next(i for i, w in enumerate(want) if w[0][0] != "Ok")
    r = _result(res)
    assert (gh.err_tuple(gh.snap().error.from_c(r.status)) if r.status.code else ("Ok", 0, 0, 0)) == want[first_bad][0]
    # the Python wrapper raises the first failing stream's error, like a decompress_vec loop
    with pytest.raises(gh.snap().Error) as ei:
        gh.snap().raw.Decoder().decompress_batch([good] + streams[2:])
    assert ei.value.as_tuple() == want[2][0]
    # a cap below the total: nothing is decoded, every unit reports BufferTooSmall{cap, total}
    gstreams = [good] * 3
    t, ptrs, lens = dev_units(torch, gstreams)
    out, offs, st, res, _ = decompress_ws(torch, ptrs, lens, 3, 3 * len(good_in) - 1)
    torch.cuda.synchronize()
    bts = ("BufferTooSmall", 3 * len(good_in) - 1, 3 * len(good_in), 0)
    assert _statuses(st, 3) == [bts] * 3 and int(offs[3]) == 3 * len(good_in)


def test_streams_compress_cap_and_total_in(torch, oracle):
    units = [_blob(200000), b"", b"a", _blob(70000)[::-1]]
    want = [oracle.compress(u) for u in units]
    total = sum(map(len, want))
    t, ptrs, lens = dev_units(torch, units)
    out, offs, st, res, _ = compress_ws(torch, ptrs, lens, 4, sum(map(len, units)), total - 1)
    torch.cuda.synchronize()
    r = _result(res)
    assert (r.status.code, r.status.a, r.status.b, r.bytes) == (2, total - 1, total, 0)
    assert int(offs[4]) == total
    out2, offs2, _, res2, _ = compress_ws(torch, ptrs, lens, 4, sum(map(len, units)), int(offs[4]))   # retry sized by the report
    torch.cuda.synchronize()
    assert _result(res2).status.code == 0 and streams_of(out2, offs2) == want
    out, offs, st, res, _ = compress_ws(torch, ptrs, lens, 4, sum(map(len, units)) - 1, total)
    torch.cuda.synchronize()
    r = _result(res)
    assert (r.status.code, r.status.a, r.status.b, r.bytes) == (202, sum(map(len, units)), sum(map(len, units)) - 1, 0)


def test_streams_limits_real_allocations(torch, oracle):
    """A 3,681,400,512-byte unit is refused with TooBig and its neighbours compress; a 3,681,400,511-byte unit of
    zeros compresses (checked block by block: every full block of zeros compresses to the same body)."""
    big, ok_n = 3681400512, 3681400511
    small = [_blob(100000), _blob(5000)[::-1]]
    t_big = torch.empty(big, dtype=torch.uint8, device="cuda")          # never read: only planned with
    t_zero = torch.zeros(ok_n, dtype=torch.uint8, device="cuda")
    t_small, p_small, l_small = dev_units(torch, small)
    ptrs = torch.stack([p_small[0], torch.tensor(t_big.data_ptr(), device="cuda"), torch.tensor(t_zero.data_ptr(), device="cuda"),
                        p_small[1]])
    lens = torch.tensor([len(small[0]), big, ok_n, len(small[1])], dtype=torch.int64, device="cuda")
    cap = sum(gh.lib().sb_max_compress_len(n) for n in (len(small[0]), ok_n, len(small[1])))
    out, offs, st, res, scr = compress_ws(torch, ptrs, lens, 4, int(lens.sum()), cap)
    torch.cuda.synchronize()
    del scr, t_big
    r = _result(res)
    assert (r.status.code, r.status.a, r.status.b) == (1, big, MAX)
    assert _statuses(st, 4) == [("Ok", 0, 0, 0), ("TooBig", big, MAX, 0), ("Ok", 0, 0, 0), ("Ok", 0, 0, 0)]
    o = [int(x) for x in offs.cpu()]
    h = out[:o[4]].cpu().numpy()
    assert bytes(h[o[0]:o[1]]) == oracle.compress(small[0]) and bytes(h[o[3]:o[4]]) == oracle.compress(small[1])
    assert o[2] == o[1]                                                 # the refused unit's stream is empty
    hdr = _varint(ok_n)
    full = oracle.compress(bytes(65536))[len(_varint(65536)):]          # body of one full block of zeros
    tail_n = ok_n % 65536
    tail_body = oracle.compress(bytes(tail_n))[len(_varint(tail_n)):]
    zero_stream = h[o[2]:o[3]]
    want_len = len(hdr) + (ok_n // 65536) * len(full) + len(tail_body)
    assert len(zero_stream) == want_len
    assert bytes(zero_stream[:len(hdr)]) == bytes(hdr)
    body = zero_stream[len(hdr):len(hdr) + (ok_n // 65536) * len(full)].reshape(-1, len(full))
    assert (body == np.frombuffer(full, dtype=np.uint8)).all()
    assert bytes(zero_stream[len(zero_stream) - len(tail_body):]) == tail_body


def test_streams_host_waves_without_allocations(torch, oracle):
    """compress_batch over several waves, one unit larger than the first wave (> 64 MiB); after sb_reserve the
    repeated calls allocate nothing."""
    s = gh.snap()
    L = gh.lib()
    units = [_blob(100 << 20)] + [_blob((1 << 20) + k)[k:] for k in range(300)]
    waves_units = len(units) + sum(len(u) for u in units) // 65536 + 64
    e = s._lib.SbError()
    assert L.sb_reserve(waves_units, 1 << 30, (1 << 30) + (1 << 28), C.byref(e)) == 0
    enc = s.raw.Encoder()
    got = enc.compress_batch(units)
    assert [i for i, (g, u) in enumerate(zip(got, units)) if g != oracle.compress(u)] == []
    before = L.sb_alloc_count()
    for _ in range(2):
        assert enc.compress_batch(units) == got
    assert L.sb_alloc_count() == before
    with pytest.raises(s.Error):                                        # empty list and errors keep the loop's behaviour
        s.raw.Decoder().decompress_batch([got[0], b""])
    assert enc.compress_batch([]) == [] and enc.compress_batch([b""]) == [b"\x00"]


def test_streams_stream_order(torch, oracle):
    """The _ws calls run on a non-default stream right after a kernel on that stream writes their input."""
    units = [_blob(3 << 20), _blob(700000)[::-1], _blob(65537)]
    key = 0x5A
    t, ptrs, lens = dev_units(torch, units)
    scrambled = t ^ key
    t.zero_()
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    n, total = len(units), sum(map(len, units))
    cap = sum(gh.lib().sb_max_compress_len(len(u)) for u in units)
    with torch.cuda.stream(side):
        torch.bitwise_xor(scrambled, key, out=t)                        # the kernel that writes the input
        cout, coffs, _, cres, _ = compress_ws(torch, ptrs, lens, n, total, cap, stream=side)
        dptrs = cout.data_ptr() + coffs[:-1]
        dlens = coffs[1:] - coffs[:-1]
        dout, doffs, dst, dres, _ = decompress_ws(torch, dptrs, dlens, n, total, stream=side)
    side.synchronize()
    assert streams_of(cout, coffs) == [oracle.compress(u) for u in units]
    assert streams_of(dout, doffs) == units
