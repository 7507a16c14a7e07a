"""Throughput of the raw-stream batch calls on device-resident text, next to the 64KB-block batch over the same bytes.

For each shape (256 KiB, 1 MiB, 8 MiB and mixed log-uniform 4 KiB-8 MiB units; >= --gib GiB per shape, larger than
L2) it times, with CUDA events and alternating:
  streams   sb_compress_streams_device_ws over all units (varint + blocks, packed back to back)
  blocks    sb_compress_batch_device over the same 64KB blocks of the same units (identical K1 work, per-block
            varint, fixed-stride slots): the gap is the cost of K7's plan, expand, scan and gather steps
  decomp    sb_decompress_streams_device_ws over the streams (sizes and places every output on the device)
Rates are uncompressed bytes / time. Parity in the same run: every stream is decoded on the device and compared with
its input; every stream equals its unit's varint followed by the block batch's outputs for its blocks with their
per-block varints removed (compared on the device); a sample of units is checked against the oracle.

    python tools/streams_bench.py --out profiles/streams_bench.json [--gib 8] [--reps 5]
"""
import argparse
import ctypes as C
import json
import math
import os
import random
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as graft  # noqa: E402

MUL = 65521
STRIDE = 76544          # K1 slot stride (>= max_compress_len(65536))


def varint(n):
    out = bytearray()
    while n >= 0x80:
        out.append((n & 0x7F) | 0x80)
        n >>= 7
    out.append(n)
    return bytes(out)


def shape_lens(name, total, rng):
    if name == "mixed":
        lens, s = [], 0
        while True:
            n = int(math.exp(rng.uniform(math.log(4096), math.log(8 << 20))))
            if s + n > total:
                return lens
            lens.append(n)
            s += n
    size = {"256KiB": 256 << 10, "1MiB": 1 << 20, "8MiB": 8 << 20}[name]
    return [size] * (total // size)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--gib", type=float, default=8.0)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--shapes", default="256KiB,1MiB,8MiB,mixed")
    args = ap.parse_args()

    import torch
    torch.cuda.set_device(0)
    snap = graft.load_package()
    L = snap._lib.lib()
    from oracle import oracle as orc
    dev = torch.device("cuda:0")
    err = snap._lib.SbError()

    def ck(rc):
        if rc:
            raise snap.error.from_c(err)

    text = b"".join(open(os.path.join(ROOT, "tests", "golden", "data", f), "rb").read()
                    for f in ("alice29.txt", "asyoulik.txt", "lcet10.txt", "plrabn12.txt", "html", "urls.10K"))
    t_text = torch.frombuffer(bytearray(text), dtype=torch.uint8).to(dev)
    total = int(args.gib * (1 << 30))
    nblk = (total + 65535) // 65536
    t_in = torch.empty(nblk * 65536, dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    ck(L.sb_generate_blocks_device(t_text.data_ptr(), len(text), t_in.data_ptr(), 65536, 65536, 0, nblk, MUL, st, C.byref(err)))
    rng = random.Random(1)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:          # the number is still reported, with the reason the limit is missing
        power = "unavailable (%s)" % e
    result = {"device": torch.cuda.get_device_name(0), "power_limit": power, "gib_per_shape": args.gib, "reps": args.reps,
              "shapes": {}}

    for shape in args.shapes.split(","):
        lens = shape_lens(shape, total, rng)
        n = len(lens)
        offs = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
        nbytes = int(offs[-1])
        assert nbytes <= t_in.numel()
        base = t_in.data_ptr()
        d_ptrs = torch.tensor(base + offs[:-1], dtype=torch.int64, device=dev)
        d_lens = torch.tensor(lens, dtype=torch.int64, device=dev)
        # the same units cut into 64KB blocks for the block batch
        nb = [max(1, (x + 65535) // 65536) for x in lens]
        b_ptr, b_len = [], []
        for o, x, k in zip(offs[:-1], lens, nb):
            for j in range(k):
                b_ptr.append(base + int(o) + 65536 * j)
                b_len.append(min(65536, x - 65536 * j))
        items = len(b_ptr)
        d_bptr = torch.tensor(b_ptr, dtype=torch.int64, device=dev)
        d_blen = torch.tensor(b_len, dtype=torch.int32, device=dev)
        cap = sum(L.sb_max_compress_len(x) for x in lens)
        out = torch.empty(cap, dtype=torch.uint8, device=dev)
        d_offs = torch.empty(n + 1, dtype=torch.int64, device=dev)
        d_res = torch.zeros(6, dtype=torch.int64, device=dev)
        sb = L.sb_compress_streams_scratch_bytes(n, nbytes)
        scr = torch.empty(sb, dtype=torch.uint8, device=dev)
        slots = torch.empty(items * STRIDE, dtype=torch.uint8, device=dev)
        b_clen = torch.zeros(items, dtype=torch.int32, device=dev)
        bt = snap._lib.SbBatch()
        bt.in_ptrs = d_bptr.data_ptr(); bt.in_lens = d_blen.data_ptr()
        bt.out_base = slots.data_ptr(); bt.out_stride = STRIDE; bt.out_cap_uniform = STRIDE
        bt.out_lens = b_clen.data_ptr(); bt.count = items
        dout = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        dd_offs = torch.empty(n + 1, dtype=torch.int64, device=dev)
        dd_st = torch.empty((n, 4), dtype=torch.int64, device=dev)
        dd_res = torch.zeros(6, dtype=torch.int64, device=dev)
        dsb = L.sb_decompress_streams_scratch_bytes(n)
        dscr = torch.empty(dsb, dtype=torch.uint8, device=dev)

        def run_streams():
            ck(L.sb_compress_streams_device_ws(d_ptrs.data_ptr(), d_lens.data_ptr(), n, nbytes, out.data_ptr(), cap,
                                               d_offs.data_ptr(), None, d_res.data_ptr(), scr.data_ptr(), sb, st, C.byref(err)))

        def run_blocks():
            ck(L.sb_compress_batch_device(C.byref(bt), st, C.byref(err)))

        def run_decomp():
            ck(L.sb_decompress_streams_device_ws(c_ptrs.data_ptr(), c_lens.data_ptr(), n, dout.data_ptr(), nbytes,
                                                 dd_offs.data_ptr(), dd_st.data_ptr(), dd_res.data_ptr(), dscr.data_ptr(), dsb,
                                                 st, C.byref(err)))

        def timed(fn):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            return a.elapsed_time(b) / 1e3

        run_streams(); run_blocks()                                          # warm-up
        torch.cuda.synchronize()
        c_ptrs = out.data_ptr() + d_offs[:-1]
        c_lens = d_offs[1:] - d_offs[:-1]
        run_decomp()
        torch.cuda.synchronize()
        ts, tb, td = [], [], []
        for _ in range(args.reps):
            ts.append(timed(run_streams))
            tb.append(timed(run_blocks))
            td.append(timed(run_decomp))
        res = snap._lib.SbFrameResult.from_buffer_copy(d_res.cpu().numpy().tobytes())
        dres = snap._lib.SbFrameResult.from_buffer_copy(dd_res.cpu().numpy().tobytes())
        comp_bytes = int(d_offs[-1])

        # ---- parity: round trip on the device
        round_trip = dres.status.code == 0 and res.status.code == 0 and bool(torch.equal(dout, t_in[:nbytes]))
        # ---- parity: stream == varint(n) + block outputs without their per-block varint
        hl = torch.where(d_blen >= 16384, 3, torch.where(d_blen >= 128, 2, 1)).to(torch.int64)
        body = b_clen.to(torch.int64) - hl
        first_item = torch.tensor(np.concatenate([[0], np.cumsum(nb)[:-1]]), dtype=torch.int64, device=dev)
        unit_of = torch.repeat_interleave(torch.arange(n, device=dev), torch.tensor(nb, device=dev))
        hdr = torch.tensor([len(varint(x)) for x in lens], dtype=torch.int64, device=dev)
        csum = torch.cumsum(body, 0) - body
        dst = d_offs[:-1][unit_of] + hdr[unit_of] + csum - csum[first_item][unit_of]
        want_len = hdr + torch.zeros(n, dtype=torch.int64, device=dev).index_add_(0, unit_of, body)
        lens_ok = bool(torch.equal(want_len, d_offs[1:] - d_offs[:-1]))
        bytes_ok = True
        chunk = 1024
        j = torch.arange(STRIDE, device=dev)
        for lo in range(0, items, chunk):
            hi = min(items, lo + chunk)
            m = j[None, :] < body[lo:hi, None]
            src = (torch.arange(lo, hi, device=dev)[:, None] * STRIDE + hl[lo:hi, None] + j[None, :])[m]
            dpos = (dst[lo:hi, None] + j[None, :])[m]
            if not torch.equal(slots[src], out[dpos]):
                bytes_ok = False
                break
        hpos = d_offs[:-1][:, None] + torch.arange(5, device=dev)[None, :]
        hbytes = out[hpos.clamp(max=cap - 1)].cpu().numpy()
        hdr_ok = all(bytes(hbytes[i, :len(varint(x))]) == varint(x) for i, x in enumerate(lens))
        # ---- parity: a sample against the oracle
        o = d_offs.cpu().numpy()
        sample = random.Random(2).sample(range(n), min(n, 8))
        oracle_ok = all(orc.compress(t_in[int(offs[i]):int(offs[i + 1])].cpu().numpy().tobytes()) ==
                        out[int(o[i]):int(o[i + 1])].cpu().numpy().tobytes() for i in sample)
        med = lambda v: sorted(v)[len(v) // 2]   # noqa: E731
        r = {"units": n, "blocks": items, "bytes": nbytes, "compressed_bytes": comp_bytes,
             "streams_compress_gbps": nbytes / med(ts) / 1e9, "blocks_compress_gbps": nbytes / med(tb) / 1e9,
             "streams_vs_blocks": med(tb) / med(ts), "decompress_gbps": nbytes / med(td) / 1e9,
             "ms": {"streams": [1e3 * x for x in ts], "blocks": [1e3 * x for x in tb], "decompress": [1e3 * x for x in td]},
             "parity": {"device_round_trip": round_trip, "lengths_match_blocks": lens_ok, "bytes_match_blocks": bytes_ok,
                        "varints": hdr_ok, "oracle_sample": oracle_ok, "oracle_sample_units": len(sample)}}
        result["shapes"][shape] = r
        print(json.dumps({shape: r}), flush=True)
        del out, scr, slots, dout, dscr
        torch.cuda.empty_cache()

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    ok = all(all(v for v in s["parity"].values() if isinstance(v, bool)) for s in result["shapes"].values())
    print("parity", "ok" if ok else "FAILED")
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
