#!/usr/bin/env python
"""bench.py -- the headline measurement for the Snappy raw-block hot path.

Workload (BASELINE.json configs[1]): `--blocks` (default 1,048,576) independent
64KB synthetic text blocks per GPU, block i = T[off_i : off_i+65536] with
T = alice29 || asyoulik || lcet10 || plrabn12 and off_i = (i*65521) mod (|T|-65536)
(SURVEY.md 8d). One step = compress every block (K1) then decompress every
compressed block (K2), device resident, in waves that reuse two staging buffers.

metric  : uncompressed GB/s over the compress+decompress round trip
          = 2 * uncompressed_bytes / (t_compress + t_decompress)
value   : device-resident (inputs already in HBM), CUDA events, max over ranks
e2e     : the same round trip through the C ABI with HOST (pinned) buffers,
          H2D/D2H inside the timed region; compress uses sb_compress_batch_host_packed
          (the library packs the streams and reports the offsets: no foreknowledge of sizes)
parity  : warm-up step: full on-device round trip + masked CRC-32C and length of EVERY
          compressed block (K3 on the device) against the oracle's fingerprints for a
          stratified sample of every wave (100% when the host is fast enough)
side workloads (--workload): urls-decompress (configs[2]), frame (configs[3]: device-resident
          FrameEncoder/FrameDecoder over a long stream in waves), frame-shard (configs[4]:
          chunk ranges per rank, wave k's NCCL size+payload all-gather overlapping wave k+1's kernels)
--impl reference : the reference's CPU implementation of the same path (the
          oracle port -- the Rust crate cannot be built here), all host threads,
          bounded sample per step.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BLOCK = 65536
STRIDE = 76544
MUL = 65521
TEXT_FILES = ("alice29.txt", "asyoulik.txt", "lcet10.txt", "plrabn12.txt")
METRIC = "uncompressed GB/s, raw 64KB-block compress+decompress round trip"
DUMP_SAMPLE, DUMP_SEED = 32, 0       # --dump-outputs: blocks of the last wave whose bytes are written, and their seed
DUMP_LIMIT = 64 << 20


def load_text():
    d = os.path.join(ROOT, "tests", "golden", "data")
    return b"".join(open(os.path.join(d, f), "rb").read() for f in TEXT_FILES)


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def effective_cores():
    """CPU time this process may actually use: the affinity mask capped by the cgroup quota (cpu.max / cfs quota).
    sched_getaffinity alone ignores container quotas (a 128-thread mask with a 16-core quota is 16 cores)."""
    n = float(host_threads())
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            quota = float(q) / float(per)
    except (OSError, ValueError):
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except (OSError, ValueError):
            pass
    return min(n, quota) if quota else n, quota


def cpu_baseline_report(orc, text, seconds):
    """Oracle port on the host cores, bounded sample, with the numbers needed to judge it: threads used, effective
    cores (cgroup quota), per-thread rate and a 1-thread figure (reference README.md:135-158: ~0.32-0.39 GB/s
    compress, ~0.9-1.1 GB/s decompress per thread on text)."""
    threads = host_threads()
    eff, quota = effective_cores()
    tc1, td1, _ = cpu_roundtrip(orc, text, 0, 256, 1)
    one = 2 * 256 * BLOCK / (tc1 + td1) / 1e9
    tc, td, _ = cpu_roundtrip(orc, text, 0, 32 * threads, threads)
    count = max(threads, int(32 * threads / (tc + td) * seconds))
    tc, td, _ = cpu_roundtrip(orc, text, 0, count, threads)
    val = 2 * count * BLOCK / (tc + td) / 1e9
    per_thread = val / threads
    return {"value": val, "unit": "GB/s", "cores": threads, "effective_cores": eff, "cgroup_cpu_quota": quota, "kind": "port",
            "sample": "%d of the same 64KB text blocks, compress+decompress, oracle C port of rust-snappy on all host threads" % count,
            "compress_gbs": count * BLOCK / tc / 1e9, "decompress_gbs": count * BLOCK / td / 1e9,
            "per_thread_gbs": per_thread, "one_thread_gbs": one,
            "one_thread_compress_gbs": 256 * BLOCK / tc1 / 1e9, "one_thread_decompress_gbs": 256 * BLOCK / td1 / 1e9,
            "oversubscribed": bool(per_thread < 0.5 * one)}, count


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:  # noqa: BLE001
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU every 200 ms via NVML."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:  # noqa: BLE001
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # noqa: BLE001
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2)
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ----------------------------------------------------------------------------- reference arm
def cpu_roundtrip(orc, text, first, count, threads):
    """Oracle port on host threads: compress `count` blocks, then decompress them."""
    tc, comp_total = orc.bench_compress_mt(text, BLOCK, first, count, MUL, threads)
    # a small fixed set of compressed streams, tiled round-robin like the GPU decode input
    span = len(text) - BLOCK
    streams = [orc.compress(text[((first + i) * MUL) % span:][:BLOCK]) for i in range(min(count, 64))]
    td, dec_total = orc.bench_decompress_mt(streams, count, threads)
    assert dec_total == count * BLOCK
    return tc, td, comp_total


def run_reference(args, rank, world):
    if rank != 0:
        return
    from oracle import oracle as orc
    orc.lib()
    text = load_text()
    threads = host_threads()
    tc1, td1, _ = cpu_roundtrip(orc, text, 0, 256, 1)
    one_thread = 2 * 256 * BLOCK / (tc1 + td1) / 1e9
    # probe speed, then size each step to ~6 s of CPU work so W+K steps end within minutes
    tc, td, _ = cpu_roundtrip(orc, text, 0, 64 * threads, threads)
    rate = 64 * threads / (tc + td)
    budget = min(6.0, 150.0 / max(1, args.steps + args.warmup))
    count = max(threads, int(rate * budget))
    for _ in range(args.warmup):
        cpu_roundtrip(orc, text, 0, count, threads)
    ttot_c = ttot_d = 0.0
    for _ in range(args.steps):
        tc, td, _ = cpu_roundtrip(orc, text, 0, count, threads)
        ttot_c += tc
        ttot_d += td
    u = count * BLOCK * args.steps
    val = 2 * u / (ttot_c + ttot_d) / 1e9
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "GB/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * (ttot_c + ttot_d) / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": "raw 64KB text blocks (BASELINE configs[1] generator), CPU sample of %d blocks per step" % count,
                   "block_bytes": BLOCK},
        "compress_gbs": u / ttot_c / 1e9, "decompress_gbs": u / ttot_d / 1e9,
        "cpu_baseline": {"value": val, "unit": "GB/s", "cores": threads, "effective_cores": effective_cores()[0],
                         "cgroup_cpu_quota": effective_cores()[1], "kind": "port", "per_thread_gbs": val / threads,
                         "one_thread_gbs": one_thread, "oversubscribed": bool(val / threads < 0.5 * one_thread),
                         "sample": "%d blocks x 64KB per step, oracle C port of rust-snappy (no rustc in image)" % count},
        "e2e": {"value": val, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- our arm
def run_ours(args, rank, local_rank, world):
    import torch
    import __graft_entry__ as graft
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        # keep stdout for the one JSON line: NCCL's banner/debug output goes to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
        # finish communicator / connection setup before the first codec kernel runs: NCCL sets transports up lazily at the
        # first collective, and nothing of that should be in flight beside K1 (the 8-GPU faults of round 2 all hit a rank
        # whose first kernels ran right after init)
        dist.barrier()
        torch.cuda.synchronize()
    snap = graft.load_package()
    L = snap._lib.lib()
    err = snap._lib.SbError()
    numa_node = {"node": None}       # filled by run_e2e: the host thread is bound to the GPU's NUMA node only while it
                                     # allocates and streams pinned memory; the CPU-side work (parity, cpu_baseline) keeps every core
    text = load_text()
    span = len(text) - BLOCK
    blocks = args.blocks
    wave = min(args.wave, blocks)
    nwaves = (blocks + wave - 1) // wave
    first_block = rank * blocks          # weak scaling: every rank owns its own range of blocks

    t_text = torch.frombuffer(bytearray(text), dtype=torch.uint8).to(dev)
    t_in = torch.empty(blocks * BLOCK, dtype=torch.uint8, device=dev)
    t_c = torch.empty(wave * STRIDE, dtype=torch.uint8, device=dev)
    t_out = torch.empty(wave * BLOCK, dtype=torch.uint8, device=dev)
    t_clen = torch.zeros(blocks, dtype=torch.int32, device=dev)
    t_ccrc = torch.zeros(blocks, dtype=torch.int32, device=dev)     # masked CRC-32C of every compressed block (parity)
    t_dlen = torch.zeros(wave, dtype=torch.int32, device=dev)
    t_st = torch.zeros(wave * 4, dtype=torch.int64, device=dev)
    stream = torch.cuda.current_stream().cuda_stream

    def ck(rc):
        if rc:
            raise snap.error.from_c(err)

    ck(L.sb_generate_blocks_device(t_text.data_ptr(), len(text), t_in.data_ptr(), BLOCK, BLOCK,
                                   first_block, blocks, MUL, stream, C.byref(err)))
    torch.cuda.synchronize()

    def batch(in_ptr, in_stride, in_len, in_lens_ptr, out_ptr, out_stride, out_cap, lens_ptr, st_ptr, count):
        b = snap._lib.SbBatch()
        b.in_base, b.in_stride, b.in_len_uniform = in_ptr, in_stride, in_len
        if in_lens_ptr:
            b.in_lens = in_lens_ptr
        b.out_base, b.out_stride, b.out_cap_uniform = out_ptr, out_stride, out_cap
        b.out_lens = lens_ptr
        if st_ptr:
            b.statuses = st_ptr
        b.count = count
        return b

    ev = torch.cuda.Event

    def one_step(verify=False):
        """compress + decompress every wave; returns (ms_compress, ms_decompress)."""
        marks = []
        for w in range(nwaves):
            lo = w * wave
            cnt = min(wave, blocks - lo)
            e0, e1, e2 = ev(enable_timing=True), ev(enable_timing=True), ev(enable_timing=True)
            bc = batch(t_in.data_ptr() + lo * BLOCK, BLOCK, BLOCK, 0, t_c.data_ptr(), STRIDE, STRIDE,
                       t_clen.data_ptr() + 4 * lo, 0, cnt)
            bd = batch(t_c.data_ptr(), STRIDE, 0, t_clen.data_ptr() + 4 * lo, t_out.data_ptr(), BLOCK, BLOCK,
                       t_dlen.data_ptr(), t_st.data_ptr(), cnt)
            e0.record()
            ck(L.sb_compress_batch_device(C.byref(bc), stream, C.byref(err)))
            e1.record()
            ck(L.sb_decompress_batch_device(C.byref(bd), stream, C.byref(err)))
            e2.record()
            marks.append((e0, e1, e2))
            if verify:
                # fingerprint of every compressed block of this wave, on the device (K3 over the slots)
                bf = batch(t_c.data_ptr(), STRIDE, 0, t_clen.data_ptr() + 4 * lo, 0, 0, 0, t_ccrc.data_ptr() + 4 * lo, 0, cnt)
                ck(L.sb_crc32c_masked_batch_device(C.byref(bf), stream, C.byref(err)))
                torch.cuda.synchronize()
                assert torch.equal(t_in[lo * BLOCK:(lo + cnt) * BLOCK], t_out[:cnt * BLOCK]), "round trip mismatch"
                assert int(t_st.view(wave, 4)[:cnt, 0].abs().sum()) == 0, "decode status != Ok"
        torch.cuda.synchronize()
        return sum(a.elapsed_time(b) for a, b, _ in marks), sum(b.elapsed_time(c) for _, b, c in marks)

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    # warm-up (first warm-up step also verifies the round trip bit-exactly on device)
    for i in range(args.warmup):
        one_step(verify=(i == 0))
    comp_bytes = int(t_clen.to(torch.int64).sum().item())
    # Parity of the ENCODER on the whole workload, outside the timed region: length + masked CRC-32C of every
    # sampled block's compressed stream against the oracle. The sample is stratified over every wave (every
    # `step`-th block); step = 1 (100%) when the host can fingerprint the rank's blocks in ~parity_seconds.
    parity = None
    if not args.no_parity:
        import numpy as np
        from oracle import oracle as orc
        threads = host_threads()
        probe = min(blocks, 8 * threads)
        secs, _l, _c = orc.fingerprint_blocks_mt(text, BLOCK, first_block, 1, probe, MUL, threads)
        rate = probe / max(secs, 1e-6)
        budget = args.parity_seconds / max(1, min(world, 8))        # ranks share the host
        step = max(1, int(-(-blocks // max(1, int(rate * budget)))))
        step = min(step, 100)                                        # never below 1% of every wave
        nsamp = (blocks + step - 1) // step
        secs, want_len, want_crc = orc.fingerprint_blocks_mt(text, BLOCK, first_block, step, nsamp, MUL, threads)
        got_len = t_clen.cpu().numpy().astype(np.uint32)[::step][:nsamp]
        got_crc = t_ccrc.cpu().numpy().astype(np.uint32)[::step][:nsamp]
        equal = int(((got_len == want_len) & (got_crc == want_crc)).sum())
        # and the bytes themselves for a few blocks of the last wave
        lo = (nwaves - 1) * wave
        cnt = blocks - lo
        idx = sorted(set([0, cnt - 1] + [(k * 7919) % cnt for k in range(args.parity_samples)]))
        clen = t_clen[lo:lo + cnt].cpu().numpy()
        ok_n = 0
        for i in idx:
            got = bytes(t_c[i * STRIDE:i * STRIDE + int(clen[i])].cpu().numpy())
            off = ((first_block + lo + i) * MUL) % span
            ok_n += int(got == orc.compress(text[off:off + BLOCK]))
        parity = {"blocks_compared": int(nsamp), "blocks_equal": equal, "coverage": nsamp / blocks, "every": step,
                  "what": "compressed length + masked CRC-32C of every sampled block vs the oracle, all waves",
                  "bytes_compared": len(idx), "bytes_equal": ok_n, "cpu_seconds": secs}
        assert equal == nsamp and ok_n == len(idx), "compressed blocks differ from the oracle: %r" % (parity,)

    sampler = ClockSampler(local_rank)
    barrier()
    launches0 = L.sb_launch_count()
    sampler.start()
    t0 = time.perf_counter()
    ms_c = ms_d = 0.0
    for _ in range(args.steps):
        c_ms, d_ms = one_step()
        ms_c += c_ms
        ms_d += d_ms
    barrier()
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    launches = L.sb_launch_count() - launches0
    if args.dump_outputs and rank == 0:
        lo = (nwaves - 1) * wave
        dump_outputs(args.dump_outputs, t_clen, t_c, t_out, t_dlen, t_st, lo, blocks - lo)

    # max over ranks of the device-timed step
    tot = torch.tensor([ms_c + ms_d, ms_c, ms_d], dtype=torch.float64, device=dev)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(tot, op=dist.ReduceOp.MAX)
        sizes = torch.tensor([comp_bytes], dtype=torch.int64, device=dev)
        gathered = [torch.zeros_like(sizes) for _ in range(world)]
        dist.all_gather(gathered, sizes)          # per-rank compressed totals -> global stream offsets
        comp_all = int(sum(int(g.item()) for g in gathered))
    else:
        comp_all = comp_bytes
    ms_tot, ms_cmax, ms_dmax = [float(x) for x in tot.tolist()]
    u_rank = blocks * BLOCK
    u_all = u_rank * world

    # ---------------- e2e: host buffers through the C ABI (H2D/D2H inside the timed region)
    e2e = None
    if not args.no_e2e:
        aff0 = os.sched_getaffinity(0)
        if not args.no_numa_bind:
            # this rank's host thread (and the pinned buffers it allocates from here on) stay on the GPU's NUMA node
            numa_node["node"] = L.sb_bind_host_thread_to_device_numa(local_rank)
        try:
            e2e = run_e2e(args, snap, L, torch, dev, t_in, t_clen, rank, world)
        finally:
            os.sched_setaffinity(0, aff0)

    # ---------------- N > 1: the frame path's exchange step (sizes + payload all-gather over NCCL), small scale
    shard = None
    if world > 1 and not args.no_shard:
        del t_c, t_out
        torch.cuda.empty_cache()
        shard = frame_shard_measure(args, snap, L, torch, dev, rank, world, t_text, len(text), gib_per_rank=args.shard_gib_per_rank,
                                    steps=max(1, min(args.steps, 2)), warmup=1)
    if rank != 0:
        return
    peak, peak_src = measured_peak()
    value = 2 * u_all * args.steps / (ms_tot / 1e3) / 1e9
    k1_bytes = (u_rank + comp_bytes) * args.steps          # algorithmic bytes moved by K1 launches
    k1_achieved = k1_bytes / (ms_c / 1e3) / 1e9
    k2_achieved = k1_bytes / (ms_d / 1e3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "k1_traffic.json")
    if os.path.exists(tp):
        try:
            traffic = json.load(open(tp)).get("dram_bytes_per_block") * min(wave, blocks)   # per launch
        except Exception:  # noqa: BLE001
            traffic = None
    line = {
        "metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_tot / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": {"workload": "batched raw block compress+decompress: %d x 64KB synthetic text blocks per GPU (BASELINE configs[1])" % blocks,
                   "blocks_per_gpu": blocks, "block_bytes": BLOCK, "wave_blocks": wave, "ratio": comp_bytes / u_rank,
                   "l2": "inputs larger than L2 (%.1f GiB per GPU per pass)" % (u_rank / 2**30), "parity": parity,
                   "wall_s_timed_region": wall, "numa_node": numa_node["node"],
                   "lib": os.path.basename(os.environ.get("SNAPB200_LIB", "libsnapb200.so")),
                   "k1_ng_env": os.environ.get("SNAPB200_K1_NG")},
        "compress_gbs": u_all * args.steps / (ms_cmax / 1e3) / 1e9,
        "decompress_gbs": u_all * args.steps / (ms_dmax / 1e3) / 1e9,
        "roofline": {"bound": "hbm", "kernel": "k1_m7_kernel (K1 compress)", "achieved": k1_achieved, "peak": peak, "unit": "GB/s",
                     "frac": k1_achieved / peak, "traffic": traffic, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": (u_rank + comp_bytes) / nwaves,
                     "k2_decompress_kernel": {"achieved": k2_achieved, "frac": k2_achieved / peak}},
        "clocks": clocks, "gpu_launches": int(launches), "compressed_bytes_all_ranks": comp_all,
    }
    if e2e is not None:
        line["e2e"] = e2e
    if shard is not None:
        line["frame_shard"] = shard
    if world == 1 and not args.no_cpu_baseline:
        from oracle import oracle as orc
        line["cpu_baseline"], _ = cpu_baseline_report(orc, text, 12.0)
    print(json.dumps(line), flush=True)


def dump_outputs(out_dir, t_clen, t_c, t_out, t_dlen, t_st, lo, cnt):
    """--dump-outputs: what the last timed step handed back, as <name>.npy in float32 (bytes, lengths) or float64
    (status records), so that two builds can be compared array for array. The compressed length covers every block;
    the staging buffers hold only the last wave (blocks lo .. lo+cnt-1), whose lengths and statuses are written in
    full and whose bytes are written for a fixed seeded sample of DUMP_SAMPLE blocks (compressed slots padded with -1
    past the stream's end, where the slot holds no output)."""
    import numpy as np
    clen = t_clen.cpu().numpy()
    pick = np.sort(np.random.default_rng(DUMP_SEED).choice(cnt, size=min(DUMP_SAMPLE, cnt), replace=False))
    comp = np.full((len(pick), STRIDE), -1.0, dtype=np.float32)
    back = np.empty((len(pick), BLOCK), dtype=np.float32)
    for k, i in enumerate(pick):
        n = int(clen[lo + i])
        comp[k, :n] = t_c[i * STRIDE:i * STRIDE + n].cpu().numpy()
        back[k] = t_out[i * BLOCK:(i + 1) * BLOCK].cpu().numpy()
    arrays = {
        "compressed_len": clen.astype(np.float32),
        "sample_block": (lo + pick).astype(np.float64),
        "compressed_sample": comp,
        "decompressed_len": t_dlen[:cnt].cpu().numpy().astype(np.float32),
        "decompressed_sample": back,
        "decompress_status": t_st.view(-1, 4)[:cnt].cpu().numpy().astype(np.float64),
    }
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_LIMIT, "--dump-outputs would write %d bytes" % total
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_e2e(args, snap, L, torch, dev, t_in, t_clen, rank, world):
    """Round trip through sb_compress_batch_host_packed / sb_decompress_batch_host with pinned host buffers.
    Nothing learned in the device-resident pass is passed in: the library packs the compressed streams and
    reports their offsets, and the decompress call consumes exactly that report."""
    import numpy as np
    avail = 0
    try:
        for ln in open("/proc/meminfo"):
            if ln.startswith("MemAvailable"):
                avail = int(ln.split()[1]) * 1024
    except OSError:
        pass
    n = min(args.e2e_blocks, args.blocks)
    while n > 1024 and avail and n * BLOCK * 3.4 * max(1, world) > 0.5 * avail:
        n //= 2
    err = snap._lib.SbError()
    h_in = torch.empty(n * BLOCK, dtype=torch.uint8).pin_memory()
    h_in.copy_(t_in[:n * BLOCK])
    cap = int(L.sb_max_compress_len(BLOCK))
    c_cap = n * cap                                              # worst case: the only bound a caller has
    h_c = torch.empty(min(c_cap, int(n * BLOCK * 1.2) + cap), dtype=torch.uint8).pin_memory()
    h_out = torch.empty(n * BLOCK, dtype=torch.uint8).pin_memory()
    in_offs = np.arange(n, dtype=np.uint64) * BLOCK
    in_lens = np.full(n, BLOCK, dtype=np.uint32)
    c_lens = np.zeros(n, dtype=np.uint32)
    d_lens = np.zeros(n, dtype=np.uint32)
    st = np.zeros(n * 4, dtype=np.uint64)
    if L.sb_reserve(1 << 15, 1 << 30, 1 << 30, C.byref(err)):       # wave-sized pools up front: no allocation while timed
        raise snap.error.from_c(err)

    # The round trip is pipelined the way a caller with a stream of data would: the blocks go through in `nb`
    # batches, batch i+1 is compressed (thread A) while batch i is decompressed (thread B). The two directions use
    # separate lanes of the library, so H2D/kernel/D2H of both are in flight at once (PCIe is full duplex).
    nb = max(1, min(args.e2e_batches, n // 4096))
    per = n // nb
    n = per * nb
    ccap = h_c.numel() // nb
    errs = [snap._lib.SbError(), snap._lib.SbError()]
    c_offs = np.zeros((nb, per + 1), dtype=np.uint64)

    def comp(i):
        lo = i * per
        rc = L.sb_compress_batch_host_packed(h_in.data_ptr(), in_offs[lo:].ctypes.data, in_lens[lo:].ctypes.data,
                                             h_c.data_ptr() + i * ccap, ccap, c_offs[i].ctypes.data, c_lens[lo:].ctypes.data, per,
                                             C.byref(errs[0]))
        if rc:
            raise snap.error.from_c(errs[0])

    def decomp(i):
        lo = i * per
        rc = L.sb_decompress_batch_host(h_c.data_ptr() + i * ccap, c_offs[i].ctypes.data, c_lens[lo:].ctypes.data, h_out.data_ptr(),
                                        in_offs[lo:].ctypes.data, in_lens[lo:].ctypes.data, d_lens[lo:].ctypes.data,
                                        st[4 * lo:].ctypes.data, per, C.byref(errs[1]))
        if rc:
            raise snap.error.from_c(errs[1])

    def step():
        done = [threading.Event() for _ in range(nb)]
        fail = []

        def a():
            try:
                for i in range(nb):
                    comp(i)
                    done[i].set()
            except BaseException as e:  # noqa: BLE001
                fail.append(e)
                for d in done:
                    d.set()

        ta = threading.Thread(target=a)
        ta.start()
        for i in range(nb):
            done[i].wait()
            if fail:
                break
            decomp(i)
        ta.join()
        if fail:
            raise fail[0]

    for _ in range(max(1, args.warmup - 1)):
        step()
    assert bool((d_lens == BLOCK).all()) and torch.equal(h_in, h_out), "e2e round trip mismatch"
    allocs0 = L.sb_alloc_count()
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    tt = torch.tensor([dt], dtype=torch.float64, device=dev)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    dt = float(tt.item())
    cbytes = int(c_lens.astype(np.uint64).sum())
    return {"value": 2 * n * BLOCK * world * args.steps / dt / 1e9, "unit": "GB/s",
            "h2d_bytes_per_step": n * BLOCK + cbytes, "d2h_bytes_per_step": cbytes + n * BLOCK,
            "blocks_per_gpu": n, "batches": nb,
            "api": "sb_compress_batch_host_packed + sb_decompress_batch_host (pinned host buffers; offsets reported by the "
                   "library, none passed in); %d batches, compress of batch i+1 overlaps decompress of batch i (two host threads)" % nb,
            "ms_per_step": 1e3 * dt / args.steps, "allocations_in_timed_region": int(L.sb_alloc_count() - allocs0)}


# ----------------------------------------------------------------------------- frame workloads
def _wave_input(L, snap, torch, t_text, text_len, t_pool, pool_waves, wave_bytes, first_chunk, w, stream, err, generated):
    """Input of wave w: slot w % pool_waves of the resident pool, generated on first use (synthetic text chunks)."""
    slot = w % pool_waves
    if slot not in generated or generated[slot] != first_chunk:
        if L.sb_generate_blocks_device(t_text.data_ptr(), text_len, t_pool.data_ptr() + slot * wave_bytes, BLOCK, BLOCK,
                                       first_chunk, wave_bytes // BLOCK, MUL, stream, C.byref(err)):
            raise snap.error.from_c(err)
        generated[slot] = first_chunk
    return t_pool.data_ptr() + slot * wave_bytes


def frame_shard_measure(args, snap, L, torch, dev, rank, world, t_text, text_len, gib_per_rank, steps, warmup,
                        wave_gib=1.0, verify=True):
    """BASELINE configs[4]: a stream of 64KB frames split across ranks. Wave w = global chunks
    [w*world*W, (w+1)*world*W); rank r encodes its r-th slice (sb_frame_encode_device_ws, stream ordered), the
    per-rank sizes are all-gathered from the device-side result record and the payload is exchanged with grouped
    NCCL send/recv straight into the wave's reassembly buffer, overlapping the next wave's kernels.
    Returns GB/s (uncompressed, all ranks) compute-only and with the exchange."""
    import torch.distributed as dist
    err = snap._lib.SbError()
    wave_bytes = int(wave_gib * (1 << 30)) // BLOCK * BLOCK
    per_rank = int(gib_per_rank * (1 << 30)) // wave_bytes * wave_bytes
    nwaves = max(1, per_rank // wave_bytes)
    W = wave_bytes // BLOCK
    free_b, _tot = torch.cuda.mem_get_info()
    pool_waves = max(1, min(nwaves, int((free_b * 0.55 - 4 * wave_bytes * world * 0.7) // wave_bytes)))
    t_pool = torch.empty(pool_waves * wave_bytes, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    generated = {}
    first_wave_hash = {}
    verdict = {"ok": None}

    fake = os.environ.get("SNAPB200_FAKE_SHARD")                     # debugging: "rank/world" whose data this single rank generates
    frank, fworld = (int(x) for x in fake.split("/")) if fake else (None, world)

    def chunk0(w, r):
        return (w * fworld + (frank if frank is not None else r)) * W   # first global chunk of (wave, rank)

    def run(exchange, check=False):
        state = {"ok": True}

        def on_wave(w, buf, offs, sizes, total):
            if not (check and w == 0):
                return
            # decode the reassembled wave on this rank and compare with every rank's regenerated input
            t_dec = torch.empty(world * wave_bytes + 64, dtype=torch.uint8, device=dev)
            res = snap._lib.SbFrameResult()
            rc = L.sb_frame_decode_device(buf.data_ptr(), total, t_dec.data_ptr(), world * wave_bytes, None, 0, 0, C.byref(res),
                                          stream, C.byref(err))
            t_ref = torch.empty(wave_bytes, dtype=torch.uint8, device=dev)
            good = rc == 0 and res.status.code == 0 and res.bytes == world * wave_bytes      # no raise: the other ranks would hang
            for r in range(world):
                L.sb_generate_blocks_device(t_text.data_ptr(), text_len, t_ref.data_ptr(), BLOCK, BLOCK, chunk0(0, r), W, MUL,
                                            stream, C.byref(err))
                good = good and bool(torch.equal(t_ref, t_dec[r * wave_bytes:(r + 1) * wave_bytes]))
            state["ok"] = good
            first_wave_hash["bytes"] = total

        pipe = snap.shard.WavePipeline(wave_bytes, dist if world > 1 else None, dev, exchange=exchange,
                                       on_wave=on_wave if check else None)
        ins = [_wave_input(L, snap, torch, t_text, text_len, t_pool, pool_waves, wave_bytes, chunk0(w, rank), w, stream, err, generated)
               if w < pool_waves else None for w in range(nwaves)]
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for w in range(nwaves):
            d_in = ins[w] if ins[w] is not None else t_pool.data_ptr() + (w % pool_waves) * wave_bytes   # pool cycles when the share exceeds HBM
            pipe.encode(w, d_in, wave_bytes)
        pipe.flush()
        e1.record()
        torch.cuda.synchronize()
        if check:
            verdict["ok"] = bool(state["ok"])        # reported, not asserted: a rank that bails out here would hang the others
        return e0.elapsed_time(e1), pipe.stream_bytes, pipe.nccl_bytes

    run(True, check=verify)                                          # warm-up + verification of wave 0
    for _ in range(max(0, warmup - 1)):
        run(True)
    ms_x = ms_c = 0.0
    sb = nb = 0
    for _ in range(steps):
        m, sb, nb = run(True)
        ms_x += m
    for _ in range(steps):
        m, _a, _b = run(False)
        ms_c += m
    tt = torch.tensor([ms_x, ms_c, 0.0 if verdict["ok"] in (True, None) else 1.0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms_x, ms_c, bad = [float(x) for x in tt.tolist()]
    all_ok = verify and bad == 0.0
    u_all = nwaves * wave_bytes * world
    del t_pool
    torch.cuda.empty_cache()
    return {"workload": "frame chunks sharded over %d ranks, %d waves x %.2f GiB per rank (BASELINE configs[4] shape), "
                        "size all-gather + grouped NCCL send/recv payload all-gather inside the timed region" % (world, nwaves, wave_bytes / 2**30),
            "uncompressed_bytes_all_ranks": u_all, "stream_bytes": sb, "nvlink_bytes_received_per_rank": nb,
            "with_allgather_gbs": u_all * steps / (ms_x / 1e3) / 1e9, "compute_only_gbs": u_all * steps / (ms_c / 1e3) / 1e9,
            "ms_per_step_with_allgather": ms_x / steps, "ms_per_step_compute_only": ms_c / steps,
            "input_pool_waves": pool_waves,
            "verified": ("wave 0 reassembled on every rank decodes (device frame decoder) to all ranks' inputs" if all_ok
                         else "FAILED: wave 0 did not decode to the ranks' inputs on at least one rank") if verify else None}


def run_frame_shard(args, rank, local_rank, world):
    """--workload frame-shard: BASELINE configs[4] as its own line (1 TiB total by default, strong scaling)."""
    import torch
    import __graft_entry__ as graft
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
        dist.barrier()                   # communicator setup done before the first codec kernel (see run_ours)
        torch.cuda.synchronize()
    snap = graft.load_package()
    L = snap._lib.lib()
    text = load_text()
    t_text = torch.frombuffer(bytearray(text), dtype=torch.uint8).to(dev)
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = L.sb_launch_count()
    res = frame_shard_measure(args, snap, L, torch, dev, rank, world, t_text, len(text), gib_per_rank=args.gib / world,
                              steps=args.steps, warmup=args.warmup, wave_gib=args.wave_gib)
    clocks = sampler.stop()
    if rank == 0:
        peak, peak_src = measured_peak()
        print(json.dumps({
            "metric": "uncompressed GB/s, frame encode sharded over ranks with NCCL all-gather reassembly",
            "value": res["with_allgather_gbs"], "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": res["ms_per_step_with_allgather"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic", "side_measurement": True,
            "config": {"workload": res["workload"], "total_gib": args.gib, "verified": res["verified"], "input_pool_waves": res["input_pool_waves"],
                       "l2": "every wave is 1 GiB per rank (larger than L2)"},
            "compute_only_gbs": res["compute_only_gbs"], "with_allgather_gbs": res["with_allgather_gbs"],
            "stream_bytes": res["stream_bytes"], "nvlink_bytes_received_per_rank": res["nvlink_bytes_received_per_rank"],
            "clocks": clocks, "gpu_launches": int(L.sb_launch_count() - launches0), "peak_source": peak_src}), flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


def run_frame(args, local_rank):
    """--workload frame: BASELINE configs[3], FrameEncoder/FrameDecoder over a long synthetic stream on one GPU,
    device resident, in waves (the 256 GiB stream and its ~155 GiB of frames do not fit 180 GB at once): every wave
    is frame-encoded (K1 with the chunk CRC in the emitter, scan, gather) and decoded again (header parse from the
    encoder's chunk index, K2, CRC verify). The first pass checks decode(encode(x)) == x for every wave."""
    import torch
    import __graft_entry__ as graft
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    snap = graft.load_package()
    L = snap._lib.lib()
    err = snap._lib.SbError()
    text = load_text()
    t_text = torch.frombuffer(bytearray(text), dtype=torch.uint8).to(dev)
    wave_bytes = int(args.wave_gib * (1 << 30)) // BLOCK * BLOCK
    W = wave_bytes // BLOCK
    nwaves = max(1, int(args.gib * (1 << 30)) // wave_bytes)
    cap = L.sb_frame_max_len(wave_bytes)
    esb, dsb = L.sb_frame_encode_scratch_bytes(wave_bytes), L.sb_frame_decode_scratch_bytes(W + 1)
    t_enc = torch.empty(cap + 16, dtype=torch.uint8, device=dev)
    t_dec = torch.empty(wave_bytes + 16, dtype=torch.uint8, device=dev)
    t_idx = torch.zeros(W + 1, dtype=torch.int64, device=dev)
    t_res = torch.zeros(16, dtype=torch.int64, device=dev)           # two sb_frame_result records
    t_scr = torch.empty(max(esb, dsb) + 256, dtype=torch.uint8, device=dev)
    free_b, _t = torch.cuda.mem_get_info()
    pool_waves = max(1, min(nwaves, int(free_b * 0.8 // wave_bytes)))
    t_pool = torch.empty(pool_waves * wave_bytes, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    generated = {}
    ev = torch.cuda.Event

    def ck(rc):
        if rc:
            raise snap.error.from_c(err)

    def one_pass(verify):
        marks, total_stream = [], 0
        for w in range(nwaves):
            d_in = _wave_input(L, snap, torch, t_text, len(text), t_pool, pool_waves, wave_bytes, w * W, w, stream, err, generated) \
                if (verify or w < pool_waves) else t_pool.data_ptr() + (w % pool_waves) * wave_bytes
            e0, e1, e2 = ev(enable_timing=True), ev(enable_timing=True), ev(enable_timing=True)
            e0.record()
            ck(L.sb_frame_encode_device_ws(d_in, wave_bytes, t_enc.data_ptr(), cap, 1 if w == 0 else 0, t_idx.data_ptr(),
                                           t_res.data_ptr(), t_scr.data_ptr(), esb + 256, stream, C.byref(err)))
            e1.record()
            # the stream length is the last entry of the index the encoder just wrote (one 8-byte read back per wave;
            # the pool cycles, so sizes from an earlier pass are not this wave's)
            n_stream = int(t_idx[W].item())
            ck(L.sb_frame_decode_device_ws(t_enc.data_ptr(), n_stream, t_dec.data_ptr(), wave_bytes, t_idx.data_ptr(), W,
                                           0 if w == 0 else 1, t_res.data_ptr() + 64, t_scr.data_ptr(), dsb + 256, W + 1, stream,
                                           C.byref(err)))
            e2.record()
            marks.append((e0, e1, e2))
            one_pass.sizes[w] = n_stream
            if verify:
                torch.cuda.synchronize()
                assert int(t_res[0].item()) & 0xFFFFFFFF == 0 and int(t_res[8].item()) & 0xFFFFFFFF == 0, \
                    "frame status != Ok: wave %d encode %r decode %r" % (w, t_res[:6].tolist(), t_res[8:14].tolist())
                assert int(t_res[12].item()) == wave_bytes, "decoder produced %d bytes" % int(t_res[12].item())
                assert torch.equal(t_dec[:wave_bytes], t_pool[(w % pool_waves) * wave_bytes:(w % pool_waves + 1) * wave_bytes]), "frame round trip mismatch"
            total_stream += one_pass.sizes[w]
        torch.cuda.synchronize()
        bad = t_res[8].item() & 0xFFFFFFFF
        assert bad == 0, "frame decode status %d in the last wave" % bad
        return sum(a.elapsed_time(b) for a, b, _ in marks), sum(b.elapsed_time(c) for _, b, c in marks), total_stream

    one_pass.sizes = [0] * nwaves
    one_pass(True)
    # first chunks of the stream against the oracle's FrameEncoder bytes
    from oracle import oracle as orc
    span = len(text) - BLOCK
    head = b"".join(text[(i * MUL) % span:][:BLOCK] for i in range(4))
    d0 = _wave_input(L, snap, torch, t_text, len(text), t_pool, pool_waves, wave_bytes, 0, 0, stream, err, generated)   # wave 0 again (the pool cycles)
    ck(L.sb_frame_encode_device_ws(d0, wave_bytes, t_enc.data_ptr(), cap, 1, t_idx.data_ptr(), t_res.data_ptr(),
                                   t_scr.data_ptr(), esb + 256, stream, C.byref(err)))
    torch.cuda.synchronize()
    want = orc.frame_encode(head)
    assert bytes(t_enc[:len(want)].cpu().numpy()) == want, "frame bytes differ from the oracle"
    for _ in range(max(0, args.warmup - 1)):
        one_pass(False)
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = L.sb_launch_count()
    ms_e = ms_d = 0.0
    for _ in range(args.steps):
        a, b, stream_bytes = one_pass(False)
        ms_e += a
        ms_d += b
    clocks = sampler.stop()
    u = nwaves * wave_bytes
    peak, peak_src = measured_peak()
    enc = u * args.steps / (ms_e / 1e3) / 1e9
    dec = u * args.steps / (ms_d / 1e3) / 1e9
    print(json.dumps({
        "metric": "uncompressed GB/s, FrameEncoder + FrameDecoder round trip (device resident)",
        "value": 2 * u * args.steps / ((ms_e + ms_d) / 1e3) / 1e9, "unit": "GB/s", "n_gpus": 1, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": (ms_e + ms_d) / args.steps, "higher_is_better": True, "dtype": "u8",
        "data": "synthetic", "side_measurement": True,
        "config": {"workload": "FrameEncoder/FrameDecoder over a %.0f GiB synthetic text stream in %d waves of %.1f GiB on 1 B200 (BASELINE configs[3])"
                               % (u / 2**30, nwaves, wave_bytes / 2**30), "stream_bytes": stream_bytes, "ratio": stream_bytes / u,
                   "input_pool_waves": pool_waves,
                   "parity": "every wave: decode(encode(x)) == x on device, statuses Ok; first 4 chunks == oracle FrameEncoder bytes"},
        "frame_encode_gbs": enc, "frame_decode_gbs": dec,
        "roofline": {"bound": "hbm", "kernel": "k1_m7_kernel (frame encode: K1 + fused CRC, scan, gather)", "achieved": (u + stream_bytes) * args.steps / (ms_e / 1e3) / 1e9,
                     "peak": peak, "unit": "GB/s", "frac": (u + stream_bytes) * args.steps / (ms_e / 1e3) / 1e9 / peak, "peak_source": peak_src, "traffic": None,
                     "k5_decode_kernel": {"achieved": (u + stream_bytes) * args.steps / (ms_d / 1e3) / 1e9,
                                          "frac": (u + stream_bytes) * args.steps / (ms_d / 1e3) / 1e9 / peak}},
        "clocks": clocks, "gpu_launches": int(L.sb_launch_count() - launches0)}), flush=True)


def run_urls(args, local_rank):
    """BASELINE configs[2]: urls.10K cut into 11 blocks, each compressed independently, tiled
    round-robin (compressed bytes physically replicated in HBM) and decoded by K2."""
    import numpy as np
    import torch
    import __graft_entry__ as graft
    from oracle import oracle as orc
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    snap = graft.load_package()
    L = snap._lib.lib()
    err = snap._lib.SbError()
    data = open(os.path.join(ROOT, "tests", "golden", "data", "urls.10K"), "rb").read()
    blocks = [data[i:i + BLOCK] for i in range(0, len(data), BLOCK)]
    comp = [orc.compress(b) for b in blocks]                  # input preparation, outside the timed region
    reps = int(args.urls_gib * (1 << 30)) // len(data)
    n = reps * len(blocks)
    clen = np.array([len(c) for c in comp], dtype=np.int64)
    tile = int(clen.sum())
    src = torch.frombuffer(bytearray(b"".join(comp)), dtype=torch.uint8).to(dev)
    t_c = src.repeat(reps)                                    # physical tiling of the compressed streams
    starts = np.concatenate([[0], np.cumsum(clen)[:-1]])
    base = (np.arange(reps, dtype=np.int64) * tile)[:, None] + starts[None, :]
    in_ptrs = torch.from_numpy(base.reshape(-1) + t_c.data_ptr()).to(dev)
    in_lens = torch.from_numpy(np.tile(clen, reps).astype(np.int32)).to(dev)
    t_out = torch.empty(n * BLOCK, dtype=torch.uint8, device=dev)
    t_dlen = torch.zeros(n, dtype=torch.int32, device=dev)
    t_st = torch.zeros(n * 4, dtype=torch.int64, device=dev)
    b = snap._lib.SbBatch()
    b.in_ptrs, b.in_lens = in_ptrs.data_ptr(), in_lens.data_ptr()
    b.out_base, b.out_stride, b.out_cap_uniform = t_out.data_ptr(), BLOCK, BLOCK
    b.out_lens, b.statuses, b.count = t_dlen.data_ptr(), t_st.data_ptr(), n
    stream = torch.cuda.current_stream().cuda_stream
    ev = torch.cuda.Event

    def step():
        e0, e1 = ev(enable_timing=True), ev(enable_timing=True)
        e0.record()
        if L.sb_decompress_batch_device(C.byref(b), stream, C.byref(err)):
            raise snap.error.from_c(err)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    for _ in range(max(3, args.warmup)):
        step()
    assert int(t_st.view(n, 4)[:, 0].abs().sum()) == 0
    view = t_out.view(reps, len(blocks), BLOCK)
    for k, blk in enumerate(blocks):                          # every tile decodes to the original bytes
        want = torch.frombuffer(bytearray(blk), dtype=torch.uint8).to(dev)
        assert bool((view[:, k, :len(blk)] == want).all())
    ms = sum(step() for _ in range(args.steps)) / args.steps
    u, c = reps * len(data), reps * tile
    peak, peak_src = measured_peak()
    print(json.dumps({
        "metric": "uncompressed GB/s, batched raw block decompress", "value": u / (ms / 1e3) / 1e9, "unit": "GB/s",
        "n_gpus": 1, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms, "higher_is_better": True,
        "dtype": "u8", "data": "data/urls.10K tiled", "side_measurement": True,
        "config": {"workload": "batched raw block decompress: data/urls.10K tiled to %.1f GiB (BASELINE configs[2])" % (u / 2**30),
                   "streams": n, "compressed_bytes": c, "ratio": c / u, "parity": "every stream equals its source block"},
        "roofline": {"bound": "hbm", "kernel": "k2_decompress_kernel", "achieved": (u + c) / (ms / 1e3) / 1e9, "peak": peak,
                     "unit": "GB/s", "frac": (u + c) / (ms / 1e3) / 1e9 / peak, "peak_source": peak_src, "traffic": None},
    }), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--blocks", type=int, default=1 << 20, help="64KB blocks per GPU (BASELINE configs[1]: 1M)")
    ap.add_argument("--wave", type=int, default=1 << 17, help="blocks per kernel launch")
    ap.add_argument("--e2e-blocks", type=int, default=1 << 18)
    ap.add_argument("--e2e-batches", type=int, default=1, help="e2e: batches pipelined through compress and decompress from two host threads (1 = sequential phases; measured: 8 batches 33.3, 16 batches 35.9, sequential 37.9 GB/s -- K1 owns every SM, so the overlap buys nothing)")
    ap.add_argument("--parity-samples", type=int, default=48)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--parity-seconds", type=float, default=20.0, help="host time budget of the full-coverage fingerprint check")
    ap.add_argument("--no-numa-bind", action="store_true")
    ap.add_argument("--no-shard", action="store_true", help="N>1: skip the frame-shard exchange sub-measurement")
    ap.add_argument("--shard-gib-per-rank", type=float, default=4.0)
    ap.add_argument("--workload", default="text-roundtrip", choices=["text-roundtrip", "urls-decompress", "frame", "frame-shard"],
                    help="side measurements: urls-decompress = BASELINE configs[2]; frame = configs[3] (--gib, default 256); "
                         "frame-shard = configs[4] (--gib total over all ranks, default 1024)")
    ap.add_argument("--urls-gib", type=float, default=64.0)
    ap.add_argument("--gib", type=float, default=None)
    ap.add_argument("--wave-gib", type=float, default=None)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="text-roundtrip: after the timed steps, write what the last step computed (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.workload != "text-roundtrip"):
        ap.error("--dump-outputs applies to --impl ours --workload text-roundtrip")
    if args.warmup < 3 and args.workload != "frame-shard":
        args.warmup = 3          # frame-shard steps are whole-stream passes (hundreds of waves each): --warmup 1 is accepted there
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.workload == "urls-decompress":
        run_urls(args, local_rank)
        return
    if args.workload == "frame":
        args.gib = args.gib or 256.0
        args.wave_gib = args.wave_gib or 4.0
        run_frame(args, local_rank)
        return
    if args.workload == "frame-shard":
        args.gib = args.gib or 1024.0
        args.wave_gib = args.wave_gib or 1.0
        run_frame_shard(args, rank, local_rank, world)
        return
    run_ours(args, rank, local_rank, world)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
