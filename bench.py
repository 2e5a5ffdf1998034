#!/usr/bin/env python3
"""bench.py -- the BASELINE.json metric: Mtexels/s of the BCn block-compression hot path.

A "step" is one pass of the hot path over one synthetic surface.  Default workload (N=1) is
BASELINE.json configs[1]: BC7 `GetProfile_slow`, 4096x4096 RGBA8 uniform-random texels.

  value     whole-job Mtexels/s with inputs resident in HBM (device-pointer entry itw_encode_device),
            timed on the device with CUDA events around every step, max over ranks.
  e2e       the same metric through the reference-facing C-ABI call CompressBlocksBC*(host surface,
            host dst): pinned host buffers, H2D + kernel + D2H inside the timed region.  With N > 1 it is
            ONE process (rank 0) issuing ONE call per step on a surface of N x 4096 rows, fanned over the N
            GPUs by the library (itw_set_devices) -- the other ranks idle at a barrier meanwhile.
  parity    the blocks the e2e call just produced, compared with what the CPU arm (oracle/_ref) produced
            for the same rows of the same surface.
  roofline  algorithmic bytes of the kernel / its CUDA-event duration, against the measured HBM peak
            in MEASURED_PEAKS.json (+ the issue-rate roofline of the compute-bound encoders).
  sweep     the rest of the metric: {BC1, BC3, BC6H slow, BC7 slow, BC7 basic} x {4096^2, 8192^2}.
  c4 / c5   BASELINE configs[3] (BC3 + mip chain 8192^2, row-sharded with ONE NCCL all-gather issued by the
            library) and configs[4] (tile stream of 1024^2 tiles through itw_encode_batch).
  cpu_baseline / --impl reference
            the reference's own encoder (oracle/_ref = kernel.ispc compiled scalar, else the oracle
            port) on the host cores, on a bounded sample of the same workload.

Multi-GPU (torchrun, one rank per GPU): blocks are independent, so for `value` each rank encodes its own
surface of the same shape (weak scaling, no data-path collective); NCCL carries the barrier, the
max-over-ranks reduction of the step times and config C4's all-gather.
"""
import argparse
import ctypes
import hashlib
import importlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
pkg = importlib.import_module("intel-texture-works-plugin_b200")
binding = importlib.import_module("intel-texture-works-plugin_b200.binding")

READ_BYTES_PER_TEXEL = {"BC1": 4, "BC3": 4, "BC4": 4, "BC5": 4, "BC7": 4, "BC6H": 8}
WRITE_BYTES_PER_TEXEL = {"BC1": 0.5, "BC4": 0.5, "BC3": 1, "BC5": 1, "BC7": 1, "BC6H": 1}
DEFAULT_PROFILE = {"BC7": "slow", "BC6H": "bc6h_slow"}
KERNEL_OF = {"BC7": "bc7_kernel", "BC6H": "bc6h_kernel", "BC1": "bc1_bc3_kernel", "BC3": "bc1_bc3_kernel",
             "BC4": "bc4_bc5_kernel", "BC5": "bc4_bc5_kernel"}
SWEEP = [("BC1", None), ("BC3", None), ("BC6H", "bc6h_slow"), ("BC7", "slow"), ("BC7", "basic")]


def make_surface(fmt, size, seed, height=None):
    h = height or size
    if fmt == "BC6H":
        return pkg.synth.random_rgba16f(h, size, seed=0xB2000003 + seed)
    return pkg.synth.random_rgba8(h, size, seed=0xB2000002 + seed)


def workload_name(fmt, prof, size):
    kind = "RGBA16F random" if fmt == "BC6H" else "RGBA8 random"
    return f"{fmt}{' ' + prof if prof else ''}, {size}x{size} {kind}"


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's own implementation on the host cores (test infrastructure under oracle/)
# ------------------------------------------------------------------------------------------------
def load_cpu_reference():
    """oracle/_ref (the reference's kernel.ispc + ispc_texcomp.cpp compiled scalar) if it exists,
    else the handwritten oracle port."""
    ref_so = os.path.join(ROOT, "oracle", "_ref", "libitw_ref.so")
    if os.path.exists(ref_so):
        return binding.EncoderApi(ref_so, ""), "reference"
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle")])
    return binding.EncoderApi(os.path.join(ROOT, "oracle", "libitw_oracle.so"), "oracle_"), "port"


def usable_cores():
    """Host threads this process may really use: the affinity mask, capped by the cgroup CPU quota
    (os.cpu_count() ignores both)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    quota = None
    try:                                                       # cgroup v2
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            quota = float(q) / float(p)
    except (OSError, ValueError):
        try:                                                   # cgroup v1
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / p
        except (OSError, ValueError):
            pass
    if quota:
        n = max(1, min(n, int(quota + 0.5)))
    return n


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def cpu_encode_mt(api, fmt, img, settings, threads):
    """Row-band split exactly like CompressImageMT (win32Threads.cpp:217-230): linesPerThread =
    ceil(h/T), bands rounded down to multiples of 4 rows, one band per thread."""
    h, w = img.shape[:2]
    bpb = binding.FORMATS[fmt][1]
    out = np.zeros((h // 4) * (w // 4) * bpb, np.uint8)
    lines = (h + threads - 1) // threads
    jobs = []
    for t in range(threads):
        y0 = (lines * t) // 4 * 4
        y1 = min((lines * (t + 1)) // 4 * 4, h)
        if y1 > y0:
            jobs.append((y0, y1))

    def work(job):
        y0, y1 = job
        api.encode_raw(fmt, img.ctypes.data + y0 * img.strides[0], w, y1 - y0, img.strides[0],
                       out.ctypes.data + (y0 // 4) * (w // 4) * bpb, settings)

    ts = [threading.Thread(target=work, args=(j,)) for j in jobs]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    return out


def cpu_sample_rows(api, fmt, img, settings, threads, target_s):
    """Rows of the workload that take about `target_s` seconds on `threads` host threads (calibrated
    on a small band first; the calibration pass doubles as warm-up)."""
    h, w = img.shape[:2]
    probe = min(h, 4 * threads)
    t0 = time.perf_counter()
    cpu_encode_mt(api, fmt, img[:probe], settings, threads)
    dt = max(time.perf_counter() - t0, 1e-4)
    rows = int(probe * target_s / dt)
    rows = max(4 * threads, min(h, rows // (4 * threads) * (4 * threads)))
    return min(rows, h // 4 * 4)


def run_cpu_arm(args, fmt, prof, size, full_json):
    """Times the CPU reference on the first `rows` rows of surface 0 of the workload.  Returns (info, median ms per
    sample step, rows, the blocks it produced) -- the blocks feed the GPU arm's parity check."""
    api, kind = load_cpu_reference()
    settings = api.profile(prof) if prof else None
    threads = usable_cores()
    img = make_surface(fmt, size, 0)
    if full_json:      # --impl reference: W + K steps of a bounded sample, about a minute in total
        per_step_s = 60.0 / max(args.steps + args.warmup, 1)
        steps, warm = args.steps, args.warmup
    else:              # cpu_baseline leg of the GPU arm: >= 3 repetitions, about 15 s in total
        per_step_s, steps, warm = 4.0, 3, 0
    rows = cpu_sample_rows(api, fmt, img, settings, threads, max(per_step_s, 0.25))
    band = img[:rows]
    out = None
    for _ in range(warm):
        cpu_encode_mt(api, fmt, band, settings, threads)
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        out = cpu_encode_mt(api, fmt, band, settings, threads)
        times.append(time.perf_counter() - t0)
    med = statistics.median(times)
    mtexels = rows * size / med / 1e6
    info = {"value": round(mtexels, 4), "unit": "Mtexels/s", "cores": threads, "kind": kind, "cpu": cpu_model(),
            "per_core": round(mtexels / threads, 5), "repetitions": steps,
            "ms_per_surface": round(med * 1e3 * size / rows, 1),
            "sample": f"first {rows} of {size} rows of surface 0 of the workload per step, median of {steps} steps, row-band split of "
                      f"CompressImageMT over {threads} threads (affinity and cgroup quota respected); scalar strict-IEEE build of the "
                      f"reference source, not the ISPC SIMD binary; ms_per_surface extrapolates the sample to all {size} rows"}
    return info, med * 1e3, rows, out


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def count(self, t0=0.0):
        return sum(1 for t, _ in self.lines if t >= t0)

    def stop(self, t0=0.0, t1=float("inf"), window="timed region"):
        """Summary of the samples that arrived in [t0, t1] (perf_counter times)."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 6 or t < t0 or t > t1:
                continue
            try:
                sm.append(float(parts[0]))
                smax = float(parts[1])
            except ValueError:
                continue
            for n, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm), "window": window}


# ------------------------------------------------------------------------------------------------
# GPU arm helpers
# ------------------------------------------------------------------------------------------------
class Gpu:
    """Everything the measurements share: the library, torch, the rank layout."""

    def __init__(self, torch, dist, lib, rank, world, local_rank):
        self.torch, self.dist, self.lib = torch, dist, lib
        self.rank, self.world, self.local_rank = rank, world, local_rank
        self.stream = torch.cuda.current_stream()
        self.host_group = dist.new_group(backend="gloo") if world > 1 else None
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            self.peak = float(json.load(open(peaks_path))["hbm_gbs"])
            self.peak_src = "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
        else:
            self.peak, self.peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
        path = os.path.join(ROOT, "profiles", "dram_traffic.json")
        self.counters = json.load(open(path)) if os.path.exists(path) else {}
        self.sms = torch.cuda.get_device_properties(local_rank).multi_processor_count

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def host_barrier(self):
        """CPU-only rendezvous (gloo): used while rank 0 drives ALL GPUs from one process -- an NCCL barrier would park a
        spinning kernel on the other ranks' GPUs and take SMs away from the work being timed."""
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier(group=self.host_group)

    def max_over_ranks(self, x):
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def to_device(self, host):
        return self.torch.from_numpy(host.view(np.uint8).reshape(-1)).cuda()

    def pin(self, host):
        return self.torch.from_numpy(host.view(np.uint8).reshape(-1)).pin_memory()

    def device_ms(self, fmt, settings, d_in, width, height, d_out, steps, warm):
        """Average CUDA-event time of `steps` device-resident encodes, rotating over the inputs in d_in."""
        torch = self.torch
        texel = binding.FORMATS[fmt][2]

        def step(i):
            self.lib.encode_device(fmt, d_in[i % len(d_in)].data_ptr(), width, height, width * texel, d_out.data_ptr(), settings,
                                   self.stream.cuda_stream)
        for i in range(warm):
            step(i)
        self.barrier()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for i in range(steps):
            evs[i][0].record(self.stream)
            step(warm + i)
            evs[i][1].record(self.stream)
        self.barrier()
        return sum(a.elapsed_time(b) for a, b in evs) / steps

    def e2e_ms(self, fmt, settings, h_in, width, height, h_out, steps, warm):
        """Wall-clock time per CompressBlocks<fmt>(host surface, host dst) call, pinned buffers."""
        texel = binding.FORMATS[fmt][2]
        for _ in range(warm):
            self.lib.encode_raw(fmt, h_in.data_ptr(), width, height, width * texel, h_out.data_ptr(), settings)
        self.torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            self.lib.encode_raw(fmt, h_in.data_ptr(), width, height, width * texel, h_out.data_ptr(), settings)
        return (time.perf_counter() - t0) / steps * 1e3

    def fractions(self, fmt, prof, size, ms, sm_mhz):
        texels = size * size
        algo = texels * (READ_BYTES_PER_TEXEL[fmt] + WRITE_BYTES_PER_TEXEL[fmt])
        hbm = algo / (ms * 1e-3) / 1e9 / self.peak
        winst = self.counters.get("warp_inst", {}).get(f"{fmt}:{prof}:{size}")
        issue = None
        if winst and sm_mhz:
            issue = winst / (ms * 1e-3) / (4.0 * self.sms * sm_mhz * 1e6)
        return algo, hbm, issue, winst


def run_sweep(g, args, hosts4096, sm_mhz, e2e_devices):
    """{BC1, BC3, BC6H slow, BC7 slow, BC7 basic} x {4096^2, 8192^2}: device-resident and end-to-end Mtexels/s,
    HBM and issue-rate fractions.  Inputs: 4096^2 RGBA8 rotates over 4 surfaces (256 MiB > L2), 4096^2 RGBA16F over 2
    (256 MiB), an 8192^2 surface (256 / 512 MiB) is larger than L2 by itself."""
    torch = g.torch
    out = []
    cache = {}

    def inputs(fmt, size):
        key = ("f16" if fmt == "BC6H" else "u8", size)
        if key not in cache:
            cache.clear()                                     # one family resident at a time (HBM and pinned host memory)
            torch.cuda.empty_cache()
            if size == 4096 and key[0] == "u8":
                hs = hosts4096
            else:
                n = 2 if size == 4096 else 1
                hs = [make_surface(fmt, size, 16 * g.rank + i) for i in range(n)]
            cache[key] = (hs, [g.to_device(h) for h in hs], g.pin(hs[0]) if g.rank == 0 else None)
        return cache[key]

    order = sorted(((f, p, s) for s in (4096, 8192) for f, p in SWEEP), key=lambda t: (t[2], t[0] == "BC6H"))
    for fmt, prof, size in order:
        hs, d_in, h_in = inputs(fmt, size)
        settings = g.lib.profile(prof) if prof else None
        bpb = binding.FORMATS[fmt][1]
        out_bytes = (size // 4) ** 2 * bpb
        d_out = torch.empty(out_bytes, dtype=torch.uint8, device="cuda")
        fast = fmt in ("BC1", "BC3")
        ms = g.device_ms(fmt, settings, d_in, size, size, d_out, steps=20 if fast else 3, warm=3)
        ms = g.max_over_ranks(ms)
        entry = {"format": fmt, "profile": prof, "size": size, "ms": round(ms, 4),
                 "mtexels_s": round(size * size * g.world / ms / 1e3, 1)}
        algo, hbm, issue, winst = g.fractions(fmt, prof, size, ms, sm_mhz)
        entry["hbm_frac"] = round(hbm, 6)
        entry["issue_frac"] = round(issue, 3) if issue else None
        entry["dram_bytes"] = g.counters.get(f"{fmt}:{prof}:{size}")
        g.host_barrier()
        if g.rank == 0:
            h_out = torch.empty(out_bytes, dtype=torch.uint8).pin_memory()
            e = g.e2e_ms(fmt, settings, h_in, size, size, h_out, steps=5 if fast else 2, warm=1)
            entry["e2e_mtexels_s"] = round(size * size / e / 1e3, 1)
            if e2e_devices > 1:                               # the same call fanned over all GPUs by the library (strong scaling)
                g.lib.set_devices(list(range(e2e_devices)))
                e = g.e2e_ms(fmt, settings, h_in, size, size, h_out, steps=5 if fast else 2, warm=1)
                g.lib.set_devices([])
                entry["e2e_all_gpus_mtexels_s"] = round(size * size / e / 1e3, 1)
            del h_out
        g.host_barrier()
        out.append(entry)
        del d_out
    cache.clear()
    torch.cuda.empty_cache()
    return out


def run_c4(g):
    """BASELINE configs[3]: BC3 + full mip chain of an 8192^2 RGBA8 texture, level 0 row-sharded over the ranks, ONE
    ncclAllGather issued by the library (itw_encode_mip_chain_sharded); rank 0 compares the chain with its own
    single-GPU encode of the whole texture (itw_dds_encode_texture payload)."""
    torch, lib = g.torch, g.lib
    sharding = importlib.import_module("intel-texture-works-plugin_b200.sharding")
    n, levels = 8192, 14
    y0, y1 = sharding.band_rows(n, g.world, g.rank)
    base = pkg.synth.mixed_rgba8(n, n) if g.rank == 0 else None
    band_host = base[y0:y1] if g.rank == 0 else _mixed_rows(n, y0, y1)   # the other ranks generate only their own rows
    band = torch.from_numpy(np.ascontiguousarray(band_host).reshape(-1)).cuda()
    if g.world > 1:
        sharding.shard_init(lib)
    chain, plan = sharding.encode_mip_chain_sharded(lib, "BC3", band, n, n, levels)
    for _ in range(2):
        sharding.encode_mip_chain_sharded(lib, "BC3", band, n, n, levels, chain=chain)
    g.barrier()
    reps = 5
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.perf_counter()
    e0.record(g.stream)
    for _ in range(reps):
        sharding.encode_mip_chain_sharded(lib, "BC3", band, n, n, levels, chain=chain)
    e1.record(g.stream)
    torch.cuda.synchronize()
    wall = (time.perf_counter() - w0) / reps * 1e3
    ms = g.max_over_ranks(e0.elapsed_time(e1) / reps)
    wall = g.max_over_ranks(wall)
    res = None
    if g.rank == 0:
        d = pkg.DdsDesc(n, n, levels, 1, 77, 0)
        whole = lib.dds_encode_texture(d, [base])
        hdr = lib.lib.itw_dds_header_bytes(ctypes.byref(d))
        got = chain.cpu().numpy()
        texels = sum(max(n >> l, 1) ** 2 for l in range(levels))
        res = {"config": f"BC3 + {levels}-level mip chain {n}x{n}, row-sharded over {g.world} GPU(s), one ncclAllGather in the library",
               "ms": round(ms, 4), "wall_ms": round(wall, 4), "mtexels_s": round(texels / ms / 1e3, 1),
               "allgather_bytes_per_rank": int(plan.slot_bytes), "band_levels": int(plan.band_levels),
               "equals_single_gpu": bool(np.array_equal(got, whole[hdr:])),
               "sha256": hashlib.sha256(got.tobytes()).hexdigest()}
    if g.world > 1:
        sharding.shard_finalize(lib)
    del chain, band
    return res


def _mixed_rows(n, y0, y1):
    """Rows [y0, y1) of synth.mixed_rgba8(n, n) without building the whole image."""
    x = np.arange(n, dtype=np.int64)[None, :]
    y = np.arange(y0, y1, dtype=np.int64)[:, None]
    img = np.empty((y1 - y0, n, 4), np.uint8)
    img[..., 0] = (x ^ y) & 255
    img[..., 1] = ((3 * x + 5 * y) >> 6) & 255
    with np.errstate(over="ignore"):
        ctr = np.uint64(0xB2000004) + (np.arange(y0 * n, y1 * n, dtype=np.uint64))
    img[..., 2] = (pkg.synth.splitmix64(ctr) & np.uint64(255)).astype(np.uint8).reshape(y1 - y0, n)
    img[..., 3] = ((x + y) >> 6) & 255
    return img


def run_c5(g, devices):
    """BASELINE configs[4]: BC7 basic, 1024 independent 1024^2 RGBA8 tiles streamed through ONE itw_encode_batch call of
    ONE process (tiles dealt round-robin over `devices` GPUs, three copy/compute lanes per GPU, no collective).  The host
    holds 64 distinct pinned tiles (even: random, odd: gradient with a per-tile phase -- SURVEY.md 8d) which the batch
    cycles through 16 times; every tile has its own pinned destination.  Parity of the first 8 tiles is checked against
    single-tile encodes."""
    torch, lib = g.torch, g.lib
    ntiles, distinct, ts = 1024, 64, 1024
    settings = lib.profile("basic")
    tiles = [pkg.synth.c5_tile(t, ts) for t in range(distinct)]
    pins = [g.pin(t) for t in tiles]
    out_bytes = (ts // 4) ** 2 * 16
    outs = torch.empty(ntiles * out_bytes, dtype=torch.uint8).pin_memory()
    surfaces = [(pins[i % distinct].data_ptr(), ts, ts, ts * 4) for i in range(ntiles)]
    dsts = [outs.data_ptr() + i * out_bytes for i in range(ntiles)]
    if devices > 1:
        lib.set_devices(list(range(devices)))
    lib.encode_batch("BC7", surfaces[:128], dsts[:128], settings)                  # warm-up: buffers, streams
    t0 = time.perf_counter()
    lib.encode_batch("BC7", surfaces, dsts, settings)
    dt = time.perf_counter() - t0
    if devices > 1:
        lib.set_devices([])
    ok = True
    for i in (0, 1, 2, 3, 64, 65, 1022, 1023):
        want = lib.encode("BC7", tiles[i % distinct], settings)
        ok = ok and np.array_equal(outs[i * out_bytes:(i + 1) * out_bytes].numpy(), want)
    return {"config": f"BC7 basic, {ntiles} tiles of {ts}x{ts} RGBA8 ({distinct} distinct pinned host tiles cycled), one itw_encode_batch call, "
                      f"{devices} GPU(s), one process", "mtexels_s": round(ntiles * ts * ts / dt / 1e6, 1), "seconds": round(dt, 3),
            "h2d_bytes": ntiles * ts * ts * 4, "d2h_bytes": ntiles * out_bytes, "tiles_equal_single_encodes": bool(ok)}


def dump_outputs(out_dir, blocks, fmt, size, bpb, limit=48 << 20):
    """What the timed device path returned in its last step, for output-for-output comparison of two builds:
    `blocks.npy` holds the encoded blocks as float32 (block rows x blocks per row x bytes per block, values 0..255).  Above
    `limit` bytes as float32 it holds a fixed sample of block rows (seed 0, sorted), whose indices `block_rows.npy` lists."""
    rows = size // 4
    grid = blocks.reshape(rows, size // 4, bpb)
    keep = np.arange(rows)
    if grid.size * 4 > limit:
        n = max(1, limit // (grid[0].size * 4))
        keep = np.sort(np.random.default_rng(0).choice(rows, size=n, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "blocks.npy"), grid[keep].astype(np.float32))
    np.save(os.path.join(out_dir, "block_rows.npy"), keep.astype(np.float64))


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--format", default="BC7", choices=sorted(binding.FORMATS))
    ap.add_argument("--profile", default=None)
    ap.add_argument("--size", type=int, default=4096)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (and with it the parity object)")
    ap.add_argument("--no-extras", action="store_true", help="skip sweep / c4 / c5 (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the blocks of the last timed step to DIR/*.npy (float32; a fixed sample of block rows above 48 MiB)")
    args = ap.parse_args()
    fmt = args.format
    prof = args.profile or DEFAULT_PROFILE.get(fmt)
    size = args.size
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # identical in both arms (the driver compares it): the workload only
    config = {"workload": workload_name(fmt, prof, size), "format": fmt, "profile": prof, "width": size, "height": size,
              "sharding": "one surface per GPU, no collective" if world > 1 else "single GPU"}

    if args.impl == "reference":
        if rank != 0:
            return
        info, ms, rows, _ = run_cpu_arm(args, fmt, prof, size, full_json=True)
        line = {"impl": "reference", "metric": "Mtexels/s", "value": info["value"], "unit": "Mtexels/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 3),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config, "cpu_baseline": info,
                "e2e": {"value": info["value"], "unit": "Mtexels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0,
                "note": f"a step encodes {rows} of {size} rows (bounded sample); ms_per_step is that sample's median time, "
                        f"cpu_baseline.ms_per_surface the extrapolation to a whole surface"}
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    lib = pkg.ItwBcn()
    lib.set_device(local_rank)
    g = Gpu(torch, dist, lib, rank, world, local_rank)
    settings = lib.profile(prof) if prof else None
    _, bpb, texel_bytes, _ = binding.FORMATS[fmt]
    out_bytes = (size // 4) * (size // 4) * bpb
    in_bytes = size * size * texel_bytes

    # Inputs resident in HBM.  A rotation of distinct surfaces larger than L2 in total, so a step
    # never finds its input in the 126 MB L2 left there by the previous step.
    nrot = max(2, -(-(256 << 20) // in_bytes))
    l2_policy = f"rotation of {nrot} distinct input surfaces ({nrot * in_bytes >> 20} MiB > 126 MB L2)"
    hosts = [make_surface(fmt, size, 16 * rank + i) for i in range(nrot)]
    d_in = [g.to_device(h) for h in hosts]
    d_out = torch.empty(out_bytes, dtype=torch.uint8, device="cuda")
    stream = g.stream

    def step(i):
        lib.encode_device(fmt, d_in[i % nrot].data_ptr(), size, size, size * texel_bytes, d_out.data_ptr(), settings,
                          stream.cuda_stream)

    # nvidia-smi needs a second or more before its first line (longer on an 8-GPU box): started before the warm-up, and only the
    # samples that arrive inside the timed region count
    sampler = ClockSampler(local_rank)
    sampler.start()
    for i in range(args.warmup):
        step(i)
    g.barrier()
    launches0 = lib.launch_count()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    wall0 = time.perf_counter()
    for i in range(args.steps):
        evs[i][0].record(stream)
        step(args.warmup + i)
        evs[i][1].record(stream)
    g.barrier()
    wall1 = time.perf_counter()
    wall = wall1 - wall0
    launches_timed = lib.launch_count() - launches0
    if sampler.count(wall0) >= 3 or not sampler.proc:
        clocks = sampler.stop(wall0, wall1)
    else:
        # a timed region shorter than a few 100 ms sampling periods: the same steps keep running (untimed) until three samples
        # have been taken under that load; they write to a spare buffer, so that d_out keeps the last timed step's blocks
        i, limit = args.warmup + args.steps, time.perf_counter() + 6.0
        d_spare = torch.empty_like(d_out)
        while sampler.count(wall1) < 3 and time.perf_counter() < limit:
            for _ in range(4):
                lib.encode_device(fmt, d_in[i % nrot].data_ptr(), size, size, size * texel_bytes, d_spare.data_ptr(), settings,
                                  stream.cuda_stream)
                i += 1
            stream.synchronize()
        del d_spare
        clocks = sampler.stop(wall0, window="timed region + the same steps continued until 3 samples")
    g.barrier()
    launches = launches_timed
    dev_ms = g.max_over_ranks(sum(a.elapsed_time(b) for a, b in evs))
    ms_per_step = dev_ms / args.steps
    texels_per_step = size * size * world
    value = texels_per_step / (ms_per_step * 1e-3) / 1e6
    last_blocks = d_out.cpu().numpy() if rank == 0 else None              # the last timed step: surface (warmup+steps-1) % nrot
    device_digest = hashlib.sha256(last_blocks.tobytes()).hexdigest() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, last_blocks, fmt, size, bpb)

    # ---- end to end through the reference-facing C-ABI with pinned host buffers: ONE process, ONE call per step ----
    # N = 1: CompressBlocks<fmt>(4096 x 4096 host surface).  N > 1: rank 0 alone calls CompressBlocks<fmt> on a surface of
    # N x 4096 rows (rows 0..4095 = surface 0 of the workload) after itw_set_devices(0..N-1); the library cuts it into one
    # band per GPU.  The other ranks wait at the barrier.
    e2e = None
    parity = None
    cpu_info = None
    e2e_steps = args.steps
    g.host_barrier()
    if rank == 0:
        tall = np.concatenate([hosts[0]] + [make_surface(fmt, size, 1000 + i) for i in range(1, world)]) if world > 1 else hosts[0]
        h_in = g.pin(tall)
        h_out = torch.empty(out_bytes * world, dtype=torch.uint8).pin_memory()
        if world > 1:
            lib.set_devices(list(range(world)))
        e2e_ms = g.e2e_ms(fmt, settings, h_in, size, size * world, h_out, steps=e2e_steps, warm=min(args.warmup, 2))
        e2e = {"value": round(texels_per_step / e2e_ms / 1e3, 3), "unit": "Mtexels/s", "h2d_bytes_per_step": in_bytes * world,
               "d2h_bytes_per_step": out_bytes * world, "steps": e2e_steps, "calls_per_step": 1, "processes": 1, "gpus": world,
               "surface": f"{size}x{size * world}"}
        got = h_out.numpy().copy()
        assert int(got[:4096].astype(np.int64).sum()) != 0, "encoder produced an empty output"
        if world > 1:                                         # the fanned-out call against the same call on ONE GPU
            lib.set_devices([])
            lib.encode_raw(fmt, h_in.data_ptr(), size, size * world, size * texel_bytes, h_out.data_ptr(), settings)
            e2e["equals_single_gpu"] = bool(np.array_equal(got, h_out.numpy()))
        # ---- parity: the CPU arm encodes the first rows of the same surface; compare block for block ----
        # N = 1: the rows of the cpu_baseline leg (>= 3 timed repetitions).  N > 1: the spec keeps the cpu_baseline leg to
        # N = 1, so a fixed 256-row (64 block rows) sample is encoded once, for the comparison only.
        if not args.no_cpu:
            if world == 1:
                cpu_info, _, rows, cpu_blocks = run_cpu_arm(args, fmt, prof, size, full_json=False)
                against = cpu_info["kind"]
            else:
                api, against = load_cpu_reference()
                rows = min(256, size)
                cpu_blocks = cpu_encode_mt(api, fmt, hosts[0][:rows], api.profile(prof) if prof else None, usable_cores())
            nblk = (rows // 4) * (size // 4)
            a = got[:nblk * bpb].reshape(nblk, bpb)
            b = cpu_blocks[:nblk * bpb].reshape(nblk, bpb)
            parity = {"blocks_checked": int(nblk), "block_rows_checked": rows // 4, "mismatches": int((a != b).any(1).sum()),
                      "against": "oracle/_ref" if against == "reference" else "oracle port",
                      "what": "output of the timed e2e call (rows of host surface 0) vs the CPU reference on the same rows",
                      "sha256_e2e_output": hashlib.sha256(got.tobytes()).hexdigest(), "sha256_last_device_output": device_digest}
            if world == 1 and (args.warmup + args.steps - 1) % nrot == 0:
                parity["device_equals_e2e"] = bool(device_digest == parity["sha256_e2e_output"])
        del h_in, h_out
    g.host_barrier()

    # ---- the rest of the metric ----
    sweep = c4 = c5 = None
    if not args.no_extras and fmt == "BC7" and size == 4096:
        hosts4 = hosts if (fmt != "BC6H" and len(hosts) >= 4) else [make_surface("BC7", 4096, 16 * rank + i) for i in range(4)]
        del d_in, d_out
        torch.cuda.empty_cache()
        sweep = run_sweep(g, args, hosts4, clocks.get("sm_mhz"), world)
        c4 = run_c4(g)
        g.host_barrier()
        if rank == 0:
            c5 = run_c5(g, world)
        g.host_barrier()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    algo_bytes, hbm_frac, issue_frac, winst = g.fractions(fmt, prof, size, ms_per_step, clocks.get("sm_mhz"))
    achieved = algo_bytes / (ms_per_step * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": round(achieved, 3), "peak": g.peak, "unit": "GB/s", "frac": round(achieved / g.peak, 6),
                "traffic": g.counters.get(f"{fmt}:{prof}:{size}"), "traffic_source": "ncu dram__bytes_read+write per launch, profiles/dram_traffic.json",
                "peak_source": g.peak_src, "kernel": KERNEL_OF[fmt], "algorithmic_bytes_per_launch": int(algo_bytes),
                "note": "read-only variant: %.3f GB/s" % (size * size * READ_BYTES_PER_TEXEL[fmt] / (ms_per_step * 1e-3) / 1e9)}
    if issue_frac:
        # The encoders are issue-bound, not HBM-bound (DESIGN.md section 4): alongside the required HBM roofline, the
        # warp-instruction issue rate against 4 schedulers x SM count x the SM clock sampled DURING the timed region.
        peak_issue = 4.0 * g.sms * clocks["sm_mhz"] * 1e6
        roofline["issue"] = {"warp_inst_per_launch": int(winst), "achieved_ginst_s": round(winst / (ms_per_step * 1e-3) / 1e9, 1),
                             "peak_ginst_s": round(peak_issue / 1e9, 1), "frac": round(issue_frac, 3),
                             "note": "4 warp schedulers/SM x SMs x median SM clock under load; instruction count from profiles/"}

    line = {"metric": "Mtexels/s", "value": round(value, 3), "unit": "Mtexels/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(ms_per_step, 4), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config, "l2_policy": l2_policy,
            "e2e": e2e, "gpu_launches": int(launches) * world, "clocks": clocks, "roofline": roofline, "parity": parity,
            "cpu_baseline": cpu_info, "wall_ms_per_step": round(wall / args.steps * 1e3, 4), "sweep": sweep, "c4": c4, "c5": c5}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
