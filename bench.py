#!/usr/bin/env python
"""bench.py -- complex IQ MSamples/s through the FFT-waterfall + 8-VFO WFM chain (BASELINE.json metric).

One "step" = one pass of the hot path over one chunk of synthetic IQ (BASELINE config 2: 100 MS/s stream,
1,048,576-point Nuttall FFT @ 20 fps, 8 WFM VFOs at +-5/15/25/35 MHz -> 250 kS/s stereo audio each).

  value     whole-job throughput with the chunks already resident in HBM (cf32), timed with CUDA events on the
            stream the kernels run on, max over ranks
  e2e       the same metric through the reference-facing C-ABI call with HOST (pinned) buffers: every step
            copies its IQ chunk host->device and its audio / FFT lines device->host inside the timed region.
            Reported for int16 IQ (file_source's native format, 4 B/sample) as the headline and for cf32.
  roofline  dominant kernel (stage 1: translate + first decimation of all VFOs, IQ read once): algorithmic bytes
            per launch / its device time measured live with CUDA events (b200_fe_s1_stats)
  cpu_baseline  the reference's own blocks (oracle/_ref/ref_pipeline: reference headers + restated VOLK/FFT leaf
            kernels, one thread per block, SpeedTester method) timed on this box's host cores

N > 1 (torchrun): N independent IQ streams, one full front end per GPU, no collective on the data path
(BASELINE config 5 style replicas) -> weak scaling, value = sum over ranks / max time.
`--impl reference` times the reference CPU path only (rank 0).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FS = 100e6
OFFSETS = [5e6, -5e6, 15e6, -15e6, 25e6, -25e6, 35e6, -35e6]
FFT_SIZE, FFT_RATE = 1 << 20, 20.0
WORKLOAD = "C2: 100 MS/s complex IQ, 1048576-pt Nuttall FFT @20 fps + 8 VFO WFM (250 kS/s, 150 kHz, mono+LPF)"
# algorithmic bytes per input sample (SURVEY.md 8d): read IQ once + 8 stereo outputs + dB lines
ALGO_BYTES_PER_SAMPLE = 8.0 + 8 * 8 * (250e3 / FS) + 4.0 * FFT_SIZE * FFT_RATE / FS     # = 9.0
# fp32 work per input sample in stage 1 as executed (complex taps): 8 VFOs * ceil-padded taps / D * 4 FMA
METRIC = "complex IQ MSamples/s through FFT + 8-VFO WFM chain"


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [c.strip() for c in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def bind_to_gpu_numa(local):
    """Run this process (and first-touch its pinned buffers) on the CPUs of the GPU's own NUMA node."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        with open("/sys/bus/pci/devices/%s/local_cpulist" % bdf) as f:
            txt = f.read().strip()
        cpus = set()
        for part in txt.split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return "%s -> cpus %s" % (bdf, txt)
    except Exception as ex:       # noqa: BLE001
        return "unbound (%r)" % (ex,)
    return "unbound"


def pcie_probe(torch, nbytes=256 << 20):
    """Plain pinned<->device copy bandwidth of this box: the ceiling of the end-to-end legs."""
    h = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    d = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    res = {}
    for name, (dst, src) in (("h2d_gbs", (d, h)), ("d2h_gbs", (h, d))):
        dst.copy_(src, non_blocking=True)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(4):
            dst.copy_(src, non_blocking=True)
        e1.record()
        torch.cuda.synchronize()
        res[name] = 4 * nbytes / (e0.elapsed_time(e1) * 1e-3) / 1e9
    return res


def measured_peak_hbm():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except (OSError, KeyError, ValueError):
        return 6650.0, "fallback (B200_PROFILING.md)"


DUMP_BYTES = 60e6


def dump_outputs(path, arrays):
    """Writes {name: float32 array} as path/<name>.npy.  Above DUMP_BYTES in all, every array keeps the same share of its
    rows, drawn with a fixed seed and kept in order, so that two builds given the same arguments write the same rows."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    keep = min(1.0, DUMP_BYTES / max(sum(a.nbytes for a in arrays.values()), 1))
    rng = np.random.default_rng(0x5D12)
    for name, a in arrays.items():
        if keep < 1.0:
            a = a[np.sort(rng.choice(a.shape[0], int(a.shape[0] * keep), replace=False))]
        np.save(os.path.join(path, name + ".npy"), a)


def cpu_reference_run(duration_ms, nvfo=8):
    """Times the reference's own blocks on the host cores.  Returns (samples_per_s, threads, kind, what)."""
    # -march=native build first (AVX-512 where the container had it); the x86-64-v3 build if that one cannot run here
    for name, flags in (("ref_pipeline", "-O3 -march=native of the build container"), ("ref_pipeline_v3", "-O3 -march=x86-64-v3")):
        exe = os.path.join(ROOT, "oracle", "_ref", name)
        if not os.path.exists(exe):
            continue
        out = subprocess.run([exe, str(FS), "500000", str(FFT_SIZE), str(FFT_RATE), str(nvfo), str(int(duration_ms)), "wfm"],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=duration_ms / 1000.0 * 3 + 120)
        rows = [l for l in out.stdout.strip().splitlines() if l and not l.startswith("[")]
        if out.returncode != 0 or not rows:
            continue
        last = rows[-1].split()
        return float(last[0]), int(last[1]), "reference", ("reference dsp headers + restated VOLK-generic/FFT leaf kernels (%s), one thread per block, "
                                                           "SpeedTester method, chunk 500000, %d ms" % (flags, duration_ms))
    # port: the plain-C restatement, single thread, bounded sample
    import numpy as np
    from oracle.oracle import Oracle, available
    o = Oracle("restatement_fast" if available("restatement_fast") else "restatement")
    n = 2000000
    rng = np.random.default_rng(0x5D12)
    x = rng.uniform(-1, 1, 2 * n).astype(np.float32)
    blocks = [(o.rxvfo(FS, 250e3, 150e3, off), o.wfm(75e3, 250e3, False, True)) for off in OFFSETS[:nvfo]]
    t0 = time.perf_counter()
    for i in range(0, n, 500000):
        seg = x[2 * i: 2 * (i + 500000)]
        for v, d in blocks:
            d.process(v.process(seg))
    o.fft_frame(FFT_SIZE, FFT_SIZE, 2, x[: 2 * FFT_SIZE].view(np.complex64))
    dt = time.perf_counter() - t0
    return n / dt, 1, "port", "plain-C restatement (oracle/liboracle), single thread, %d samples" % n


def run_reference(args):
    rank = env_int("RANK", 0)
    if rank != 0:
        return 0
    total = args.steps + args.warmup
    step_ms = max(500, min(3000, int(150000 / max(total, 1))))
    vals = []
    threads = kind = what = None
    for i in range(total):
        v, threads, kind, what = cpu_reference_run(step_ms)
        if i >= args.warmup:
            vals.append(v)
    v = sum(vals) / len(vals) / 1e6
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "MS/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "chunk_samples": 500000, "note": "reference chunk cap STREAM_BUFFER_SIZE=1e6"},
            "cpu_baseline": {"value": v, "unit": "MS/s", "cores": threads, "host_cpus": os.cpu_count(), "kind": kind, "sample": what},
            "e2e": {"value": v, "unit": "MS/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line))
    return 0


C4_FS = 1.024e9
C4_WORKLOAD = "C4: 1.024 GS/s complex IQ, 64 mixed AM/NFM/USB VFOs on a 12.5 MHz grid (+ 1048576-pt FFT on rank 0), VFO groups per GPU, raw IQ broadcast over NCCL"


def c4_vfos(sb, lib):
    """BASELINE config 4: 64 VFOs, offsets k * 12.5 MHz (k = -32..-1, 1..32), modes cycling AM / NFM / USB."""
    ks = list(range(-32, 0)) + list(range(1, 33))
    mk = [lambda o: sb.VfoConfig.am(o), lambda o: sb.VfoConfig.nfm(o), lambda o: sb.VfoConfig.ssb(o, lib.DEMOD_USB)]
    return [mk[i % 3](12.5e6 * k) for i, k in enumerate(ks)]


def c4_leg(torch, dist, sb, lib, rank, world, local, steps, warm=3, chunk=1 << 23):
    """Strong scaling of ONE stream: the same 64 VFOs + FFT whatever the GPU count; rank 0 owns the stream, the library
    broadcasts every raw chunk (b200_shard_*), every rank demodulates its VFO group.  value = samples / max-over-ranks time."""
    import ctypes as C
    from sdrplusplus_b200.sharding import ShardedFrontEnd, make_unique_id, partition_vfos
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        cfgs = c4_vfos(sb, lib)
        mine = partition_vfos(len(cfgs), world, rank)
        fe = sb.FrontEnd(C4_FS, chunk)
        fe.set_stream(stream.cuda_stream)
        if rank == 0:
            fe.set_fft(FFT_SIZE, FFT_RATE, lib.WIN_NUTTALL)
        ids = [fe.add_vfo(cfgs[i]) for i in mine]
        uid = [make_unique_id() if rank == 0 else None]
        if world > 1:
            dist.broadcast_object_list(uid, src=0)
        sh = ShardedFrontEnd(fe, rank, world, uid[0])
        gen = torch.Generator(device="cuda")
        gen.manual_seed(0xC4)
        ins = [(torch.rand(2 * chunk, device="cuda", generator=gen, dtype=torch.float32) * 2.0 - 1.0) for _ in range(3)] if rank == 0 else []
        outs = []
        for _ in range(2):
            o = lib.Outputs()
            keep = []
            for v in ids:
                cap = fe.vfo_max_out(v, chunk)
                t = torch.empty(2 * cap, device="cuda", dtype=torch.float32)
                keep.append(t)
                o.vfo_out[v] = t.data_ptr()
                o.vfo_cap[v] = cap
            nl = max(1, fe.fft_max_lines(chunk))
            t = torch.empty(nl * FFT_SIZE, device="cuda", dtype=torch.float32)
            keep.append(t)
            o.fft_out = t.data_ptr()
            o.fft_cap_lines = nl
            o.out_mem = lib.MEM_DEVICE
            outs.append((o, keep))

        def loop(n):
            infl = 0
            for i in range(n):
                ptr = ins[i % 3].data_ptr() if rank == 0 else 0
                sh.submit_ptr(ptr, chunk, lib.FMT_CF32, lib.MEM_DEVICE, outs[i % 2][0])
                infl += 1
                if infl == 2:
                    sh.wait()
                    infl -= 1
            while infl:
                sh.wait()
                infl -= 1

        loop(warm)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        b0 = sh.bytes_broadcast()
        l0 = fe.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        loop(steps)
        e1.record(stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            dist.barrier()
            t = torch.tensor([ms], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t[0])
        res = {"workload": C4_WORKLOAD, "scaling": "strong", "value": chunk * steps / (ms * 1e-3) / 1e6, "unit": "MS/s", "n_gpus": world,
               "ms_per_step": ms / steps, "steps": steps, "chunk_samples": chunk, "vfos_total": len(cfgs), "vfos_this_rank": len(ids),
               "collective": "ncclBroadcast of the raw chunk from rank 0 (b200_shard_submit), one chunk ahead of the compute" if world > 1 else "none (one GPU)",
               "nvlink_bytes_per_step_per_receiver": (sh.bytes_broadcast() - b0) // max(steps, 1), "gpu_launches_rank0": int(fe.launch_count() - l0),
               "timing": "CUDA events on each rank's stream, max over ranks"}
        sh.close()
        fe.close()
    return res


def c3_leg(torch, lib, steps=60, chunk=1 << 20):
    """BASELINE config 3: 256-channel polyphase filter-bank channelizer, 127 taps per branch (500 MS/s class stream), chunks of
    1 Mi samples resident in HBM, outputs to HBM.  Algorithmic bytes 16 per input sample (SURVEY 8d: 8 in + 8 out)."""
    import ctypes as C
    L = lib.load()
    L.b200_chan_create.restype = C.c_void_p
    ch = L.b200_chan_create(256, 127, chunk)
    if not ch:
        raise RuntimeError(L.b200_last_error().decode())
    ch = C.c_void_p(ch)
    ins = [torch.rand(2 * chunk, device="cuda") * 2.0 - 1.0 for _ in range(20)]          # 160 MB in rotation: larger than L2
    out = torch.empty(2 * chunk, device="cuda")
    for i in range(5):
        lib.check(L.b200_chan_process(ch, C.c_void_p(ins[i].data_ptr()), chunk, lib.MEM_DEVICE, C.c_void_p(out.data_ptr()), lib.MEM_DEVICE))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(steps):
        lib.check(L.b200_chan_process(ch, C.c_void_p(ins[i % 20].data_ptr()), chunk, lib.MEM_DEVICE, C.c_void_p(out.data_ptr()), lib.MEM_DEVICE))
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    peak, src = measured_peak_hbm()
    v = chunk * steps / dt
    L.b200_chan_destroy(ch)
    return {"workload": "C3: 256-channel critically sampled polyphase filter bank, 127 taps per branch (32512-tap Nuttall windowed-sinc prototype), 1 Mi-sample chunks",
            "value": v / 1e6, "unit": "MS/s", "target_stream_rate_msps": 500.0, "chunks": steps, "chunk_samples": chunk,
            "timing": "wall clock over synchronous b200_chan_process calls (device in, device out; includes the D2D placement behind the history and the carry)",
            "roofline": {"bound": "hbm", "algorithmic_bytes_per_sample": 16.0, "achieved": v * 16.0 / 1e9, "peak": peak, "peak_source": src, "unit": "GB/s",
                         "frac": v * 16.0 / 1e9 / peak,
                         "note": "127 packed FMAs per input sample: the fp32 issue roof (about 17 T FFMA2/s) caps this kernel near 138 GS/s = 0.34 of the HBM roof"}}


def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import sdrplusplus_b200 as sb
    from sdrplusplus_b200 import lib

    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    # libraries (NCCL's version banner) write to fd 1: keep stdout clean for the single JSON line
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- libb200dsp has no CPU fallback")
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    L = lib.load()
    lib.check(L.b200_init(local))

    chunk = args.chunk
    nbuf = 3
    # stage 1 runs on this stream: between the chain behind it (highest priority, csrc/api.cpp) and the spectrum branch (lowest)
    stream = torch.cuda.Stream(priority=args.main_prio)
    with torch.cuda.stream(stream):
        offsets = OFFSETS if args.offsets == "sym" else [5e6, -7e6, 15e6, -17e6, 25e6, -27e6, 35e6, -37e6]
        fe = sb.FrontEnd(FS, chunk)
        fe.set_stream(stream.cuda_stream)
        fe.set_option("overlap", args.overlap)
        fe.set_option("pair", args.pair)
        fe.set_option("s1", args.s1)
        fe.set_option("s1_mt", args.s1_mt)
        fe.set_option("s1_stages", args.s1_stages)
        fe.set_option("tails", args.tails)
        for kv in [a for a in args.ft.split(",") if a]:
            fe.set_option(kv.split("=")[0], int(kv.split("=")[1]))
        fe.set_fft(FFT_SIZE, FFT_RATE, lib.WIN_NUTTALL)
        ids = [fe.add_vfo(sb.VfoConfig.wfm(o)) for o in offsets]
        gen = torch.Generator(device="cuda")
        gen.manual_seed(0x5D12 + rank)
        # synthetic inputs, SpeedTester distribution: i.i.d. uniform[-1,1) re/im; distinct per buffer and per rank
        dev_in = [(torch.rand(2 * chunk, device="cuda", generator=gen, dtype=torch.float32) * 2.0 - 1.0) for _ in range(nbuf)]
        cap = {v: fe.vfo_max_out(v, chunk) for v in ids}
        nl = fe.fft_max_lines(chunk)

        L.b200_host_alloc.restype = C.c_void_p

        class Pinned:
            """Pinned host buffer from the library's own allocator (b200_host_alloc == what dsp::stream<T> uses in the
            adapters).  torch's pinned allocator handed out an occasional buffer that DMAs at 11 GB/s on this box
            (tools/diag_pinned.py); cudaHostAlloc is consistent at 55 / 57 GB/s."""

            def __init__(self, nbytes):
                self.nbytes = nbytes
                self.ptr = L.b200_host_alloc(nbytes)
                if not self.ptr:
                    raise MemoryError("b200_host_alloc(%d) failed" % nbytes)

            def array(self, dtype):
                n = self.nbytes // np.dtype(dtype).itemsize
                return np.ctypeslib.as_array(C.cast(self.ptr, C.POINTER(C.c_uint8)), shape=(self.nbytes,)).view(dtype)[:n]

            def data_ptr(self):
                return self.ptr

            def free(self):
                if self.ptr:
                    L.b200_host_free(C.c_void_p(self.ptr))
                    self.ptr = None

        def make_outputs(pinned):
            o = lib.Outputs()
            keep = []
            for v in ids:
                t = Pinned(8 * cap[v]) if pinned else torch.empty(2 * cap[v], device="cuda", dtype=torch.float32)
                keep.append(t)
                o.vfo_out[v] = t.data_ptr()
                o.vfo_cap[v] = cap[v]
            t = Pinned(4 * nl * FFT_SIZE) if pinned else torch.empty(nl * FFT_SIZE, device="cuda", dtype=torch.float32)
            keep.append(t)
            o.fft_out = t.data_ptr()
            o.fft_cap_lines = nl
            o.out_mem = lib.MEM_HOST if pinned else lib.MEM_DEVICE
            return o, keep

        def barrier():
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()

        def timed_loop(ptrs, fmt, mem, outs, steps, warm, cps=1):
            """pipelined submit/wait (two chunks in flight); a step = `cps` chunks.  Returns (ms by CUDA events on `stream`,
            wall ms, d2h bytes of one chunk)."""
            inflight = 0
            for i in range(warm * cps):
                fe.submit_ptr(ptrs[i % len(ptrs)], chunk, fmt, mem, outs[i % 2][0])
                inflight += 1
                if inflight == 2:
                    fe.wait()
                    inflight -= 1
            while inflight:
                fe.wait()
                inflight -= 1
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record(stream)
            d2h = 0
            host_submit = 0.0
            for i in range(steps * cps):
                o = outs[i % 2][0]
                th = time.perf_counter()
                fe.submit_ptr(ptrs[i % len(ptrs)], chunk, fmt, mem, o)
                host_submit += time.perf_counter() - th
                d2h = sum(o.vfo_count[v] for v in ids) * 8 + o.fft_lines * FFT_SIZE * 4
                inflight += 1
                if inflight == 2:
                    fe.wait()
                    inflight -= 1
            while inflight:
                fe.wait()
                inflight -= 1
            e1.record(stream)
            torch.cuda.synchronize()
            wall = (time.perf_counter() - t0) * 1e3
            ms = e0.elapsed_time(e1)
            barrier()
            if world > 1:
                t = torch.tensor([ms, wall], device="cuda", dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms, wall = float(t[0]), float(t[1])
            timed_loop.host_submit_ms = host_submit * 1e3 / max(steps * cps, 1)
            return ms, wall, d2h

        probe = pcie_probe(torch)
        clocks = ClockSampler(local)
        # ---------------- device-resident leg ----------------
        outs_dev = [make_outputs(False), make_outputs(False)]
        ptrs = [t.data_ptr() for t in dev_in]
        fe.set_option("time_s1", 0)
        l0 = fe.launch_count()
        cps = max(1, min(args.chunks_per_step, 32) if args.quick else args.chunks_per_step)
        timed_loop(ptrs, lib.FMT_CF32, lib.MEM_DEVICE, outs_dev, 0, args.warmup, cps)       # warm-up only
        fe.set_option("time_s1", 1)
        if not args.no_clocks:
            clocks.start()
        l0 = fe.launch_count()
        ms, wall, _ = timed_loop(ptrs, lib.FMT_CF32, lib.MEM_DEVICE, outs_dev, args.steps, 0, cps)
        launches = fe.launch_count() - l0
        host_submit_ms = timed_loop.host_submit_ms
        s1_ms, s1_n = fe.group_stats(0)
        tail_ms, tail_n = fe.group_stats(1)
        fft_ms, fft_n = fe.group_stats(2)
        tma_launches = fe.stat("s1_tma_launches")
        fe.set_option("time_s1", 0)
        value = world * chunk * cps * args.steps / (ms * 1e-3) / 1e6
        if args.dump_outputs and rank == 0:
            # what the caller received for the last chunk of the last step (the buffers of earlier chunks have been reused):
            # each VFO's stereo audio and the spectrum lines
            o, keep = outs_dev[(args.steps * cps - 1) % 2]
            got = {"vfo%d_audio" % k: keep[k][: 2 * o.vfo_count[v]].view(-1, 2).cpu().numpy() for k, v in enumerate(ids)}
            got["fft_lines"] = keep[-1][: o.fft_lines * FFT_SIZE].view(-1, FFT_SIZE).cpu().numpy()
            dump_outputs(args.dump_outputs, got)

        # ---------------- end-to-end legs (host pinned in, host pinned out) ----------------
        outs_host = [make_outputs(True), make_outputs(True)]
        e2e = {}
        for name, fmt, bps in (("cs16", lib.FMT_CS16, 4), ("cf32", lib.FMT_CF32, 8), ("cs8", lib.FMT_CS8, 2)):
            if args.quick and name != "cs16":
                e2e[name] = {"value": None}
                continue
            host_in = [Pinned(chunk * bps) for _ in range(2)]
            for k, t in enumerate(host_in):
                if name == "cs16":
                    t.array(np.int16)[:] = (dev_in[k] * 32767.0).to(torch.int16).cpu().numpy()
                elif name == "cs8":
                    t.array(np.int8)[:] = (dev_in[k] * 127.0).to(torch.int8).cpu().numpy()
                else:
                    t.array(np.float32)[:] = dev_in[k].cpu().numpy()
            hp = [t.data_ptr() for t in host_in]
            steps = args.steps
            ecps = max(1, cps // 8)
            ems, ewall, d2h = timed_loop(hp, fmt, lib.MEM_HOST, outs_host, steps, 3, ecps)
            e2e[name] = {"value": world * chunk * ecps * steps / (ewall * 1e-3) / 1e6, "unit": "MS/s", "h2d_bytes_per_step": chunk * bps * ecps,
                         "d2h_bytes_per_step": int(d2h) * ecps, "steps": steps, "chunks_per_step": ecps, "ms_per_step_wall": ewall / steps,
                         "ms_per_step_events": ems / steps}
            for t in host_in:
                t.free()
        clk = clocks.stop()
        fe.close()
        # ---------------- the dominant kernel with nothing else running (explains roofline.frac) ----------------
        s1_alone = None
        if rank == 0:
            try:                                     # an explanatory extra: never let it take the bench line down
                fe2 = sb.FrontEnd(FS, chunk)
                fe2.set_stream(stream.cuda_stream)
                fe2.set_option("overlap", 0)
                fe2.set_option("pair", args.pair)
                fe2.set_option("s1", args.s1)
                fe2.set_option("tails", args.tails)
                for o in offsets:
                    fe2.add_vfo(sb.VfoConfig.wfm(o))
                o2 = make_outputs(False)
                for k in range(3):
                    fe2.submit_ptr(ptrs[k % nbuf], chunk, lib.FMT_CF32, lib.MEM_DEVICE, o2[0]); fe2.wait()
                fe2.set_option("time_s1", 1)
                for k in range(10):
                    fe2.submit_ptr(ptrs[k % nbuf], chunk, lib.FMT_CF32, lib.MEM_DEVICE, o2[0]); fe2.wait()
                a_ms, a_n = fe2.s1_stats()
                fe2.close()
                s1_alone = a_ms / max(a_n, 1)
            except Exception as ex:                  # noqa: BLE001
                print("roofline.alone skipped: %r" % (ex,), file=sys.stderr)
                s1_alone = None

        # ---------------- the small-chunk regime (SURVEY 8d: the reference's own chunk sizes at 100 MS/s) ----------------
        sweep = None
        if rank == 0 and not args.quick:
            sweep = {}
            for csz, nchunks in ((500000, 400), (1000000, 300), (1 << 22, 120)):
                try:
                    fe3 = sb.FrontEnd(FS, csz)
                    fe3.set_stream(stream.cuda_stream)
                    fe3.set_fft(FFT_SIZE, FFT_RATE, lib.WIN_NUTTALL)
                    ids3 = [fe3.add_vfo(sb.VfoConfig.wfm(o)) for o in offsets]
                    o3 = []
                    for _ in range(2):
                        oo = lib.Outputs()
                        keep3 = []
                        for v in ids3:
                            c3 = fe3.vfo_max_out(v, csz)
                            t3 = torch.empty(2 * c3, device="cuda", dtype=torch.float32)
                            keep3.append(t3); oo.vfo_out[v] = t3.data_ptr(); oo.vfo_cap[v] = c3
                        nl3 = max(1, fe3.fft_max_lines(csz))
                        t3 = torch.empty(nl3 * FFT_SIZE, device="cuda", dtype=torch.float32)
                        keep3.append(t3); oo.fft_out = t3.data_ptr(); oo.fft_cap_lines = nl3; oo.out_mem = lib.MEM_DEVICE
                        o3.append((oo, keep3))
                    nslots = (2 * chunk) // (2 * csz)                      # walk through the big device buffers: larger than L2

                    def run3(n):
                        infl = 0
                        for i in range(n):
                            b = dev_in[(i // nslots) % nbuf]
                            fe3.submit_ptr(b.data_ptr() + (i % nslots) * csz * 8, csz, lib.FMT_CF32, lib.MEM_DEVICE, o3[i % 2][0])
                            infl += 1
                            if infl == 2:
                                fe3.wait(); infl -= 1
                        while infl:
                            fe3.wait(); infl -= 1
                    run3(20)
                    torch.cuda.synchronize()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream); run3(nchunks); e1.record(stream)
                    torch.cuda.synchronize()
                    sweep[str(csz)] = {"value": csz * nchunks / (e0.elapsed_time(e1) * 1e-3) / 1e6, "unit": "MS/s", "chunks": nchunks,
                                       "us_per_chunk": e0.elapsed_time(e1) * 1e3 / nchunks}
                    fe3.close()
                    # the same chunk size end to end: int16 IQ in pinned host memory -> H2D -> kernels -> audio and dB lines
                    # in pinned host memory, four chunks in flight (the copy engine fed a few chunks ahead)
                    fe4 = sb.FrontEnd(FS, csz)
                    fe4.set_option("inflight", 4)
                    fe4.set_fft(FFT_SIZE, FFT_RATE, lib.WIN_NUTTALL)
                    ids4 = [fe4.add_vfo(sb.VfoConfig.wfm(o)) for o in offsets]
                    o4, keep4 = [], []
                    for _ in range(4):
                        oo = lib.Outputs()
                        for v in ids4:
                            c4s = fe4.vfo_max_out(v, csz)
                            t4 = Pinned(8 * c4s); keep4.append(t4); oo.vfo_out[v] = t4.data_ptr(); oo.vfo_cap[v] = c4s
                        nl4 = max(1, fe4.fft_max_lines(csz))
                        t4 = Pinned(4 * nl4 * FFT_SIZE); keep4.append(t4); oo.fft_out = t4.data_ptr(); oo.fft_cap_lines = nl4; oo.out_mem = lib.MEM_HOST
                        o4.append(oo)
                    hin = Pinned(64 << 20)
                    hin.array(np.int16)[:] = (np.random.default_rng(7).standard_normal((64 << 20) // 2) * 3000).astype(np.int16)
                    hslots = (64 << 20) // (4 * csz)

                    def run4(n):
                        infl = 0
                        for i in range(n):
                            fe4.submit_ptr(hin.data_ptr() + (i % hslots) * csz * 4, csz, lib.FMT_CS16, lib.MEM_HOST, o4[i % 4])
                            infl += 1
                            if infl == 4:
                                fe4.wait(); infl -= 1
                        while infl:
                            fe4.wait(); infl -= 1
                    run4(40)
                    t0 = time.perf_counter(); run4(nchunks); wall4 = time.perf_counter() - t0
                    sweep[str(csz)]["e2e_int16"] = {"value": csz * nchunks / wall4 / 1e6, "unit": "MS/s", "us_per_chunk": wall4 * 1e6 / nchunks,
                                                    "inflight": 4, "timing": "wall clock around the pipelined submit/wait loop (H2D, kernels, outputs in pinned host memory)"}
                    fe4.close()
                    hin.free()
                    for t4 in keep4:
                        t4.free()
                except Exception as ex:              # noqa: BLE001
                    sweep[str(csz)] = {"value": None, "error": repr(ex)}
        numa_all = [numa]
        if world > 1:
            numa_all = [None] * world
            dist.all_gather_object(numa_all, numa)

    c4 = None
    if args.c4 and not args.quick:
        try:
            c4 = c4_leg(torch, dist, sb, lib, rank, world, local, args.steps)
        except Exception as ex:                      # noqa: BLE001 -- a secondary leg: never take the bench line down (all ranks fail alike)
            c4 = {"workload": C4_WORKLOAD, "value": None, "error": repr(ex)}
    c3 = None
    if rank == 0 and args.c3 and not args.quick:
        try:
            c3 = c3_leg(torch, lib)
        except Exception as ex:                      # noqa: BLE001
            c3 = {"value": None, "error": repr(ex)}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0
    peak, peak_src = measured_peak_hbm()
    algo_bytes = ALGO_BYTES_PER_SAMPLE * chunk
    s1_avg = s1_ms / max(s1_n, 1)
    achieved = algo_bytes / (s1_avg * 1e-3) / 1e9 if s1_n else None
    nchunks_timed = cps * args.steps
    s1_kernel = ("k_xd_tma" if tma_launches > 0 else ("k_xd_pfb" if args.s1 >= 7 and args.offsets == "sym" else "k_xd_pipe"))
    # DRAM traffic of the dominant kernel: from the tracked ncu capture of this round, never a constant in this file
    traffic, traffic_src = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
            tj = json.load(f)
        if tj.get("kernel", "").startswith(s1_kernel) and tj.get("chunk_samples") == chunk:
            traffic = int(tj["dram_bytes_read"] + tj["dram_bytes_write"])
            traffic_src = "ncu --set full, %s: dram__bytes_read.sum %.2f MB + dram__bytes_write.sum %.2f MB per launch (%s)" % (
                tj.get("kernel"), tj["dram_bytes_read"] / 1e6, tj["dram_bytes_write"] / 1e6, tj.get("source"))
    except (OSError, ValueError, KeyError):
        pass
    # useful fp32 multiply-adds behind stage 1, per VFO output sample of the C2 chain (real FMA; a packed FFMA2 counts 2):
    # audio FIR 237 + channel FIR 2*126 + polyphase 2*119 + (2,69) stage 2*69*1.5625 + (4,27) stage 2*27*3.125
    tail_fma = 8 * chunk * (250e3 / FS) * (237 + 2 * 126 + 2 * 119 + 2 * 69 * 1.5625 + 2 * 27 * 3.125)
    fma_peak = 35.0e12                      # measured FFMA / FFMA2 issue peak of this part (tools/ubench.cu), FMA/s
    tail_avg = tail_ms / max(tail_n, 1)
    fft_avg = fft_ms / max(fft_n, 1)
    fft_bytes = chunk * (FFT_RATE / FS) * FFT_SIZE * (8 + 8 + 8 + 4)          # frames per chunk x (read IQ, work out, work in, dB out)
    groups = [
        {"group": "stage 1", "kernels": s1_kernel, "avg_ms": s1_avg, "timed": s1_n, "bound": "hbm", "achieved": achieved, "peak": peak,
         "unit": "GB/s", "frac": (achieved / peak) if achieved else None},
        {"group": "behind stage 1", "kernels": "k_dfir_reg x2, k_poly_reg, k_fir_reg, k_quad, k_firr_reg, k_carry (six dependent launches)", "avg_ms": tail_avg, "timed": tail_n, "bound": "fp32 FMA issue",
         "achieved": (tail_fma / (tail_avg * 1e-3) / 1e12) if tail_n else None, "peak": fma_peak / 1e12, "unit": "TFMA/s",
         "frac": (tail_fma / (tail_avg * 1e-3) / fma_peak) if tail_n else None, "useful_fma_per_chunk": tail_fma},
        {"group": "spectrum branch", "kernels": "k_fftr_p1, k_fftr_p2 (frames of a chunk batched)", "avg_ms": fft_avg, "timed": fft_n, "bound": "hbm / L2",
         "achieved": (fft_bytes / (fft_avg * 1e-3) / 1e9) if fft_n else None, "peak": peak, "unit": "GB/s",
         "frac": (fft_bytes / (fft_avg * 1e-3) / 1e9 / peak) if fft_n else None,
         "bytes_per_chunk": fft_bytes},
    ]
    timed = [g for g in groups if g["timed"]]
    dominant_by_time = max(timed, key=lambda g: g["avg_ms"])["group"] if timed else None
    line = {
        "metric": METRIC, "value": value, "unit": "MS/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "ms_per_step_wall": wall / args.steps, "host_ms_per_submit": host_submit_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": WORKLOAD, "chunk_samples": chunk, "chunks_per_step": cps, "samples_per_step": chunk * cps, "samplerate": FS,
                   "parallelism": "replicas x%d (one IQ stream per GPU, no collective)" % world,
                   "l2": "inputs larger than L2: %d MiB cf32 chunk, %d rotating device buffers" % (chunk * 8 >> 20, nbuf),
                   "value_input": "cf32 resident in HBM, outputs to HBM", "e2e_input": "int16 IQ in pinned host memory (file_source format); cf32 and int8 also reported",
                   "pipelining": "b200_fe_submit/wait, 2 chunks in flight", "s1_variant": args.s1, "tails_variant": args.tails,
                   "vfo_offsets_hz": offsets, "conjugate_pair_sharing": bool(args.pair) and args.offsets == "sym",
                   "tails_overlap_next_chunk": bool(args.overlap),
                   "chain_launch": "chain behind stage 1 replayed as a CUDA graph; programmatic dependent launch (B200_PDL=%s) for launches of at most 2 CTAs per SM" % os.environ.get("B200_PDL", "2"),
                   "chunk_sweep": sweep, "chunk_sweep_note": "the same graph at the reference's own chunk sizes (STREAM_BUFFER_SIZE caps a chunk at 1e6 samples, core/src/dsp/stream.h:9): device-resident MS/s, and end to end from int16 IQ in pinned host memory"},
        "e2e": dict(e2e["cs16"], format="cs16", cf32=e2e["cf32"], cs8=e2e["cs8"], pcie_probe=probe, numa=numa, numa_per_rank=numa_all,
                    host_buffers="b200_host_alloc (cudaHostAlloc)"),
        "gpu_launches": int(launches),
        "clocks": clk,
        "roofline": {"bound": "hbm", "kernel": s1_kernel + " (stage 1: translate + first decimating FIR of all VFOs, IQ read once; the kernel that moves the algorithmic bytes)",
                     "achieved": achieved, "peak": peak, "peak_source": peak_src, "unit": "GB/s",
                     "frac": (achieved / peak) if achieved else None,
                     "traffic": traffic, "traffic_source": traffic_src,
                     "algorithmic_bytes_per_launch": algo_bytes, "avg_launch_ms": s1_avg, "launches_timed": s1_n,
                     "share_of_step": (s1_avg * nchunks_timed / ms) if ms else None,
                     "step_level": {"achieved": algo_bytes * nchunks_timed / (ms * 1e-3) / 1e9, "frac": algo_bytes * nchunks_timed / (ms * 1e-3) / 1e9 / peak},
                     "alone": ({"avg_launch_ms": s1_alone, "achieved": algo_bytes / (s1_alone * 1e-3) / 1e9,
                                "frac": algo_bytes / (s1_alone * 1e-3) / 1e9 / peak,
                                "what": "same kernel, same inputs, no spectrum branch and no overlapped tail kernels on the GPU"} if s1_alone else None),
                     "by_group": groups, "dominant_by_time": dominant_by_time,
                     "note": "avg_launch_ms of every group is measured live with CUDA events on the stream the group runs on, inside the timed region, "
                             "where the three streams (stage 1 | behind stage 1 | spectrum) share the SMs; 'alone' times stage 1 with nothing else running. "
                             "Timed: the first %d chunks of the region per group." % s1_n},
    }
    if c4 is not None:
        line["c4"] = c4
    if c3 is not None:
        line["c3"] = c3
    if world == 1 and not args.no_cpu:
        try:
            v, threads, kind, what = cpu_reference_run(args.cpu_ms)
            line["cpu_baseline"] = {"value": v / 1e6, "unit": "MS/s", "cores": threads, "host_cpus": os.cpu_count(), "kind": kind, "sample": what}
        except Exception as ex:          # noqa: BLE001
            line["cpu_baseline"] = {"value": None, "unit": "MS/s", "cores": 0, "kind": "reference", "sample": "failed: %r" % (ex,)}
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    print(json.dumps(line))
    sys.stdout.flush()
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--chunk", type=int, default=1 << 24, help="IQ samples per chunk (default 16 Mi = 128 MiB cf32 > L2)")
    ap.add_argument("--chunks-per-step", type=int, default=512, help="a step = this many chunks through the pipelined submit/wait API (default 512: about 75 ms of device time per step)")
    ap.add_argument("--s1", type=int, default=8, help="stage-1 kernel variant (8 = filter-bank form fed by the TMA engine, 7 = filter bank on cp.async tiles, when the VFO plan allows it; else 6 = per-VFO complex taps)")
    ap.add_argument("--tails", type=int, default=2, help="2 = one fused tail launch per <= 16 VFOs (default), 1 = shared-memory tiled kernel per stage, 0 = one thread per output")
    ap.add_argument("--ft", default="", help="fused-tail tuning, e.g. ft_threads=256,ft_obmax=1024,ft_smem_kb=72")
    ap.add_argument("--s1-stages", type=int, default=2, help="ring depth of the TMA stage 1 (2 = leaves shared memory for the kernels of the other streams, 3)")
    ap.add_argument("--s1-mt", type=int, default=0, help="force the stage-1 tile size (outputs per tile), 0 = automatic")
    ap.add_argument("--overlap", type=int, default=1, help="1 = tails of chunk k overlap stage 1 of chunk k+1 (default)")
    ap.add_argument("--pair", type=int, default=1, help="1 = VFOs at +f/-f share their stage-1 multiply-accumulates (default)")
    ap.add_argument("--offsets", default="sym", choices=["sym", "asym"],
                    help="sym = BASELINE config 2 (+-5/15/25/35 MHz); asym = 8 offsets without conjugate pairs")
    ap.add_argument("--cpu-ms", type=int, default=12000, help="duration of the CPU reference sample")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--quick", action="store_true", help="diagnostic: only the int16 end-to-end leg")
    ap.add_argument("--c4", type=int, default=1, help="1 = also time BASELINE config 4 (one 1.024 GS/s stream, 64 VFOs sharded over the GPUs with an NCCL broadcast) and report it under 'c4'")
    ap.add_argument("--c3", type=int, default=1, help="1 = also time BASELINE config 3 (256-channel polyphase filter-bank channelizer) on rank 0 and report it under 'c3'")
    ap.add_argument("--main-prio", type=int, default=-1, help="CUDA priority of the stream stage 1 runs on (0 = lowest; the library's own streams: B200_STREAM_PRIO)")
    ap.add_argument("--no-clocks", action="store_true", help="do not poll nvidia-smi during the timed region (diagnostic)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last chunk of the last step returned "
                    "(vfo<k>_audio.npy: stereo audio of each VFO, fft_lines.npy: spectrum lines in dB; float32) to DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
