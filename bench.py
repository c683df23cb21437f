#!/usr/bin/env python
"""bench.py -- OFDM symbols/s through the TX -> AWGN -> RX chain (BASELINE.json metric).

Workload (configs[1]): batched QPSK BER/EVM sweep, 1,000,000 frames x 2 data symbols, 21 SNR points
0..20 dB, injected standard-normal draws (one per sample, reused across SNR points), EXACT mode
(bit-exact error counts versus OFDM.c).  One "step" = one whole sweep: Transmitter once, then channel +
receiver at every SNR point.  A counted OFDM symbol is one data symbol that went through TX, the channel and
RX at one SNR point: symbols/step = frames x n_sym x n_snr.

  value   inputs resident in HBM, CUDA-event timed on the launching stream.  The SNR loop runs in ONE kernel
          (k_sweep_lin: FFT(x + sigma g) = FFT(x) + sigma FFT(g), so each frame and its draws are transformed once
          and every SNR point costs a multiply-add per bin plus the verified decision stage).
  e2e     the same sweep through ofdm_sweep_inject_host: HOST (pinned) bits + draws, H2D copies,
          kernels and the D2H of the counters inside the timed region
  roofline  the HBM-bound kernel of the path: k_stream_quad<checked,inject>, the fused channel + receiver of ONE SNR
            point, one frame per 8-lane group (what the stage API ofdm_awgn_rx_inject launches, and what the sweep
            launched 21 times before k_sweep_lin existed): algorithmic bytes (3100 B per frame, DESIGN.md) / mean launch
            time, CUDA events around each launch of a dedicated loop of steps x 21 launches in this run.  sweep_kernel
            describes k_sweep_lin, which is bound by instruction issue, not by HBM.
  configs   configs[2] (streaming TX / RX of 16 Mi HBM-resident symbols, HBM GB/s fraction), configs[3] (fused on-chip
            Philox Monte-Carlo, fixed frame count and the until-100-errors-or-1e-7-budget rule), configs[4] (8-tap
            multipath): per-config throughput and roofline; at N > 1 configs[3] / [4] are sharded by global frame index
            with the NCCL all-reduce of the counters inside the timed region (time = max over ranks).
  cpu_baseline  the compiled reference (oracle/_ref) stage chain on a bounded sample, one thread

--impl reference: the reference's own CPU implementation of the path (oracle/_ref, else the oracle
port) on all host cores, each step a bounded sample of the same workload (Transmitter once per frame, then
channel + receiver per SNR point, as main() arranges it).
Multi-GPU (torchrun): frames are sharded across ranks (weak scaling: 1M frames per rank), one NCCL
all-reduce of the counters per sweep; time = max over ranks.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import __graft_entry__ as entry  # noqa: E402

N_SYM = 2
SNRS = [float(s) for s in range(0, 21)]
BYTES_PER_FRAME_PASS = (128 + 64 * N_SYM) * 8 + (128 + 64 * N_SYM) * 4 + 12 * N_SYM + 4   # 3100
METRIC = "OFDM symbols/s, TX+AWGN+RX chain (BER/EVM sweep)"
UNIT = "symbols/s"


def workload_name(n_frames):
    return ("cfg1: batched QPSK BER/EVM sweep, %d frames x %d data symbols x %d SNR points (0..20 dB), "
            "injected normals, exact mode" % (n_frames, N_SYM, len(SNRS)))


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.t = threading.Thread(target=self._read, daemon=True)
        self.t.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except (ValueError, IndexError):
                continue
            for name, v in zip(self.NAMES, r[3:7]):
                if v == "Active":
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ----------------------------------------------------------------------------- CPU reference legs
_W = {}


def _worker_init():
    po = entry.load_oracle()
    _W["impl"] = po.Ref() if po.have_ref() else po.Port()


def _worker_run(args):
    bits, g, snrs = args
    impl = _W["impl"]
    return sum(c.bit_errors for c in impl.chain_sweep(bits, g, N_SYM, snrs))


def sample_inputs(n_frames, seed):
    rng = np.random.default_rng(seed)
    bits = rng.integers(0, 2, (n_frames, 96 * N_SYM), dtype=np.uint8)
    g = rng.standard_normal((n_frames, 160 + 80 * N_SYM)).astype(np.float32)
    return bits, g


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def host_cores():
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


def cpu_baseline_single(sample_frames):
    """oracle/_ref (kind reference) or the port, one thread, bounded sample of the same workload."""
    po = entry.load_oracle()
    po.build()
    kind = "reference" if po.have_ref() else "port"
    impl = po.Ref() if kind == "reference" else po.Port()
    bits, g = sample_inputs(sample_frames, 1234)
    impl.chain(bits[:64], g[:64], N_SYM, 10.0)          # warm
    t0 = time.perf_counter()
    impl.chain_sweep(bits, g, N_SYM, SNRS)              # Transmitter once per frame, 21 x (channel + receiver): main()'s loop
    dt = time.perf_counter() - t0
    return {"value": sample_frames * N_SYM * len(SNRS) / dt, "unit": UNIT, "cores": 1, "kind": kind,
            "sample": "%d frames x %d symbols x %d SNR points, injected normals, %.1f s" % (sample_frames, N_SYM, len(SNRS), dt),
            "host": "%s, %d cores available" % (cpu_model(), host_cores())}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import multiprocessing as mp
    po = entry.load_oracle()
    po.build()
    kind = "reference" if po.have_ref() else "port"
    cores = host_cores()
    per_core = 192
    n_frames = per_core * cores
    bits, g = sample_inputs(n_frames, 4321)
    tasks = [(bits[i * per_core:(i + 1) * per_core], g[i * per_core:(i + 1) * per_core], SNRS) for i in range(cores)]
    ctx = mp.get_context("fork")
    with ctx.Pool(cores, initializer=_worker_init) as pool:
        for _ in range(args.warmup):
            pool.map(_worker_run, tasks, chunksize=1)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            pool.map(_worker_run, tasks, chunksize=1)
        dt = time.perf_counter() - t0
    ms = dt / args.steps * 1e3
    value = n_frames * N_SYM * len(SNRS) / (dt / args.steps)
    sample = "%d frames x %d symbols x %d SNR points per step, %d processes" % (n_frames, N_SYM, len(SNRS), cores)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32+f64", "data": "synthetic",
            "config": {"workload": workload_name(args.frames), "reference_arm_sample": sample},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample,
                             "host": "%s, %d cores available" % (cpu_model(), cores)},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)
    return 0


# ----------------------------------------------------------------------------- GPU arm
def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def run_extras(o, pkg, torch, dev, args, rank, world):
    """Secondary configurations (not the headline): configs[2] streaming TX / RX of HBM-resident frames in fast
    mode as HBM GB/s, configs[3] fused on-chip Philox Monte-Carlo as symbols/s.  Per-rank numbers (rank 0 reports)."""
    import torch.distributed as dist
    out = {}
    peak, _ = peaks()

    def timed(fn, reps=5):
        fn(); torch.cuda.synchronize()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record(); torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    n = args.stream_frames
    bits = torch.randint(-2 ** 31, 2 ** 31 - 1, (n * N_SYM * 3,), dtype=torch.int32, device=dev)
    frames = torch.empty((n, pkg.frame_len(N_SYM), 2), dtype=torch.float32, device=dev)
    cnt = o.new_counters(1)
    lib, h = o.lib, o.h
    ms_tx = timed(lambda: o._check(lib.ofdm_tx_frames(h, bits.data_ptr(), frames.data_ptr(), None, n, N_SYM, pkg.MODE_FAST)))
    ms_rx = timed(lambda: o._check(lib.ofdm_rx_frames(h, frames.data_ptr(), bits.data_ptr(), n, N_SYM, pkg.MODE_FAST, cnt.data_ptr(), None)))
    tx_bytes, rx_bytes = n * (24 + 2560), n * (2048 + 24)
    out["cfg2_streaming_fast"] = {
        "frames": n, "data_symbols": n * N_SYM,
        "tx_ms": ms_tx, "tx_GBps": tx_bytes / ms_tx / 1e6, "tx_frac_of_hbm_peak": tx_bytes / ms_tx / 1e6 / peak,
        "rx_ms": ms_rx, "rx_GBps": rx_bytes / ms_rx / 1e6, "rx_frac_of_hbm_peak": rx_bytes / ms_rx / 1e6 / peak,
        "symbols_per_s_tx_plus_rx": n * N_SYM / ((ms_tx + ms_rx) * 1e-3),
        "bytes_per_frame": {"tx": 24 + 2560, "rx": 2048 + 24},
        "note": "rx reads only the LTS halves and symbol bodies (2048 B of the 2560 B frame) + 24 B of bits"}
    # the same in EXACT mode (bit-exact IQ from the transmitter; the receiver's totals through the checked arithmetic)
    ms_txe = timed(lambda: o._check(lib.ofdm_tx_frames(h, bits.data_ptr(), frames.data_ptr(), None, n, N_SYM, pkg.MODE_EXACT)))
    ms_rxe = timed(lambda: o._check(lib.ofdm_rx_frames(h, frames.data_ptr(), bits.data_ptr(), n, N_SYM, pkg.MODE_EXACT, cnt.data_ptr(), None)))
    out["cfg2_streaming_exact"] = {
        "frames": n, "tx_ms": ms_txe, "tx_GBps": tx_bytes / ms_txe / 1e6, "tx_frac_of_hbm_peak": tx_bytes / ms_txe / 1e6 / peak,
        "rx_ms": ms_rxe, "rx_GBps": rx_bytes / ms_rxe / 1e6, "rx_frac_of_hbm_peak": rx_bytes / ms_rxe / 1e6 / peak,
        "symbols_per_s_tx_plus_rx": n * N_SYM / ((ms_txe + ms_rxe) * 1e-3)}
    del frames, bits
    torch.cuda.empty_cache()
    nm = args.mc_frames
    mc = o.new_counters(len(SNRS))
    for mode, name in ((pkg.MODE_FAST, "fast"), (pkg.MODE_EXACT, "exact")):
        ms = timed(lambda: o.mc_sweep_philox(7, rank * nm, nm, N_SYM, SNRS, mode, counters=mc), reps=2)
        out["cfg3_mc_philox_" + name] = {"frames": nm, "snr_points": len(SNRS), "ms": ms,
                                         "symbols_per_s": nm * N_SYM * len(SNRS) / (ms * 1e-3),
                                         "fft_gflops": nm * len(SNRS) * 4 * 1920 / (ms * 1e-3) / 1e9}
    # other frame shapes (n_sym != 2) through the multi-pass streaming receiver, injected draws, 4 M windows each
    shapes = {}
    for ns in (1, 4, 16):
        nf = 4_000_000 // (2 + ns)
        fl = 160 + 80 * ns
        b = torch.randint(-2 ** 31, 2 ** 31 - 1, (nf * 3 * ns,), dtype=torch.int32, device=dev)
        fr = torch.empty((nf, fl, 2), dtype=torch.float32, device=dev)
        gg = torch.randn((nf, fl), dtype=torch.float32, device=dev)
        pw = torch.empty((nf,), dtype=torch.float32, device=dev)
        for mode, name in ((pkg.MODE_EXACT, "exact"), (pkg.MODE_FAST, "fast")):
            o._check(lib.ofdm_tx_frames(h, b.data_ptr(), fr.data_ptr(), pw.data_ptr(), nf, ns, mode))
            ms = timed(lambda: o._check(lib.ofdm_awgn_rx_inject(h, fr.data_ptr(), gg.data_ptr(), pw.data_ptr(), b.data_ptr(), 8.0, nf, ns, mode,
                                                                  cnt.data_ptr(), None)), reps=3)
            shapes["n_sym_%d_%s" % (ns, name)] = {"frames": nf, "ms": ms, "data_symbols_per_s": nf * ns / (ms * 1e-3),
                                                  "windows_per_s": nf * (2 + ns) / (ms * 1e-3)}
        del b, fr, gg, pw
    out["other_frame_shapes_rx"] = shapes
    torch.cuda.empty_cache()
    out["next_rows_full_receiver_path"] = run_next_rows(o, pkg, torch, dev, peak)
    torch.cuda.empty_cache()
    # configs[4]: per-frame random multipath (8 taps drawn on chip) + LTS estimate + ZF equaliser, Philox noise;
    # frames staged in HBM once per chunk (TX, fading, power), then one receiver pass per SNR point
    mp = o.new_counters(len(SNRS))
    for mode, name in ((pkg.MODE_FAST, "fast"), (pkg.MODE_EXACT, "exact")):
        ms = timed(lambda: o.mc_sweep_multipath(11, rank * nm, nm, N_SYM, 8, SNRS, mode, counters=mp), reps=2)
        out["cfg4_multipath_" + name] = {"frames": nm, "taps": 8, "snr_points": len(SNRS), "ms": ms,
                                         "symbols_per_s": nm * N_SYM * len(SNRS) / (ms * 1e-3)}
    return out


def run_next_rows(o, pkg, torch, dev, peak, n=32768):
    """SURVEY 8(f) rows, measured: the reference's whole over-the-air path, batched (STS || LTS || data, x2 RRC pulse shaping,
    x10 repetition, AWGN over all 9800 samples, capture window, packet detection / selection, matched filter + decimation,
    coarse + fine CFO, receiver).  Per stage: time (CUDA events) and algorithmic bytes (what the stage must read + write)."""
    def timed(fn, reps=3):
        out = fn(); out = fn(); torch.cuda.synchronize()        # twice: the stage outputs ping-pong between two cached allocations
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            out = fn()
        e1.record(); torch.cuda.synchronize()
        return out, e0.elapsed_time(e1) / reps

    gen = torch.Generator(device=dev); gen.manual_seed(31)
    packed = torch.randint(-2 ** 31, 2 ** 31 - 1, (n * N_SYM * 3,), dtype=torch.int32, device=dev, generator=gen)
    starts = torch.randint(0, 9800 - 3008, (n,), dtype=torch.int32, device=dev, generator=gen)
    stages = []

    def stage(name, fn, nbytes):
        out, ms = timed(fn)
        stages.append({"stage": name, "ms": ms, "GBps": nbytes / ms / 1e6, "frac_of_hbm_peak": nbytes / ms / 1e6 / peak})
        return out

    frames = stage("tx_frames (exact)", lambda: o.tx_frames(packed, N_SYM, pkg.MODE_EXACT, with_power=False), n * (24 + 2560))
    full = stage("prepend_sts", lambda: o.prepend_sts(frames), n * (2560 + 3840))
    shaped = stage("rrc_tx (x2 zero-stuff + 21-tap RRC)", lambda: o.rrc_tx(full), n * (3840 + 980 * 8))
    rep = stage("gather (x10 repetition)", lambda: o.gather(shaped, 0, 9800), n * (980 * 8 + 9800 * 8))
    ota = stage("awgn_philox_len (power + noise, 9800 samples)", lambda: o.awgn_philox_len(rep, 12.0, 5, 0, 0, pkg.MODE_FAST), n * (2 * 9800 * 8 + 9800 * 8))
    del rep
    cap = stage("gather (capture window, 3008 samples)", lambda: o.gather(ota, starts, 3008), n * 2 * 3008 * 8)
    corr = stage("packet_detect", lambda: o.packet_detect(cap), n * (3008 * 8 + 2961 * 4))
    idx = stage("packet_select", lambda: o.packet_select(corr), n * (2961 * 4 + 4))
    fr = stage("rrc_rx_idx (matched filter + decimation)", lambda: o.rrc_rx_idx(cap, idx, 480), n * (3008 * 8 + 3840))
    c1 = stage("cfo_coarse", lambda: o.cfo(fr, fine=False)[0], n * 2 * 3840)
    c2 = stage("cfo_fine", lambda: o.cfo(c1, fine=True)[0], n * 2 * 3840)
    lts_data = stage("gather (drop the STS)", lambda: o.gather(c2, 160, 320), n * (3840 + 2560))
    stage("rx_frames (exact, totals)", lambda: o.rx_frames(lts_data, packed, N_SYM, pkg.MODE_EXACT)[0], n * (2048 + 24))
    total_ms = sum(st["ms"] for st in stages)
    res = {"frames": n, "stages": stages, "total_ms": total_ms, "frames_per_s": n / (total_ms * 1e-3),
           "symbols_per_s": n * N_SYM / (total_ms * 1e-3)}
    # the reference's own main() body for one SNR point (Transmitter + channel + Receiver), one host core
    try:
        po = entry.load_oracle(); po.build()
        if po.have_ref():
            r = po.Ref(); r.full_point(1, 2, 12.0)
            t0 = time.perf_counter(); k = 0
            while time.perf_counter() - t0 < 3.0:
                r.full_point(10 + k, 20 + k, 12.0); k += 1
            dt = time.perf_counter() - t0
            res["cpu_reference_full_point"] = {"frames_per_s": k / dt, "cores": 1, "kind": "reference",
                                               "sample": "%d single-frame points of the reference's main() body, %.1f s" % (k, dt)}
    except Exception as exc:                   # the CPU figure is informational
        res["cpu_reference_full_point"] = {"unavailable": type(exc).__name__}
    return res


def bind_near_gpu(local):
    """Pin this rank to the host cores next to its GPU (NVML's CPU affinity) before any pinned host memory is
    allocated, so that the e2e path's H2D copies stay on the GPU's own NUMA node.  Returns a short description."""
    if os.environ.get("OFDM_BENCH_AFFINITY", "1") == "0":
        return "off"
    try:
        import pynvml
        pynvml.nvmlInit()
        hnd = pynvml.nvmlDeviceGetHandleByIndex(local)
        words = pynvml.nvmlDeviceGetCpuAffinity(hnd, (os.cpu_count() + 63) // 64)
        cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1}
        allowed = os.sched_getaffinity(0)
        use = cpus & allowed
        if not use or use == allowed:
            return "all %d cores are local" % len(allowed)
        os.sched_setaffinity(0, use)
        return "%d of %d cores" % (len(use), len(allowed))
    except Exception as e:                      # affinity is an optimisation, never a requirement
        return "unavailable (%s)" % type(e).__name__


def kernel_metrics():
    """ncu-derived pipe / issue utilisation of the kernels that are not HBM-bound (profiles/r2b_kernel_metrics.json, written by
    tools/ncu_summary.py from the committed ncu captures); None when the file is absent"""
    path = os.path.join(ROOT, "profiles", "r2b_kernel_metrics.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f)
    return {}


def run_configs(o, pkg, torch, dist, dev, args, rank, world):
    """configs[2], [3], [4] of BASELINE.json, each with its own roofline statement.  Returns the dict on every rank
    (aggregates are over all ranks: time = max over ranks, work = sum)."""
    peak, _ = peaks()
    km = kernel_metrics()
    lib, h = o.lib, o.h
    out = {}

    def timed(fn, reps):
        fn(); torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record(); torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / reps], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- configs[2]: streaming TX + RX of HBM-resident frames (16 Mi data symbols per GPU), HBM-bound
    n = args.stream_frames
    bits = torch.randint(-2 ** 31, 2 ** 31 - 1, (n * N_SYM * 3,), dtype=torch.int32, device=dev)
    frames = torch.empty((n, pkg.frame_len(N_SYM), 2), dtype=torch.float32, device=dev)
    cnt = o.new_counters(1)
    tx_bytes, rx_bytes = n * (24 + 2560), n * (2048 + 24)
    c2 = {"frames_per_gpu": n, "data_symbols_per_gpu": n * N_SYM, "bytes_per_frame": {"tx": 24 + 2560, "rx": 2048 + 24},
          "note": "rx reads only the LTS halves and the symbol bodies (2048 B of the 2560 B frame) + 24 B of bits; inputs larger than L2; the peak is the "
                  "measured COPY bandwidth (read + write): the read-only receiver can run a little above it (nominal HBM3e: 7.7 TB/s)"}
    for mode, name in ((pkg.MODE_FAST, "fast"), (pkg.MODE_EXACT, "exact")):
        ms_tx = timed(lambda: o._check(lib.ofdm_tx_frames(h, bits.data_ptr(), frames.data_ptr(), None, n, N_SYM, mode)), 5)
        cnt.zero_()
        ms_rx = timed(lambda: o._check(lib.ofdm_rx_frames(h, frames.data_ptr(), bits.data_ptr(), n, N_SYM, mode, cnt.data_ptr(), None)), 5)
        assert int(o.read_counters(cnt)[0].bit_errors) == 0            # noise-free round trip
        rx_kernel = "k_stream_quad<%s,none>" % ("fast" if name == "fast" else "checked")
        c2[name] = {"tx": {"ms": ms_tx, "roofline": {"bound": "hbm", "kernel": "k_tx_frames2<%s>" % name, "achieved": tx_bytes / ms_tx / 1e6, "peak": peak,
                                                      "unit": "GB/s", "frac": tx_bytes / ms_tx / 1e6 / peak}},
                    "rx": {"ms": ms_rx, "roofline": dict({"bound": "hbm", "kernel": rx_kernel, "achieved": rx_bytes / ms_rx / 1e6, "peak": peak,
                                                           "unit": "GB/s", "frac": rx_bytes / ms_rx / 1e6 / peak},
                                                          **{k: v for k, v in km.get("k_stream_quad_%s_none" % ("fast" if name == "fast" else "checked"), {}).items()
                                                             if k in ("warp_instructions_per_unit", "smem_wavefronts_per_unit", "issue_active_pct", "ipc", "registers", "source")})},
                    "symbols_per_s_tx_plus_rx": world * n * N_SYM / ((ms_tx + ms_rx) * 1e-3)}
    out["cfg2_streaming"] = c2
    del frames, bits
    torch.cuda.empty_cache()

    # ---- configs[3] / configs[4]: on-chip Philox Monte-Carlo, sharded by global frame index, all-reduce inside the timed region
    nm = args.mc_frames
    mc = o.new_counters(len(SNRS))

    def mc_step(mode, n_taps):
        mc.zero_()
        o.mc_sweep_points(7, rank * nm, nm, N_SYM, n_taps, SNRS, None, mode, mc)
        if world > 1:
            pkg.sweep.allreduce_counter_tensor(mc)

    for key, n_taps in (("cfg3_philox_mc", 0), ("cfg4_multipath_8taps", 8)):
        c = {"frames_per_gpu": nm, "snr_points": len(SNRS), "taps": n_taps,
             "parallelism": "global frame index sharded over %d GPU(s), one NCCL all-reduce of the counters per sweep (inside the timed region)" % world}
        for mode, name in ((pkg.MODE_FAST, "fast"), (pkg.MODE_EXACT, "exact")):
            ms = timed(lambda: mc_step(mode, n_taps), 2)
            tot = o.read_counters(mc)
            assert all(t.frames == world * nm and t.bits == world * nm * 96 * N_SYM for t in tot), "all-reduced totals"
            sym = world * nm * N_SYM * len(SNRS) / (ms * 1e-3)
            c[name] = {"ms": ms, "symbols_per_s": sym, "symbols_per_s_per_gpu": sym / world,
                       # transforms actually executed per frame and SNR point: three (one frame per lane group, the LTS halves are added
                       # in time); 1920 flop per 64-point transform
                       "fft_tflops_per_gpu": nm * len(SNRS) * 3 * 1920 / (ms * 1e-3) / 1e12,
                       "ber_0_10_14dB": [tot[0].bit_errors / tot[0].bits, tot[10].bit_errors / tot[10].bits, tot[14].bit_errors / tot[14].bits],
                       "roofline": dict({"bound": "issue (on-chip: no HBM traffic beyond the counters)",
                                         "kernel": ("k_mc_quad<fast,multipath>" if n_taps and name == "fast" else
                                                    "staged: k_tx_frames2 + k_multipath + k_frame_power + k_stream_quad<checked,philox> per point" if n_taps else
                                                    "k_mc_quad<%s>" % ("fast" if name == "fast" else "checked"))},
                                        **km.get("k_mc_quad_fast_multipath" if n_taps and name == "fast" else
                                                 "k_mc_quad_%s" % ("fast" if name == "fast" else "checked") if not n_taps else "", {}))}
        out[key] = c

    # ---- configs[3] as stated: every SNR point until >= 100 bit errors or the BER-1e-7 budget (1e9 bits), rounds sharded over the ranks
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    round_frames = args.until_round_frames * world          # a round keeps every GPU busy for the same time as at N = 1
    tot, rounds = pkg.sweep.mc_sweep_until(o, 11, N_SYM, SNRS, pkg.MODE_FAST, 100, 10 ** 9, round_frames, 0, rank, world)
    torch.cuda.synchronize()
    dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    work = sum(t.frames for t in tot)
    out["cfg3_philox_mc"]["until_100_errors_or_1e-7"] = {
        "seconds": float(dt.item()), "rounds": rounds, "round_frames": round_frames, "mode": "fast",
        "frame_points": int(work), "symbols_per_s": work * N_SYM / float(dt.item()),
        "points": [{"snr_db": s, "bit_errors": int(t.bit_errors), "bits": int(t.bits), "ber": t.bit_errors / t.bits} for s, t in zip(SNRS, tot)],
        "parallelism": "every round's frame range split over %d GPU(s) for every still-active SNR point; one all-reduce per round" % world}
    return out


def run_gpu(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    affinity = bind_near_gpu(local)
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    pkg = entry.load_pkg()
    o = pkg.Ofdm(local)
    n_frames, n_snr = args.frames, len(SNRS)
    flen = pkg.frame_len(N_SYM)
    gen = torch.Generator(device=dev)
    gen.manual_seed(1000 + rank)
    bits = torch.randint(-2 ** 31, 2 ** 31 - 1, (n_frames * N_SYM * 3,), dtype=torch.int32, device=dev, generator=gen)
    g = torch.randn((n_frames, flen), dtype=torch.float32, device=dev, generator=gen)
    frames = torch.empty((n_frames, flen, 2), dtype=torch.float32, device=dev)
    power = torch.empty((n_frames,), dtype=torch.float32, device=dev)
    counters = o.new_counters(n_snr)
    host_cnt = torch.empty(counters.shape, dtype=torch.int64).pin_memory()
    bits_h = torch.empty(bits.shape, dtype=torch.int32).pin_memory(); bits_h.copy_(bits)
    g_h = torch.empty(g.shape, dtype=torch.float32).pin_memory(); g_h.copy_(g)
    snr_arr = np.ascontiguousarray(SNRS, dtype=np.float32)
    torch.cuda.synchronize()
    lib, h = o.lib, o.h

    def sweep_resident(record):
        """Transmitter once, then the whole SNR list in one kernel; returns the (start, end) events around the sweep kernel"""
        counters.zero_()
        o._check(lib.ofdm_tx_frames(h, bits.data_ptr(), frames.data_ptr(), power.data_ptr(), n_frames, N_SYM, pkg.MODE_EXACT))
        ev = None
        if record:
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True); e0.record()
        o._check(lib.ofdm_awgn_rx_inject_sweep(h, frames.data_ptr(), g.data_ptr(), power.data_ptr(), bits.data_ptr(), snr_arr.ctypes.data, n_snr,
                                               n_frames, N_SYM, pkg.MODE_EXACT, counters.data_ptr()))
        if record:
            e1.record(); ev = (e0, e1)
        if world > 1:
            pkg.sweep.allreduce_counter_tensor(counters)
        host_cnt.copy_(counters, non_blocking=True)
        return ev

    def sweep_host():
        res = o.sweep_inject_host(bits_h, g_h, n_frames, N_SYM, SNRS, pkg.MODE_EXACT)
        if world > 1:
            res = pkg.sweep.allreduce_counters(res, device=dev)
        return res

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    sampler = ClockSampler(local)
    for _ in range(args.warmup):
        sweep_resident(False)
    barrier()
    if rank == 0:
        sampler.start()
    launches0 = o.launch_count
    o.replayed_frames(reset=True)
    t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
    t0.record()
    sweep_evs = []
    for _ in range(args.steps):
        sweep_evs.append(sweep_resident(True))
    t1.record()
    barrier()
    launches = o.launch_count - launches0
    replayed = o.replayed_frames() / max(1, args.steps)
    ms_total = t0.elapsed_time(t1)
    sweep_kernel_ms = float(np.mean([a.elapsed_time(b) for a, b in sweep_evs]))
    resident_counts = o.read_counters(host_cnt)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, pkg, torch, frames, power, host_cnt)

    # the HBM-bound kernel of the path, one SNR point per launch (stage API): steps x 21 launches, events around each
    # (after one second of idle: the first sweep of the loop then shows the kernel at full clocks, the mean over the whole loop
    # shows it under the power cap the box applies after ~100 ms of this load -- tools/sustained_probe.py)
    staged_cnt = o.new_counters(n_snr)
    point_evs = []
    torch.cuda.synchronize()
    time.sleep(1.0)
    for rep in range(args.steps + 1):
        staged_cnt.zero_()
        for i, s in enumerate(SNRS):
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True); e0.record()
            o._check(lib.ofdm_awgn_rx_inject(h, frames.data_ptr(), g.data_ptr(), power.data_ptr(), bits.data_ptr(), s,
                                             n_frames, N_SYM, pkg.MODE_EXACT, staged_cnt[i].data_ptr(), None))
            e1.record()
            point_evs.append((e0, e1))
    torch.cuda.synchronize()
    kernel_ms_all = [a.elapsed_time(b) for a, b in point_evs]
    kernel_ms_burst = kernel_ms_all[3:n_snr]          # first sweep after the idle second, less its first launches (cold instruction cache)
    kernel_ms = kernel_ms_all[n_snr:]                 # the remaining `steps` sweeps: sustained
    staged_counts = o.read_counters(staged_cnt)

    # end to end through the public host-buffer API
    for _ in range(max(1, args.warmup // 2)):
        sweep_host()
    barrier()
    w0 = time.perf_counter()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        e2e_counts = sweep_host()
    e1.record()
    barrier()
    e2e_ms_total = max(e0.elapsed_time(e1), (time.perf_counter() - w0) * 1e3)   # wall clock covers the host side of the call
    clocks = sampler.stop() if rank == 0 else None

    g_h = bits_h = None              # release the pinned host buffers
    configs = run_configs(o, pkg, torch, dist, dev, args, rank, world) if not args.no_configs else None
    extras = run_extras(o, pkg, torch, dev, args, rank, world) if args.extras else None
    tm = torch.tensor([ms_total, e2e_ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    ms_total, e2e_ms_total = tm.tolist()
    # every route must agree on every integer total: all-SNR kernel == one launch per point (this rank's frames), and the
    # all-reduced totals of the resident and the host-buffer sweeps (all ranks' frames)
    local_res = resident_counts if world == 1 else None
    for i, b in enumerate(staged_counts):
        assert b.frames == n_frames and b.bits == n_frames * 96 * N_SYM
        if local_res is not None:
            a = local_res[i]
            assert (a.bit_errors, a.rail_errors, a.frames_in_error) == (b.bit_errors, b.rail_errors, b.frames_in_error), "fused vs per-point"
    for a, b in zip(resident_counts, e2e_counts):
        assert a.frames == world * n_frames and a.bits == world * n_frames * 96 * N_SYM, "all-reduced frame / bit totals"
        assert (a.bit_errors, a.rail_errors, a.frames_in_error, a.frames, a.bits) == (b.bit_errors, b.rail_errors, b.frames_in_error, b.frames, b.bits), \
            "resident vs host-buffer sweep"
    if rank == 0:
        symbols = n_frames * N_SYM * n_snr * world
        ms_step = ms_total / args.steps
        value = symbols / (ms_step * 1e-3)
        e2e_value = symbols / (e2e_ms_total / args.steps * 1e-3)
        k_ms = float(np.mean(kernel_ms))
        peak, peak_src = peaks()
        achieved = BYTES_PER_FRAME_PASS * n_frames / (k_ms * 1e-3) / 1e9
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            with open(tpath) as f:
                traffic = json.load(f).get("k_stream_quad_checked_inject_bytes_per_launch")
                if traffic is not None and n_frames != 1_000_000:
                    traffic = traffic * n_frames / 1_000_000        # captured on the 1 M-frame launch
        ber = [c.bit_errors / max(1, c.bits) for c in resident_counts]
        km = kernel_metrics()
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32+f64", "data": "synthetic",
                "config": {"workload": workload_name(n_frames), "frames_per_gpu": n_frames, "n_sym": N_SYM, "snr_db": [SNRS[0], SNRS[-1]],
                           "mode": "exact", "l2": "inputs larger than L2 (%.2f GB of draws + %.2f GB of TX IQ per sweep)"
                                                   % (g.numel() * 4 / 1e9, frames.numel() * 4 / 1e9),
                           "parallelism": "frames sharded across %d GPU(s), one NCCL all-reduce of the counters" % world,
                           "host_affinity": affinity},
                "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": e2e_ms_total / args.steps,
                        # the draws of the guard interval / cyclic prefixes are never read by the receiver and stay on the host
                        "h2d_bytes_per_step": int(n_frames * N_SYM * 12 + n_frames * (128 + 64 * N_SYM) * 4),
                        "host_buffer_bytes": int(n_frames * N_SYM * 12 + n_frames * flen * 4),
                        "d2h_bytes_per_step": int(n_snr * pkg.COUNTERS_BYTES)},
                "gpu_launches": int(launches),
                "roofline": {"bound": "hbm", "kernel": "k_stream_quad<checked,inject>", "achieved": achieved, "peak": peak,
                             "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                             # the measured peak is a copy (read + write); this kernel only reads, and a read-only stream can run a
                             # little above a copy's rate: the nominal HBM3e figure beside it, for context
                             "nominal_GBps": 7700.0, "frac_of_nominal": achieved / 7700.0,
                             "kernel_ms_burst": float(np.mean(kernel_ms_burst)),
                             "frac_burst": BYTES_PER_FRAME_PASS * n_frames / (float(np.mean(kernel_ms_burst)) * 1e-3) / 1e9 / peak,
                             "burst_vs_sustained": "kernel_ms / frac: mean over %d back-to-back launches (sustained: the box power-caps this kernel after ~100 ms, "
                                                   "a plain copy is not affected); kernel_ms_burst / frac_burst: the first sweep's launches after 1 s of idle" % len(kernel_ms),
                             "bytes_per_launch": BYTES_PER_FRAME_PASS * n_frames, "kernel_ms": k_ms,
                             "timed": "%d launches (one per SNR point, %d sweeps) through ofdm_awgn_rx_inject in this run, CUDA events per launch"
                                      % (len(kernel_ms), args.steps),
                             "sweep_ms_if_launched_per_point": k_ms * n_snr,
                             "kernel_ms_by_snr_point": [round(float(np.mean(kernel_ms[i::n_snr])), 4) for i in range(n_snr)]},
                "sweep_kernel": dict({"kernel": "k_sweep_lin<checked>", "kernel_ms": sweep_kernel_ms, "share_of_step": sweep_kernel_ms / ms_step,
                                      "bound": "instruction issue (the frame and its draws cross HBM once per sweep)",
                                      "hbm_GBps": BYTES_PER_FRAME_PASS * n_frames / (sweep_kernel_ms * 1e-3) / 1e9,
                                      "frame_points_per_s": n_frames * n_snr / (sweep_kernel_ms * 1e-3),
                                      "points_replayed_exactly_per_sweep": replayed, "frame_points_per_sweep": n_frames * n_snr},
                                     **km.get("k_sweep_lin_checked", {})),
                "clocks": clocks,
                "ber_0_10_20dB": [ber[0], ber[10], ber[20]]}
        if configs:
            line["configs"] = configs
        if extras:
            line["extras"] = extras
        if not args.no_cpu and world == 1:
            line["cpu_baseline"] = cpu_baseline_single(args.cpu_sample)
        emit(line)
    o.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


DUMP_SAMPLE_FRAMES = 8192


def dump_outputs(out_dir, pkg, torch, frames, power, counters):
    """Write what the last timed step returned to its caller, so that two builds can be compared output for output:
    counters.npy (one row per SNR point, columns as ofdm_counters, float64: the integer totals stay exact) and, for a
    fixed, seeded sample of frames, the TX IQ and frame power (sample_*.npy; about 21 MB at any frame count)."""
    os.makedirs(out_dir, exist_ok=True)
    n_frames = frames.shape[0]
    idx = np.sort(np.random.default_rng(0).choice(n_frames, min(DUMP_SAMPLE_FRAMES, n_frames), replace=False))
    sel = torch.from_numpy(idx).to(frames.device)
    raw = counters.cpu().numpy()
    n_int = pkg.sweep.N_INT_FIELDS
    cnt = np.concatenate([raw[:, :n_int].astype(np.float64), raw[:, n_int:].copy().view(np.float64)], axis=1)
    arrays = {"counters": cnt, "sample_frame_index": idx.astype(np.float64),
              "sample_tx_frames": frames.index_select(0, sel).cpu().numpy(), "sample_tx_power": power.index_select(0, sel).cpu().numpy()}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def emit(line):
    """print the one JSON line on the real stdout (libraries such as NCCL may write to fd 1 meanwhile)"""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)            # anything else that prints to stdout goes to stderr
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--frames", type=int, default=1_000_000, help="frames per GPU")
    ap.add_argument("--cpu-sample", type=int, default=12000, help="frames in the single-thread CPU baseline sample")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--extras", action="store_true", help="also measure configs[2] (streaming) and configs[3] (Philox MC)")
    ap.add_argument("--stream-frames", type=int, default=8_388_608, help="frames for the streaming extra (16 Mi data symbols)")
    ap.add_argument("--mc-frames", type=int, default=2_000_000, help="frames per GPU of the configs[3] / configs[4] Monte-Carlo sweeps")
    ap.add_argument("--until-round-frames", type=int, default=1 << 20, help="frames per round and GPU of the until-rule sweep")
    ap.add_argument("--no-configs", action="store_true", help="skip configs[2] / [3] / [4] (A/B runs of the headline only)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the b200 path")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        return run_reference(args)
    return run_gpu(args)


if __name__ == "__main__":
    sys.exit(main())
