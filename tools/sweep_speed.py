"""Time the all-SNR sweep kernel k_sweep_lin (ofdm_awgn_rx_inject_sweep on 1 M transmitter frames) in both arithmetics at
21 and 64 SNR points, CUDA events around `reps` calls after one warm-up call.  Seeded inputs, so two builds can be compared
point for point: the integer totals of every point and the exactly replayed (frame, point) count are printed too.
    python tools/sweep_speed.py [reps]                 (OFDM_B200_LIB=<other build> for an A/B run)
Prints one JSON line."""
import hashlib
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import __graft_entry__ as e

pkg = e.load_pkg()
o = pkg.Ofdm(0)
dev, lib, h = o.device, o.lib, o.h
reps = int(sys.argv[1]) if len(sys.argv) > 1 else 20
N = 1_000_000
gen = torch.Generator(device=dev)
gen.manual_seed(2024)
out = {"lib": os.path.relpath(pkg.binding.LIB_PATH if not os.environ.get("OFDM_B200_LIB") else os.environ["OFDM_B200_LIB"]),
       "gpu": torch.cuda.get_device_name(dev), "frames": N, "reps": reps}
bits = torch.randint(-2 ** 31, 2 ** 31 - 1, (N * 6,), dtype=torch.int32, device=dev, generator=gen)
g = torch.randn((N, 320), dtype=torch.float32, device=dev, generator=gen)
frames = torch.empty((N, 320, 2), dtype=torch.float32, device=dev)
power = torch.empty((N,), dtype=torch.float32, device=dev)
for mode_name, mode in (("exact", pkg.MODE_EXACT), ("fast", pkg.MODE_FAST)):
    o._check(lib.ofdm_tx_frames(h, bits.data_ptr(), frames.data_ptr(), power.data_ptr(), N, 2, mode))
    for n_snr in (21, 64):
        snrs = np.ascontiguousarray(np.linspace(-4.0, 26.0, n_snr) if n_snr != 21 else np.arange(21.0), dtype=np.float32)
        cnt = o.new_counters(n_snr)

        def call():
            o._check(lib.ofdm_awgn_rx_inject_sweep(h, frames.data_ptr(), g.data_ptr(), power.data_ptr(), bits.data_ptr(),
                                                   snrs.ctypes.data, n_snr, N, 2, mode, cnt.data_ptr()))
        cnt.zero_()
        o.replayed_frames(reset=True)
        call()
        torch.cuda.synchronize()
        replayed = o.replayed_frames(reset=True)
        res = o.read_counters(cnt)
        ints = [(c.bit_errors, c.rail_errors, c.frames_in_error, c.frames, c.bits) for c in res]
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            call()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        out["%s_%d" % (mode_name, n_snr)] = {"kernel_ms": round(ms, 4), "frame_points_per_s": N * n_snr / ms * 1e3,
                                              "replayed": int(replayed), "bit_errors": int(sum(c.bit_errors for c in res)),
                                              "integer_totals_sha1": hashlib.sha1(repr(ints).encode()).hexdigest()[:12],
                                              "sum_err2": [float(c.sum_err2) for c in res]}
print(json.dumps(out), flush=True)
o.close()
