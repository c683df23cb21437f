"""Speed of the Monte-Carlo sweep per channel, in one process on one GPU: 1 M frames x 21 SNR points (0..20 dB), two-symbol
frames, payload and noise drawn on chip.  The reference channel's fused sweep (configs[3]) runs first in the same call as the
control.  CUDA events around each sweep, best of --repeats after a warm-up of every route.  Prints one JSON line with data
symbols per second per run, the device name and its power limit.

    python tools/channel_speed.py [--frames N] [--repeats R]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import __graft_entry__ as entry  # noqa: E402

# name -> (mode, noise, snr_def, n_taps, force_generic_rx)
RUNS = {
    "reference_fused_fast": ("fast", "real", "frame_power", 0, 0),
    "complex_esn0_fused_fast": ("fast", "complex", "esn0", 0, 0),
    "complex_esn0_staged_fast": ("fast", "complex", "esn0", 0, 1),
    "complex_esn0_exact": ("exact", "complex", "esn0", 0, 0),
    "complex_esn0_taps8_fused_fast": ("fast", "complex", "esn0", 8, 0),
}


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                             timeout=30).stdout.strip()
        return out or None
    except (OSError, subprocess.SubprocessError):
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1 << 20)
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    import torch
    pkg = entry.load_pkg()
    o = pkg.Ofdm(0)
    snrs = np.arange(21, dtype=np.float32)
    n_sym = 2
    cnt = o.new_counters(len(snrs))

    def sweep(spec, n_frames, frame0=0):
        mode, noise, snr_def, n_taps, generic = spec
        o.set_option("force_generic_rx", generic)
        try:
            o.mc_sweep_channel(7, frame0, n_frames, n_sym, snrs, pkg.MODE_FAST if mode == "fast" else pkg.MODE_EXACT, noise, snr_def, n_taps,
                               counters=cnt)
        finally:
            o.set_option("force_generic_rx", 0)

    for spec in RUNS.values():                       # module load, scratch allocation
        sweep(spec, 4096)
    torch.cuda.synchronize()
    result = {"device": torch.cuda.get_device_name(0), "power_limit": power_limit(), "frames": args.frames, "snr_points": len(snrs),
              "n_sym": n_sym, "runs": {}}
    for name, spec in RUNS.items():
        best = None
        for r in range(args.repeats):
            cnt.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            sweep(spec, args.frames, frame0=r * args.frames)
            b.record()
            b.synchronize()
            ms = a.elapsed_time(b)
            best = ms if best is None else min(best, ms)
        c = o.read_counters(cnt)
        result["runs"][name] = {"mode": spec[0], "noise": spec[1], "snr_def": spec[2], "n_taps": spec[3], "staged": bool(spec[4]),
                                "ms": round(best, 3), "data_symbols_per_s": args.frames * n_sym * len(snrs) / (best * 1e-3),
                                "ber_0db": c[0].bit_errors / c[0].bits, "ber_10db": c[10].bit_errors / c[10].bits}
    o.close()
    print(json.dumps(result))


if __name__ == "__main__":
    main()
