"""Speed of the coded link on one GPU, in one process: k_viterbi alone over the receiver's dumps of 1 M two-symbol frames for
{1/2, 3/4} x {soft, hard}, then the coded Monte-Carlo sweep at 1 M frames x 21 Eb/N0 points (0..20 dB, complex noise) and, as
the control in the same run, the uncoded sweep through the same staged route (force_generic_rx = 1: Philox bits, transmitter,
per point the channel into HBM and the receiver).  CUDA events, best of --repeats after a warm-up of every shape.  Writes one JSON
file with the card's name and power limit read in the same call, data symbols per second, and the decoder's share of a sweep
(its stand-alone time x 21 points over the sweep's time).

    python tools/coded_speed.py [--frames N] [--repeats R] [--out profiles/coded_speed_b200.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import __graft_entry__ as entry  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                             timeout=30).stdout.strip()
        name, limit = [x.strip() for x in out.split(",")]
        return name, limit
    except (OSError, subprocess.SubprocessError, ValueError):
        return None, None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1 << 20)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "coded_speed_b200.json"))
    args = ap.parse_args()
    import torch
    pkg = entry.load_pkg()
    o = pkg.Ofdm(0)
    n, n_sym, seed = args.frames, 2, 7
    snrs = np.arange(21, dtype=np.float32)

    def timed(fn):
        best = None
        for r in range(args.repeats):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn(r)
            b.record()
            b.synchronize()
            best = a.elapsed_time(b) if best is None else min(best, a.elapsed_time(b))
        return best

    name, limit = card()
    result = {"device": name or torch.cuda.get_device_name(0), "power_limit": limit, "frames": n, "n_sym": n_sym, "snr_points": len(snrs),
              "decoder": {}, "sweeps": {}}

    # ---- the decoder alone on the receiver's dumps (complex noise, Eb/N0 = 3 dB)
    for rate in ("1/2", "3/4"):
        words = o.random_bits(seed, 0, n, n_sym)
        payload = o.conv_encode(words, n_sym, rate)
        tx = o.tx_frames(payload, n_sym, pkg.MODE_FAST, with_power=False)
        ota = o.awgn_philox_ex(tx, 3.0, seed, 0, 0, n_sym, pkg.MODE_FAST, "complex", "ebn0")
        del tx
        _, bufs = o.rx_frames(ota, payload, n_sym, pkg.MODE_FAST, want=("H", "eq"))
        del ota
        H, eq = bufs["H"], bufs["eq"]
        cnt = o.new_counters()
        for decision in ("soft", "hard"):
            cd = pkg.code(rate, decision)

            def dec(_r):
                o._check(o.lib.ofdm_viterbi_decode(o.h, C.byref(cd), H.data_ptr(), eq.data_ptr(), words.data_ptr(), None, n, n_sym, cnt.data_ptr()))
            dec(0)
            torch.cuda.synchronize()
            cnt.zero_()
            ms = timed(dec)
            c = o.read_counters(cnt)[0]
            result["decoder"]["%s_%s" % (rate, decision)] = {
                "ms": round(ms, 3), "frames_per_s": n / (ms * 1e-3), "data_symbols_per_s": n * n_sym / (ms * 1e-3),
                "trellis_steps_per_s": n * n_sym * pkg.DATA_BITS_PER_SYM[rate] / (ms * 1e-3), "ber_3db_ebn0": c.bit_errors / c.bits}
        del H, eq, bufs

    # ---- whole sweeps: coded (staged by definition) and the uncoded staged control, FAST and EXACT
    coded = o.new_counters(len(snrs))
    raw = o.new_counters(len(snrs))
    runs = {}
    for mode_name, mode in (("fast", pkg.MODE_FAST), ("exact", pkg.MODE_EXACT)):
        runs["uncoded_staged_%s" % mode_name] = ("uncoded", mode, None)
        for rate in ("1/2", "3/4"):
            runs["coded_%s_soft_%s" % (rate, mode_name)] = ("coded", mode, rate)

    def sweep(spec, frames, frame0):
        kind, mode, rate = spec
        if kind == "uncoded":
            o.set_option("force_generic_rx", 1)
            try:
                o.mc_sweep_channel(seed, frame0, frames, n_sym, snrs, mode, "complex", "ebn0", counters=coded)
            finally:
                o.set_option("force_generic_rx", 0)
        else:
            o.mc_sweep_coded(seed, frame0, frames, n_sym, snrs, mode, rate, "soft", "complex", "ebn0", counters=(coded, raw))

    for spec in runs.values():                    # module load, scratch allocation at the full size
        sweep(spec, n, 0)
    torch.cuda.synchronize()
    for key, spec in runs.items():
        coded.zero_()
        ms = timed(lambda r: sweep(spec, n, (r + 1) * n))
        c = o.read_counters(coded)
        entry_ = {"mode": "fast" if spec[1] == pkg.MODE_FAST else "exact", "ms": round(ms, 3),
                  "data_symbols_per_s": n * n_sym * len(snrs) / (ms * 1e-3),
                  "ber_4db": c[4].bit_errors / c[4].bits, "per_4db": c[4].frames_in_error / c[4].frames}
        if spec[0] == "coded":
            dec_ms = result["decoder"]["%s_soft" % spec[2]]["ms"]
            entry_["decoder_share"] = round(dec_ms * len(snrs) / ms, 3)
        result["sweeps"][key] = entry_
    o.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
