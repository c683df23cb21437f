"""What a replay costs in the one-frame-per-lane-group kernels, as tools/replay_cost.py measures it for the all-SNR kernel:
k_stream_quad<checked, inject> (ofdm_awgn_rx_inject on 1 M two-symbol frames, one SNR point) and k_mc_quad<checked>
(ofdm_mc_sweep_philox, 200 k frames x 21 points), each timed normally and with every frame, or (frame, point), replayed.
CUDA events around `reps` calls after one warm-up call; seeded inputs.
    python tools/replay_cost_quad.py [reps]            (OFDM_B200_LIB=<other build> for an A/B run)
Prints one JSON line."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import __graft_entry__ as e

pkg = e.load_pkg()
o = pkg.Ofdm(0)
dev = o.device
reps = int(sys.argv[1]) if len(sys.argv) > 1 else 10
out = {"lib": os.environ.get("OFDM_B200_LIB", "default"), "gpu": torch.cuda.get_device_name(dev), "reps": reps}


def timed(call):
    call()
    torch.cuda.synchronize()
    a = torch.cuda.Event(enable_timing=True)
    b = torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        call()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def cost(name, call, units):
    """time `call` normally and with every unit replayed; ns of kernel time per replay"""
    res = {}
    for force in (0, 1):
        o.set_option("force_replay", force)
        o.replayed_frames(reset=True)
        call()
        torch.cuda.synchronize()
        replayed = o.replayed_frames(reset=True)
        res[force] = (timed(call), replayed)
    o.set_option("force_replay", 0)
    (t0, r0), (t1, r1) = res[0], res[1]
    assert r1 == units, (name, r1, units)
    out[name] = {"normal_ms": round(t0, 4), "replayed_normally": int(r0), "every_unit_replayed_ms": round(t1, 4),
                 "ns_per_replay": round((t1 - t0) / (r1 - r0) * 1e6, 3)}


gen = torch.Generator(device=dev)
gen.manual_seed(2024)
N = 1_000_000
bits = torch.randint(-2 ** 31, 2 ** 31 - 1, (N * 6,), dtype=torch.int32, device=dev, generator=gen)
g = torch.randn((N, 320), dtype=torch.float32, device=dev, generator=gen)
frames, power = o.tx_frames(bits, 2, pkg.MODE_EXACT)
cnt = o.new_counters(1)
cost("k_stream_quad_checked_inject", lambda: o.awgn_rx_inject(frames, g, bits, 4.0, 2, pkg.MODE_EXACT, power=power, counters=cnt), N)

N_MC = 200_000
snr = [float(s) for s in range(21)]
cnt_mc = o.new_counters(len(snr))
cost("k_mc_quad_checked", lambda: o.mc_sweep_philox(2024, 0, N_MC, 2, snr, pkg.MODE_EXACT, counters=cnt_mc), N_MC * len(snr))
print(json.dumps(out), flush=True)
o.close()
