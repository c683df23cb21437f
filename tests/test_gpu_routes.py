"""Which kernels one call runs.  The receiver entry points, the SNR sweep on resident frames and the Monte-Carlo sweeps pick a
kernel family, a template build and the receiver's params from the mode, the noise source, the frame shape, the buffers and the
context's options (csrc/ofdm_b200.cu: rx_family / rx_policy, ofdm_mc_sweep_channel_dev; DESIGN.md "Routing").  Each case runs
one call under torch.profiler and checks the kernels it launched, by name, against the routing tables written out below, the
context's launch count, and the replay counter: a kernel that gets the caller's raw params (the generic receiver, the all-exact
arithmetic, the fused sweeps of the non-reference channels) never counts a replay, even with "force_replay" on."""
import json
import os
import re
import tempfile

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

EXACT, FAST = 0, 1
A_FAST, A_EXACT, A_CHECKED = 0, 1, 2                    # kArith*
N_NONE, N_INJECT, N_PHILOX = 0, 1, 2                    # kNoise*
SEED = 77
DEFAULTS = {"force_generic_rx": 0, "exact_speculation": 1, "force_replay": 0, "general_stream": 0, "stream_layout": 0,
            "stream_warps": 6, "multipath_path": 0, "fused_sweep": 1}
# each option alone on top of the defaults; "dump" (per-frame outputs) and "unaligned" (input a view offset by 2 floats) are
# properties of the call
RX_VARIANTS = [{}, {"force_generic_rx": 1}, {"exact_speculation": 0}, {"force_replay": 1}, {"general_stream": 1},
               {"stream_layout": 1}, {"stream_warps": 8}, {"dump": 1}, {"unaligned": 1}]
MC_VARIANTS = [{}, {"force_generic_rx": 1}, {"exact_speculation": 0}, {"force_replay": 1}, {"general_stream": 1},
               {"stream_layout": 1}, {"stream_warps": 8}, {"multipath_path": 1}, {"multipath_path": 2}]
SWEEP_VARIANTS = [{}, {"fused_sweep": 0}, {"force_generic_rx": 1}, {"exact_speculation": 0}, {"general_stream": 1},
                  {"stream_layout": 1}, {"unaligned": 1}]
CHANNELS = [("real", "frame_power"), ("complex", "frame_power"), ("real", "esn0"), ("complex", "esn0"), ("real", "ebn0"),
            ("complex", "ebn0")]


def b(x):
    return "true" if x else "false"


def opt(v, name):
    return v.get(name, DEFAULTS.get(name, 0))


def arith_of(mode, v):
    return A_FAST if mode == FAST else A_CHECKED if opt(v, "exact_speculation") else A_EXACT


# ---- the routing tables
def rx_route(mode, noise, n_sym, v, dump=False, aligned=True):
    """(kernel, gets the policy params) of one receiver call"""
    arith = arith_of(mode, v)
    if dump or not aligned or opt(v, "force_generic_rx"):
        return "k_rx_frames<%s,%d,%s>" % (b(mode == EXACT), noise, b(dump)), False
    if opt(v, "stream_layout") == 0 and arith != A_EXACT:
        w, nsym2 = (8, False) if opt(v, "stream_warps") == 8 else (6, n_sym == 2 and not opt(v, "general_stream"))
        return "k_stream_quad<%d,%d,%d,%s>" % (arith, noise, w, b(nsym2)), True
    if n_sym != 2 or opt(v, "general_stream"):
        return "k_stream_rxn<%d,%d>" % (arith, noise), arith != A_EXACT
    return "k_stream_rx2<%d,%d>" % (arith, noise), arith != A_EXACT


def tx_kernels(mode, n_sym, v, power):
    e = b(mode == EXACT)
    ks = ["k_tx_frames2<%s>" % e if n_sym == 2 and not opt(v, "force_generic_rx") else "k_tx_frames<%s>" % e]
    if power:
        ks.append("k_frame_power_tiled" if mode == EXACT else "k_frame_power_fast")
    return ks


def mc_route(noise, snr_def, n_taps, mode, n_sym, v, n_points):
    """(kernels, the sweep's kernels all take the raw params) of one Monte-Carlo sweep"""
    ref, mp, fast, arith = (noise, snr_def) == ("real", "frame_power"), n_taps > 0, mode == FAST, arith_of(mode, v)
    per_frame, generic = snr_def == "frame_power", opt(v, "force_generic_rx")
    if not ref:
        fused = n_sym == 2 and fast and not generic
    elif not mp:
        fused = n_sym == 2
    else:
        fused = n_sym == 2 and not generic and (opt(v, "multipath_path") == 2 or (opt(v, "multipath_path") == 0 and fast))
    if fused:
        layout0 = opt(v, "stream_layout") == 0
        if not ref:
            ch = (1 if noise == "complex" else 0) | (0 if per_frame else 2)
            return ["k_mc_quad<0,%s,%d>" % (b(mp), ch)], True
        if (arith == A_FAST and layout0) or (arith == A_CHECKED and layout0 and not mp):
            return ["k_mc_quad<%d,%s,0>" % (arith, b(mp))], False
        return ["k_mc_philox<%d,%s>" % (arith, b(mp))], False
    ks = ["k_philox_bits"] + tx_kernels(mode, n_sym, v, per_frame and not mp)
    if mp:
        ks += ["k_multipath<true>"] + (tx_kernels(mode, n_sym, v, True)[1:] if per_frame else [])
    raw = True
    for _ in range(n_points):
        if ref:
            k, policy = rx_route(mode, N_PHILOX, n_sym, v)
        else:
            ks.append("k_awgn_channel<%s,%s>" % (b(mode == EXACT), b(noise == "complex")))
            k, policy = rx_route(mode, N_NONE, n_sym, v)
        ks.append(k)
        raw = raw and not policy
    return ks, raw


def sweep_route(mode, n_sym, v, n_points, aligned=True):
    arith = arith_of(mode, v)
    if (opt(v, "fused_sweep") and n_sym == 2 and aligned and not opt(v, "force_generic_rx") and not opt(v, "general_stream")
            and arith != A_EXACT):
        return ["k_sweep_lin<%d>" % arith], False
    k, policy = rx_route(mode, N_INJECT, n_sym, v, aligned=aligned)
    return [k] * n_points, not policy


# ---- one call, observed
def kernel_name(name):
    name = re.sub(r"^void ", "", name).replace("(anonymous namespace)::", "").replace("ofdm::", "")
    name = re.sub(r"\((int|bool)\)", "", name)
    return name.split("(")[0].replace(" ", "")


def observe(o, call):
    """(kernel names in launch order, launch count delta, replay count delta) of call()"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    o.replayed_frames(reset=True)
    l0 = o.launch_count
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        call()
        torch.cuda.synchronize()
    launches = o.launch_count - l0
    replayed = o.replayed_frames(reset=True)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    kernels = sorted((e["ts"], kernel_name(e["name"])) for e in events if e.get("cat") == "kernel")
    return [k for _, k in kernels], launches, replayed


def set_options(o, v):
    for name, default in DEFAULTS.items():
        o.set_option(name, v.get(name, default))


def rx_call(o, pkg, mode, noise, n_sym, v, n_frames=96):
    """the receiver entry point of `noise` on n_frames seeded frames: a closure that runs it, and the counters"""
    torch = o.torch
    bits = o.random_bits(SEED, 0, n_frames, n_sym)
    tx, power = o.tx_frames(bits, n_sym, mode)
    if noise == N_NONE:
        tx = o.awgn_philox(tx, 6.0, SEED, 3, 0, n_sym, mode, power=power)
    if v.get("unaligned"):
        buf = o.empty((tx.numel() + 2,), torch.float32)
        buf[2:].copy_(tx.reshape(-1))
        tx = buf[2:]
    g = torch.randn((n_frames, pkg.frame_len(n_sym)), dtype=torch.float32, device=o.device,
                    generator=torch.Generator(device=o.device).manual_seed(SEED))
    cnt = o.new_counters()
    d, _ = o._dump(n_frames, n_sym, ("bits", "frame_bit_errors") if v.get("dump") else ())
    lib, h, C = o.lib, o.h, pkg.binding.C
    if noise == N_NONE:
        fn = lambda: o._check(lib.ofdm_rx_frames(h, tx.data_ptr(), bits.data_ptr(), n_frames, n_sym, mode, cnt.data_ptr(), C.byref(d)))
    elif noise == N_INJECT:
        fn = lambda: o._check(lib.ofdm_awgn_rx_inject(h, tx.data_ptr(), g.data_ptr(), power.data_ptr(), bits.data_ptr(), 4.0, n_frames,
                                                      n_sym, mode, cnt.data_ptr(), C.byref(d)))
    else:
        fn = lambda: o._check(lib.ofdm_awgn_rx_philox(h, tx.data_ptr(), power.data_ptr(), bits.data_ptr(), 4.0, SEED, 1, 0, n_frames,
                                                      n_sym, mode, cnt.data_ptr(), C.byref(d)))
    return fn, cnt


def sweep_call(o, pkg, mode, n_sym, v, snrs, n_frames=96):
    torch = o.torch
    bits = o.random_bits(SEED, 0, n_frames, n_sym)
    tx, power = o.tx_frames(bits, n_sym, mode)
    g = torch.randn((n_frames * pkg.frame_len(n_sym) + 4,), dtype=torch.float32, device=o.device,
                    generator=torch.Generator(device=o.device).manual_seed(SEED))
    g = g[2:] if v.get("unaligned") else g[:-4]
    cnt = o.new_counters(len(snrs))
    return (lambda: o.awgn_rx_inject_sweep(tx, g, bits, snrs, n_sym, mode, power=power, counters=cnt)), cnt


def mc_call(o, noise, snr_def, n_taps, mode, n_sym, snrs, n_frames=200):
    cnt = o.new_counters(len(snrs))
    return (lambda: o.mc_sweep_channel(SEED, 1000, n_frames, n_sym, snrs, mode, noise=noise, snr_def=snr_def, n_taps=n_taps,
                                       counters=cnt)), cnt


# ---- the matrix (also read by tools/route_digest.py)
def cases():
    out = []
    for mode in (EXACT, FAST):
        for n_sym in (1, 2, 3):
            for noise in (N_NONE, N_INJECT, N_PHILOX):
                for v in RX_VARIANTS:
                    out.append(("rx", mode, n_sym, noise, v))
            for v in SWEEP_VARIANTS:
                out.append(("sweep", mode, n_sym, None, v))
            for ch in CHANNELS:
                for n_taps in (0, 4):
                    for v in (MC_VARIANTS if n_sym != 1 else [{}]):
                        out.append(("mc", mode, n_sym, (ch, n_taps), v))
    return out


def case_id(c):
    kind, mode, n_sym, what, v = c
    w = "" if what is None else "-%s" % (what if kind == "rx" else "%s_%s_%dtaps" % (what[0][0], what[0][1], what[1]))
    return "%s-%s-nsym%d%s-%s" % (kind, "exact" if mode == EXACT else "fast", n_sym, w, "+".join("%s=%s" % kv for kv in v.items()) or "default")


SNRS = [2.0, 9.0]


def run_case(o, pkg, c):
    """set the case's options, run its call once under the profiler: (kernels, launches, replayed, counters, expected route)"""
    kind, mode, n_sym, what, v = c
    set_options(o, v)
    try:
        if kind == "rx":
            fn, cnt = rx_call(o, pkg, mode, what, n_sym, v)
            k, policy = rx_route(mode, what, n_sym, v, dump=bool(v.get("dump")), aligned=not v.get("unaligned"))
            want = ([k], not policy)
        elif kind == "sweep":
            fn, cnt = sweep_call(o, pkg, mode, n_sym, v, SNRS)
            want = sweep_route(mode, n_sym, v, len(SNRS), aligned=not v.get("unaligned"))
        else:
            (noise, snr_def), n_taps = what
            fn, cnt = mc_call(o, noise, snr_def, n_taps, mode, n_sym, SNRS)
            want = mc_route(noise, snr_def, n_taps, mode, n_sym, v, len(SNRS))
        kernels, launches, replayed = observe(o, fn)
        return kernels, launches, replayed, o.read_counters(cnt), want
    finally:
        set_options(o, {})


@pytest.fixture(scope="module")
def octx(pkg, lib):
    o = pkg.Ofdm(0, lib=lib)
    yield o
    o.close()


@pytest.mark.parametrize("case", cases(), ids=case_id)
def test_route(octx, pkg, case):
    kernels, launches, replayed, counters, (want, raw) = run_case(octx, pkg, case)
    assert kernels == want
    assert launches == len(want)
    assert all(c.frames > 0 for c in counters)
    if raw:
        assert replayed == 0                       # raw params: no replay counter
    v, mode = case[4], case[1]
    if v.get("force_replay") and mode == EXACT and not raw and arith_of(mode, v) == A_CHECKED:
        assert replayed > 0                        # the error radii reached the speculating kernel
