"""Generates tests/golden/stage_vectors.npz and tests/golden/chain_totals.npz from the COMPILED, UNMODIFIED
reference (oracle/_ref/libofdm_ref.so, built by oracle/Makefile from $REF_ROOT/src/OFDM.c, REF_ROOT being a
checkout of the original simulator):

    REF_ROOT=<checkout of the original> python tests/golden/make_golden.py

Contents: per-stage vectors of the reference stage chain for a few frames (bits, QPSK points, grid,
TX IQ, the noise draw g_keep captured from the reference's rand()/Box-Muller stream, OTA IQ, H_est,
equalised points, slicer output, demodulated bits, per-frame EVM / bit errors) at several SNRs and
two frame lengths; in chain_totals.npz, whole-chain totals for a 256-frame batch per SNR.  Two files keep
each well under 1 MB.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import pyoracle as po  # noqa: E402


def main():
    ref_root = os.environ.get("REF_ROOT")
    if not ref_root or not os.path.isfile(os.path.join(ref_root, "src", "OFDM.c")):
        raise SystemExit("set REF_ROOT to a checkout of the original simulator (it must contain src/OFDM.c)")
    po.build(force=True)                # oracle/Makefile takes REF_ROOT from the environment
    ref = po.Ref()
    out = {}
    out["lts_freq"] = ref.lts_freq()
    out["lts_time"] = ref.lts_time()
    rng = np.random.default_rng(20261018)
    x = rng.standard_normal((16, 64, 2)).astype(np.float32)
    out["fft_in"] = x
    out["fft_out"] = ref.fft64(x)
    out["ifft_out"] = ref.ifft64(x)
    for n_sym, n_frames in ((2, 24), (5, 6)):
        tag = "n%d_" % n_sym
        L = 160 + 80 * n_sym
        bits = rng.integers(0, 2, (n_frames, 96 * n_sym), dtype=np.uint8)
        # frame 0 of the n_sym=2 set carries the reference repo's own golden bits (data/Matlab_Output.txt) as symbol 0
        if n_sym == 2:
            mo = os.path.join(ref_root, "data", "Matlab_Output.txt")
            b96 = np.array(open(mo).read().split(), dtype=np.float64).astype(np.uint8)
            assert b96.size == 96
            bits[0, :96] = b96
            out["matlab_output_bits"] = b96
        out[tag + "bits"] = bits
        mod = ref.qpsk_mod(bits)
        out[tag + "mod"] = mod
        out[tag + "grid"] = ref.map_grid(mod)
        out[tag + "sym_time"] = ref.ifft64(out[tag + "grid"])
        tx = ref.tx_frames(bits, n_sym)
        out[tag + "tx"] = tx
        out[tag + "power"] = np.array([ref.frame_power(f) for f in tx], np.float32)
        snrs = np.array([0.0, 4.0, 9.0, 15.0, 30.0], np.float32)
        out[tag + "snr"] = snrs
        g = ref.capture_gkeep(n_frames * L, seed=4242 + n_sym).reshape(n_frames, L)
        out[tag + "g"] = g
        for i, s in enumerate(snrs):
            # OTA through the reference's own Transmission_Over_Air with the same libc stream
            ref.seed(4242 + n_sym)
            ota = np.stack([ref.awgn(tx[f], float(s), seed=None) for f in range(n_frames)])
            ota_inj = ref.awgn_inject(tx, g, float(s))
            assert np.array_equal(ota, ota_inj), "captured g does not reproduce Transmission_Over_Air"
            r = ref.rx_frames(ota, bits, n_sym)
            out[tag + "ota_%d" % i] = ota
            for k in ("H", "eq", "sliced", "bits", "evm_lin", "evm_db", "evm_agc_lin", "evm_agc_db", "ber", "bit_errors", "rail_errors"):
                out[tag + "rx_%s_%d" % (k, i)] = r[k]
    # the reference's own over-the-air waveform (Transmitter(): STS, LTS, 2 symbols of "Hey! I am Vivaswan", x2, RRC, x10)
    out["ref_tx_waveform"] = ref.transmit_full()
    # whole-chain totals
    n_sym, n_frames = 2, 256
    bits = rng.integers(0, 2, (n_frames, 96 * n_sym), dtype=np.uint8)
    g = ref.capture_gkeep(n_frames * 320, seed=777).reshape(n_frames, 320)
    out["chain_bits"], out["chain_g"] = bits, g
    snrs = np.arange(0, 21, 2, dtype=np.float32)
    out["chain_snr"] = snrs
    tot = []
    for s in snrs:
        a = ref.chain(bits, g, n_sym, float(s))
        tot.append([a.bit_errors, a.bits, a.frames_in_error, a.rail_errors, a.frames, a.sum_err2, a.sum_ref2, a.sum_evm_lin])
    out["chain_totals"] = np.array(tot, np.float64)
    chain = {k: out.pop(k) for k in [k for k in out if k.startswith("chain_")]}
    for name, arrays in (("stage_vectors.npz", out), ("chain_totals.npz", chain)):
        path = os.path.join(ROOT, "tests", "golden", name)
        np.savez_compressed(path, **arrays)
        print("wrote", path, os.path.getsize(path), "bytes,", len(arrays), "arrays")


if __name__ == "__main__":
    main()
