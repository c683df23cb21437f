"""ctypes front-end of tests/channel_oracle.c (TEST INFRASTRUCTURE ONLY): the channels of ofdm_channel on the CPU, plus an
independent float64 numpy model of the complex-noise Es/N0 channel as seen by the receiver.

The library is compiled once per process into a temporary directory with the pinned oracle's flags, so running the tests
writes nothing into the tree."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
NOISE = {"real": 0, "complex": 1}
SNR_DEF = {"frame_power": 0, "esn0": 1, "ebn0": 2}
DOMAIN_NOISE, DOMAIN_NOISE_Q = 0, 4


class Counters(C.Structure):
    _fields_ = [("bit_errors", C.c_uint64), ("bits", C.c_uint64), ("frames_in_error", C.c_uint64),
                ("rail_errors", C.c_uint64), ("frames", C.c_uint64),
                ("sum_err2", C.c_double), ("sum_ref2", C.c_double), ("sum_evm_lin", C.c_double)]


def _p(a, t=C.c_float):
    return None if a is None else a.ctypes.data_as(C.POINTER(t))


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


class ChannelOracle:
    def __init__(self):
        self._dir = tempfile.mkdtemp(prefix="ofdm_channel_oracle_")
        so = os.path.join(self._dir, "libchannel_oracle.so")
        subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-w",
                               "-o", so, os.path.join(HERE, "channel_oracle.c"), "-lm"])
        self.lib = C.CDLL(so)
        self.lib.orc_init()

    @staticmethod
    def frame_len(n_sym):
        return 160 + 80 * n_sym

    def philox_bits(self, seed, frame0, n_frames, n_sym):
        bits = np.zeros((n_frames, 96 * n_sym), np.uint8)
        self.lib.orc_philox_bits(C.c_uint32(seed), C.c_uint64(frame0), C.c_long(n_frames), C.c_int(n_sym), _p(bits, C.c_uint8))
        return bits

    def philox_normals(self, seed, stream, frame0, n_frames, length, domain=DOMAIN_NOISE):
        g = np.zeros((n_frames, length), np.float32)
        self.lib.orc_philox_normals_domain(C.c_uint32(seed), C.c_uint32(stream), C.c_uint64(frame0), C.c_long(n_frames), C.c_int(length),
                                           C.c_uint32(domain), _p(g))
        return g

    def philox_taps(self, seed, frame0, n_frames, n_taps):
        t = np.zeros((n_frames, n_taps, 2), np.float32)
        self.lib.orc_philox_taps(C.c_uint32(seed), C.c_uint64(frame0), C.c_long(n_frames), C.c_int(n_taps), _p(t))
        return t

    def tx_frames(self, bits, n_sym):
        bits = np.ascontiguousarray(bits, dtype=np.uint8).reshape(-1, 96 * n_sym)
        out = np.zeros((bits.shape[0], self.frame_len(n_sym), 2), np.float32)
        for i in range(bits.shape[0]):
            self.lib.orc_tx_frame(_p(bits[i], C.c_uint8), C.c_int(n_sym), _p(out[i]))
        return out

    def awgn_channel(self, tx, g0, g1, snr_db, noise, snr_def):
        frames = _f32(tx).reshape(-1, np.shape(tx)[-2], 2)
        n, length = frames.shape[:2]
        g0 = _f32(g0).reshape(n, length)
        g1 = None if g1 is None else _f32(g1).reshape(n, length)
        out = np.zeros_like(frames)
        for i in range(n):
            self.lib.orc_awgn_channel(_p(frames[i]), _p(g0[i]), None if g1 is None else _p(g1[i]), _p(out[i]), C.c_float(snr_db),
                                      C.c_int(NOISE[noise]), C.c_int(SNR_DEF[snr_def]), C.c_int(length))
        return out

    def chain_channel(self, bits, g0, g1, taps, n_sym, snr_db, noise, snr_def, per_frame=False):
        bits = np.ascontiguousarray(bits, dtype=np.uint8).reshape(-1, 96 * n_sym)
        n = bits.shape[0]
        g0 = _f32(g0).reshape(n, self.frame_len(n_sym))
        g1 = None if g1 is None else _f32(g1).reshape(n, self.frame_len(n_sym))
        n_taps = 0 if taps is None else taps.shape[1]
        taps = None if taps is None else _f32(taps)
        acc = Counters()
        fe = np.zeros(n, np.int32) if per_frame else None
        fv = np.zeros(n, np.float32) if per_frame else None
        self.lib.orc_chain_channel(_p(bits, C.c_uint8), _p(g0), _p(g1), _p(taps), C.c_int(n_taps), C.c_long(n), C.c_int(n_sym),
                                   C.c_float(snr_db), C.c_int(NOISE[noise]), C.c_int(SNR_DEF[snr_def]), C.byref(acc),
                                   _p(fe, C.c_int), _p(fv))
        return (acc, fe, fv) if per_frame else acc

    def mc_sweep(self, seed, frame0, n_frames, n_sym, snr_db, noise, snr_def, n_taps=0, streams=None, per_frame=False):
        """what ofdm_mc_sweep_channel_dev computes in EXACT mode, point by point: list of Counters (or (Counters, fe, fv))"""
        bits = self.philox_bits(seed, frame0, n_frames, n_sym)
        taps = self.philox_taps(seed, frame0, n_frames, n_taps) if n_taps > 0 else None
        out = []
        for i, s in enumerate(snr_db):
            stream = i if streams is None else int(streams[i])
            L = self.frame_len(n_sym)
            g0 = self.philox_normals(seed, stream, frame0, n_frames, L, DOMAIN_NOISE)
            g1 = self.philox_normals(seed, stream, frame0, n_frames, L, DOMAIN_NOISE_Q) if noise == "complex" else None
            out.append(self.chain_channel(bits, g0, g1, taps, n_sym, float(s), noise, snr_def, per_frame))
        return out


def model_complex_esn0(snr_db, n_frames, n_sym, rng):
    """Independent float64 model of the complex / Es/N0 AWGN channel at the receiver's data bins, written from the definitions
    alone: a data bin carries X (|X| = 1) plus CN(0, 64 np) noise, np = 1 / (64 Es/N0); the LTS estimate is the average of two
    halves, so H = 1 + CN(0, 32 np) per data bin; the rails are decided on F conj(H), bits through the non-Gray map
    (I error 1 bit, Q error 2, both 1).  Returns per-frame bit errors [n_frames] (errors within a frame are correlated by H)."""
    esn0 = 10.0 ** (snr_db / 10.0)
    var_f = 1.0 / esn0                                     # 64 np
    var_h = 0.5 / esn0                                     # 32 np

    def cn(var, shape):
        return np.sqrt(var / 2.0) * (rng.standard_normal(shape) + 1j * rng.standard_normal(shape))

    x = ((rng.integers(0, 2, (n_frames, n_sym, 48)) * 2 - 1) + 1j * (rng.integers(0, 2, (n_frames, n_sym, 48)) * 2 - 1)) / np.sqrt(2.0)
    H = 1.0 + cn(var_h, (n_frames, 1, 48))
    F = x + cn(var_f, x.shape)
    d = F * np.conj(H)
    ei = np.sign(d.real) != np.sign(x.real)
    eq = np.sign(d.imag) != np.sign(x.imag)
    bits = np.where(ei & eq, 1, np.where(ei, 1, 0) + np.where(eq, 2, 0))
    return bits.reshape(n_frames, -1).sum(axis=1)
