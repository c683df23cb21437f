"""ctypes front-end of tests/coded_oracle.c (TEST INFRASTRUCTURE ONLY): the coded link of ofdm_code on the CPU, plus independent
numpy models written from the 802.11a definitions alone (shift-register encoder, float64 Viterbi) to check the oracle against.

The library is compiled once per process into a temporary directory with the pinned oracle's flags, so running the tests writes
nothing into the tree."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from channel_oracle import ChannelOracle, Counters, NOISE, SNR_DEF, _p, _f32

HERE = os.path.dirname(os.path.abspath(__file__))
RATE = {"1/2": 1, "3/4": 2}
DECISION = {"soft": 0, "hard": 1}
DBPS = {"1/2": 48, "3/4": 72}


def k_info(rate, n_sym):
    return n_sym * DBPS[rate] - 6


class CodedOracle(ChannelOracle):
    """ChannelOracle (same Philox streams, transmitter, channels) with the coded link on top"""

    def __init__(self):
        self._dir = tempfile.mkdtemp(prefix="ofdm_coded_oracle_")
        so = os.path.join(self._dir, "libcoded_oracle.so")
        subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-w",
                               "-o", so, os.path.join(HERE, "coded_oracle.c"), "-lm"])
        self.lib = C.CDLL(so)
        self.lib.orc_init()

    def interleave(self, k):
        return int(self.lib.orc_interleave(C.c_int(k)))

    def qpsk_mod(self, bits, n_sym):
        bits = np.ascontiguousarray(bits, dtype=np.uint8)
        out = np.zeros((n_sym * 48, 2), np.float32)
        self.lib.orc_qpsk_mod(_p(bits, C.c_uint8), C.c_int(n_sym), _p(out))
        return out

    def conv_encode(self, info, n_sym, rate):
        """info bits [n_frames, >= K_info] (one byte per bit) -> payload bits [n_frames, 96 n_sym]"""
        info = np.ascontiguousarray(info, dtype=np.uint8).reshape(-1, np.shape(info)[-1])
        out = np.zeros((info.shape[0], 96 * n_sym), np.uint8)
        for i in range(info.shape[0]):
            self.lib.orc_conv_encode(C.c_int(RATE[rate]), _p(info[i], C.c_uint8), C.c_int(n_sym), _p(out[i], C.c_uint8))
        return out

    def viterbi(self, H, eq, n_sym, rate, decision):
        """H [n, 64, 2], eq [n, 48 n_sym, 2] -> decoded information bits [n, K_info]"""
        H = _f32(H).reshape(-1, 64, 2)
        eq = _f32(eq).reshape(H.shape[0], 48 * n_sym, 2)
        out = np.zeros((H.shape[0], k_info(rate, n_sym)), np.uint8)
        for i in range(H.shape[0]):
            self.lib.orc_viterbi(C.c_int(RATE[rate]), C.c_int(DECISION[decision]), _p(H[i]), _p(eq[i]), C.c_int(n_sym), _p(out[i], C.c_uint8))
        return out

    def coded_chain(self, info, g0, g1, taps, n_sym, snr_db, noise, snr_def, rate, decision):
        """(coded Counters, raw Counters) of the whole coded chain over the frames, on the given draws and taps"""
        info = np.ascontiguousarray(info, dtype=np.uint8).reshape(-1, 96 * n_sym)
        n = info.shape[0]
        g0 = _f32(g0).reshape(n, self.frame_len(n_sym))
        g1 = None if g1 is None else _f32(g1).reshape(n, self.frame_len(n_sym))
        n_taps = 0 if taps is None else taps.shape[1]
        taps = None if taps is None else _f32(taps)
        coded, raw = Counters(), Counters()
        self.lib.orc_coded_chain(C.c_int(RATE[rate]), C.c_int(DECISION[decision]), _p(info, C.c_uint8), _p(g0), _p(g1), _p(taps),
                                 C.c_int(n_taps), C.c_long(n), C.c_int(n_sym), C.c_float(snr_db), C.c_int(NOISE[noise]),
                                 C.c_int(SNR_DEF[snr_def]), C.byref(coded), C.byref(raw))
        return coded, raw


# ---- independent numpy models (from the standard's text, not from the oracle)
G0, G1 = (1, 0, 1, 1, 0, 1, 1), (1, 1, 1, 1, 0, 0, 1)          # 133, 171 octal: taps on x[n], x[n-1], ..., x[n-6]


def np_encode(info, rate, n_sym):
    """coded bits [n_frames, 96 n_sym] of information bits [n_frames, >= K_info], before the interleaver"""
    info = np.asarray(info, dtype=np.int64)
    T, K = n_sym * DBPS[rate], k_info(rate, n_sym)
    x = np.zeros((info.shape[0], T + 6), np.int64)          # 6 leading zeros: the encoder starts in state 0
    x[:, 6:6 + K] = info[:, :K]
    a = sum(G0[d] * x[:, 6 - d:6 - d + T] for d in range(7)) % 2
    b = sum(G1[d] * x[:, 6 - d:6 - d + T] for d in range(7)) % 2
    ab = np.stack([a, b], axis=-1).reshape(info.shape[0], 2 * T)
    if rate == "1/2":
        return ab.astype(np.uint8)
    keep = np.tile(np.array([1, 1, 1, 0, 0, 1], bool), T // 3)     # A0 B0 A1 (B1) (A2) B2
    return ab[:, keep].astype(np.uint8)


def _branch_outputs():
    """outputs (A, B) of the transition from state s (the last 6 inputs, x[n-1] in bit 5 .. x[n-6] in bit 0) with input u"""
    a = np.zeros((64, 2), np.int64)
    b = np.zeros((64, 2), np.int64)
    for s in range(64):
        for u in range(2):
            hist = [u] + [(s >> (5 - d)) & 1 for d in range(6)]     # x[n], x[n-1] .. x[n-6]
            a[s, u] = sum(g * h for g, h in zip(G0, hist)) % 2
            b[s, u] = sum(g * h for g, h in zip(G1, hist)) % 2
    return a, b


def np_viterbi(La, Lb):
    """float64 maximum-likelihood paths through the tail-terminated trellis (start and end in state 0), vectorised over frames:
    La, Lb [n, T] branch inputs -> (input bits [n, T], best correlations [n])."""
    La, Lb = np.atleast_2d(np.asarray(La, np.float64)), np.atleast_2d(np.asarray(Lb, np.float64))
    n, T = La.shape
    out_a, out_b = _branch_outputs()
    t = np.arange(64)
    u = t >> 5
    preds = np.stack([((t << 1) & 63), ((t << 1) & 63) | 1])         # the two states whose successor with input u is t
    sa = 2 * out_a[preds, u] - 1                                      # [2, 64]
    sb = 2 * out_b[preds, u] - 1
    M = np.full((n, 64), -np.inf)
    M[:, 0] = 0.0
    choice = np.zeros((T, n, 64), np.int8)
    for k in range(T):
        cand = M[:, preds] + La[:, k, None, None] * sa + Lb[:, k, None, None] * sb     # [n, 2, 64]
        c = np.argmax(cand, axis=1)
        choice[k] = c
        M = np.take_along_axis(cand, c[:, None, :], axis=1)[:, 0, :]
    bits = np.zeros((n, T), np.int64)
    s = np.zeros(n, np.int64)
    rows = np.arange(n)
    for k in range(T - 1, -1, -1):
        bits[:, k] = s >> 5
        s = preds[choice[k, rows, s], s]
    return bits, M[:, 0]


def np_inputs(H, eq, n_sym, rate, decision):
    """float64 depunctured branch inputs (La, Lb) [n, T] from H [n, 64, 2] (centred) and eq [n, 48 n_sym, 2], from the definitions:
    data point d sits on the d-th data subcarrier (-26 .. 26 without 0 and the pilots), coded bit k of a symbol at interleaver
    position 6 (k mod 16) + k // 16 (I rail if even, Q if odd); stolen bits are 0"""
    H = np.asarray(H, np.float64).reshape(-1, 64, 2)
    eq = np.asarray(eq, np.float64).reshape(H.shape[0], n_sym, 48, 2)
    sub = [k for k in range(-26, 27) if k not in (0, -21, -7, 7, 21)]
    centred = np.array([k + 32 for k in sub])
    w = (H[:, centred, 0] ** 2 + H[:, centred, 1] ** 2)[:, None, :]                       # [n, 1, 48]
    with np.errstate(invalid="ignore", over="ignore"):
        if decision == "hard":
            L = np.where(eq > 0, 1.0, -1.0)
        else:
            L = w[..., None] * eq
        L = np.where(np.isfinite(L), L, 0.0)
    pos = L.reshape(H.shape[0], n_sym, 96)                                                  # position i = 2 d + rail
    k = np.arange(96)
    coded = pos[:, :, 6 * (k % 16) + k // 16].reshape(H.shape[0], -1)
    T = n_sym * DBPS[rate]
    if rate == "1/2":
        return coded[:, 0::2], coded[:, 1::2]
    full = np.zeros((H.shape[0], 2 * T))
    full[:, np.tile(np.array([1, 1, 1, 0, 0, 1], bool), T // 3)] = coded
    return full[:, 0::2], full[:, 1::2]


def correlation(coded, La, Lb, rate):
    """float64 sum L (2c - 1) of a coded (punctured) bit sequence against the depunctured inputs"""
    T = len(La)
    coded = np.asarray(coded, np.int64)
    if rate == "1/2":
        a, b = coded[0::2], coded[1::2]
    else:
        full = np.zeros(2 * T, np.int64)
        keep = np.tile(np.array([1, 1, 1, 0, 0, 1], bool), T // 3)
        full[keep] = coded
        a, b = full[0::2], full[1::2]
        a = np.where(np.tile([1, 1, 0], T // 3) == 1, a, 0)
        b = np.where(np.tile([1, 0, 1], T // 3) == 1, b, 0)
    La, Lb = np.asarray(La, np.float64), np.asarray(Lb, np.float64)
    return float(np.sum(La * (2 * a - 1)) + np.sum(Lb * (2 * b - 1)))
