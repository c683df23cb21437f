"""ctypes front-end of tests/ota_oracle.c (TEST INFRASTRUCTURE ONLY): the C driver's default over-the-air path on the CPU, plus
the driver's own bookkeeping restated in Python (message codec, buffer lengths, capture starts from the C library's rand()).

The library is compiled once per process into a temporary directory with the pinned oracle's flags, so running the tests
writes nothing into the tree."""
import ctypes as C
import math
import os
import subprocess
import tempfile

import numpy as np

from channel_oracle import ChannelOracle, _f32, _p

HERE = os.path.dirname(os.path.abspath(__file__))
DOMAIN_FLAT = 3


class RxStats(C.Structure):
    """orc_rx_stats"""
    _fields_ = [("evm_lin", C.c_float), ("evm_db", C.c_float), ("evm_agc_lin", C.c_float),
                ("evm_agc_db", C.c_float), ("ber", C.c_float), ("bit_errors", C.c_int), ("rail_errors", C.c_int)]


class OtaOracle(ChannelOracle):
    """ChannelOracle (same Philox streams and oracle stages) with the flat noise layout and the driver's whole path"""

    def __init__(self):
        self._dir = tempfile.mkdtemp(prefix="ofdm_ota_oracle_")
        so = os.path.join(self._dir, "libota_oracle.so")
        subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-w",
                               "-o", so, os.path.join(HERE, "ota_oracle.c"), "-lm"])
        self.lib = C.CDLL(so)
        self.lib.orc_init()
        self.lib.orc_cfo_freq.restype = C.c_float

    def philox_normals_flat(self, seed, stream, frame0, n_frames, length, domain=DOMAIN_FLAT):
        g = np.zeros((n_frames, length), np.float32)
        self.lib.orc_philox_normals_flat(C.c_uint32(seed), C.c_uint32(stream), C.c_uint64(frame0), C.c_long(n_frames), C.c_int(length),
                                         C.c_uint32(domain), _p(g))
        return g

    def noise_slot(self, n):
        blk, j = C.c_int(0), C.c_int(0)
        self.lib.orc_noise_slot(C.c_int(n), C.byref(blk), C.byref(j))
        return blk.value, j.value

    def cfo_freq(self, rx, fine):
        return float(self.lib.orc_cfo_freq(_p(_f32(rx)), C.c_int(int(fine))))

    def waveform(self, bits, n_sym):
        """(STS || LTS || data [len480], after x2 + RRC [len_shaped], tiled 10x [len_rep]) of one message, as the driver builds them"""
        length, len480, len_shaped, len_rep, _ = lengths(n_sym)
        sts = np.zeros((160, 2), np.float32)
        self.lib.orc_sts_time(_p(sts))
        full = np.ascontiguousarray(np.concatenate([sts, self.tx_frames(bits, n_sym)[0]]))
        shaped = np.zeros((len_shaped, 2), np.float32)
        self.lib.orc_rrc_tx(_p(full), C.c_int(len480), _p(shaped))
        return full, shaped, np.tile(shaped, (10, 1))

    def ota_point(self, rep, g, snr_db, rx_start, len_cap, bits, n_sym):
        """(selected index or -1 where the matched filter would leave the capture, RxStats) of one point of the driver's path"""
        rep, g = _f32(rep), _f32(g)
        bits = np.ascontiguousarray(bits, dtype=np.uint8)
        st = RxStats()
        idx = self.lib.orc_ota_point(_p(rep), C.c_int(rep.shape[0]), _p(g), C.c_float(snr_db), C.c_int(rx_start), C.c_int(len_cap),
                                     _p(bits, C.c_uint8), C.c_int(n_sym), C.byref(st))
        return int(idx), st


# ---- the driver's bookkeeping (host/ofdm_main.c)
def encode_message(msg):
    """encode_message: 8 bits per character, MSB first, padded with spaces to whole 96-bit symbols -> (bits [96 n_sym], n_sym)"""
    raw = msg.encode("latin-1")
    n_sym = max(1, math.ceil(8 * len(raw) / 96.0))
    padded = raw + b" " * (12 * n_sym - len(raw))
    return np.unpackbits(np.frombuffer(padded, np.uint8)), n_sym


def lengths(n_sym):
    """(len, len480, len_shaped, len_rep, len_cap) of the driver's whole path for n_sym-symbol frames"""
    length = 160 + 80 * n_sym
    len480 = 160 + length
    len_shaped = 2 * len480 + 20
    len_rep = 10 * len_shaped
    return length, len480, len_shaped, len_rep, int(len_rep * 0.307)


def capture_starts(seed, n, len_rep, len_cap):
    """srand(seed), then rand() % (len_rep - len_cap) once per SNR point, through the C library the driver links"""
    libc = C.CDLL(None)
    libc.srand(C.c_uint(seed))
    return [libc.rand() % (len_rep - len_cap) for _ in range(n)]
