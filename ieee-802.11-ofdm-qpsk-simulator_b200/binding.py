"""ctypes binding of libofdm_b200.so (the C-ABI declared in include/ofdm_b200.h).

This is plumbing only: torch supplies device memory and the stream, every computation happens in
the hand-written sm_100a kernels behind the C-ABI.  There is no CPU or PyTorch fallback: if the
shared library is missing, or there is no CUDA device, construction fails loudly.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libofdm_b200.so")

MODE_EXACT, MODE_FAST = 0, 1
NFFT, CP, SYM_LEN, LTS_LEN, DATA_PER_SYM, BITS_PER_SYM, WORDS_PER_SYM = 64, 16, 80, 160, 48, 96, 3


def frame_len(n_sym):
    return LTS_LEN + SYM_LEN * n_sym


class Counters(C.Structure):
    """ofdm_counters"""
    _fields_ = [("bit_errors", C.c_uint64), ("bits", C.c_uint64), ("frames_in_error", C.c_uint64),
                ("rail_errors", C.c_uint64), ("frames", C.c_uint64),
                ("sum_err2", C.c_double), ("sum_ref2", C.c_double), ("sum_evm_lin", C.c_double)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}

    def __iadd__(self, o):
        for k, _ in self._fields_:
            setattr(self, k, getattr(self, k) + getattr(o, k))
        return self


COUNTER_FIELDS = [k for k, _ in Counters._fields_]
COUNTERS_BYTES = C.sizeof(Counters)


class RxDump(C.Structure):
    """ofdm_rx_dump"""
    _fields_ = [("H", C.c_void_p), ("eq", C.c_void_p), ("sliced", C.c_void_p), ("bits", C.c_void_p),
                ("frame_bit_errors", C.c_void_p), ("frame_evm_lin", C.c_void_p)]


class Channel(C.Structure):
    """ofdm_channel"""
    _fields_ = [("noise", C.c_int), ("snr_def", C.c_int), ("n_taps", C.c_int)]


# ofdm_channel's enums under the names the Python methods take; ("real", "frame_power") is the reference's channel
NOISE = {"real": 0, "complex": 1}
SNR_DEF = {"frame_power": 0, "esn0": 1, "ebn0": 2}


def channel(noise="real", snr_def="frame_power", n_taps=0):
    """Channel from names: noise "real" | "complex", snr_def "frame_power" | "esn0" | "ebn0" (include/ofdm_b200.h)."""
    if noise not in NOISE:
        raise ValueError("noise must be one of %s, not %r" % (sorted(NOISE), noise))
    if snr_def not in SNR_DEF:
        raise ValueError("snr_def must be one of %s, not %r" % (sorted(SNR_DEF), snr_def))
    return Channel(NOISE[noise], SNR_DEF[snr_def], int(n_taps))


class Code(C.Structure):
    """ofdm_code"""
    _fields_ = [("rate", C.c_int), ("decision", C.c_int)]


# ofdm_code's enums under the names the Python methods take (DESIGN.md section 6.2)
CODE = {"1/2": 1, "3/4": 2}
DECISION = {"soft": 0, "hard": 1}
DATA_BITS_PER_SYM = {"1/2": 48, "3/4": 72}


def code(rate="1/2", decision="soft"):
    """Code from names: rate "1/2" | "3/4", decision "soft" | "hard" (include/ofdm_b200.h)."""
    if rate not in CODE:
        raise ValueError("rate must be one of %s, not %r" % (sorted(CODE), rate))
    if decision not in DECISION:
        raise ValueError("decision must be one of %s, not %r" % (sorted(DECISION), decision))
    return Code(CODE[rate], DECISION[decision])


def info_bits(rate, n_sym):
    """K_info: the information bits of a coded frame of n_sym OFDM symbols (the last 6 of n_sym * N_DBPS are the tail)."""
    return n_sym * DATA_BITS_PER_SYM[rate] - 6


class OfdmError(RuntimeError):
    pass


_VP, _I, _L, _F, _U32, _U64, _SZ = C.c_void_p, C.c_int, C.c_long, C.c_float, C.c_uint32, C.c_uint64, C.c_size_t

# name -> (restype, argtypes); must list every symbol include/ofdm_b200.h declares
SIGNATURES = {
    "ofdm_version": (_I, []),
    "ofdm_strerror": (C.c_char_p, [_I]),
    "ofdm_ctx_create": (_I, [C.POINTER(_VP), _I]),
    "ofdm_ctx_destroy": (_I, [_VP]),
    "ofdm_last_error": (C.c_char_p, [_VP]),
    "ofdm_ctx_set_stream": (_I, [_VP, _VP]),
    "ofdm_ctx_stream": (_VP, [_VP]),
    "ofdm_ctx_sync": (_I, [_VP]),
    "ofdm_ctx_set_option": (_I, [_VP, C.c_char_p, _I]),
    "ofdm_ctx_replayed_frames": (_I, [_VP, C.POINTER(_U64), _I]),
    "ofdm_ctx_sm_count": (_I, [_VP]),
    "ofdm_ctx_launch_count": (_U64, [_VP]),
    "ofdm_dev_alloc": (_I, [_VP, C.POINTER(_VP), _SZ]),
    "ofdm_dev_free": (_I, [_VP, _VP]),
    "ofdm_host_alloc": (_I, [_VP, C.POINTER(_VP), _SZ]),
    "ofdm_host_free": (_I, [_VP, _VP]),
    "ofdm_memcpy_h2d": (_I, [_VP, _VP, _VP, _SZ]),
    "ofdm_memcpy_d2h": (_I, [_VP, _VP, _VP, _SZ]),
    "ofdm_memset_dev": (_I, [_VP, _VP, _I, _SZ]),
    "ofdm_pack_bits": (_I, [_VP, _VP, _VP, _L]),
    "ofdm_unpack_bits": (_I, [_VP, _VP, _VP, _L]),
    "ofdm_qpsk_modulate": (_I, [_VP, _VP, _VP, _L]),
    "ofdm_map_subcarriers": (_I, [_VP, _VP, _VP, _L]),
    "ofdm_ifft64": (_I, [_VP, _VP, _VP, _L, _I]),
    "ofdm_fft64": (_I, [_VP, _VP, _VP, _L, _I]),
    "ofdm_add_cp": (_I, [_VP, _VP, _VP, _L]),
    "ofdm_lts": (_I, [_VP, _VP, _VP]),
    "ofdm_tx_frames": (_I, [_VP, _VP, _VP, _VP, _L, _I, _I]),
    "ofdm_frame_power": (_I, [_VP, _VP, _VP, _L, _I, _I]),
    "ofdm_awgn_inject": (_I, [_VP, _VP, _VP, _VP, _F, _VP, _L, _I, _I]),
    "ofdm_awgn_philox": (_I, [_VP, _VP, _VP, _F, _U32, _U32, _U64, _VP, _L, _I, _I]),
    "ofdm_awgn_philox_ex": (_I, [_VP, _I, _I, _VP, _VP, _F, _U32, _U32, _U64, _VP, _L, _I, _I]),
    "ofdm_rx_frames": (_I, [_VP, _VP, _VP, _L, _I, _I, _VP, C.POINTER(RxDump)]),
    "ofdm_awgn_rx_inject": (_I, [_VP, _VP, _VP, _VP, _VP, _F, _L, _I, _I, _VP, C.POINTER(RxDump)]),
    "ofdm_awgn_rx_philox": (_I, [_VP, _VP, _VP, _VP, _F, _U32, _U32, _U64, _L, _I, _I, _VP, C.POINTER(RxDump)]),
    "ofdm_awgn_rx_inject_sweep": (_I, [_VP, _VP, _VP, _VP, _VP, _VP, _I, _L, _I, _I, _VP]),
    "ofdm_strip_cp": (_I, [_VP, _VP, _VP, _L, _I, _I, _I]),
    "ofdm_channel_estimate": (_I, [_VP, _VP, _VP, _L, _I, _I, _I]),
    "ofdm_equalize": (_I, [_VP, _VP, _VP, _VP, _L, _I, _I]),
    "ofdm_demap": (_I, [_VP, _VP, _VP, _L]),
    "ofdm_agc_slicer": (_I, [_VP, _VP, _VP, _L]),
    "ofdm_qpsk_demodulate": (_I, [_VP, _VP, _VP, _L]),
    "ofdm_sweep_inject_host": (_I, [_VP, _VP, _VP, _L, _I, _VP, _I, _I, C.POINTER(Counters)]),
    "ofdm_sweep_inject_dev": (_I, [_VP, _VP, _VP, _L, _I, _VP, _I, _I, C.POINTER(Counters)]),
    "ofdm_random_bits": (_I, [_VP, _U32, _U64, _L, _I, _VP]),
    "ofdm_mc_sweep_philox_dev": (_I, [_VP, _U32, _U64, _L, _I, _VP, _I, _I, _VP]),
    "ofdm_mc_sweep_points_dev": (_I, [_VP, _U32, _U64, _L, _I, _I, _VP, _VP, _I, _I, _VP]),
    "ofdm_mc_sweep_until": (_I, [_VP, _U32, _U64, _I, _I, _VP, _I, _I, _U64, _U64, _L, C.POINTER(Counters), C.POINTER(_I)]),
    "ofdm_mc_sweep_channel_dev": (_I, [_VP, C.POINTER(Channel), _U32, _U64, _L, _I, _VP, _VP, _I, _I, _VP]),
    "ofdm_mc_sweep_channel_until": (_I, [_VP, C.POINTER(Channel), _U32, _U64, _I, _VP, _I, _I, _U64, _U64, _L, C.POINTER(Counters),
                                         C.POINTER(_I)]),
    "ofdm_mc_sweep_philox": (_I, [_VP, _U32, _U64, _L, _I, _VP, _I, _I, C.POINTER(Counters)]),
    "ofdm_conv_encode": (_I, [_VP, _I, _VP, _VP, _L, _I]),
    "ofdm_viterbi_decode": (_I, [_VP, C.POINTER(Code), _VP, _VP, _VP, _VP, _L, _I, _VP]),
    "ofdm_mc_sweep_coded_dev": (_I, [_VP, C.POINTER(Channel), C.POINTER(Code), _U32, _U64, _L, _I, _VP, _VP, _I, _I, _VP, _VP]),
    "ofdm_mc_sweep_coded_until": (_I, [_VP, C.POINTER(Channel), C.POINTER(Code), _U32, _U64, _I, _VP, _I, _I, _U64, _U64, _L,
                                       C.POINTER(Counters), C.POINTER(Counters), C.POINTER(_I)]),
    "ofdm_multipath_taps": (_I, [_VP, _VP, _VP, _I, _VP, _L, _I]),
    "ofdm_multipath_philox": (_I, [_VP, _VP, _U32, _U64, _I, _VP, _VP, _L, _I]),
    "ofdm_mc_sweep_multipath_dev": (_I, [_VP, _U32, _U64, _L, _I, _I, _VP, _I, _I, _VP]),
    "ofdm_rrc_tx": (_I, [_VP, _VP, _VP, _L, _I]),
    "ofdm_rrc_rx": (_I, [_VP, _VP, _VP, _L, _I, _I, _I]),
    "ofdm_awgn_inject_len": (_I, [_VP, _VP, _VP, _VP, _F, _VP, _L, _I, _I]),
    "ofdm_packet_detect": (_I, [_VP, _VP, _VP, _L, _I]),
    "ofdm_packet_select": (_I, [_VP, _VP, _VP, _L, _I]),
    "ofdm_sts": (_I, [_VP, _VP]),
    "ofdm_prepend_sts": (_I, [_VP, _VP, _VP, _L, _I]),
    "ofdm_gather": (_I, [_VP, _VP, _VP, _I, _VP, _L, _I, _I]),
    "ofdm_rrc_rx_idx": (_I, [_VP, _VP, _VP, _VP, _L, _I, _I]),
    "ofdm_cfo_coarse": (_I, [_VP, _VP, _VP, _VP, _L, _I]),
    "ofdm_cfo_fine": (_I, [_VP, _VP, _VP, _VP, _L, _I]),
    "ofdm_awgn_philox_len": (_I, [_VP, _VP, _VP, _F, _U32, _U32, _U64, _VP, _L, _I, _I]),
    "ofdm_counters_pack": (_I, [_VP, _VP, _I, _VP, _VP]),
    "ofdm_counters_unpack": (_I, [_VP, _VP, _I, _VP, _VP]),
    "ofdm_counters_finalize": (_I, [C.POINTER(Counters), C.POINTER(_F)]),
    "ofdm_write_float_array_to_file": (_I, [_VP, _I, C.c_char_p]),
    "ofdm_write_complex_array_to_file": (_I, [_VP, _I, C.c_char_p, _I]),
}


def load_library(path=None):
    """dlopen the C-ABI library and attach the prototypes.  Raises if the library is not built.
    OFDM_B200_LIB overrides the path (A/B runs of two builds on the same box)."""
    path = path or os.environ.get("OFDM_B200_LIB") or LIB_PATH
    if not os.path.exists(path):
        raise OfdmError("%s is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(there is no CPU fallback)" % path)
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here == header/library mismatch
        fn.restype, fn.argtypes = res, args
    return lib


def _ptr(t):
    if t is None:
        return None
    return t.data_ptr()


class Ofdm:
    """One context on one GPU.  Device buffers are torch CUDA tensors (contiguous); every method
    forwards to the C-ABI entry point of the same name."""

    def __init__(self, device=0, lib=None):
        import torch
        self.torch = torch
        self.lib = lib or load_library()
        if not torch.cuda.is_available():
            raise OfdmError("no CUDA device visible: libofdm_b200 has no CPU fallback")
        self.device = torch.device("cuda", device)
        h = _VP()
        self._check(self.lib.ofdm_ctx_create(C.byref(h), device), None)
        self.h = h
        # order this context's work on torch's current stream of that device
        self.use_stream(torch.cuda.current_stream(self.device))

    # ---- plumbing
    def _check(self, status, h="self"):
        if status != 0:
            msg = self.lib.ofdm_strerror(status).decode()
            if h == "self" and getattr(self, "h", None):
                msg += ": " + self.lib.ofdm_last_error(self.h).decode()
            raise OfdmError(msg)

    def use_stream(self, stream):
        self._check(self.lib.ofdm_ctx_set_stream(self.h, _VP(stream.cuda_stream)))

    def set_option(self, name, value):
        self._check(self.lib.ofdm_ctx_set_option(self.h, name.encode(), int(value)))

    def replayed_frames(self, reset=False):
        """frames the speculating EXACT kernels replayed in the reference's arithmetic (process-wide counter)"""
        v = _U64(0)
        self._check(self.lib.ofdm_ctx_replayed_frames(self.h, C.byref(v), int(bool(reset))))
        return int(v.value)

    def sync(self):
        self._check(self.lib.ofdm_ctx_sync(self.h))

    def close(self):
        if getattr(self, "h", None):
            self.lib.ofdm_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def sm_count(self):
        return self.lib.ofdm_ctx_sm_count(self.h)

    @property
    def launch_count(self):
        return int(self.lib.ofdm_ctx_launch_count(self.h))

    def empty(self, shape, dtype):
        return self.torch.empty(shape, dtype=dtype, device=self.device)

    def zeros(self, shape, dtype):
        return self.torch.zeros(shape, dtype=dtype, device=self.device)

    def to_dev(self, a):
        return self.torch.from_numpy(np.ascontiguousarray(a)).to(self.device)

    def new_counters(self, n=1):
        return self.zeros((n, COUNTERS_BYTES // 8), self.torch.int64)

    def read_counters(self, t):
        raw = t.cpu().numpy()
        out = []
        for row in raw:
            c = Counters.from_buffer_copy(row.tobytes())
            out.append(c)
        return out

    def _dump(self, n_frames, n_sym, want):
        t = self.torch
        bufs, d = {}, RxDump()
        spec = {"H": ((n_frames, 64, 2), t.float32), "eq": ((n_frames, n_sym * 48, 2), t.float32),
                "sliced": ((n_frames, n_sym * 48, 2), t.float32), "bits": ((n_frames, n_sym * 3), t.int32),
                "frame_bit_errors": ((n_frames,), t.int32), "frame_evm_lin": ((n_frames,), t.float32)}
        for k in want:
            shape, dt = spec[k]
            bufs[k] = self.zeros(shape, dt)
            setattr(d, k, bufs[k].data_ptr())
        return d, bufs

    # ---- stage-level
    def pack_bits(self, bits_u8):
        n_symbols = bits_u8.numel() // 96
        out = self.empty((n_symbols * 3,), self.torch.int32)
        self._check(self.lib.ofdm_pack_bits(self.h, _ptr(bits_u8), _ptr(out), n_symbols))
        return out

    def unpack_bits(self, packed):
        n_symbols = packed.numel() // 3
        out = self.empty((n_symbols * 96,), self.torch.uint8)
        self._check(self.lib.ofdm_unpack_bits(self.h, _ptr(packed), _ptr(out), n_symbols))
        return out

    def qpsk_modulate(self, packed):
        n_symbols = packed.numel() // 3
        out = self.empty((n_symbols, 48, 2), self.torch.float32)
        self._check(self.lib.ofdm_qpsk_modulate(self.h, _ptr(packed), _ptr(out), n_symbols))
        return out

    def map_subcarriers(self, mod):
        n_symbols = mod.numel() // 96
        out = self.empty((n_symbols, 64, 2), self.torch.float32)
        self._check(self.lib.ofdm_map_subcarriers(self.h, _ptr(mod), _ptr(out), n_symbols))
        return out

    def ifft64(self, x, mode):
        n = x.numel() // 128
        out = self.empty((n, 64, 2), self.torch.float32)
        self._check(self.lib.ofdm_ifft64(self.h, _ptr(x), _ptr(out), n, mode))
        return out

    def fft64(self, x, mode):
        n = x.numel() // 128
        out = self.empty((n, 64, 2), self.torch.float32)
        self._check(self.lib.ofdm_fft64(self.h, _ptr(x), _ptr(out), n, mode))
        return out

    def add_cp(self, sym):
        n = sym.numel() // 128
        out = self.empty((n, 80, 2), self.torch.float32)
        self._check(self.lib.ofdm_add_cp(self.h, _ptr(sym), _ptr(out), n))
        return out

    def lts(self):
        f = np.zeros((64, 2), np.float32)
        t = np.zeros((160, 2), np.float32)
        self._check(self.lib.ofdm_lts(self.h, f.ctypes.data, t.ctypes.data))
        return f, t

    def tx_frames(self, packed, n_sym, mode, with_power=True):
        n_frames = packed.numel() // (3 * n_sym)
        frames = self.empty((n_frames, frame_len(n_sym), 2), self.torch.float32)
        power = self.empty((n_frames,), self.torch.float32) if with_power else None
        self._check(self.lib.ofdm_tx_frames(self.h, _ptr(packed), _ptr(frames), _ptr(power), n_frames, n_sym, mode))
        return (frames, power) if with_power else frames

    def frame_power(self, frames, mode):
        n_frames, length = frames.shape[0], frames.shape[1]
        power = self.empty((n_frames,), self.torch.float32)
        self._check(self.lib.ofdm_frame_power(self.h, _ptr(frames), _ptr(power), n_frames, length, mode))
        return power

    def awgn_inject(self, tx, g, snr_db, n_sym, mode, power=None):
        n_frames = tx.shape[0]
        ota = self.empty(tuple(tx.shape), self.torch.float32)
        self._check(self.lib.ofdm_awgn_inject(self.h, _ptr(tx), _ptr(g), _ptr(power), snr_db, _ptr(ota), n_frames, n_sym, mode))
        return ota

    def awgn_philox(self, tx, snr_db, seed, stream, frame0, n_sym, mode, power=None):
        n_frames = tx.shape[0]
        ota = self.empty(tuple(tx.shape), self.torch.float32)
        self._check(self.lib.ofdm_awgn_philox(self.h, _ptr(tx), _ptr(power), snr_db, seed, stream, frame0, _ptr(ota),
                                              n_frames, n_sym, mode))
        return ota

    def awgn_philox_ex(self, tx, snr_db, seed, stream, frame0, n_sym, mode, noise="real", snr_def="frame_power", power=None):
        """the channel (noise, snr_def) on LTS||data frames with on-chip draws; ("real", "frame_power") is awgn_philox"""
        ch = channel(noise, snr_def)
        ota = self.empty(tuple(tx.shape), self.torch.float32)
        self._check(self.lib.ofdm_awgn_philox_ex(self.h, ch.noise, ch.snr_def, _ptr(tx), _ptr(power), snr_db, seed, stream, frame0,
                                                 _ptr(ota), tx.shape[0], n_sym, mode))
        return ota

    def rx_frames(self, ota, tx_packed, n_sym, mode, want=()):
        n_frames = ota.shape[0]
        cnt = self.new_counters()
        d, bufs = self._dump(n_frames, n_sym, want)
        self._check(self.lib.ofdm_rx_frames(self.h, _ptr(ota), _ptr(tx_packed), n_frames, n_sym, mode, _ptr(cnt), C.byref(d)))
        return self.read_counters(cnt)[0], bufs

    def awgn_rx_inject(self, tx, g, tx_packed, snr_db, n_sym, mode, power=None, want=(), counters=None):
        n_frames = tx.shape[0]
        cnt = counters if counters is not None else self.new_counters()
        d, bufs = self._dump(n_frames, n_sym, want)
        self._check(self.lib.ofdm_awgn_rx_inject(self.h, _ptr(tx), _ptr(g), _ptr(power), _ptr(tx_packed), snr_db, n_frames,
                                                 n_sym, mode, _ptr(cnt), C.byref(d)))
        if counters is not None:
            return None, bufs
        return self.read_counters(cnt)[0], bufs

    def awgn_rx_philox(self, tx, tx_packed, snr_db, seed, stream, frame0, n_sym, mode, power=None, want=(), counters=None):
        n_frames = tx.shape[0]
        cnt = counters if counters is not None else self.new_counters()
        d, bufs = self._dump(n_frames, n_sym, want)
        self._check(self.lib.ofdm_awgn_rx_philox(self.h, _ptr(tx), _ptr(power), _ptr(tx_packed), snr_db, seed, stream, frame0,
                                                 n_frames, n_sym, mode, _ptr(cnt), C.byref(d)))
        if counters is not None:
            return None, bufs
        return self.read_counters(cnt)[0], bufs

    def awgn_rx_inject_sweep(self, tx, g, tx_packed, snr_db, n_sym, mode, power=None, counters=None):
        """channel + receiver over a list of SNR points on resident frames; counters [n_snr] device tensor (accumulated into)"""
        snr = np.ascontiguousarray(snr_db, dtype=np.float32)
        cnt = counters if counters is not None else self.new_counters(len(snr))
        self._check(self.lib.ofdm_awgn_rx_inject_sweep(self.h, _ptr(tx), _ptr(g), _ptr(power), _ptr(tx_packed), snr.ctypes.data, len(snr),
                                                       tx.shape[0], n_sym, mode, _ptr(cnt)))
        return None if counters is not None else self.read_counters(cnt)

    # ---- the receiver's stages one by one
    def strip_cp(self, frames, n_sym, data_off=160):
        n, length = frames.shape[0], frames.shape[1]
        out = self.empty((n, n_sym, 64, 2), self.torch.float32)
        self._check(self.lib.ofdm_strip_cp(self.h, _ptr(frames), _ptr(out), n, n_sym, length, data_off))
        return out

    def channel_estimate(self, frames, mode, lts_off=0):
        n, length = frames.shape[0], frames.shape[1]
        out = self.empty((n, 64, 2), self.torch.float32)
        self._check(self.lib.ofdm_channel_estimate(self.h, _ptr(frames), _ptr(out), n, length, lts_off, mode))
        return out

    def equalize(self, F, H, mode):
        n, n_sym = F.shape[0], F.shape[1]
        out = self.empty(tuple(F.shape), self.torch.float32)
        self._check(self.lib.ofdm_equalize(self.h, _ptr(F), _ptr(H), _ptr(out), n, n_sym, mode))
        return out

    def demap(self, grid):
        n_symbols = grid.numel() // 128
        out = self.empty((n_symbols, 48, 2), self.torch.float32)
        self._check(self.lib.ofdm_demap(self.h, _ptr(grid), _ptr(out), n_symbols))
        return out

    def agc_slicer(self, points):
        n_symbols = points.numel() // 96
        out = self.empty((n_symbols, 48, 2), self.torch.float32)
        self._check(self.lib.ofdm_agc_slicer(self.h, _ptr(points), _ptr(out), n_symbols))
        return out

    def qpsk_demodulate(self, points):
        n_symbols = points.numel() // 96
        out = self.empty((n_symbols * 3,), self.torch.int32)
        self._check(self.lib.ofdm_qpsk_demodulate(self.h, _ptr(points), _ptr(out), n_symbols))
        return out

    # ---- sweeps
    def sweep_inject_host(self, bits_packed_host, g_host, n_frames, n_sym, snr_db, mode):
        """bits_packed_host / g_host: numpy arrays or pinned CPU torch tensors (HOST memory)."""
        snr = np.ascontiguousarray(snr_db, dtype=np.float32)
        out = (Counters * len(snr))()
        bp = bits_packed_host.data_ptr() if hasattr(bits_packed_host, "data_ptr") else bits_packed_host.ctypes.data
        gp = g_host.data_ptr() if hasattr(g_host, "data_ptr") else g_host.ctypes.data
        self._check(self.lib.ofdm_sweep_inject_host(self.h, bp, gp, n_frames, n_sym, snr.ctypes.data, len(snr), mode, out))
        return list(out)

    def sweep_inject_dev(self, bits_packed, g, n_frames, n_sym, snr_db, mode):
        snr = np.ascontiguousarray(snr_db, dtype=np.float32)
        out = (Counters * len(snr))()
        self._check(self.lib.ofdm_sweep_inject_dev(self.h, _ptr(bits_packed), _ptr(g), n_frames, n_sym, snr.ctypes.data,
                                                   len(snr), mode, out))
        return list(out)

    def random_bits(self, seed, frame0, n_frames, n_sym):
        out = self.empty((n_frames * n_sym * 3,), self.torch.int32)
        self._check(self.lib.ofdm_random_bits(self.h, seed, frame0, n_frames, n_sym, _ptr(out)))
        return out

    def mc_sweep_philox(self, seed, frame0, n_frames, n_sym, snr_db, mode, counters=None):
        """counters=None: returns host totals (synchronises); else accumulates into the device counters tensor."""
        snr = np.ascontiguousarray(snr_db, dtype=np.float32)
        if counters is not None:
            self._check(self.lib.ofdm_mc_sweep_philox_dev(self.h, seed, frame0, n_frames, n_sym, snr.ctypes.data, len(snr), mode,
                                                          _ptr(counters)))
            return None
        out = (Counters * len(snr))()
        self._check(self.lib.ofdm_mc_sweep_philox(self.h, seed, frame0, n_frames, n_sym, snr.ctypes.data, len(snr), mode, out))
        return list(out)

    def mc_sweep_points(self, seed, frame0, n_frames, n_sym, n_taps, snr_db, streams, mode, counters):
        """Monte-Carlo over an explicit list of points (streams: their Philox noise streams, None = 0..n-1); n_taps = 0 is AWGN only.
        Accumulates into the device counters tensor."""
        snr = np.ascontiguousarray(snr_db, dtype=np.float32)
        st = None if streams is None else np.ascontiguousarray(streams, dtype=np.uint32)
        self._check(self.lib.ofdm_mc_sweep_points_dev(self.h, seed, frame0, n_frames, n_sym, n_taps, snr.ctypes.data,
                                                      None if st is None else st.ctypes.data, len(snr), mode, _ptr(counters)))

    def mc_sweep_until(self, seed, frame0, n_sym, n_taps, snr_db, mode, target_errors=100, max_bits=10 ** 9, round_frames=1 << 20):
        """configs[3]'s stop rule on one GPU: returns (host totals, rounds)"""
        snr = np.ascontiguousarray(snr_db, dtype=np.float32)
        out = (Counters * len(snr))()
        rounds = _I(0)
        self._check(self.lib.ofdm_mc_sweep_until(self.h, seed, frame0, n_sym, n_taps, snr.ctypes.data, len(snr), mode, target_errors, max_bits,
                                                 round_frames, out, C.byref(rounds)))
        return list(out), int(rounds.value)

    def mc_sweep_channel(self, seed, frame0, n_frames, n_sym, snr_db, mode, noise="real", snr_def="frame_power", n_taps=0, streams=None,
                         counters=None):
        """Monte-Carlo sweep through the channel (noise, snr_def, n_taps); ("real", "frame_power") is mc_sweep_points.
        counters=None: returns host totals (synchronises); else accumulates into the device counters tensor."""
        ch = channel(noise, snr_def, n_taps)
        snr = np.ascontiguousarray(snr_db, dtype=np.float32)
        st = None if streams is None else np.ascontiguousarray(streams, dtype=np.uint32)
        cnt = counters if counters is not None else self.new_counters(len(snr))
        self._check(self.lib.ofdm_mc_sweep_channel_dev(self.h, C.byref(ch), seed, frame0, n_frames, n_sym, snr.ctypes.data,
                                                       None if st is None else st.ctypes.data, len(snr), mode, _ptr(cnt)))
        return None if counters is not None else self.read_counters(cnt)

    def mc_sweep_channel_until(self, seed, frame0, n_sym, snr_db, mode, noise="real", snr_def="frame_power", n_taps=0, target_errors=100,
                               max_bits=10 ** 9, round_frames=1 << 20):
        """configs[3]'s stop rule through the channel (noise, snr_def, n_taps) on one GPU: returns (host totals, rounds)"""
        ch = channel(noise, snr_def, n_taps)
        snr = np.ascontiguousarray(snr_db, dtype=np.float32)
        out = (Counters * len(snr))()
        rounds = _I(0)
        self._check(self.lib.ofdm_mc_sweep_channel_until(self.h, C.byref(ch), seed, frame0, n_sym, snr.ctypes.data, len(snr), mode,
                                                         target_errors, max_bits, round_frames, out, C.byref(rounds)))
        return list(out), int(rounds.value)

    # ---- the coded link (DESIGN.md section 6.2)
    def conv_encode(self, info, n_sym, rate="1/2"):
        """information words [n_frames * n_sym * 3] (int32) -> payload words of the same shape for tx_frames"""
        n_frames = info.numel() // (3 * n_sym)
        out = self.empty((n_frames * n_sym * 3,), self.torch.int32)
        self._check(self.lib.ofdm_conv_encode(self.h, CODE[rate] if rate in CODE else -1, _ptr(info), _ptr(out), n_frames, n_sym))
        return out

    def viterbi_decode(self, H, eq, n_sym, rate="1/2", decision="soft", info=None, want_decoded=True):
        """decode the receiver's H [n_frames, 64, 2] and eq [n_frames, n_sym * 48, 2] dumps; returns (coded Counters or None when
        info is None, decoded words [n_frames * n_sym * 3] or None)"""
        cd = code(rate, decision)
        n_frames = H.shape[0]
        cnt = self.new_counters() if info is not None else None
        dec = self.zeros((n_frames * n_sym * 3,), self.torch.int32) if want_decoded else None
        self._check(self.lib.ofdm_viterbi_decode(self.h, C.byref(cd), _ptr(H), _ptr(eq), _ptr(info), _ptr(dec), n_frames, n_sym, _ptr(cnt)))
        return (self.read_counters(cnt)[0] if cnt is not None else None), dec

    def mc_sweep_coded(self, seed, frame0, n_frames, n_sym, snr_db, mode, rate="1/2", decision="soft", noise="real", snr_def="frame_power",
                       n_taps=0, streams=None, counters=None):
        """Monte-Carlo sweep of the coded link through the channel (noise, snr_def, n_taps).  counters=None: returns host totals
        (coded, raw); else counters is a pair of device tensors (coded, raw or None) accumulated into, and None is returned."""
        ch, cd = channel(noise, snr_def, n_taps), code(rate, decision)
        snr = np.ascontiguousarray(snr_db, dtype=np.float32)
        st = None if streams is None else np.ascontiguousarray(streams, dtype=np.uint32)
        coded, raw = counters if counters is not None else (self.new_counters(len(snr)), self.new_counters(len(snr)))
        self._check(self.lib.ofdm_mc_sweep_coded_dev(self.h, C.byref(ch), C.byref(cd), seed, frame0, n_frames, n_sym, snr.ctypes.data,
                                                     None if st is None else st.ctypes.data, len(snr), mode, _ptr(coded), _ptr(raw)))
        if counters is not None:
            return None
        return self.read_counters(coded), self.read_counters(raw)

    def mc_sweep_coded_until(self, seed, frame0, n_sym, snr_db, mode, rate="1/2", decision="soft", noise="real", snr_def="frame_power",
                             n_taps=0, target_errors=100, max_bits=10 ** 9, round_frames=1 << 20):
        """configs[3]'s stop rule on the coded counters, on one GPU: returns (coded host totals, raw host totals, rounds)"""
        ch, cd = channel(noise, snr_def, n_taps), code(rate, decision)
        snr = np.ascontiguousarray(snr_db, dtype=np.float32)
        coded, raw = (Counters * len(snr))(), (Counters * len(snr))()
        rounds = _I(0)
        self._check(self.lib.ofdm_mc_sweep_coded_until(self.h, C.byref(ch), C.byref(cd), seed, frame0, n_sym, snr.ctypes.data, len(snr), mode,
                                                       target_errors, max_bits, round_frames, coded, raw, C.byref(rounds)))
        return list(coded), list(raw), int(rounds.value)

    def multipath_taps(self, tx, taps, n_sym):
        out = self.empty(tuple(tx.shape), self.torch.float32)
        self._check(self.lib.ofdm_multipath_taps(self.h, _ptr(tx), _ptr(taps), taps.shape[1], _ptr(out), tx.shape[0], n_sym))
        return out

    def multipath_philox(self, tx, seed, frame0, n_taps, n_sym):
        out = self.empty(tuple(tx.shape), self.torch.float32)
        taps = self.empty((tx.shape[0], n_taps, 2), self.torch.float32)
        self._check(self.lib.ofdm_multipath_philox(self.h, _ptr(tx), seed, frame0, n_taps, _ptr(out), _ptr(taps), tx.shape[0], n_sym))
        return out, taps

    def mc_sweep_multipath(self, seed, frame0, n_frames, n_sym, n_taps, snr_db, mode, counters=None):
        snr = np.ascontiguousarray(snr_db, dtype=np.float32)
        cnt = counters if counters is not None else self.new_counters(len(snr))
        self._check(self.lib.ofdm_mc_sweep_multipath_dev(self.h, seed, frame0, n_frames, n_sym, n_taps, snr.ctypes.data, len(snr), mode,
                                                         _ptr(cnt)))
        return None if counters is not None else self.read_counters(cnt)

    def rrc_tx(self, frames):
        n, length = frames.shape[0], frames.shape[1]
        out = self.empty((n, 2 * length + 20, 2), self.torch.float32)
        self._check(self.lib.ofdm_rrc_tx(self.h, _ptr(frames), _ptr(out), n, length))
        return out

    def rrc_rx(self, x, packet_idx, frame_len_):
        n, in_len = x.shape[0], x.shape[1]
        out = self.empty((n, frame_len_, 2), self.torch.float32)
        self._check(self.lib.ofdm_rrc_rx(self.h, _ptr(x), _ptr(out), n, in_len, packet_idx, frame_len_))
        return out

    def awgn_inject_len(self, tx, g, snr_db, mode, power=None):
        ota = self.empty(tuple(tx.shape), self.torch.float32)
        self._check(self.lib.ofdm_awgn_inject_len(self.h, _ptr(tx), _ptr(g), _ptr(power), snr_db, _ptr(ota), tx.shape[0], tx.shape[1], mode))
        return ota

    def packet_detect(self, rx):
        n, length = rx.shape[0], rx.shape[1]
        corr = self.empty((n, length - 47), self.torch.float32)
        self._check(self.lib.ofdm_packet_detect(self.h, _ptr(rx), _ptr(corr), n, length))
        return corr

    def packet_select(self, corr):
        idx = self.empty((corr.shape[0],), self.torch.int32)
        self._check(self.lib.ofdm_packet_select(self.h, _ptr(corr), _ptr(idx), corr.shape[0], corr.shape[1]))
        return idx

    def sts(self):
        t = np.zeros((160, 2), np.float32)
        self._check(self.lib.ofdm_sts(self.h, t.ctypes.data))
        return t

    def prepend_sts(self, frames):
        n, length = frames.shape[0], frames.shape[1]
        out = self.empty((n, 160 + length, 2), self.torch.float32)
        self._check(self.lib.ofdm_prepend_sts(self.h, _ptr(frames), _ptr(out), n, length))
        return out

    def gather(self, x, start, out_len):
        """start: int (same for all) or an int32 device tensor [n]"""
        n, in_len = x.shape[0], x.shape[1]
        out = self.empty((n, out_len, 2), self.torch.float32)
        if isinstance(start, int):
            self._check(self.lib.ofdm_gather(self.h, _ptr(x), None, start, _ptr(out), n, in_len, out_len))
        else:
            self._check(self.lib.ofdm_gather(self.h, _ptr(x), _ptr(start), 0, _ptr(out), n, in_len, out_len))
        return out

    def rrc_rx_idx(self, x, idx, frame_len_):
        n, in_len = x.shape[0], x.shape[1]
        out = self.empty((n, frame_len_, 2), self.torch.float32)
        self._check(self.lib.ofdm_rrc_rx_idx(self.h, _ptr(x), _ptr(idx), _ptr(out), n, in_len, frame_len_))
        return out

    def cfo(self, x, fine):
        n, length = x.shape[0], x.shape[1]
        out = self.empty((n, length, 2), self.torch.float32)
        freq = self.empty((n,), self.torch.float32)
        fn = self.lib.ofdm_cfo_fine if fine else self.lib.ofdm_cfo_coarse
        self._check(fn(self.h, _ptr(x), _ptr(out), _ptr(freq), n, length))
        return out, freq

    def awgn_philox_len(self, tx, snr_db, seed, stream, frame0, mode, power=None):
        ota = self.empty(tuple(tx.shape), self.torch.float32)
        self._check(self.lib.ofdm_awgn_philox_len(self.h, _ptr(tx), _ptr(power), snr_db, seed, stream, frame0, _ptr(ota), tx.shape[0],
                                                  tx.shape[1], mode))
        return ota

    def finalize(self, counters):
        res = (_F * 3)()
        self._check(self.lib.ofdm_counters_finalize(C.byref(counters), res))
        return float(res[0]), float(res[1]), float(res[2])


def pack_bits_host(bits_u8):
    """numpy helper: [..., 96*k] bytes (0/1) -> [..., 3*k] uint32 words, bit j at word j>>5, position j&31."""
    b = np.ascontiguousarray(bits_u8, dtype=np.uint8)
    assert b.shape[-1] % 32 == 0
    w = b.reshape(b.shape[:-1] + (b.shape[-1] // 32, 32)).astype(np.uint32)
    return (w << np.arange(32, dtype=np.uint32)).sum(axis=-1, dtype=np.uint64).astype(np.uint32)


def unpack_bits_host(words):
    w = np.ascontiguousarray(words, dtype=np.uint32)
    return ((w[..., None] >> np.arange(32, dtype=np.uint32)) & 1).astype(np.uint8).reshape(w.shape[:-1] + (w.shape[-1] * 32,))


def write_float_array_to_file(lib, a, fname):
    a = np.ascontiguousarray(a, dtype=np.float32)
    return lib.ofdm_write_float_array_to_file(a.ctypes.data, a.size, fname.encode())


def write_complex_array_to_file(lib, a_iq, fname, fmt):
    a = np.ascontiguousarray(a_iq, dtype=np.float32).reshape(-1, 2)
    return lib.ofdm_write_complex_array_to_file(a.ctypes.data, a.shape[0], fname.encode(), fmt)
