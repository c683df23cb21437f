"""The C driver's default mode -- the reference's own main() body, STS + x2 RRC shaping, 10x repetition, flat Philox noise, capture
window, packet detection and selection, matched filter, coarse and fine CFO, receiver -- against the CPU oracle at every message
length, stage by stage: each GPU stage is given the GPU's previous output and compared with the oracle applied to that same input,
so that differences cannot compound and a failure names its kernel.  Then the oracle runs the path end to end on the GPU's draws,
and the driver's result files must be the replay's, byte for byte."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from ota_oracle import OtaOracle, capture_starts, encode_message, lengths

pytestmark = pytest.mark.gpu

SEED = 17
DRIVER_NSYM = (1, 2, 5, 39)
MESSAGES = ["OFDM on B200", "Hey! I am Vivaswan", "The quick brown fox jumps over the lazy dog, and back again.",
            "802.11a OFDM QPSK " * 26]


@pytest.fixture(scope="module")
def oo():
    return OtaOracle()


def same(a, b):
    return np.array_equal(np.asarray(a), np.asarray(b), equal_nan=True)


def dev(ofdm, a, offset=False):
    """a on the device, 16-byte aligned, or (offset) in a view whose base is 8 bytes off a 16-byte boundary"""
    torch = ofdm.torch
    a = np.ascontiguousarray(a, dtype=np.float32)
    if not offset:
        return ofdm.to_dev(a)
    buf = ofdm.zeros((a.size + 2,), torch.float32)
    t = buf[2:].view(a.shape)
    assert t.data_ptr() % 16 == 8
    t.copy_(torch.from_numpy(a))
    return t


def flat_channel(ofdm, tx, snr_db, seed, stream, frame0, mode, power=None, out=None):
    """ofdm_awgn_philox_len into `out` (default: a fresh aligned tensor)"""
    out = ofdm.empty(tuple(tx.shape), ofdm.torch.float32) if out is None else out
    ofdm._check(ofdm.lib.ofdm_awgn_philox_len(ofdm.h, tx.data_ptr(), None if power is None else power.data_ptr(), snr_db, seed, stream,
                                              frame0, out.data_ptr(), tx.shape[0], tx.shape[1], mode))
    return out


def gpu_flat_draws(ofdm, pkg, seed, stream, frame0, n_frames, length):
    """the GPU's flat normals, bit for bit: at 0 dB with power 1.0, sigma = 1 exactly and the I rail is the draw itself; the Q
    rail must come back untouched"""
    torch = ofdm.torch
    gen = torch.Generator(device=ofdm.device)
    gen.manual_seed(seed ^ stream)
    tx = ofdm.zeros((n_frames, length, 2), torch.float32)
    tx[..., 1] = torch.randn((n_frames, length), device=ofdm.device, generator=gen)
    ones = torch.ones((n_frames,), dtype=torch.float32, device=ofdm.device)
    out = flat_channel(ofdm, tx, 0.0, seed, stream, frame0, pkg.MODE_EXACT, power=ones)
    assert torch.equal(out[..., 1], tx[..., 1])
    return out[..., 0].cpu().numpy()


# ---- 1. the flat Philox channel (ofdm_awgn_philox_len, k_awgn_philox_flat)
@pytest.mark.parametrize("length", [1, 3, 5, 6, 4097, 8200])
def test_flat_draws_are_the_oracles_layout(ofdm, pkg, oo, length):
    frame0 = (1 << 32) - 2                                     # the frames cross the carry into the counter's high word
    g = gpu_flat_draws(ofdm, pkg, SEED, 5, frame0, 5, length)
    assert np.max(np.abs(g - oo.philox_normals_flat(SEED, 5, frame0, 5, length))) < 2e-5       # MUFU vs libm
    for f in range(5):
        assert same(g[f], gpu_flat_draws(ofdm, pkg, SEED, 5, frame0 + f, 1, length)[0])
    # the scalar branch (buffers 8 bytes off a 16-byte boundary) hands out the same draws as the vector branch
    torch = ofdm.torch
    tx = dev(ofdm, np.zeros((5, length, 2), np.float32), offset=True)
    out = dev(ofdm, np.full((5, length, 2), 7.0, np.float32), offset=True)
    ones = torch.ones((5,), dtype=torch.float32, device=ofdm.device)
    flat_channel(ofdm, tx, 0.0, SEED, 5, frame0, pkg.MODE_EXACT, power=ones, out=out)
    o = out.cpu().numpy()
    assert same(o[..., 0], g) and not o[..., 1].any()


def test_flat_draws_statistics(ofdm, pkg, oo):
    n = 1 << 20
    g = gpu_flat_draws(ofdm, pkg, SEED, 0, 0, 4, n).astype(np.float64)
    z = g.ravel()
    assert abs(z.mean()) < 5 / np.sqrt(z.size) and abs(z.var() - 1) < 5e-3
    assert abs(np.mean(z ** 4) / np.mean(z ** 2) ** 2 - 3) < 0.02
    q = g.reshape(4, -1, 4)
    for a, b in ((0, 1), (2, 3)):                                # the two normals of a Box-Muller pair
        assert abs(np.corrcoef(q[..., a].ravel(), q[..., b].ravel())[0, 1]) < 0.01
    m = 1 << 16
    base = g[:, :m].ravel()
    for other in (gpu_flat_draws(ofdm, pkg, SEED, 1, 0, 4, m), gpu_flat_draws(ofdm, pkg, SEED + 1, 0, 0, 4, m)):
        assert abs(np.corrcoef(base, other.ravel())[0, 1]) < 0.03
    # domain 3 against the frame layout's domain 0 of the same (seed, stream, frame)
    length = 160 + 80 * 100
    d0 = oo.philox_normals(SEED, 0, 0, 8, length, 0)
    d3 = gpu_flat_draws(ofdm, pkg, SEED, 0, 0, 8, length)
    assert abs(np.corrcoef(d0.ravel(), d3.ravel())[0, 1]) < 0.03


FLAT_LENGTHS = [8200, 9800, 14600, 69000, 1, 3, 5, 4097, 2023]


def channel_inputs(oo, length, rng, n_frames=3):
    """the driver's repeated waveform at its own lengths (a message per frame, scaled), else noise-like frames over many binades"""
    for n_sym in DRIVER_NSYM:
        if lengths(n_sym)[3] == length:
            bits = rng.integers(0, 2, (n_frames, 96 * n_sym), dtype=np.uint8)
            reps = [oo.waveform(b[None], n_sym)[2] for b in bits]
            return np.stack(reps) * np.float32(2.0) ** rng.integers(-6, 6, (n_frames, 1, 1)).astype(np.float32)
    return (rng.standard_normal((n_frames, length, 2)) * 2.0 ** rng.integers(-20, 20, (n_frames, 1, 1))).astype(np.float32)


@pytest.mark.parametrize("length", FLAT_LENGTHS)
def test_flat_channel_against_oracle(ofdm, pkg, port, oo, length):
    """EXACT = the oracle's awgn_inject on the GPU's draws, with the frame power measured inside the call (the driver's case),
    bit for bit, whatever the alignment; FAST within 1e-5 of each frame's peak"""
    rng = np.random.default_rng(length)
    tx = channel_inputs(oo, length, rng)
    n = tx.shape[0]
    for stream, frame0, snr in ((0, 0, 4.0), (3, 1 << 33, 17.5), (11, 5, -2.0)):
        g = gpu_flat_draws(ofdm, pkg, SEED, stream, frame0, n, length)
        want = port.awgn_inject(tx, g, snr)
        got = []
        for offset in (False, True):
            out = dev(ofdm, np.zeros_like(tx), offset) if offset else None
            got.append(flat_channel(ofdm, dev(ofdm, tx, offset), snr, SEED, stream, frame0, pkg.MODE_EXACT, out=out).cpu().numpy())
        assert same(got[0], want), (stream, np.argwhere(got[0] != want)[:5])
        assert same(got[1], want), (stream, np.argwhere(got[1] != want)[:5])
        fast = flat_channel(ofdm, dev(ofdm, tx), snr, SEED, stream, frame0, pkg.MODE_FAST).cpu().numpy()
        peak = np.abs(want).max(axis=(1, 2), keepdims=True)
        assert np.all(np.abs(fast - want) <= 1e-5 * peak)


# ---- 2. the exact frame power on the path's lengths (ofdm_frame_power: k_frame_power_exact<true> / <false>)
def hard_frames(rng, n, length):
    """the inputs of test_margins_agree_on_hard_inputs at any length: random binades, zeros, tiny and huge samples, frames among
    the float subnormals, real-only frames"""
    x = rng.standard_normal((n, length, 2)).astype(np.float32) * np.float32(2.0) ** rng.integers(-20, 20, (n, 1, 1)).astype(np.float32)
    x[::7, 5:40] = 0.0
    x[::11, length // 3] = 3.0e-23
    x[1::11, length // 2, 0] = 3.0e19
    x[2::11] *= np.float32(1.0e-22)
    x[3::11, :, 1] = 0.0
    x[4] = 0.0
    return x


@pytest.mark.parametrize("length", [1, 2, 15, 17, 321, 8200, 9800, 21183])
def test_exact_frame_power_against_oracle(ofdm, pkg, port, length):
    rng = np.random.default_rng(1000 + length)
    x = hard_frames(rng, 45, length)
    want = np.array([port.frame_power(f) for f in x], np.float32)
    assert np.isinf(want[1::11]).all() and (want[2::11] < 1e-30).all() and want[4] == 0
    for offset in (False, True):
        got = ofdm.frame_power(dev(ofdm, x, offset), pkg.MODE_EXACT).cpu().numpy()
        assert same(got, want), (offset, np.flatnonzero(got != want)[:10])


# ---- 3. packet detection across tiles of 4096 lags (k_packet_detect)
DETECT_LENGTHS = [48, 4143, 4144, 4175, 8239, 8240, 4482, 21183]


def noisy_captures(golden, length, n, rng):
    """windows of the reference's own over-the-air waveform (repeated, as the driver repeats it) with real-rail noise"""
    tx = golden["ref_tx_waveform"]
    p = np.mean(np.sum(tx.astype(np.float64) ** 2, axis=1))
    caps = []
    for k in range(n):
        snr_db = [2.0, 6.0, 10.0, 20.0][k % 4]
        start = int(rng.integers(0, tx.shape[0]))
        cap = np.take(tx, np.arange(start, start + length), axis=0, mode="wrap").copy()
        cap[:, 0] += (rng.standard_normal(length) * np.sqrt(p / 10 ** (snr_db / 10))).astype(np.float32)
        caps.append(cap)
    return caps


def degenerate_captures(caps, length, rng):
    """test_gpu_detect's degenerate captures, with the bad samples in the halo of a tile boundary (lags 4096 k)"""
    near = [4096 * k + d for k in range(1, 6) for d in (0, 20, 46) if 4096 * k + d < length] or [length // 2]
    out = [np.zeros((length, 2), np.float32), rng.standard_normal((length, 2)).astype(np.float32)]
    for i, scale in enumerate((1e-25, 3e-19, 1e17, 1e20)):
        out.append((caps[i % len(caps)] * np.float32(scale)).astype(np.float32))
    bad = caps[0].copy(); bad[near, 0] = np.nan; out.append(bad)
    bad = caps[1 % len(caps)].copy(); bad[near[-1], 1] = np.inf; out.append(bad)
    bad = caps[2 % len(caps)].copy(); bad[[max(0, k - 47) for k in near], 0] = -np.inf; out.append(bad)
    mixed = caps[3 % len(caps)].copy(); mixed[::3] *= np.float32(1e-24); out.append(mixed)
    return out


def check_detection(ofdm, port, caps):
    corr = ofdm.packet_detect(ofdm.to_dev(np.stack(caps)))
    idx = ofdm.packet_select(corr).cpu().numpy()
    got = corr.cpu().numpy()
    found = 0
    for i, cap in enumerate(caps):
        want = port.packet_detection(cap)
        assert same(got[i], want[:, 0]), (i, np.flatnonzero(~((got[i] == want[:, 0]) | (np.isnan(got[i]) & np.isnan(want[:, 0]))))[:10])
        want_idx = port.packet_selection(want)
        assert idx[i] == want_idx, (i, idx[i], want_idx)
        found += want_idx > 0
    return found


@pytest.mark.parametrize("length", DETECT_LENGTHS)
def test_packet_detection_across_tiles(ofdm, pkg, port, golden, length):
    rng = np.random.default_rng(length)
    caps = noisy_captures(golden, length, 8, rng)
    caps += degenerate_captures(caps, length, rng)
    found = check_detection(ofdm, port, caps)                 # 18 captures: fewer than the resident blocks
    if length >= 3008:
        assert found >= 4


def test_packet_detection_more_captures_than_blocks(ofdm, pkg, port, golden):
    """more captures than the persistent grid holds (at most 3 blocks of 66 KB per SM): blocks take several captures each"""
    rng = np.random.default_rng(3)
    n = 8 * ofdm.sm_count + 3
    assert check_detection(ofdm, port, noisy_captures(golden, 4144, n, rng)) >= n // 4


# ---- 4. packet selection edges (k_packet_select)
T_UP = np.nextafter(np.float32(0.75), np.float32(1))


def row(length, lags, fill=0.1):
    r = np.full(length, fill, np.float32)
    for p in lags:
        p, v = p if isinstance(p, tuple) else (p, 0.9)
        r[p] = v
    return r


def selection_rows(length=2000):
    """(row, what it exercises); a front is an above-threshold lag more than 300 after the previous one (the first one: more than
    300 after lag -1); all fronts but the last are tried, in order, on the lag 230 after them"""
    rows = []
    for v in (0.75, T_UP, -0.8, np.nan, np.inf, -np.inf, -0.75):
        rows.append((row(length, [(400, v), 630, 1500]), "front value %r" % v))
        rows.append((row(length, [400, (630, v), 1500]), "look-ahead value %r" % v))
    for first in (299, 300, 301):
        rows.append((row(length, [first, first + 230, 1000, 1230, 1600]), "first lag %d" % first))
        rows.append((row(length, [first, 1000, 1230, 1600]), "first lag %d, failing" % first))
    for gap in (299, 300, 301):
        b = 500 + gap
        rows.append((row(length, [500, b, b + 230, 1400, 1630, 1950]), "gap %d" % gap))
        rows.append((row(length, list(range(500, 540)) + [539 + gap, 539 + gap + 230, 1500]), "gap %d after a run" % gap))
    for front in (640, 671, 672, 703):                          # lanes 0 and 31 of consecutive 32-lag steps
        for gap in (300, 301):
            rows.append((row(length, [front - gap, front, front + 230, 1600]), "front %d, gap %d" % (front, gap)))
    rows.append((row(length, [383, 384, 614, 1500]), "lane 31 then lane 0 of the next step: one front, its look-ahead fails"))
    rows.append((row(length, [383, 384, 613, 1500]), "lane 31 then lane 0 of the next step: one front, its look-ahead passes"))
    rows.append((row(length, [31, 32, 262, 700]), "first lags 31, 32 (no front), then one front, the last"))
    rows.append((row(length, [100, 700, 930, 1400, length - 100]), "the last front's look-ahead lies beyond the row"))
    rows.append((row(length, [100, 700, 930, length - 230, length - 1]), "the look-ahead of the last front is the last lag"))
    rows.append((row(length, [400, 1100, 1330]), "the only passing front is the last"))
    rows.append((row(length, [1100, 1330]), "one front only"))
    rows.append((row(length, []), "nothing above the threshold"))
    rows.append((np.full(length, 0.9, np.float32), "everything above the threshold"))
    rows.append((row(length, [0, 230, 600, 830, 1300]), "a front at lag 0 is not one (gap 1)"))
    rows.append((row(length, [301, 531, 900]), "a front at lag 301"))
    return rows


def random_rows(rng, n, length):
    """sparse runs of above-threshold lags (some exactly at the threshold, negative or NaN) with gaps around 230 and 300"""
    vals = np.array([0.8, 0.95, 1.0, -0.9, 0.75, T_UP, np.nan, 0.5], np.float32)
    out = np.empty((n, length), np.float32)
    for k in range(n):
        r = rng.uniform(-0.74, 0.74, length).astype(np.float32)
        p = int(rng.integers(0, min(420, length)))
        while p < length:
            run = min(int(rng.integers(1, 40)), length - p)
            r[p:p + run] = vals[rng.choice(len(vals), run, p=[0.3, 0.25, 0.15, 0.14, 0.05, 0.05, 0.03, 0.03])]
            u = rng.random()
            if u < 0.35:
                p += int(rng.integers(222, 232))                # the next run starts around this one's look-ahead
            else:
                p += run - 1 + (int(rng.integers(297, 304)) if u < 0.7 else int(rng.integers(1, 700)))     # a gap around 300, or any
        out[k] = r
    return out


def check_selection(ofdm, port, rows):
    rows = np.ascontiguousarray(rows, dtype=np.float32)
    got = ofdm.packet_select(ofdm.to_dev(rows)).cpu().numpy()
    want = np.array([port.packet_selection(np.stack([r, np.zeros_like(r)], axis=-1)) for r in rows])
    return got, want


def test_packet_selection_edges(ofdm, pkg, port):
    rows = selection_rows()
    got, want = check_selection(ofdm, port, [r for r, _ in rows])
    for g, w, (_, what) in zip(got, want, rows):
        assert g == w, (what, g, w)
    assert (want > 0).sum() >= 15 and (want == 0).sum() >= 15
    # the rules as stated, on a few of the rows
    named = dict((what, w) for (_, what), w in zip(rows, want))
    assert named["first lag 299"] == 1011 and named["first lag 300"] == 311 and named["first lag 301"] == 312
    assert named["gap 300"] == 1411 and named["gap 301"] == 812
    assert named["the only passing front is the last"] == 0
    assert named["lane 31 then lane 0 of the next step: one front, its look-ahead fails"] == 0
    assert named["lane 31 then lane 0 of the next step: one front, its look-ahead passes"] == 394


@pytest.mark.parametrize("length", [1, 31, 32, 33, 2000, 21136])
def test_packet_selection_random_rows(ofdm, pkg, port, length):
    rng = np.random.default_rng(length)
    n = {2000: 3000, 21136: 300}.get(length, 200)
    rows = random_rows(rng, n, length)
    got, want = check_selection(ofdm, port, rows)
    bad = np.flatnonzero(got != want)
    assert bad.size == 0, [(int(i), int(got[i]), int(want[i])) for i in bad[:5]]
    if length == 2000:
        assert 0.1 * n < (want > 0).sum() < 0.9 * n
    if length == 21136:
        assert (want > 0).sum() > 0.5 * n


# ---- 5. glue and CFO at every length
@pytest.mark.parametrize("in_len", [1, 3, 31, 32, 33, 480])
def test_gather_against_numpy(ofdm, pkg, in_len):
    rng = np.random.default_rng(in_len)
    n = 6
    x = rng.standard_normal((n, in_len, 2)).astype(np.float32)
    xd = ofdm.to_dev(x)
    starts = np.array([0, in_len, in_len - 1, 7 * in_len + 5, (1 << 31) - 1, int(rng.integers(0, 1000))], np.int32)
    for out_len in sorted({1, max(1, in_len // 2), 31, 33, 37 * in_len + 3}):
        got = ofdm.gather(xd, ofdm.to_dev(starts), out_len).cpu().numpy()
        for f in range(n):
            want = np.take(x[f], (np.arange(out_len, dtype=np.int64) + int(starts[f])) % in_len, axis=0, mode="wrap")
            assert same(got[f], want), (in_len, out_len, f, int(starts[f]))
        for s in (0, in_len, 3 * in_len + 2):
            got = ofdm.gather(xd, s, out_len).cpu().numpy()
            assert same(got, np.take(x, (np.arange(out_len, dtype=np.int64) + s) % in_len, axis=1, mode="wrap"))


@pytest.mark.parametrize("n_sym", [1, 3, 5, 39])
def test_prepend_and_shaping_at_every_length(ofdm, pkg, port, n_sym):
    rng = np.random.default_rng(n_sym)
    n = 3
    bits = rng.integers(0, 2, (n, 96 * n_sym), dtype=np.uint8)
    frames = ofdm.tx_frames(ofdm.to_dev(pkg.pack_bits_host(bits).view(np.int32)), n_sym, pkg.MODE_EXACT, with_power=False)
    full = ofdm.prepend_sts(frames)
    want_full = np.concatenate([np.broadcast_to(port.sts_time(), (n, 160, 2)), port.tx_frames(bits, n_sym)], axis=1)
    assert same(full.cpu().numpy(), want_full)
    assert same(ofdm.rrc_tx(full).cpu().numpy(), port.rrc_tx(want_full))


def check_cfo(got, want):
    """the CFO contract: within 1e-6 of the peak, in practice bit-identical almost everywhere (double libm on both sides)"""
    assert np.max(np.abs(got - want)) <= 1e-6 * np.abs(want).max()
    return np.sum(got == want), got.size


@pytest.mark.parametrize("length", [400, 480, 720, 3440])
def test_cfo_at_every_length(ofdm, pkg, port, oo, length):
    n_sym = (length - 320) // 80
    rng = np.random.default_rng(length)
    ident = total = 0
    for batch in (1, 7, 65):
        bits = rng.integers(0, 2, (batch, 96 * n_sym), dtype=np.uint8)
        full = np.concatenate([np.broadcast_to(port.sts_time(), (batch, 160, 2)), port.tx_frames(bits, n_sym)], axis=1)
        off = np.where(np.arange(batch) % 2 == 0, 40e3, -40e3)[:, None]
        rot = np.exp(2j * np.pi * off * np.arange(length) / 20e6)
        x = (full[..., 0] + 1j * full[..., 1]) * rot + 0.002 * (rng.standard_normal((batch, length)) + 1j * rng.standard_normal((batch, length)))
        x = np.stack([x.real, x.imag], axis=-1).astype(np.float32)
        c1, f1 = ofdm.cfo(ofdm.to_dev(x), fine=False)
        c2, f2 = ofdm.cfo(c1, fine=True)
        c1, f1, c2, f2 = c1.cpu().numpy(), f1.cpu().numpy(), c2.cpu().numpy(), f2.cpu().numpy()
        assert np.all(np.abs(f1 - off[:, 0]) < 4e3)
        for f in range(batch):
            for got, want in ((c1[f], port.cfo_coarse(x[f])), (c2[f], port.cfo_fine(c1[f]))):
                a, b = check_cfo(got, want)
                ident += a; total += b
            for got, want in ((f1[f], oo.cfo_freq(x[f], False)), (f2[f], oo.cfo_freq(c1[f], True))):
                assert abs(got - want) <= 1e-6 * abs(want), (f, got, want)
    assert ident >= 0.999 * total


# ---- 6. the whole chain and the driver's default run
SNR_START, SNR_STEP, SNR_COUNT = 4.0, 2.0, 19


def snr_points():
    return [np.float32(SNR_START) + np.float32(SNR_STEP) * np.float32(i) for i in range(SNR_COUNT)]


def replay(ofdm, pkg, msg, seed, mode):
    """the driver's loop (host/ofdm_main.c, full_chain) through the binding, one SNR point at a time as the driver runs it"""
    bits, n_sym = encode_message(msg)
    length, len480, len_shaped, len_rep, len_cap = lengths(n_sym)
    packed = ofdm.to_dev(pkg.pack_bits_host(bits[None]).view(np.int32))
    frame, _ = ofdm.tx_frames(packed, n_sym, mode)
    full = ofdm.prepend_sts(frame)
    shaped = ofdm.rrc_tx(full)
    rep = ofdm.gather(shaped, 0, len_rep)
    starts = capture_starts(seed, SNR_COUNT, len_rep, len_cap)
    points = []
    for i, snr in enumerate(snr_points()):
        ota = ofdm.awgn_philox_len(rep, float(snr), seed, i, 0, mode)
        cap = ofdm.gather(ota, starts[i], len_cap)
        corr = ofdm.packet_detect(cap)
        idx = ofdm.packet_select(corr)
        rxf = ofdm.rrc_rx_idx(cap, idx, len480)
        c1, _ = ofdm.cfo(rxf, fine=False)
        c2, _ = ofdm.cfo(c1, fine=True)
        ld = ofdm.gather(c2, 160, length)
        cnt, d = ofdm.rx_frames(ld, packed, n_sym, mode, want=("bits",))
        points.append(dict(start=starts[i], ota=ota, cap=cap, corr=corr, idx=idx, rxf=rxf, c1=c1, c2=c2, ld=ld, cnt=cnt, rx_bits=d["bits"],
                           res=ofdm.finalize(cnt)))
    return dict(bits=bits, n_sym=n_sym, frame=frame, full=full, shaped=shaped, rep=rep, points=points)


def driver_files(r):
    """what the driver writes for the replayed points: write_float_array_to_file's "%.2e", tab-separated, one newline"""
    fmt = lambda v: "\t".join("%.2e" % float(np.float32(x)) for x in v) + "\n"              # noqa: E731
    res = [p["res"] for p in r["points"]]
    return {"Output_SNR.txt": fmt(snr_points()), "Output_EVM_AGC.txt": fmt([x[0] for x in res]),
            "Output_EVM_AGC_DB.txt": fmt([x[1] for x in res]), "Output_BER.txt": fmt([x[2] for x in res])}


def run_driver(msg, seed, mode, outdir):
    exe = os.path.join(ROOT, "ieee-802.11-ofdm-qpsk-simulator_b200", "ofdm_sweep")
    os.makedirs(outdir, exist_ok=True)
    cmd = [exe, "--quiet", "--message", msg, "--seed", str(seed), "--snr-start", "%g" % SNR_START, "--snr-count", str(SNR_COUNT),
           "--snr-step", "%g" % SNR_STEP, "--outdir", str(outdir)] + (["--mode", "fast"] if mode == "fast" else [])
    r = subprocess.run(cmd, capture_output=True, timeout=600)
    assert r.returncode == 0, r.stdout.decode("latin-1") + r.stderr.decode("latin-1")
    return {k: open(os.path.join(outdir, k)).read() for k in ("Output_SNR.txt", "Output_EVM_AGC.txt", "Output_EVM_AGC_DB.txt", "Output_BER.txt")}


@pytest.mark.parametrize("msg", MESSAGES, ids=["1sym", "2sym", "5sym", "39sym"])
def test_whole_path_against_oracle_and_driver(ofdm, pkg, port, oo, msg, tmp_path):
    bits, n_sym = encode_message(msg)
    assert n_sym in DRIVER_NSYM
    length, len480, len_shaped, len_rep, len_cap = lengths(n_sym)
    seed = 100 + n_sym
    r = replay(ofdm, pkg, msg, seed, pkg.MODE_EXACT)
    # the transmitter side, stage by stage
    want_full, want_shaped, want_rep = oo.waveform(bits[None], n_sym)
    assert same(r["full"].cpu().numpy()[0], want_full)
    assert same(r["shaped"].cpu().numpy()[0], port.rrc_tx(r["full"].cpu().numpy())[0])
    assert same(r["rep"].cpu().numpy()[0], want_rep)
    rep = r["rep"].cpu().numpy()[0]
    checked = clean = with_errors = ident = total = 0
    port_ber = {}
    for i, (snr, p) in enumerate(zip(snr_points(), r["points"])):
        g = gpu_flat_draws(ofdm, pkg, seed, i, 0, 1, len_rep)[0]
        ota = p["ota"].cpu().numpy()[0]
        assert same(ota, port.awgn_inject(rep, g, float(snr))), i                       # flat channel + exact power
        cap = p["cap"].cpu().numpy()[0]
        assert same(cap, ota[p["start"]:p["start"] + len_cap]), i                         # capture window
        want_corr = port.packet_detection(cap)
        assert same(p["corr"].cpu().numpy()[0], want_corr[:, 0]), i                      # detection
        idx = int(p["idx"].cpu().numpy()[0])
        assert idx == port.packet_selection(want_corr), i                                 # selection
        e2e_idx, e2e = oo.ota_point(want_rep, g, float(snr), p["start"], len_cap, bits, n_sym)
        if idx + 2 * (len480 - 1) >= len_cap + 20:
            assert e2e_idx == -1
            continue                                                                       # the reference reads past its buffer here
        checked += 1
        assert e2e_idx == idx
        rxf = p["rxf"].cpu().numpy()[0]
        assert same(rxf, port.rrc_rx(cap, idx, len480)[0]), i                             # matched filter at the selected index
        c1, c2 = p["c1"].cpu().numpy()[0], p["c2"].cpu().numpy()[0]
        for got, want in ((c1, port.cfo_coarse(rxf)), (c2, port.cfo_fine(c1))):           # coarse, fine CFO
            a, b = check_cfo(got, want)
            ident += a; total += b
        ld = p["ld"].cpu().numpy()[0]
        assert same(ld, c2[160:])
        want_rx = port.rx_frames(ld, bits, n_sym)                                          # receiver on the GPU's input
        errs, evm_db = int(p["cnt"].bit_errors), p["res"][0]
        assert errs == int(want_rx["bit_errors"][0]), i
        assert evm_db == pytest.approx(float(want_rx["evm_db"][0]), abs=2e-3), i
        assert errs == e2e.bit_errors, i                                                  # the oracle's own path, end to end
        assert evm_db == pytest.approx(e2e.evm_db, abs=2e-3), i
        port_ber[i] = np.float32(e2e.bit_errors / (96 * n_sym))
        clean += errs == 0
        with_errors += errs > 0
        if errs == 0:
            words = p["rx_bits"].cpu().numpy().view(np.uint32)
            assert np.packbits(pkg.unpack_bits_host(words)[0]).tobytes()[:len(msg)] == msg.encode()
    assert checked >= 0.7 * SNR_COUNT and clean >= 3 and with_errors >= 1, (checked, clean, with_errors)
    assert ident >= 0.999 * total
    # the driver's default run writes the replay's values, byte for byte, in both arithmetic modes
    files = run_driver(msg, seed, "exact", tmp_path / "exact")
    assert files == driver_files(r)
    ber = files["Output_BER.txt"].rstrip("\n").split("\t")
    for i, b in port_ber.items():
        assert ber[i] == "%.2e" % float(b), (i, ber[i], b)
    fast = replay(ofdm, pkg, msg, seed, pkg.MODE_FAST)
    assert run_driver(msg, seed, "fast", tmp_path / "fast") == driver_files(fast)


KERNELS_SCRIPT = """
import json
import __graft_entry__ as entry
from test_gpu_routes import observe
from test_gpu_ota import replay
pkg = entry.load_pkg()
o = pkg.Ofdm(0)
msg = "The quick brown fox jumps over the lazy dog, and back again."
replay(o, pkg, msg, 3, pkg.MODE_EXACT)
kernels, launches, _ = observe(o, lambda: replay(o, pkg, msg, 3, pkg.MODE_EXACT))
print(json.dumps({"kernels": kernels, "launches": launches}))
"""


def test_driver_path_kernels():
    """the replay runs the driver's kernels: the exact power of the 14600-sample repeated waveform (not whole 16-sample chunks),
    the flat Philox channel, and packet detection on 4482-sample captures (two tiles); in a process of its own, as the other
    profiler tests"""
    here = os.path.dirname(os.path.abspath(__file__))
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([ROOT, here, os.environ.get("PYTHONPATH", "")]))
    r = subprocess.run([sys.executable, "-c", KERNELS_SCRIPT], cwd=here, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    got = json.loads(r.stdout.strip().splitlines()[-1])
    names = [k.split("<")[0] for k in got["kernels"] if k.startswith("k_")]        # without torch's own fills of fresh buffers
    assert got["launches"] == len(names)
    point = ["k_frame_power_exact", "k_awgn_philox_flat", "k_gather", "k_packet_detect", "k_packet_select", "k_rrc_rx", "k_cfo", "k_cfo",
             "k_gather"]
    first = names.index(point[0])
    assert names[first - 3:first] == ["k_prepend", "k_rrc_tx", "k_gather"], names
    per_point = names[first:]
    assert len(per_point) % SNR_COUNT == 0, names
    k = len(per_point) // SNR_COUNT
    for i in range(SNR_COUNT):
        assert per_point[i * k:i * k + len(point)] == point, per_point[i * k:(i + 1) * k]
