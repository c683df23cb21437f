"""The CPU side of the over-the-air path tests (tests/ota_oracle.c): the flat Philox layout of k_awgn_philox_flat against the raw
Philox blocks and against the LTS||data layout of the other channels, the driver's bookkeeping restated in Python, and the
oracle's whole path on its own draws.  No GPU needed."""
import numpy as np
import pytest

from ota_oracle import DOMAIN_FLAT, OtaOracle, capture_starts, encode_message, lengths

SEED = 23


@pytest.fixture(scope="module")
def oo():
    return OtaOracle()


def philox(oo, ctr, key):
    import ctypes as C
    c, k, o = (C.c_uint32 * 4)(*ctr), (C.c_uint32 * 2)(*key), (C.c_uint32 * 4)()
    oo.lib.orc_philox4x32_10(c, k, o)
    return list(o)


def box_muller64(r):
    """float64 Box-Muller of one block's four words, with the uniforms formed as the oracle forms them in float32"""
    z = []
    for h in range(2):
        u1 = np.float32(np.float32(r[2 * h]) * np.float32(2.0 ** -32) + np.float32(2.0 ** -33))
        u2 = np.float32(np.float32(r[2 * h + 1]) * np.float32(2.0 ** -32))
        rad = np.sqrt(-2.0 * np.log(np.float64(u1)))
        ang = 2.0 * np.pi * np.float64(u2)
        z += [rad * np.cos(ang), rad * np.sin(ang)]
    return np.array(z)


@pytest.mark.parametrize("frame0", [0, 7, (1 << 32) - 2])
def test_flat_layout_is_four_consecutive_samples_per_block(oo, frame0):
    """block b = samples 4b .. 4b+3, counter (frame_lo, frame_hi, b, 3), key (seed, stream); a tail shorter than a block takes
    the block's first normals"""
    stream, n_frames, length = 9, 4, 4097
    g = oo.philox_normals_flat(SEED, stream, frame0, n_frames, length)
    for f in range(n_frames):
        fr = frame0 + f
        for b in (0, 1, 511, 1023, 1024):
            r = philox(oo, [fr & 0xFFFFFFFF, fr >> 32, b, DOMAIN_FLAT], [SEED, stream])
            want = box_muller64(r)[: min(4, length - 4 * b)]
            assert np.max(np.abs(g[f, 4 * b: 4 * b + 4] - want)) < 1e-5, (f, b)
    # frame f of an n-frame call is a one-frame call at frame0 + f; a longer buffer only appends samples
    for f in range(n_frames):
        assert np.array_equal(g[f], oo.philox_normals_flat(SEED, stream, frame0 + f, 1, length)[0])
    assert np.array_equal(g, oo.philox_normals_flat(SEED, stream, frame0, n_frames, 4100)[:, :length])


@pytest.mark.parametrize("domain", [0, 3, 4])
@pytest.mark.parametrize("n_sym", [1, 2, 5])
def test_flat_and_frame_layouts_share_the_philox_blocks(oo, domain, n_sym):
    """sample n of an LTS||data frame (noise_slot: block blk, normal j) is sample 4 blk + j of the flat layout of the same
    (seed, stream, frame, domain): the two layouts deal out the same Philox blocks, and the guard / CP samples (consecutive
    quadruples) sit at the same place in both"""
    length = 160 + 80 * n_sym
    slots = [oo.noise_slot(n) for n in range(length)]
    flat_len = 4 * (max(b for b, _ in slots) + 1)
    frame0 = (1 << 32) - 1
    framed = oo.philox_normals(SEED, 3, frame0, 2, length, domain)
    flat = oo.philox_normals_flat(SEED, 3, frame0, 2, flat_len, domain)
    pos = np.array([4 * b + j for b, j in slots])
    assert len(set(pos.tolist())) == length                                         # every sample has a slot of its own
    assert np.array_equal(framed, flat[:, pos])
    assert np.array_equal(framed[:, :32], flat[:, :32])
    for s in range(n_sym):
        cp = 160 + 80 * s
        b0 = slots[cp][0]
        assert np.array_equal(framed[:, cp:cp + 16], flat[:, 4 * b0: 4 * b0 + 16])


def test_driver_bookkeeping():
    """the message codec and the buffer lengths of host/ofdm_main.c, and the capture starts of the C library's rand()"""
    bits, n_sym = encode_message("Hey! I am Vivaswan")
    want = np.unpackbits(np.frombuffer(b"Hey! I am Vivaswan      ", np.uint8))
    assert n_sym == 2 and np.array_equal(bits, want)
    assert encode_message("")[1] == 1 and encode_message("x" * 12)[1] == 1 and encode_message("x" * 13)[1] == 2
    assert np.array_equal(encode_message("A")[0][:16], [0, 1, 0, 0, 0, 0, 0, 1, 0, 0, 1, 0, 0, 0, 0, 0])    # 'A' then ' '
    assert [lengths(n)[3:] for n in (1, 2, 5, 39)] == [(8200, 2517), (9800, 3008), (14600, 4482), (69000, 21183)]
    a, b = capture_starts(5, 30, 9800, 3008), capture_starts(5, 30, 9800, 3008)
    assert a == b and all(0 <= s < 9800 - 3008 for s in a) and len(set(a)) > 20
    assert capture_starts(6, 30, 9800, 3008) != a


def test_whole_path_on_the_oracles_draws(oo):
    """the oracle's own path finds the packet and decodes a clean point, and not a noisy one"""
    bits, n_sym = encode_message("Hey! I am Vivaswan")
    _, len480, _, len_rep, len_cap = lengths(n_sym)
    full, shaped, rep = oo.waveform(bits, n_sym)
    assert full.shape == (len480, 2) and rep.shape == (len_rep, 2) and np.array_equal(rep[len_rep // 10:2 * len_rep // 10], shaped)
    g = oo.philox_normals_flat(SEED, 0, 0, 1, len_rep)[0]
    idx, st = oo.ota_point(rep, g, 40.0, 100, len_cap, bits, n_sym)
    assert 0 < idx and idx + 2 * (len480 - 1) < len_cap + 20
    assert st.bit_errors == 0 and st.evm_db < -20
    _, st = oo.ota_point(rep, g, -5.0, 100, len_cap, bits, n_sym)
    assert st.bit_errors > 0
