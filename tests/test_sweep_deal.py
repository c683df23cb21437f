"""The dealing of a frame's 96 data items over the lanes of k_sweep_lin (csrc/ofdm_sweep.cuh, c_sweep_pair / c_sweep_single,
make_sweep_items), checked without a GPU: every data bin of both symbols is owned by exactly one (lane, item), items 0 and 1
of a lane are the two symbols of one subcarrier (they share its channel estimate), the payload word and shift select the
item's bit pair as pack_bits_host lays the frame's 192 bits out (bit j at word j >> 5, position j & 31: symbol s, data
index d -> bits 96 s + 2 d, + 1), and the item loads from the exchange tiles cost one extra shared-memory wavefront per frame."""
import os
import re
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_quad_tables import tables  # noqa: E402  (the reference's data map, restated from OFDM.c)

SRC = os.path.join(ROOT, "ieee-802.11-ofdm-qpsk-simulator_b200", "csrc", "ofdm_sweep.cuh")


def deal():
    src = open(SRC).read()

    def table(name, n):
        m = re.search(r"__constant__ unsigned char %s\[%d\] = \{([^}]*)\};" % (name, n), src)
        assert m, name
        vals = [int(x) for x in m.group(1).replace("\n", " ").split(",")]
        assert len(vals) == n
        return vals

    return table("c_sweep_pair", 32), table("c_sweep_single", 16)


def items(lane, pair, single):
    """make_sweep_items: (bin, symbol) of items 0, 1, 2"""
    bins = [pair[lane], single[(lane >> 4) * 8 + (lane & 7)]]
    return [(bins[t >> 1], (lane >> 3) & 1 if t == 2 else t) for t in range(3)]


def test_every_data_item_has_one_owner_and_its_word_and_shift():
    bin_data, bin_lts = tables()
    pair, single = deal()
    owned = {}
    for lane in range(32):
        its = items(lane, pair, single)
        assert its[0][0] == its[1][0] and (its[0][1], its[1][1]) == (0, 1)     # one subcarrier, both symbols
        for t, (p, sym) in enumerate(its):
            d = bin_data[p]
            assert d >= 0 and bin_lts[p] != 0, (lane, t, p)
            assert (p, sym) not in owned, (lane, t, p, sym)
            owned[(p, sym)] = (lane, t)
            word, shift = sym * 3 + (d >> 4), 2 * (d & 15)                         # what make_sweep_items computes
            j = 96 * sym + 2 * d
            assert (word, shift) == (j >> 5, j & 31) and shift <= 30
    data = [p for p in range(64) if bin_data[p] >= 0]
    assert len(data) == 48 and sorted(owned) == sorted((p, s) for p in data for s in (0, 1))


def test_item_loads_are_bank_conflict_free_but_one_wavefront():
    """64-bit loads, one half-warp per wavefront, bank pair = element index mod 16; the symbol tiles are kWin = 72 elements apart"""
    pair, single = deal()

    def extra(elems):
        by_bank = {}
        for e in elems:
            by_bank.setdefault(e % 16, set()).add(e)
        return max(len(v) for v in by_bank.values()) - 1

    total = 0
    for hw in range(2):
        lanes = range(16 * hw, 16 * hw + 16)
        its = [items(lane, pair, single) for lane in lanes]
        pair_bins = [it[0][0] for it in its]
        assert extra(pair_bins) == 0                        # the LTS tiles and both symbol tiles, estimate 0
        total += extra([it[2][0] for it in its])            # LTS tiles, estimate 1 (8 bins, each read by two lanes)
        total += extra([72 * it[2][1] + it[2][0] for it in its])
    assert total == 1


def test_the_header_states_the_same_dealing():
    """make_sweep_items is the restatement's source: keep them in step"""
    src = open(SRC).read()
    assert "c.bin[0] = c_sweep_pair[lane];" in src
    assert "c.bin[1] = c_sweep_single[(lane >> 4) * 8 + (lane & 7)];" in src
    assert "const int bin = c.bin[t >> 1], sym = t == 2 ? (lane >> 3) & 1 : t;" in src
    assert "c.word[t] = sym * 3 + (d >> 4);" in src and "c.shift[t] = 2 * (d & 15);" in src
