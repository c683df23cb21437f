#!/usr/bin/env python
"""Search for the dealing of a frame's 96 data bins to (round, half-warp, lane) that minimises shared-memory bank conflicts of
the item loads of the fused receivers (csrc/ofdm_chain.cuh: c_deal_bin; `deal_search.py sweep`: c_sweep_pair / c_sweep_single of
csrc/ofdm_sweep.cuh, where each lane takes both symbols of one bin plus one single item).  Model: 64-bit loads, one half-warp per wavefront,
bank pair = element index mod 16; LTS tiles at element offsets 288 / 360, symbol tiles at 0 / 72 (72 = 8 mod 16)."""
import random
from collections import defaultdict

C = list(range(6, 11)) + list(range(12, 25)) + list(range(26, 32)) + list(range(33, 39)) + list(range(40, 53)) + list(range(54, 59))
DATA_BIN = [(x + 32) % 64 for x in C]          # data index -> natural FFT bin


def wavefronts(elems):
    m = defaultdict(set)
    for e in elems:
        m[e % 16].add(e)
    return max(len(v) for v in m.values())


def group_cost(items):                          # 16 x (bin, symbol)
    a = [288 + b for b, s in items]
    b_ = [360 + b for b, s in items]
    f = [s * 72 + b for b, s in items]
    return wavefronts(a) - 1 + wavefronts(b_) - 1 + wavefronts(f) - 1


def total(groups):
    return sum(group_cost([(b, 0) for b in g] + [(b, 1) for b in g]) for g in groups)


def main():
    in_order = [[(DATA_BIN[(hw * 16 + l + 32 * r) % 48], (hw * 16 + l + 32 * r) // 48) for l in range(16)] for r in range(3) for hw in range(2)]
    print("data indices in order:", sum(group_cost(g) for g in in_order), "extra wavefronts per frame")
    random.seed(1)
    bins = list(DATA_BIN)
    random.shuffle(bins)
    groups = [bins[8 * k:8 * k + 8] for k in range(6)]
    cur = total(groups)
    for _ in range(400000):
        a, b = random.sample(range(6), 2)
        i, j = random.randrange(8), random.randrange(8)
        groups[a][i], groups[b][j] = groups[b][j], groups[a][i]
        t = total(groups)
        if t <= cur:
            cur = t
        else:
            groups[a][i], groups[b][j] = groups[b][j], groups[a][i]
        if cur <= 1:
            break
    print("8 bins x both symbols per half-warp:", cur, "extra wavefronts per frame")
    for g in groups:
        print("   ", ", ".join("%2d" % b for b in sorted(g)))


def sweep_cost(pairs, singles):
    c = 0
    for g in pairs:                             # 16 lanes, both symbols of one bin each: LTS A, LTS B, symbol 0, symbol 1 loads
        c += 4 * (wavefronts(g) - 1)
    for g in singles:                           # lanes 0..7 symbol 0, lanes 8..15 symbol 1 of the same 8 bins
        c += 2 * (wavefronts(g) - 1) + wavefronts(g + [72 + b for b in g]) - 1
    return c


def sweep():
    """k_sweep_lin: per half-warp 16 pair bins (both symbols, one channel estimate) and 8 single bins (symbol 0 on lanes 0..7,
    symbol 1 on lanes 8..15).  The pair bins can be made conflict-free; residues 2 and 10 mod 16 hold three single items each,
    so one extra wavefront per frame is the least possible.  Local search with restarts."""
    for seed in range(1000):
        random.seed(seed)
        bins = list(DATA_BIN)
        random.shuffle(bins)
        groups = [bins[0:16], bins[16:32], bins[32:40], bins[40:48]]
        cur = sweep_cost(groups[:2], groups[2:])
        for _ in range(20000):
            a, b = random.sample(range(4), 2)
            i, j = random.randrange(len(groups[a])), random.randrange(len(groups[b]))
            groups[a][i], groups[b][j] = groups[b][j], groups[a][i]
            t = sweep_cost(groups[:2], groups[2:])
            if t <= cur:
                cur = t
            else:
                groups[a][i], groups[b][j] = groups[b][j], groups[a][i]
            if cur <= 1:
                break
        if cur <= 1:
            break
    print("sweep: pairs + singles per half-warp:", cur, "extra wavefronts per frame (seed %d)" % seed)
    for name, g in zip(("pairs hw0", "pairs hw1", "singles hw0", "singles hw1"), groups):
        print("   ", name, ", ".join("%2d" % b for b in sorted(g)))


if __name__ == "__main__":
    import sys
    sweep() if sys.argv[1:] == ["sweep"] else main()
