"""Host-side logic of a multi-GPU sweep: one process per GPU, frames sharded by global frame index,
one all-reduce of the per-SNR counters (the only exchange the path has -- SURVEY.md section 8(e)).
Works with any torch.distributed backend: nccl on the GPUs, gloo in the CPU tests."""
import ctypes as C
import math

import numpy as np

from .binding import Counters, COUNTERS_BYTES

N_INT_FIELDS = 5          # bit_errors, bits, frames_in_error, rail_errors, frames ; then 3 doubles


def shard_range(n_frames, rank, world):
    """Contiguous shard [lo, hi) of the global frame range for ``rank``; sizes differ by at most one."""
    base, rem = divmod(n_frames, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def counters_to_arrays(counters):
    """list of Counters -> (int64 [n,5], float64 [n,3])"""
    ints = np.array([[c.bit_errors, c.bits, c.frames_in_error, c.rail_errors, c.frames] for c in counters], dtype=np.int64)
    dbls = np.array([[c.sum_err2, c.sum_ref2, c.sum_evm_lin] for c in counters], dtype=np.float64)
    return ints.reshape(-1, 5), dbls.reshape(-1, 3)


def arrays_to_counters(ints, dbls):
    out = []
    for i, d in zip(np.asarray(ints), np.asarray(dbls)):
        c = Counters()
        c.bit_errors, c.bits, c.frames_in_error, c.rail_errors, c.frames = (int(x) for x in i)
        c.sum_err2, c.sum_ref2, c.sum_evm_lin = (float(x) for x in d)
        out.append(c)
    return out


def allreduce_counters(counters, device=None, group=None):
    """Sum a list of Counters over all ranks of the process group (integers exactly; doubles in rank order
    of the backend's reduction).  No-op without an initialised group."""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return counters
    ints, dbls = counters_to_arrays(counters)
    ti = torch.from_numpy(ints)
    td = torch.from_numpy(dbls)
    if device is not None:
        ti, td = ti.to(device), td.to(device)
    dist.all_reduce(ti, group=group)
    dist.all_reduce(td, group=group)
    return arrays_to_counters(ti.cpu().numpy(), td.cpu().numpy())


def allreduce_counter_tensor(t, group=None):
    """In-place all-reduce of a device counters tensor [n_snr, 8] (int64 view of ofdm_counters)."""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return t
    ints = t[:, :N_INT_FIELDS].contiguous()
    dist.all_reduce(ints, group=group)
    dbls = t[:, N_INT_FIELDS:].contiguous().view(torch.float64)
    dist.all_reduce(dbls, group=group)
    t[:, :N_INT_FIELDS] = ints
    t[:, N_INT_FIELDS:] = dbls.view(torch.int64)
    return t


def mc_sweep_sharded(ofdm, seed, n_frames_total, n_sym, snr_db, mode, rank=0, world=1, group=None):
    """configs[3]: Philox Monte-Carlo sweep over ``n_frames_total`` frames split across ``world`` ranks by
    global frame index (so the totals do not depend on the GPU count), counters all-reduced.  Returns the
    global per-SNR Counters on every rank."""
    lo, hi = shard_range(n_frames_total, rank, world)
    cnt = ofdm.new_counters(len(snr_db))
    ofdm.mc_sweep_philox(seed, lo, hi - lo, n_sym, snr_db, mode, counters=cnt)
    allreduce_counter_tensor(cnt, group)
    return ofdm.read_counters(cnt)


def until_loop(run_round, n_points, target_errors, max_bits, round_frames, rank=0, world=1, allreduce=None, frame0=0, max_rounds=None):
    """The stop rule of configs[3] over any number of ranks: every point runs until it has >= target_errors bit errors or
    >= max_bits bits.  Round r covers the global frames [frame0 + r * round_frames, + round_frames), split across the ranks
    by shard_range; ``run_round(points, lo, n)`` returns this rank's (int64 [len(points), 5], float64 [len(points), 3]) totals
    for the points still active on frames [lo, lo + n); ``allreduce(ints, dbls)`` sums them over the ranks (None: single
    rank).  Stop decisions are taken on the all-reduced totals at round boundaries, so every rank takes the same decisions
    and the result is the single-rank result (ofdm_mc_sweep_until) whatever the world size.  Returns (ints, dbls, rounds)."""
    ints = np.zeros((n_points, N_INT_FIELDS), np.int64)
    dbls = np.zeros((n_points, 3), np.float64)
    active = list(range(n_points))
    rounds = 0
    while active and (max_rounds is None or rounds < max_rounds):
        lo, hi = shard_range(round_frames, rank, world)
        pi, pd = run_round(active, frame0 + rounds * round_frames + lo, hi - lo)
        pi, pd = np.array(pi, dtype=np.int64).reshape(len(active), N_INT_FIELDS), np.array(pd, dtype=np.float64).reshape(len(active), 3)
        if allreduce is not None and world > 1:
            pi, pd = allreduce(pi, pd)
        ints[active] += pi
        dbls[active] += pd
        active = [i for i in active if ints[i, 0] < target_errors and ints[i, 1] < max_bits]
        rounds += 1
    return ints, dbls, rounds


def mc_sweep_until(ofdm, seed, n_sym, snr_db, mode, target_errors=100, max_bits=10 ** 9, round_frames=1 << 22, n_taps=0, rank=0, world=1,
                   group=None, frame0=0, noise="real", snr_def="frame_power"):
    """configs[3] as stated, on ``world`` GPUs: SNR points x frame ranges are sharded by rounds (every rank works on every
    still-active point, on its own slice of the round's frames -- so the slow high-SNR points use all GPUs), one all-reduce
    of the counters per round.  ``noise`` / ``snr_def`` choose the channel (binding.channel; the default is the reference's).
    Returns (list of global Counters, rounds) on every rank."""
    import torch
    import torch.distributed as dist
    snr = np.asarray(snr_db, dtype=np.float32)
    cnt = ofdm.new_counters(len(snr))

    def run_round(points, lo, n):
        c = cnt[:len(points)]
        c.zero_()
        if n > 0:
            ofdm.mc_sweep_channel(seed, lo, n, n_sym, snr[points], mode, noise, snr_def, n_taps, np.asarray(points, dtype=np.uint32), c)
        if world > 1:
            allreduce_counter_tensor(c, group)              # on the device: NCCL over NVLink
        raw = c.cpu().numpy()
        return raw[:, :N_INT_FIELDS].copy(), raw[:, N_INT_FIELDS:].copy().view(np.float64)

    ints, dbls, rounds = until_loop(run_round, len(snr), target_errors, max_bits, round_frames, rank, world, None, frame0)
    return arrays_to_counters(ints, dbls), rounds


def ber_table(snr_db, counters):
    rows = []
    for s, c in zip(snr_db, counters):
        ber = c.bit_errors / c.bits if c.bits else float("nan")
        evm = np.sqrt(c.sum_err2 / c.sum_ref2) if c.sum_ref2 else float("nan")
        rows.append((float(s), int(c.bit_errors), int(c.bits), ber, 20 * np.log10(evm) if evm > 0 else -np.inf, int(c.frames_in_error)))
    return rows


def qpsk_ber_awgn(snr_db, snr_def="esn0"):
    """BER of this project's QPSK map over an AWGN channel with perfect channel knowledge: the textbook curve to lay the
    measured one over.  snr_def "esn0" (Es/N0 per data subcarrier) or "ebn0" (Eb/N0 = Es/N0 / 2), as in binding.channel.

    Each rail is decided alone with error probability p = Q(sqrt(Es/N0)).  The map (QPSK_Modulator, OFDM.c:415-433:
    00 -> (+,+), 01 -> (-,+), 10 -> (-,-), 11 -> (+,-)) is not Gray coded: an I-rail error costs 1 bit, a Q-rail error 2 and
    both together 1, so BER = (p (1-p) + 2 p (1-p) + p^2) / 2 = (3p - 2p^2) / 2.

    The receiver does not know the channel: it estimates it from the two LTS halves, whose noise (half the variance of a data
    bin's) goes into every equalised point.  The measured curve therefore lies to the right of this one."""
    if snr_def not in ("esn0", "ebn0"):
        raise ValueError("qpsk_ber_awgn needs snr_def 'esn0' or 'ebn0', not %r (the frame-power SNR depends on the frame)" % (snr_def,))
    esn0 = 10.0 ** (np.asarray(snr_db, dtype=np.float64) / 10.0) * (2.0 if snr_def == "ebn0" else 1.0)
    p = 0.5 * np.vectorize(math.erfc)(np.sqrt(esn0 / 2.0))  # Q(x) = erfc(x / sqrt(2)) / 2
    return (3.0 * p - 2.0 * p * p) / 2.0
