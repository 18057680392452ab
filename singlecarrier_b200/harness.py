"""Loop-back harness: synthetic workloads of BASELINE.json configs 2-5 and BER / lock statistics.

The reference only has the ``FOFFSET`` macro and ``rand()`` data bits (src/qpsk.c:67,395); the
configs ask for frequency/phase offsets, AWGN sweeps, drift and 2-tap multipath over thousands of
streams (SURVEY.md section 8 row f-1).  Everything here is host-side orchestration: the samples are
synthesised by the library's TX/channel kernels and demodulated by its RX kernels; the statistics are
computed with torch ops on the device.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Optional

import numpy as np

from .modem import FRAME_SIZE, N_PACKET_BER_COUNTERS, REFERENCE_GAP, ModemBank, keystream_word
from .taps import modem_taps

PERIOD = FRAME_SIZE + REFERENCE_GAP          # 2783 samples: one packet + dead air (qpsk.c:384,405,410-412)
GROUP_DELAY = 48                             # TX RRC (24) + RX RRC (24) samples
# RMS of the real TX signal over the data section, i.e. of each component of the analytic one: +-1 QPSK
# symbols, one in five filter inputs, x 2.2 (fir.c:42) x 16384 (qpsk.c:319).  7,207 LSB for the default
# alpha = 0.35 taps; the alpha = 0.5 taps give 7,205.
DATA_RMS_LSB = 16384.0 * 2.2 * math.sqrt(float((modem_taps(0.35).astype(np.float64) ** 2).sum()) / 5.0)


@dataclass
class Workload:
    samples: "object"            # CUDA int16 [n_streams, samples_per_stream]
    tx_bits: "object"            # CUDA uint8 [n_streams, n_packets, 8, 62]
    lead: "object"               # CUDA int32 [n_streams]
    gap: int
    ebn0_db: Optional["object"]  # CUDA float [n_streams] or None
    n_packets: int
    channel: Optional[dict] = None   # the per-stream channel parameter tensors that were applied


def awgn_sigma(ebn0_db, torch):
    """Real AWGN: sigma^2 = P_sig * Fs / (2 * Rs * Es/N0), Es/N0 = 2 Eb/N0 (SURVEY section 8d)."""
    p_sig = DATA_RMS_LSB ** 2                 # power of the real passband signal = |analytic|^2 / 2 = rms_component^2
    esn0 = 2.0 * torch.pow(torch.tensor(10.0, device=ebn0_db.device), ebn0_db / 10.0)
    return torch.sqrt(p_sig * 8000.0 / (2.0 * 1600.0 * esn0)).float()


def synthesize(bank: ModemBank, samples_per_stream: int, seed: int, *, config: int, gap: int = REFERENCE_GAP,
               ebn0_db=None) -> Workload:
    """config 2: clean channel, random df/phase, lead-in 80+5m (preamble lands on decimated index m).
    config 3: + AWGN at ebn0_db[s] (default: 13 points 0..12 dB, striped by stream index).
    config 4: bench workload (config 3 channel, random lead-in).
    config 5: + linear drift (+-2 Hz/s) and a 2-tap echo (a 0.1..0.5, delay 1..10 samples) at 10 dB."""
    import torch
    dev = torch.device("cuda", bank.device)
    n = bank.n_streams
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    period = FRAME_SIZE + gap
    n_packets = max(1, (samples_per_stream + period - 1) // period)
    if config == 2:
        lead = (80 + 5 * torch.randint(0, 101, (n,), generator=g, device=dev)).int()
    else:
        lead = torch.randint(0, period, (n,), generator=g, device=dev, dtype=torch.int32)
    ch = {"df_hz": (torch.rand(n, generator=g, device=dev) * 40.0 - 20.0).float(),
          "phi_rad": (torch.rand(n, generator=g, device=dev) * (2 * math.pi)).float()}
    eb = None
    if config in (3, 4, 5):
        if ebn0_db is not None:
            eb = ebn0_db.float().to(dev)
        elif config == 5:
            eb = torch.full((n,), 10.0, device=dev)
        else:
            eb = (torch.arange(n, device=dev) % 13).float()
        ch["sigma_lsb"] = awgn_sigma(eb, torch)
    if config == 5:
        ch["drift_hz_s"] = (torch.rand(n, generator=g, device=dev) * 4.0 - 2.0).float()
        ch["echo_amp"] = (0.1 + 0.4 * torch.rand(n, generator=g, device=dev)).float()
        ch["echo_theta"] = (torch.rand(n, generator=g, device=dev) * (2 * math.pi)).float()
        ch["echo_delay"] = torch.randint(1, 11, (n,), generator=g, device=dev, dtype=torch.int32)
    out = torch.empty((n, samples_per_stream), dtype=torch.int16, device=dev)
    bits = torch.empty((n, n_packets, 8, 62), dtype=torch.uint8, device=dev)
    bank.tx_packets_dev(out, n_packets, gap_samples=gap, seed=seed, bits_out=bits, lead_in=lead, channel=ch)
    torch.cuda.synchronize(dev)
    return Workload(out, bits, lead, gap, eb, n_packets, ch)


def demodulate(bank: ModemBank, samples, n_frames: int):
    """Cold-start RX of the whole bank on the device; returns a CUDA uint8 tensor viewable as RESULT_DTYPE."""
    import torch
    res = torch.zeros((bank.n_streams, n_frames * 32), dtype=torch.uint8, device=samples.device)
    bank.reset()
    bank.rx_frames_dev(samples, n_frames, res)
    torch.cuda.synchronize(samples.device)
    return res


def ber_and_lock(res, n_frames: int, wl: Workload, group=None, n_groups: int = 1):
    """Bit errors of the 62 decided bits of every valid call against the transmitted bits, and lock counts.

    A valid call n found its preamble at decimated index max_index of the window taken from frame n-2
    with timing rx_timing(n-1); that is filtered sample (n-2)*1880 + 5*max_index + T, which is packet
    j = round((that - 48 - lead) / period).  The decoded symbols are the first 31 data symbols of packet j
    (SURVEY F5).  TX does not scramble (qpsk.c:397) but RX descrambles, so decided = bits ^ keystream(n).
    Returns dict of numpy arrays per group: calls, valid, bits, errors, preambles (packets wholly inside).
    """
    import torch
    dev = res.device
    n = res.shape[0]
    r = res.view(n, n_frames, 32)
    lo = r[:, :, 0:4].contiguous().view(torch.int32).view(n, n_frames).long() & 0xffffffff
    hi = r[:, :, 4:8].contiguous().view(torch.int32).view(n, n_frames).long() & 0xffffffff
    bits = lo | (hi << 32)
    i16 = r[:, :, 16:22].contiguous().view(torch.int16).view(n, n_frames, 3).long()
    max_index, rx_timing = i16[:, :, 0], i16[:, :, 2]
    valid = r[:, :, 22] != 0
    calls = torch.arange(n_frames, device=dev).view(1, -1).expand(n, -1)
    t_prev = torch.cat([torch.full((n, 2), 128, device=dev, dtype=torch.long), rx_timing[:, :-2]], dim=1)
    # timing used to decimate the searched window = rx_timing at entry of call n-1 = value after call n-2
    pos = (calls - 2) * FRAME_SIZE + 5 * max_index + t_prev - GROUP_DELAY - wl.lead.long().view(-1, 1)
    period = FRAME_SIZE + wl.gap
    pkt = torch.div(pos + period // 2, period, rounding_mode="floor")
    ok = valid & (calls >= 2) & (pkt >= 0) & (pkt < wl.n_packets) & ((pos - pkt * period).abs() <= 10)
    pk = pkt.clamp(0, wl.n_packets - 1)
    txb = wl.tx_bits[:, :, 0, :].long()                                       # first data frame of each packet
    weights = (1 << torch.arange(62, device=dev, dtype=torch.long))
    tx_words = (txb * weights).sum(-1)                                         # [n, n_packets]
    tx_sel = torch.gather(tx_words, 1, pk)
    ks = torch.tensor([keystream_word(c) for c in range(n_frames)], device=dev, dtype=torch.long).view(1, -1)
    diff = (bits ^ ks ^ tx_sel) & ((1 << 62) - 1)
    errs = torch.zeros_like(diff)
    for b in range(62):
        errs += (diff >> b) & 1
    if group is None:
        group = torch.zeros(n, device=dev, dtype=torch.long)
    out = {k: np.zeros(n_groups, np.int64) for k in ("calls", "valid", "aligned", "bits", "errors")}
    for gi in range(n_groups):
        m = (group == gi).view(-1, 1)
        out["calls"][gi] = int((m & (calls >= 2)).sum())
        out["valid"][gi] = int((m & valid & (calls >= 2)).sum())
        out["aligned"][gi] = int((m & ok).sum())
        out["bits"][gi] = 62 * out["aligned"][gi]
        out["errors"][gi] = int((errs * (m & ok)).sum())
    return out


def ber_and_lock_dev(bank: ModemBank, res, n_frames: int, wl: Workload, group=None, n_groups: int = 1, comm=None):
    """The same statistics as ber_and_lock(), computed by one kernel (sc_ber_stats_dev) and, when ``comm`` (an
    NcclComm) is given, summed over all ranks with sc_reduce_stats -- the form a multi-GPU caller uses."""
    import torch
    cnt = torch.zeros((n_groups, 8), dtype=torch.int64, device=res.device)
    g = None if group is None else group.to(torch.int32).contiguous()
    bank.ber_stats(res, n_frames, wl.tx_bits, wl.lead, wl.gap, cnt, group=g, n_groups=n_groups)
    if comm is not None:
        comm.all_reduce_counters(cnt)
    torch.cuda.synchronize(res.device)
    c = cnt.cpu().numpy()
    return {name: c[:, k].copy() for k, name in enumerate(("calls", "valid", "aligned", "bits", "errors"))}


def packet_counters(c) -> dict:
    """Named views of sc_packet_ber_stats_dev's counters (int64 [n_groups, 32])."""
    c = np.asarray(c)
    return {"records": c[:, 0].copy(), "aligned": c[:, 1].copy(), "bits": c[:, 2].copy(), "errors": c[:, 3].copy(),
            "frame_errors": c[:, 8:16].copy(), "frames_in_error": c[:, 16:24].copy(),
            "error_histogram": c[:, 24:32].copy()}


def packet_ber_dev(bank: ModemBank, packets, n_found, res, n_frames: int, wl: Workload, group=None, n_groups: int = 1,
                   comm=None):
    """The packet counterpart of ber_and_lock_dev: bit errors of the packet records that rx_packets_dev left in
    ``packets`` / ``n_found`` (sc_packet_ber_stats_dev), summed over all ranks with sc_reduce_stats when ``comm`` is
    given.  Returns numpy arrays per group: records, aligned, bits, errors, frame_errors [n_groups, 8],
    frames_in_error [n_groups, 8] and error_histogram [n_groups, 8] (bins 0 | 1 | 2-3 | ... | 32-63 | >= 64)."""
    import torch
    cnt = torch.zeros((n_groups, N_PACKET_BER_COUNTERS), dtype=torch.int64, device=res.device)
    g = None if group is None else group.to(torch.int32).contiguous()
    bank.packet_ber_stats(packets, n_found, res, n_frames, wl.tx_bits, wl.lead, wl.gap, cnt, group=g,
                          n_groups=n_groups)
    if comm is not None:
        comm.all_reduce_counters(cnt)
    torch.cuda.synchronize(res.device)
    return packet_counters(cnt.cpu().numpy())
