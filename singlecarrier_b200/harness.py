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

from .modem import (FRAME_SIZE, N_PACKET_BER_COUNTERS, PACKET_CODED_BITS, PACKET_DTYPE, PAYLOAD_BYTES, PAYLOAD_DTYPE,
                    PAYLOAD_EX_DTYPE, PAYLOAD_MAX, REFERENCE_GAP, ModemBank, keystream_word, payload_bytes)
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
    payload: Optional["object"] = None   # CUDA uint8 [n_streams, n_packets, 27] when the packets carry coded payloads
    stream_code: Optional["object"] = None   # CUDA uint8 [n_streams] with per-stream code rates (payload [.., 41])
    packet_code: Optional["object"] = None   # CUDA uint8 [n_streams, n_packets] with per-packet code rates (the same)


def awgn_sigma(ebn0_db, torch):
    """Real AWGN: sigma^2 = P_sig * Fs / (2 * Rs * Es/N0), Es/N0 = 2 Eb/N0 (SURVEY section 8d)."""
    p_sig = DATA_RMS_LSB ** 2                 # power of the real passband signal = |analytic|^2 / 2 = rms_component^2
    esn0 = 2.0 * torch.pow(torch.tensor(10.0, device=ebn0_db.device), ebn0_db / 10.0)
    return torch.sqrt(p_sig * 8000.0 / (2.0 * 1600.0 * esn0)).float()


def synthesize(bank: ModemBank, samples_per_stream: int, seed: int, *, config: int, gap: int = REFERENCE_GAP,
               ebn0_db=None, payload=None, stream_code=None, packet_code=None) -> Workload:
    """config 2: clean channel, random df/phase, lead-in 80+5m (preamble lands on decimated index m).
    config 3: + AWGN at ebn0_db[s] (default: 13 points 0..12 dB, striped by stream index).
    config 4: bench workload (config 3 channel, random lead-in).
    config 5: + linear drift (+-2 Hz/s) and a 2-tap echo (a 0.1..0.5, delay 1..10 samples) at 10 dB.
    payload: None (random bits), or CUDA uint8 [n_streams, n_packets, 27]: the packets carry these payloads through the
    packet code (sc_packet_encode_dev); n_packets must be the number the stream's length gives.
    stream_code: None, or CUDA uint8 [n_streams]: each stream's code rate; payload is then [n_streams, n_packets, 41]
    and goes through sc_packet_encode_ex_dev.
    packet_code: None, or CUDA uint8 [n_streams, n_packets]: each packet's code rate (not with stream_code); payload is
    [n_streams, n_packets, 41] and goes through sc_packet_encode_ex_dev with one packet per stream."""
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
    if payload is None:
        bank.tx_packets_dev(out, n_packets, gap_samples=gap, seed=seed, bits_out=bits, lead_in=lead, channel=ch)
    else:
        assert stream_code is None or packet_code is None, "stream_code and packet_code are exclusive"
        width = PAYLOAD_BYTES if stream_code is None and packet_code is None else PAYLOAD_MAX
        assert tuple(payload.shape) == (n, n_packets, width) and payload.dtype == torch.uint8, "payload shape"
        payload = payload.to(dev).contiguous()
        if stream_code is not None:
            stream_code = stream_code.to(dev, torch.uint8).contiguous()
            assert stream_code.numel() == n, "stream_code shape"
            bank.packet_encode_ex(payload, stream_code, bits)
        elif packet_code is not None:
            packet_code = packet_code.to(dev, torch.uint8).contiguous()
            assert tuple(packet_code.shape) == (n, n_packets), "packet_code shape"
            # each packet a stream of its own: the bits land in the [n_streams][n_packets][8][62] layout all the same
            bank.packet_encode_ex(payload.view(n * n_packets, 1, PAYLOAD_MAX), packet_code.view(-1), bits)
        else:
            bank.packet_encode(payload, bits)
        bank.tx_packets_dev(out, n_packets, gap_samples=gap, seed=seed, bits=bits, lead_in=lead, channel=ch)
    torch.cuda.synchronize(dev)
    return Workload(out, bits, lead, gap, eb, n_packets, ch, payload, stream_code, packet_code)


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


def _host(x):
    return x.cpu().numpy() if hasattr(x, "cpu") else np.asarray(x)


def _packed_words(tx_bits, chunk: int = 8192):
    """uint8 [n, n_packets, 8, 62] of 0/1 -> uint64 [n, n_packets, 8], bit k of word f = bit k of frame f"""
    n = tx_bits.shape[0]
    out = np.zeros(tuple(tx_bits.shape[:3]), np.uint64)
    for a in range(0, n, chunk):
        t = _host(tx_bits[a:a + chunk])
        t = np.concatenate([t, np.zeros(t.shape[:3] + (2,), np.uint8)], axis=-1)
        out[a:a + chunk] = np.packbits(t, axis=-1, bitorder="little").view("<u8")[..., 0]
    return out


def packet_fec(packets, n_found: int, decoded, res, n_frames: int, wl: Workload, group=None, n_groups: int = 1):
    """Host recount of the coded payloads of packet records against the workload's payloads (wl.payload).

    packets: the records (PACKET_DTYPE, or the CUDA uint8 buffer rx_packets_*_dev filled), n_found: their number (the
    first min(n_found, capacity) are counted), decoded: the matching sc_packet_payload records (PAYLOAD_DTYPE or a
    CUDA uint8 buffer), res: the batch's results (CUDA uint8 [n_streams, >= n_frames * 32] or RESULT_DTYPE).
    Records are counted and aligned to transmitted packet j by the rule of sc_packet_ber_stats_dev (grid_sample when it
    is not 0, else call index, max_index and rx_timing).  Returns numpy int64 arrays per group: records, aligned,
    crc_ok (aligned records whose CRC checks), correct (aligned, crc_ok and the payload transmitted), undetected
    (aligned, crc_ok and another payload), raw_errors (hard-decision errors over the coded bits 0..475 of aligned
    records) and raw_packet_errors (aligned records with at least one).

    A workload with per-stream codes (wl.stream_code) takes the sc_packet_payload_ex records (PAYLOAD_EX_DTYPE) of
    sc_packet_decode_ex_dev: the payloads compare over the first payload_bytes(code) bytes, raw errors count over the
    code's N transmitted positions only, and payload_bytes (the sum of the payload bytes of correct records) is added.

    A workload with per-packet codes (wl.packet_code, records of sc_packet_decode_blind_dev) does the same with the
    code of the aligned packet j; correct also needs the record's code to be that code, and wrong_code (aligned records
    whose CRC passes at another code, counted in undetected as well) is added."""
    assert wl.payload is not None, "the workload carries no coded payload"
    per_packet = wl.packet_code is not None
    coded = wl.stream_code is not None or per_packet
    pay = _host(wl.payload).reshape(-1, wl.n_packets, PAYLOAD_MAX if coded else PAYLOAD_BYTES)
    pk = _host(packets).view(PACKET_DTYPE).reshape(-1)
    dec = _host(decoded).view(PAYLOAD_EX_DTYPE if coded else PAYLOAD_DTYPE).reshape(-1)
    kept = min(int(n_found), pk.size, dec.size)
    pk, dec = pk[:kept], dec[:kept]
    s, j, ok, al = packet_alignment(pk, kept, res, n_frames, wl)
    grp = np.zeros(pay.shape[0], np.int64) if group is None else _host(group).astype(np.int64)
    g = grp[s]
    ok &= (g >= 0) & (g < n_groups)
    al &= ok
    crc = dec["crc_ok"] != 0
    # hard decisions against the transmitted bits, packed like the records' words (bit k of word f = bit 62 f + k)
    txw = _packed_words(wl.tx_bits)[s, j]
    if coded:
        code = _host(wl.packet_code).astype(np.int64)[s, j] if per_packet else _host(wl.stream_code).astype(np.int64)[s]
        n_bytes = np.array([payload_bytes(c) for c in range(256)], np.int64)[code]
        same = ((dec["data"] == pay[s, j]) | (np.arange(PAYLOAD_MAX) >= n_bytes[:, None])).all(axis=1)
        mask = coded_position_masks()[np.minimum(code, 3)]
        if per_packet:
            wrong = dec["code"].astype(np.int64) != code
            same &= ~wrong
    else:
        same = (dec["data"] == pay[s, j]).all(axis=1)
        mask = np.array([(1 << 62) - 1] * 7 + [(1 << (PACKET_CODED_BITS - 7 * 62)) - 1], np.uint64)
    raw = np.bitwise_count((pk["bits"] ^ txw) & mask).sum(axis=1).astype(np.int64)
    names = ("records", "aligned", "crc_ok", "correct", "undetected", "raw_errors", "raw_packet_errors")
    names += (("payload_bytes",) if coded else ()) + (("wrong_code",) if per_packet else ())
    out = {k: np.zeros(n_groups, np.int64) for k in names}
    rows = [("records", ok, None), ("aligned", al, None), ("crc_ok", al & crc, None),
            ("correct", al & crc & same, None), ("undetected", al & crc & ~same, None),
            ("raw_errors", al, raw), ("raw_packet_errors", al & (raw > 0), None)]
    if coded:
        rows.append(("payload_bytes", al & crc & same, n_bytes))
    if per_packet:
        rows.append(("wrong_code", al & crc & wrong, None))
    for name, m, w in rows:
        np.add.at(out[name], g[m], 1 if w is None else w[m])
    return out


def packet_alignment(packets, n_found: int, res, n_frames: int, wl: Workload):
    """The rule of sc_packet_ber_stats_dev for the first min(n_found, len) packet records: their stream s and packet j
    (int64, both 0 and clipped into range where not counted), counted (a stream in range and a call 2..n_frames-1) and
    aligned (counted, and within +-10 samples of packet j of its stream; j from grid_sample when it is not 0, else from
    call index, max_index and rx_timing)."""
    pk = _host(packets).view(PACKET_DTYPE).reshape(-1)
    pk = pk[:min(int(n_found), pk.size)]
    n_streams = wl.tx_bits.shape[0]
    r = _host(res)
    timing = r.view(np.uint8).reshape(n_streams, -1, 32)[:, :, 20:22].copy().view("<i2")[..., 0].astype(np.int64)
    lead = _host(wl.lead).astype(np.int64)
    s = pk["stream"].astype(np.int64)
    n = pk["call_index"].astype(np.int64)
    ok = (s >= 0) & (s < n_streams) & (n >= 2) & (n < n_frames)
    s, n = np.where(ok, s, 0), np.where(ok, n, 2)
    gs = pk["grid_sample"].astype(np.int64)
    pos = np.where(gs != 0, gs, (n - 2) * FRAME_SIZE + 5 * pk["max_index"].astype(np.int64) + timing[s, n - 2]) \
        - GROUP_DELAY - lead[s]
    period = FRAME_SIZE + wl.gap
    j = np.floor_divide(pos + period // 2, period)
    al = ok & (j >= 0) & (j < wl.n_packets) & (np.abs(pos - j * period) <= 10)
    return s, np.clip(j, 0, wl.n_packets - 1), ok, al


def coded_position_masks() -> np.ndarray:
    """uint64 [4, 8]: row c (code 0..2) has the packet bit positions pi(n), n < N(c), that carry transmitted bits, in
    the records' word layout (bit k of word f = bit 62 f + k); row 3 (any other code) is empty."""
    out = np.zeros((4, 8), np.uint64)
    for c, n_coded in enumerate((476, 465, 467)):
        for n in range(n_coded):
            p = 17 * (n % 28) + n // 28
            out[c, p // 62] |= np.uint64(1 << (p % 62))
    return out
