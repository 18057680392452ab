"""GPU: the loop-back channel generator (sc_tx_channel_dev) against the float64 reference of oracle/channel_ref.py,
and the bit-error counters (sc_ber_stats_dev, harness.ber_and_lock) against a plain loop on hand-made records.

Comparison rule for the channel: with y the reference before rounding, the device output must equal rint(y)
wherever |frac(y) - 1/2| > 0.05, and may differ from it by at most 1 LSB inside that band.  The kernel's float32
work is the echo product, sincospif of a float32 phase in [0, 2) (the phase itself is kept in cycles in double),
and Box-Muller in float32; at |y| < 40,000 together they stay below ~0.03 LSB, so only samples whose exact value
lies within 0.05 of a rounding boundary may round the other way.
"""
import numpy as np
import pytest

from oracle import channel_ref as cr

pytestmark = pytest.mark.gpu

BAND = 0.05
_tally = {"samples": 0, "in_band": 0, "max_abs_diff": 0}


@pytest.fixture(scope="module")
def sc():
    import singlecarrier_b200 as m
    assert m.lib.sc_device_count() > 0
    return m


@pytest.fixture(scope="module", autouse=True)
def band_report():
    yield
    print(f"\nchannel vs float64 reference: {_tally['samples']} samples compared, {_tally['in_band']} inside the "
          f"+-{BAND} rounding band, largest |difference| {_tally['max_abs_diff']} LSB")


def assert_matches(got, y, what=""):
    got = np.asarray(got).astype(np.int64)
    want = np.rint(y).astype(np.int64)
    band = np.abs(y - np.floor(y) - 0.5) <= BAND
    diff = got - want
    _tally["samples"] += got.size
    _tally["in_band"] += int(band.sum())
    _tally["max_abs_diff"] = max(_tally["max_abs_diff"], int(np.abs(diff).max(initial=0)))
    bad = np.nonzero((diff != 0) & ~band)[0]
    assert bad.size == 0, f"{what}: {bad.size} samples differ outside the band, first at p={bad[0]}: " \
                          f"got {got[bad[0]]}, reference {y[bad[0]]!r}"
    assert np.abs(diff).max(initial=0) <= 1, what
    assert not (got == -32768).any(), what


def run_tx(sc, n_streams, n_packets, gap, samples, *, channel=None, bits=None, seed=0, lead=None, wide=False,
           packet=False, stride=None, sentinel=-12345):
    """One sc_tx_channel_dev (channel = dict of per-stream numpy arrays, {} = every array NULL) or
    sc_tx_packets_dev (channel None) call.  Returns (out [n, stride] int16 with the part past samples_per_stream
    included, bits_out [n, n_packets, 8, 62])."""
    import torch
    stride = stride or samples
    bank = sc.ModemBank(n_streams, wide=wide, packet=packet)
    full = torch.full((n_streams, stride), sentinel, dtype=torch.int16, device="cuda")
    out = full[:, :samples]
    bits_out = torch.empty((n_streams, n_packets, 8, 62), dtype=torch.uint8, device="cuda")
    ch = None
    if channel is not None:
        ch = {k: torch.from_numpy(np.asarray(v, np.int32 if k == "echo_delay" else np.float32)).cuda()
              for k, v in channel.items()}
    d_bits = torch.from_numpy(bits).cuda() if bits is not None else None
    d_lead = torch.from_numpy(np.asarray(lead, np.int32)).cuda() if lead is not None else None
    bank.tx_packets_dev(out, n_packets, gap_samples=gap, bits=d_bits, bits_out=bits_out, seed=seed, lead_in=d_lead,
                        channel=ch)
    torch.cuda.synchronize()
    bank.close()
    return full.cpu().numpy(), bits_out.cpu().numpy()


def reference(oracle, bits, channel, s, *, n_packets, gap, lead, samples, wide=False, packet=False, seed=0,
              s_global=None):
    params = {k: np.asarray(v)[s] for k, v in (channel or {}).items()}
    return cr.stream(oracle, bits, params, n_packets=n_packets, gap=gap, lead=0 if lead is None else int(lead[s]),
                     samples_per_stream=samples, wide=wide, scramble=packet, seed=seed,
                     stream_index=s if s_global is None else s_global)


@pytest.mark.parametrize("wide", [False, True])
def test_every_array_null_is_the_plain_transmitter(sc, oracle, wide):
    """A channel with every array NULL rounds Re(z) (exact: no float work is left); without a channel the output is
    the reference transmitter's truncation of the same float."""
    npk, gap, samples = 3, 500, 3 * 2380 + 700
    lead = [0, 37, 1234]
    y_ch, bits = run_tx(sc, 3, npk, gap, samples, channel={}, seed=4, lead=lead, wide=wide)
    y_tx, bits2 = run_tx(sc, 3, npk, gap, samples, channel=None, seed=4, lead=lead, wide=wide)
    assert np.array_equal(bits, bits2)
    for s in range(3):
        z = cr.clean(oracle, bits[s], n_packets=npk, gap=gap, lead=lead[s], samples_per_stream=samples, wide=wide)
        assert np.array_equal(y_ch[s], np.rint(z.real).astype(np.int16)), s
        assert np.array_equal(y_tx[s], np.trunc(z.real).astype(np.int16)), s
        assert not np.array_equal(y_ch[s], y_tx[s])


# one call per case: per-stream parameter arrays (missing key = NULL array) and the call's geometry
SWEEP = {
    "phase_only": dict(channel={"phi_rad": [1.0]}),
    "df_+20": dict(channel={"df_hz": [20.0], "phi_rad": [0.3]}),
    "df_-20": dict(channel={"df_hz": [-20.0], "phi_rad": [5.9]}),
    "df_small": dict(channel={"df_hz": [0.01, -0.37, 1e-3]}, lead=[0, 5, 700]),
    "df_zero_array": dict(channel={"df_hz": [0.0], "phi_rad": [2.5], "drift_hz_s": [0.0]}),
    "drift_+2": dict(channel={"df_hz": [5.0], "drift_hz_s": [2.0]}),
    "drift_-2": dict(channel={"drift_hz_s": [-2.0], "phi_rad": [0.7]}),
    "drift_+-50": dict(channel={"df_hz": [0.0, -3.0], "drift_hz_s": [50.0, -50.0]}, npk=4, samples=4 * 2783 + 2000),
    "echo_0.1_d1": dict(channel={"echo_amp": [0.1], "echo_theta": [0.5], "echo_delay": [1]}),
    "echo_0.5_d2": dict(channel={"echo_amp": [0.5], "echo_theta": [2.0], "echo_delay": [2], "df_hz": [7.0]}),
    "echo_1.0_d10": dict(channel={"echo_amp": [1.0], "echo_theta": [-1.0], "echo_delay": [10], "df_hz": [20.0]}),
    "echo_d16_beyond_gap": dict(channel={"echo_amp": [0.5], "echo_theta": [3.0], "echo_delay": [16],
                                         "df_hz": [-11.0]}, gap=8),
    "echo_gap0_into_next": dict(channel={"echo_amp": [0.9], "echo_theta": [1.1], "echo_delay": [10],
                                         "phi_rad": [0.2]}, gap=0),
    "echo_delay_null": dict(channel={"echo_amp": [0.5], "echo_theta": [0.8], "df_hz": [3.0]}),
    "echo_theta_null": dict(channel={"echo_amp": [0.3], "echo_delay": [5]}),
    "echo_amp_zero": dict(channel={"echo_amp": [0.0], "echo_theta": [0.8], "echo_delay": [9], "df_hz": [1.0]}),
    "sigma_0_30_300_3000": dict(channel={"sigma_lsb": [0.0, 30.0, 300.0, 3000.0], "df_hz": [1.0, -2.0, 3.0, -4.0]},
                                lead=[10, 0, 2999, 3000]),
    "sigma_only": dict(channel={"sigma_lsb": [300.0]}),
    "lead_in_null": dict(channel={"df_hz": [12.5], "sigma_lsb": [30.0]}, lead=None),
    "short_stream": dict(channel={"df_hz": [-6.0], "echo_amp": [0.4], "echo_delay": [3], "sigma_lsb": [30.0]},
                         npk=3, samples=1000, lead=[300]),
    "long_tail": dict(channel={"df_hz": [9.0], "echo_amp": [0.6], "echo_theta": [2.2], "echo_delay": [16],
                               "sigma_lsb": [30.0]}, npk=2, samples=2 * 2783 + 5000, lead=[100]),
    "stride_sentinel": dict(channel={"df_hz": [4.0, -4.0], "sigma_lsb": [300.0, 30.0], "echo_amp": [0.2, 0.7],
                                     "echo_delay": [16, 1]}, stride=9000, samples=8000, lead=[3, 1500]),
    "everything": dict(channel={"df_hz": [-17.0, 0.5, 19.9], "phi_rad": [0.1, 3.0, 6.2],
                                "drift_hz_s": [2.0, -1.0, 0.5], "sigma_lsb": [30.0, 300.0, 3000.0],
                                "echo_amp": [0.1, 0.5, 1.0], "echo_theta": [0.0, -2.0, 3.1],
                                "echo_delay": [1, 16, 7]}, lead=[0, 2000, 999], seed=123456789),
    "caller_bits": dict(channel={"df_hz": [-8.0], "echo_amp": [0.25], "echo_delay": [4]}, caller_bits=True),
    "packet_mode": dict(channel={"df_hz": [3.0, -15.0], "sigma_lsb": [0.0, 300.0], "echo_amp": [0.3, 0.0],
                                 "echo_delay": [6, 1]}, packet=True, lead=[40, 2100]),
}


@pytest.mark.parametrize("wide", [False, True])
@pytest.mark.parametrize("case", sorted(SWEEP))
def test_channel_sweep(sc, oracle, case, wide):
    c = SWEEP[case]
    channel = c["channel"]
    ns = len(next(iter(channel.values())))
    npk, gap = c.get("npk", 3), c.get("gap", 903)
    samples = c.get("samples", npk * (1880 + gap) + 3100)
    lead = c.get("lead", [1234] * ns)
    seed = c.get("seed", 77)
    stride = c.get("stride")
    bits = None
    if c.get("caller_bits"):
        bits = np.random.default_rng(3).integers(0, 2, (ns, npk, 8, 62)).astype(np.uint8)
    y, bits_out = run_tx(sc, ns, npk, gap, samples, channel=channel, bits=bits, seed=seed, lead=lead, wide=wide,
                         packet=c.get("packet", False), stride=stride)
    if bits is not None:
        assert np.array_equal(bits_out, bits)
    else:                                                   # bits_out is the payload, also in packet mode
        for s in range(ns):
            assert np.array_equal(bits_out[s], cr.data_bits(seed, s, npk)), s
    for s in range(ns):
        want = reference(oracle, bits_out[s], channel, s, n_packets=npk, gap=gap, lead=lead, samples=samples,
                         wide=wide, packet=c.get("packet", False), seed=seed)
        assert_matches(y[s, :samples], want, f"{case} stream {s}")
        if stride:
            assert (y[s, samples:] == -12345).all(), f"{case}: wrote past samples_per_stream"
    if "sigma_lsb" not in channel and "echo_amp" in channel:
        # no noise: the tail past the last packet's echo is silent
        end = (0 if lead is None else max(lead)) + (npk - 1) * (1880 + gap) + 1880 + 16
        assert not y[:, end:samples].any()


def test_slice_boundary_bank(sc, oracle):
    """65,836 streams x 4,000 samples (grid.y is cut into slices of 65,535 streams): every parameter array, the
    lead-in, the output row and the noise key of a stream must be those of its index in the whole bank."""
    import torch
    ns, samples, npk, gap, seed = 65836, 4000, 2, 100, 2024
    s = np.arange(ns)
    ch = {"df_hz": ((s * 7919) % 4001) / 100.0 - 20.0,
          "phi_rad": (s % 628) / 100.0,
          "drift_hz_s": ((s * 13) % 401) / 100.0 - 2.0,
          "sigma_lsb": 10.0 + (s % 97) * 5.0,
          "echo_amp": 0.1 + (s % 5) * 0.2,
          "echo_theta": (s * 0.37) % 6.28,
          "echo_delay": 1 + (s * 3) % 16}
    lead = (s * 37) % 1500
    bank = sc.ModemBank(ns)
    out = torch.empty((ns, samples), dtype=torch.int16, device="cuda")
    bits_out = torch.empty((ns, npk, 8, 62), dtype=torch.uint8, device="cuda")
    d_ch = {k: torch.from_numpy(np.asarray(v, np.int32 if k == "echo_delay" else np.float32)).cuda()
            for k, v in ch.items()}
    bank.tx_packets_dev(out, npk, gap_samples=gap, seed=seed, bits_out=bits_out,
                        lead_in=torch.from_numpy(lead.astype(np.int32)).cuda(), channel=d_ch)
    torch.cuda.synchronize()
    bank.close()
    rng = np.random.default_rng(6)
    pick = np.unique(np.concatenate([[0, 1, 65534, 65535, 65536, 65537, ns - 1], rng.integers(0, ns, 200)]))
    idx = torch.from_numpy(pick).cuda()
    y = out[idx].cpu().numpy()
    b = bits_out[idx].cpu().numpy()
    del out, bits_out
    for i, si in enumerate(pick):
        assert np.array_equal(b[i], cr.data_bits(seed, int(si), npk)), si
        want = reference(oracle, b[i], ch, int(si), n_packets=npk, gap=gap, lead=lead, samples=samples, seed=seed)
        assert_matches(y[i], want, f"stream {si}")


def test_saturation(sc, oracle):
    """sigma = 20,000 LSB: the output saturates at +-32767 (never -32768) as often as 2 Q(32767 / sigma) says."""
    from scipy import stats
    n = 400_000
    sigma = 20000.0
    y, _ = run_tx(sc, 1, 0, 903, n, channel={"sigma_lsb": [sigma]}, seed=5)
    clipped = float(np.mean(np.abs(y[0]) == 32767))
    p = 2.0 * stats.norm.sf(32767.0 / sigma)
    assert abs(clipped / p - 1.0) < 0.05, (clipped, p)
    assert (y[0] == 32767).any() and (y[0] == -32767).any()
    want = reference(oracle, np.zeros((0, 8, 62), np.uint8), {"sigma_lsb": [sigma]}, 0, n_packets=0, gap=903,
                     lead=None, samples=n, seed=5)
    assert_matches(y[0], want, "saturation")


def test_determinism_and_generated_bits(sc):
    """The same seed gives byte-identical output and bits; another seed changes both; bits_out is the restated
    generator mix64(seed ^ mix64(w)) & (2^62 - 1)."""
    ch = {"df_hz": [3.0, -5.0, 11.0], "sigma_lsb": [300.0, 300.0, 3000.0], "echo_amp": [0.5, 0.5, 0.5]}
    a = run_tx(sc, 3, 3, 903, 9000, channel=ch, seed=99, lead=[1, 2, 3])
    b = run_tx(sc, 3, 3, 903, 9000, channel=ch, seed=99, lead=[1, 2, 3])
    c = run_tx(sc, 3, 3, 903, 9000, channel=ch, seed=100, lead=[1, 2, 3])
    assert a[0].tobytes() == b[0].tobytes() and a[1].tobytes() == b[1].tobytes()
    assert not np.array_equal(a[0], c[0]) and not np.array_equal(a[1], c[1])
    for s in range(3):
        assert np.array_equal(a[1][s], cr.data_bits(99, s, 3))
        assert np.array_equal(c[1][s], cr.data_bits(100, s, 3))


def test_awgn_calibration_end_to_end(sc):
    """harness.synthesize(config=3): the Es/N0 measured from the noise it added (noisy - clean, the clean run being
    the same call without sigma_lsb) and the clean data-section power is 2 Eb/N0 of the stream's label, within
    0.1 dB at every point 0..12 dB."""
    import torch
    from singlecarrier_b200 import harness
    ns, samples, seed = 2600, 3 * 2783, 17
    bank = sc.ModemBank(ns)
    wl = harness.synthesize(bank, samples, seed, config=3)
    clean_ch = {k: v for k, v in wl.channel.items() if k != "sigma_lsb"}
    clean = torch.empty_like(wl.samples)
    bits = torch.empty_like(wl.tx_bits)
    bank.tx_packets_dev(clean, wl.n_packets, gap_samples=wl.gap, seed=seed, bits_out=bits, lead_in=wl.lead,
                        channel=clean_ch)
    torch.cuda.synchronize()
    bank.close()
    assert torch.equal(bits, wl.tx_bits)
    x = clean.double().cpu().numpy()
    nz = wl.samples.double().cpu().numpy() - x
    lead = wl.lead.cpu().numpy()
    eb = wl.ebn0_db.cpu().numpy()
    u = np.stack([cr.filter_time(np.arange(samples), int(lead[s]), wl.gap, wl.n_packets) for s in range(ns)])
    data = (u >= 0) & (u % 1880 >= 640)
    got = []
    for k in range(13):
        m = np.isclose(eb, k)
        assert m.sum() == 200
        p_sig = np.mean(x[m][data[m]] ** 2)
        esn0 = p_sig * 8000.0 / (2.0 * 1600.0 * np.var(nz[m]))
        got.append(10.0 * np.log10(esn0))
    want = np.arange(13) + 10.0 * np.log10(2.0)
    assert np.abs(np.array(got) - want).max() < 0.1, np.round(np.array(got) - want, 3).tolist()


# ---- bit-error counters -----------------------------------------------------------------------------------------

def ber_expected(rec, n_frames, tx_bits, n_packets, lead, gap, group, n_groups):
    """The counters of sc_ber_stats_dev written from its header (include/singlecarrier_b200.h), one call at a time."""
    ks = cr.keystream_words(n_frames)
    period = 1880 + gap
    c = np.zeros((n_groups, 8), np.int64)
    for s in range(rec.shape[0]):
        g = 0 if group is None else int(group[s])
        if not 0 <= g < n_groups:
            continue
        for n in range(2, n_frames):
            c[g, 0] += 1
            if not rec["valid"][s, n]:
                continue
            c[g, 1] += 1
            pos = (n - 2) * 1880 + 5 * int(rec["max_index"][s, n]) + int(rec["rx_timing"][s, n - 2]) - 48
            pos -= 0 if lead is None else int(lead[s])
            for j in range(n_packets):
                if abs(pos - j * period) <= 10:
                    tx = sum(int(tx_bits[s, j, 0, i]) << i for i in range(62))
                    c[g, 2] += 1
                    c[g, 3] += 62
                    c[g, 4] += bin((int(rec["bits"][s, n]) ^ ks[n] ^ tx) & ((1 << 62) - 1)).count("1")
    return c


def ber_records(sc, rng, ns, n_frames, stride, n_packets, gap, lead):
    """Records whose calls land on packet starts -1..n_packets at offsets -11, -10, -1, 0, 1, +10, +11 (or anywhere),
    at negative positions too, with bits = tx ^ keystream ^ (a known number of flipped bits)."""
    period = 1880 + gap
    ks = cr.keystream_words(n_frames)
    rec = np.zeros((ns, stride), sc.RESULT_DTYPE)
    rec["valid"] = rng.random((ns, stride)) < 0.85
    rec["max_index"] = rng.integers(-20, 128, (ns, stride))
    rec["rx_timing"] = rng.integers(-300, 300, (ns, stride))
    rec["matches"] = rng.integers(0, 129, (ns, stride))
    rec["bits"] = rng.integers(0, 2 ** 63, (ns, stride), dtype=np.uint64) * np.uint64(2) + \
        rng.integers(0, 2, (ns, stride), dtype=np.uint64)
    tx_bits = rng.integers(0, 2, (ns, n_packets, 8, 62)).astype(np.uint8)
    weights = np.uint64(1) << np.arange(62, dtype=np.uint64)
    tx_words = (tx_bits[:, :, 0, :].astype(np.uint64) * weights).sum(-1, dtype=np.uint64)       # [ns, n_packets]
    offsets = np.array([-11, -10, -1, 0, 1, 10, 11])
    for n in range(2, n_frames):
        aim = rng.random(ns) < 0.75
        j = rng.integers(-1, n_packets + 1, ns)
        off = np.where(rng.random(ns) < 0.8, offsets[rng.integers(0, offsets.size, ns)], rng.integers(-1500, 1500, ns))
        pos = j * period + off
        t = pos + 48 + (0 if lead is None else lead) - (n - 2) * 1880 - 5 * rec["max_index"][:, n].astype(np.int64)
        assert np.abs(t).max() < 32768
        rec["rx_timing"][:, n - 2] = np.where(aim, t, rec["rx_timing"][:, n - 2])
        n_flips = rng.integers(0, 63, ns)
        flip = rng.random((ns, 62)).argsort(1).argsort(1) < n_flips[:, None]          # n_flips random bits
        flips = (flip.astype(np.uint64) * weights).sum(-1, dtype=np.uint64)
        hi = rng.integers(0, 4, ns).astype(np.uint64) << np.uint64(62)      # bits 62, 63 are not compared
        jc = np.clip(j, 0, n_packets - 1)
        bits = tx_words[np.arange(ns), jc] ^ np.uint64(ks[n]) ^ flips ^ hi
        rec["bits"][:, n] = np.where(aim, bits, rec["bits"][:, n])
    return rec, tx_bits


@pytest.mark.parametrize("with_lead", [True, False])
def test_ber_counters_on_hand_made_records(sc, with_lead):
    """sc_ber_stats_dev and harness.ber_and_lock against the loop above: packet offsets -11..+11 around the
    +-10-sample window, negative positions, packets -1 and n_packets, calls 0 and 1, groups -1 and n_groups,
    result_stride > n_frames, NULL and non-NULL lead_in, more (stream, call) pairs than the grid has threads,
    counters that already hold values."""
    import torch
    from singlecarrier_b200 import harness
    rng = np.random.default_rng(40 + with_lead)
    ns, nf, stride, npk, gap, n_groups = 40_000, 9, 11, 4, 903, 3
    lead = rng.integers(0, 3000, ns) if with_lead else None
    assert ns * nf > 148 * 8 * 256
    rec, tx_bits = ber_records(sc, rng, ns, nf, stride, npk, gap, lead)
    group = rng.integers(-1, n_groups + 1, ns)
    want = ber_expected(rec, nf, tx_bits, npk, lead, gap, group, n_groups)
    assert want[:, 2].sum() > 1000 and want[:, 4].sum() > 0 and (want[:, 1] > want[:, 2]).all()
    prior = rng.integers(0, 2 ** 40, (n_groups, 8))
    d_rec = torch.from_numpy(rec.view(np.uint8).reshape(ns, stride * 32)).cuda()
    d_tx = torch.from_numpy(tx_bits).cuda()
    d_lead = torch.from_numpy(lead.astype(np.int32)).cuda() if with_lead else None
    d_group = torch.from_numpy(group.astype(np.int32)).cuda()
    cnt = torch.from_numpy(prior.copy()).cuda()
    bank = sc.ModemBank(ns)
    bank.ber_stats(d_rec, nf, d_tx, d_lead, gap, cnt, group=d_group, n_groups=n_groups)
    torch.cuda.synchronize()
    got = cnt.cpu().numpy() - prior
    assert got.tolist() == want.tolist()
    # group NULL: every stream in group 0
    cnt0 = torch.zeros((1, 8), dtype=torch.int64, device="cuda")
    bank.ber_stats(d_rec, nf, d_tx, d_lead, gap, cnt0, group=None, n_groups=1)
    torch.cuda.synchronize()
    bank.close()
    assert cnt0.cpu().numpy().tolist() == ber_expected(rec, nf, tx_bits, npk, lead, gap, None, 1).tolist()
    # the torch recount of harness.py (lead_in given as zeros where the kernel had NULL)
    wl = harness.Workload(None, d_tx, d_lead if with_lead else torch.zeros(ns, dtype=torch.int32, device="cuda"),
                          gap, None, npk)
    h = harness.ber_and_lock(d_rec[:, :nf * 32].contiguous(), nf, wl, group=d_group.long(), n_groups=n_groups)
    for k, name in enumerate(("calls", "valid", "aligned", "bits", "errors")):
        assert h[name].tolist() == want[:, k].tolist(), name
    assert [w for w in cr.keystream_words(nf)] == [sc.keystream_word(n) for n in range(nf)]
