"""GPU: a batch that the CUDA runtime refuses leaves the bank as documented (include/singlecarrier_b200.h, SC_ESTATE).

Both cases ask for an allocation larger than the whole device (a B200 has 180 GB); the runtime refuses such a request
with an API error before anything is allocated or launched.  They pin where a batch is "in flight": from its first
queued work in the device path (a failure after that poisons the bank until sc_reset), and only after the staging of
the host packet path has grown (a failure there leaves the bank as it was).  Both also check that a refused
allocation does not fail the launches of the next batch."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

FRAME = 1880


@pytest.fixture(scope="module")
def sc():
    import singlecarrier_b200 as m
    assert m.lib.sc_device_count() > 0
    return m


def loopback(sc, ns, n_frames, seed, packet=False):
    """ns streams of n_frames frames from the library's own TX and channel, on the device."""
    import torch
    bank = sc.ModemBank(ns, packet=packet)
    g = torch.Generator(device="cuda").manual_seed(seed)
    lead = torch.randint(0, 2783, (ns,), generator=g, device="cuda", dtype=torch.int32)
    df = (torch.rand(ns, generator=g, device="cuda") * 10 - 5).float()
    sigma = (torch.arange(ns, device="cuda") % 4).float() * 300.0
    d_in = torch.empty((ns, n_frames * FRAME), dtype=torch.int16, device="cuda")
    bank.tx_packets_dev(d_in, n_frames // 2 + 1, gap_samples=903, seed=seed, lead_in=lead,
                        channel={"df_hz": df, "sigma_lsb": sigma})
    torch.cuda.synchronize()
    bank.close()
    return d_in


def test_refused_device_batch_poisons_until_reset(sc):
    """sc_rx_frames_dev whose phasor table (about 250 GB) cannot be allocated: SC_ENOMEM after the batch was queued
    behind the caller's stream, so the bank refuses work (SC_ESTATE) until sc_reset; then it equals a fresh bank."""
    import torch
    ns, nf = 4, 3
    d_in = loopback(sc, ns, nf, seed=11)
    fresh = sc.ModemBank(ns)
    want = torch.zeros((ns, nf * 32), dtype=torch.uint8, device="cuda")
    fresh.rx_frames_dev(d_in, nf, want)
    torch.cuda.synchronize()
    fresh.close()

    bank = sc.ModemBank(ns)
    got = torch.zeros_like(want)
    huge = 1 << 24                          # neither the input nor the results are ever touched
    rc = sc.lib.sc_rx_frames_dev(bank._h, d_in.data_ptr(), huge * FRAME, huge, got.data_ptr(), huge, None, None)
    assert rc == sc._lib.SC_ENOMEM, sc.lib.sc_last_error()
    assert bank.call_index == 0
    rc = sc.lib.sc_rx_frames_dev(bank._h, d_in.data_ptr(), d_in.stride(0), nf, got.data_ptr(), nf, None, None)
    assert rc == sc._lib.SC_ESTATE, sc.lib.sc_last_error()
    bank.reset()
    bank.rx_frames_dev(d_in, nf, got)
    torch.cuda.synchronize()
    assert bank.call_index == nf
    assert torch.equal(got, want)
    bank.close()


def test_refused_host_packet_staging_leaves_the_bank_as_it_was(sc):
    """sc_rx_packets_host whose packet staging (capacity 2^36 records) cannot be allocated: SC_ENOMEM before anything
    was queued, so the call index, the descrambler and the poisoning are untouched and the next batch, without a
    reset, equals the same batch on a fresh bank."""
    ns, nf1, nf2 = 4, 3, 4
    samples = loopback(sc, ns, nf1 + nf2, seed=12, packet=True).cpu().numpy()
    first, second = samples[:, : nf1 * FRAME], samples[:, nf1 * FRAME:]

    fresh = sc.ModemBank(ns, packet=True)
    _, _, n_first = fresh.rx_packets_host(first)
    want = fresh.rx_packets_host(second)
    fresh.close()

    bank = sc.ModemBank(ns, packet=True)
    bank.rx_packets_host(first)
    results = np.zeros((ns, nf2), sc.RESULT_DTYPE)
    record = np.zeros(1, sc.PACKET_DTYPE)
    n = C.c_uint64(12345)
    rc = sc.lib.sc_rx_packets_host(bank._h, second.ctypes.data, second.strides[0] // 2, nf2, results.ctypes.data, nf2,
                                   record.ctypes.data, 1 << 36, C.byref(n))
    assert rc == sc._lib.SC_ENOMEM, sc.lib.sc_last_error()
    assert bank.call_index == nf1
    assert n.value == 0                     # the count is cleared before the staging is made
    got = bank.rx_packets_host(second)
    assert bank.call_index == nf1 + nf2
    assert got[0].tobytes() == want[0].tobytes()
    assert got[2] == want[2]
    assert got[1].tobytes() == want[1].tobytes()
    assert n_first + want[2] > 0
    bank.close()
