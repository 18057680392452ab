"""GPU: packet-mode banks fed through the host entry point in several blocks of frames.  A block after the first reads
the frames before it (and their phasor tables) from what the previous block saved; per-call results, records and
symbols must equal those of one device batch of the same samples on a fresh bank."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from test_packet_acq_gpu import acq_streams  # noqa: E402
from test_soft_gpu import u32  # noqa: E402

FRAME = 1880


@pytest.fixture(scope="module")
def sc():
    import singlecarrier_b200 as m
    assert m.lib.sc_device_count() > 0, "no CUDA device"
    return m


def keyed(pk, psym, field):
    out = {}
    for p, ps in zip(pk, psym):
        key = (int(p["stream"]), int(p[field]))
        assert key not in out, key
        out[key] = (p.tobytes(), u32(ps).tobytes())
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["packet", "dd", "acq"])
def test_host_blocks_equal_one_device_batch(sc, kind):
    import torch
    ns, nf = 130, 60
    samples, _, _ = acq_streams(sc, ns, 39, 0xB1C)
    samples = np.ascontiguousarray(samples[:, :nf * FRAME])
    flags = dict(packet=True, dd=kind != "packet", acq=kind == "acq")

    # Rows wider than the batch: the host entry point then stages whole frames of 4,096-stream slabs (the floor of its
    # slab size), 52 frames of which fill its 768 MiB staging buffer, so the batch runs as blocks of 52 and 8 frames.
    wide = np.zeros((ns, (nf + 1) * FRAME), np.int16)
    wide[:, :nf * FRAME] = samples
    bank = sc.ModemBank(ns, **flags)
    res, csym, pk, psym, n = bank.rx_packets_soft_host(wide[:, :nf * FRAME], nf, call_symbols=True)
    bank.close()
    assert n == len(pk) > 0

    bank = sc.ModemBank(ns, **flags)
    cap = ns * nf
    d_res = torch.zeros((ns, nf * 32), dtype=torch.uint8, device="cuda")
    d_csym = torch.zeros((ns, nf * 62), dtype=torch.float32, device="cuda")
    d_pk = torch.zeros(cap * 96, dtype=torch.uint8, device="cuda")
    d_psym = torch.zeros(cap * 496, dtype=torch.float32, device="cuda")
    d_n = torch.zeros(1, dtype=torch.int64, device="cuda")
    bank.rx_packets_soft_dev(torch.from_numpy(samples).cuda(), nf, d_res, d_pk, d_n, d_psym, symbols=d_csym)
    torch.cuda.synchronize()
    bank.close()
    m = int(d_n.item())
    assert m == n
    assert d_res.cpu().numpy().tobytes() == res.tobytes()
    assert np.array_equal(d_csym.cpu().numpy().view(np.uint32).reshape(-1), u32(csym).reshape(-1))
    field = "grid_sample" if kind == "acq" else "call_index"
    dev = keyed(d_pk.cpu().numpy()[:m * 96].view(sc.PACKET_DTYPE),
                d_psym.cpu().numpy()[:m * 496].view(np.complex64).reshape(m, 248), field)
    assert dev == keyed(pk, psym, field)
