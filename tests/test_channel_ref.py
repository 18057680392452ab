"""CPU: the float64 channel reference (oracle/channel_ref.py) and the oracle's analytic TX sample it is built on,
the statistics of the restated noise generator, and the signal power the AWGN of harness.py is calibrated to."""
import numpy as np
import pytest
from scipy import stats

from oracle import channel_ref as cr

N_DRAWS = 2_000_000
SEED = 9
# stream 65,535 is the first stream of the second grid slice of the channel kernel
STREAMS = (0, 1, 65534, 65535, 65536)


@pytest.fixture(scope="module")
def draws():
    p = np.arange(N_DRAWS)
    d = {s: cr.noise(SEED, s, p) for s in STREAMS}
    d["seed+1"] = cr.noise(SEED + 1, 0, p)
    return d


@pytest.mark.parametrize("wide", [False, True])
def test_analytic_tx_truncates_to_the_int16_tx(oracle, wide):
    """trunc(Re(analytic)) of the oracle's transmitter is its int16 output, bit for bit, across packets (the filter
    memory and the TX phasor persist) for the preamble and the data frames."""
    rng = np.random.default_rng(21)
    st_i, st_a = oracle.new_state(wide=wide), oracle.new_state(wide=wide)
    for _ in range(5):
        pairs = [(oracle.tx_preamble(st_i), oracle.tx_preamble_analytic(st_a))]
        for _ in range(8):
            b = rng.integers(0, 2, 62).astype(np.uint8)
            pairs.append((oracle.tx_data(st_i, b), oracle.tx_data_analytic(st_a, b)))
        for i16, z in pairs:
            assert z.dtype == np.complex64 and z.size == i16.size
            assert np.array_equal(np.trunc(z.real).astype(np.int16), i16)
            assert np.abs(z.imag).max() > 1000.0                 # a quadrature component is really there


@pytest.mark.parametrize("s", [0, 1, 65535, 65536])
def test_noise_moments_and_ks(draws, s):
    n = draws[s]
    N = n.size
    tol = 5.0 / np.sqrt(N)
    assert abs(n.mean()) < tol
    assert abs(n.var() - 1.0) < tol * np.sqrt(2.0)
    assert abs(stats.skew(n)) < tol * np.sqrt(6.0)
    assert abs(stats.kurtosis(n)) < tol * np.sqrt(24.0)
    assert stats.kstest(n, "norm").statistic < 2.0 / np.sqrt(N)


@pytest.mark.parametrize("s", [0, 1, 65535, 65536])
def test_noise_tail_and_truncation(draws, s):
    """P(|n| > 4) = 6.33e-5 within 5 sigma of the binomial count; the draw never exceeds sqrt(-2 ln 2^-25) = 5.887
    (the smallest u1 is 2^-25), so the generator has no tail beyond 5.9 sigma (a probability of 4e-9)."""
    n = draws[s]
    p4 = 2.0 * stats.norm.sf(4.0)
    k = int((np.abs(n) > 4.0).sum())
    assert abs(k - p4 * n.size) < 5.0 * np.sqrt(p4 * n.size)
    assert np.abs(n).max() <= cr.NOISE_BOUND
    assert abs(cr.NOISE_BOUND - 5.8870) < 1e-4


def _corr(a, b):
    a = a - a.mean()
    b = b - b.mean()
    return float(np.dot(a, b) / np.sqrt(np.dot(a, a) * np.dot(b, b)))


@pytest.mark.parametrize("s", [0, 1, 65535, 65536])
def test_noise_autocorrelation(draws, s):
    n = draws[s]
    tol = 5.0 / np.sqrt(n.size)
    worst = max(abs(_corr(n[:-k], n[k:])) for k in range(1, 65))
    assert worst < tol, worst


@pytest.mark.parametrize("a,b", [(0, 1), (65534, 65535), (65535, 65536), (0, "seed+1")])
def test_noise_independent_across_streams_and_seeds(draws, a, b):
    """Neighbouring streams, the two streams on either side of the grid-slice boundary, and two seeds."""
    assert abs(_corr(draws[a], draws[b])) < 5.0 / np.sqrt(N_DRAWS)
    assert not np.array_equal(draws[a][:64], draws[b][:64])


def test_data_bits_restatement_layout():
    """bits_out[s, P, f, j] is bit j of word (s * n_packets + P) * 8 + f."""
    b = cr.data_bits(77, 3, 2)
    assert b.shape == (2, 8, 62) and set(np.unique(b)) == {0, 1}
    w = int(cr.data_words(77, np.array([(3 * 2 + 1) * 8 + 5], np.uint64))[0])
    assert b[1, 5].tolist() == [(w >> j) & 1 for j in range(62)]
    assert w < 2 ** 62


@pytest.mark.parametrize("wide", [False, True])
def test_data_section_rms_is_the_awgn_calibration(oracle, wide):
    """harness.DATA_RMS_LSB is the P_sig of SURVEY section 8d: the RMS of the data section of the transmitted
    signal.  Measured on 200 packets of the oracle's TX with random bits it must agree within 0.5 %."""
    from singlecarrier_b200 import harness
    rng = np.random.default_rng(8)
    st = oracle.new_state(wide=wide)
    data = []
    for _ in range(200):
        oracle.tx_preamble(st)
        for _ in range(8):
            data.append(oracle.tx_data(st, rng.integers(0, 2, 62).astype(np.uint8)))
    x = np.concatenate(data).astype(np.float64)
    ratio = np.sqrt(np.mean(x ** 2)) / harness.DATA_RMS_LSB
    assert abs(ratio - 1.0) < 0.005, ratio
