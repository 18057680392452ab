"""Float64 reference of the loop-back channel generator (sc_tx_channel_dev) -- TEST INFRASTRUCTURE ONLY.

The product package (``singlecarrier_b200``) never imports this module.

The transmitted signal is the oracle's own transmitter stopped before the real part is taken
(``Oracle.tx_preamble_analytic`` / ``tx_data_analytic``); its real part truncated is the int16 output that
tests/test_oracle_vs_ref.py and the golden vectors pin to the reference.  Everything after it is computed here
in float64 from the per-stream parameters widened from float32.

Order of the channel operations (include/singlecarrier_b200.h states the same):

  1. z[p]   the analytic TX sample at filter time u(p), and 0 in the lead-in, the dead air and the tail
            (they bypass the filter and the NCO, qpsk.c:410-412);
  2. echo   e[p] = z[p] + a exp(j theta) z[p - d]            (NULL echo_delay means d = 1);
  3. offset e[p] exp(j (2 pi (df + drift t / 2) t + phi)),  t = p / 8000 s, p the output index counted from the
            stream's first sample, lead-in included: the offset is that of the receiver's oscillator;
  4. noise  Re(.) + sigma n[s, p];
  5. clip to +-32767, then round half to even.

The two counter-based generators (``noise`` and ``data_words``) are restated from the kernels: they pin the
implementation, not a specification.  If the generator in csrc/sc_tx_kernels.cu changes, these functions change
with it.
"""
from __future__ import annotations

import numpy as np

FRAME_SIZE = 1880
FS = 8000.0
BITS_PER_CALL = 62
CLIP = 32767.0
# the smallest u1 of the Box-Muller draw is 2^-25, so |n| <= sqrt(-2 ln 2^-25) = 5.887
NOISE_BOUND = float(np.sqrt(-2.0 * np.log(2.0 ** -25)))

_U64 = np.uint64
_MASK62 = _U64((1 << 62) - 1)


def mix64(z) -> np.ndarray:
    """splitmix64 finaliser on uint64 arrays (wrapping arithmetic)."""
    z = np.asarray(z, np.uint64) + _U64(0x9E3779B97F4A7C15)
    z = (z ^ (z >> _U64(30))) * _U64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> _U64(27))) * _U64(0x94D049BB133111EB)
    return z ^ (z >> _U64(31))


def noise(seed: int, stream: int, p) -> np.ndarray:
    """The unit-variance draw n[stream, p] of the AWGN (``stream`` is the stream's index in the whole bank):
    key ((stream << 34) ^ p ^ 0xA5A5A5A5), hashed, xor the seed, hashed; two 24-bit uniforms; the cos branch of
    Box-Muller, evaluated in float64.

    u1 = (x + 1/2) 2^-24 is rounded to float32 as the kernel's sum is: for x >= 2^23 the half rounds to even.
    That is invisible in the distribution, but near u1 = 1, where -2 ln u1 is 2 (1 - u1), it moves a small draw
    by tens of percent (0.66 LSB of a 24-LSB sample at sigma = 20,000)."""
    p = np.asarray(p, np.uint64)
    key = (_U64(stream) << _U64(34)) ^ p ^ _U64(0xA5A5A5A5)
    h = mix64(_U64(seed) ^ mix64(key))
    u1 = ((h >> _U64(40)).astype(np.float64) + 0.5).astype(np.float32).astype(np.float64) / 16777216.0
    u2 = ((h >> _U64(8)) & _U64(0xFFFFFF)).astype(np.float64) / 16777216.0
    return np.sqrt(-2.0 * np.log(u1)) * np.cos(2.0 * np.pi * u2)


def data_words(seed: int, w) -> np.ndarray:
    """The 62-bit payload word of global word index w = (stream * n_packets + packet) * 8 + frame when the caller
    passes no bits: mix64(seed ^ mix64(w)) & (2^62 - 1); bit j is bits_out[..][j]."""
    return mix64(_U64(seed) ^ mix64(np.asarray(w, np.uint64))) & _MASK62


def data_bits(seed: int, stream: int, n_packets: int) -> np.ndarray:
    """bits_out of one stream (global index) of a bank whose bits were drawn: uint8 [n_packets, 8, 62]."""
    v = data_words(seed, stream * n_packets * 8 + np.arange(n_packets * 8, dtype=np.uint64))
    b = (v[:, None] >> np.arange(BITS_PER_CALL, dtype=np.uint64)[None, :]) & _U64(1)
    return b.astype(np.uint8).reshape(n_packets, 8, BITS_PER_CALL)


def keystream_words(n: int) -> list:
    """Descrambler keystream words of calls 0..n-1 (integer LFSR, src/scramble.c:57-69, SEED 0x4A80): bit j of
    word n is the keystream bit of the j-th decided bit of call n.  Packet mode scrambles data frame f of every
    packet with word f."""
    m, out = 0x4A80, []
    for _ in range(n):
        w = 0
        for j in range(BITS_PER_CALL):
            o = ((m >> 1) ^ m) & 1
            m = (m >> 1) | (o << 14)
            w |= o << j
        out.append(w)
    return out


def word_bits(w: int) -> np.ndarray:
    return np.array([(w >> j) & 1 for j in range(BITS_PER_CALL)], np.uint8)


def analytic_packets(oracle, bits: np.ndarray, wide: bool = False, scramble: bool = False) -> np.ndarray:
    """The oracle's analytic TX signal of n_packets packets (bits uint8 [n_packets, 8, 62], the payload) as one
    complex128 array over filter time u, [n_packets * 1880].  scramble: packet mode, data frame f sent as
    bits ^ keystream word f."""
    st = oracle.new_state(wide=wide)
    keys = [word_bits(w) for w in keystream_words(8)] if scramble else None
    parts = []
    for P in range(bits.shape[0]):
        parts.append(oracle.tx_preamble_analytic(st))
        for f in range(8):
            b = bits[P, f] ^ keys[f] if scramble else bits[P, f]
            parts.append(oracle.tx_data_analytic(st, b))
    if not parts:
        return np.zeros(0, np.complex128)
    return np.concatenate(parts).astype(np.complex128)


def filter_time(p, lead: int, gap: int, n_packets: int) -> np.ndarray:
    """Output index p -> filter time u, or -1 in the lead-in, the dead air and the tail."""
    pp = np.asarray(p, np.int64) - lead
    period = FRAME_SIZE + gap
    P = np.floor_divide(pp, period)
    r = pp - P * period
    ok = (pp >= 0) & (P < n_packets) & (r < FRAME_SIZE)
    return np.where(ok, P * FRAME_SIZE + r, -1)


def clean(oracle, bits, *, n_packets: int, gap: int, lead: int, samples_per_stream: int, wide: bool = False,
          scramble: bool = False) -> np.ndarray:
    """z[p] of one stream: complex128 [samples_per_stream]."""
    za = analytic_packets(oracle, bits[:n_packets], wide=wide, scramble=scramble)
    u = filter_time(np.arange(samples_per_stream), lead, gap, n_packets)
    z = np.zeros(samples_per_stream, np.complex128)
    z[u >= 0] = za[u[u >= 0]]
    return z


def channel(z: np.ndarray, params: dict, *, seed: int = 0, stream: int = 0) -> np.ndarray:
    """Steps 2-5 on z (complex128 [samples]) for one stream.  params: scalar per-stream values of the sc_channel
    arrays, a missing key standing for a NULL array.  Returns y (float64, clipped, before rounding); the device
    output is np.rint(y)."""
    f = {k: float(np.float32(params[k])) if k in params else 0.0
         for k in ("df_hz", "phi_rad", "drift_hz_s", "sigma_lsb", "echo_amp", "echo_theta")}
    e = z.copy()
    if f["echo_amp"] != 0.0:
        d = int(params.get("echo_delay", 1))
        if d < len(z):
            e[d:] += f["echo_amp"] * np.exp(1j * f["echo_theta"]) * z[:len(z) - d]
    t = np.arange(len(z)) / FS
    y = (e * np.exp(1j * (2.0 * np.pi * (f["df_hz"] + 0.5 * f["drift_hz_s"] * t) * t + f["phi_rad"]))).real
    if f["sigma_lsb"] != 0.0:
        y = y + f["sigma_lsb"] * noise(seed, stream, np.arange(len(z)))
    return np.clip(y, -CLIP, CLIP)


def stream(oracle, bits, params: dict, *, n_packets: int, gap: int, lead: int, samples_per_stream: int,
           wide: bool = False, scramble: bool = False, seed: int = 0, stream_index: int = 0) -> np.ndarray:
    """y of one stream of sc_tx_channel_dev (see ``channel``)."""
    z = clean(oracle, bits, n_packets=n_packets, gap=gap, lead=lead, samples_per_stream=samples_per_stream,
              wide=wide, scramble=scramble)
    return channel(z, params, seed=seed, stream=stream_index)
