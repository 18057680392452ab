"""singlecarrier_b200 -- B200-native (sm_100a) batched 1600-baud QPSK modem chain.

Drop-in for the RX/TX hot path of srsampson/SingleCarrier (qpsk_rx_frame / qpsk_tx_frame and the
fir / equalizer / kalman / scramble primitives underneath), processing thousands of independent
8 kHz streams per launch.  The product is the C-ABI library ``libsinglecarrier_b200.so``
(``include/singlecarrier_b200.h``); this package is the thin Python host mirror used by the tests
and ``bench.py``.  PyTorch is used only for device memory, streams and ``torch.distributed``.
"""
from ._lib import LIB_PATH, SingleCarrierError, lib  # noqa: F401
from .modem import (BITS_PER_CALL, CODE_R12, CODE_R23, CODE_R34, DATA_SYMBOLS, FRAME_SIZE,  # noqa: F401
                    PACKET_DATA_SYMBOLS, PACKET_DTYPE, PAYLOAD_DTYPE, PAYLOAD_EX_DTYPE, PAYLOAD_MAX, RESULT_DTYPE,
                    payload_bytes,
                    SYMBOLS_PER_FRAME, ModemBank, NcclComm, PinnedBuffer, h2d_probe, keystream_word, launch_count,
                    packet_keystream_word, packet_soft_bits, soft_bits, unpack_bits, unpack_packet_bits)

__all__ = ["ModemBank", "NcclComm", "PinnedBuffer", "h2d_probe", "RESULT_DTYPE", "PACKET_DTYPE", "PAYLOAD_DTYPE",
           "unpack_packet_bits", "FRAME_SIZE", "BITS_PER_CALL",
           "SYMBOLS_PER_FRAME", "DATA_SYMBOLS", "PACKET_DATA_SYMBOLS", "unpack_bits", "soft_bits", "packet_soft_bits",
           "keystream_word", "packet_keystream_word", "launch_count", "SingleCarrierError", "lib", "LIB_PATH",
           "PAYLOAD_EX_DTYPE", "PAYLOAD_MAX", "CODE_R12", "CODE_R23", "CODE_R34", "payload_bytes"]
