"""Loader for libsinglecarrier_b200.so (the C ABI declared in include/singlecarrier_b200.h).

There is no CPU fallback: if the shared library is missing the import fails loudly, and every
compute entry point of the library itself fails with SC_ECUDA when no CUDA device is present.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libsinglecarrier_b200.so")

SC_OK, SC_EINVAL, SC_ECUDA, SC_ENOMEM, SC_ESTATE = 0, -1, -2, -3, -4
SC_FLAG_WIDE, SC_FLAG_DEBUG_EQ, SC_FLAG_PACKET, SC_FLAG_PACKET_DD = 0x1, 0x2, 0x4, 0x8


class SingleCarrierError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"singlecarrier_b200 error {code}: {msg}")
        self.code = code


class Channel(C.Structure):
    """sc_channel (include/singlecarrier_b200.h): device pointers, 0 = not used."""
    _fields_ = [("df_hz", C.c_void_p), ("phi_rad", C.c_void_p), ("drift_hz_s", C.c_void_p),
                ("sigma_lsb", C.c_void_p), ("echo_amp", C.c_void_p), ("echo_theta", C.c_void_p),
                ("echo_delay", C.c_void_p)]


def _load() -> C.CDLL:
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `make -C singlecarrier_b200/csrc` "
            "(or `python -c 'import __graft_entry__ as g; g.build()'`). "
            "singlecarrier_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, u32, u64, f32 = C.c_void_p, C.c_int, C.c_int64, C.c_uint32, C.c_uint64, C.c_float

    def sig(name, restype, *argtypes):
        fn = getattr(lib, name)
        fn.restype = restype
        fn.argtypes = list(argtypes)

    sig("sc_create", i32, C.POINTER(vp), i32, i64, u32, f32)
    sig("sc_destroy", None, vp)
    sig("sc_reset", i32, vp)
    sig("sc_n_streams", i64, vp)
    sig("sc_call_index", u32, vp)
    sig("sc_last_error", C.c_char_p)
    sig("sc_version", C.c_char_p)
    sig("sc_device_count", i32)
    sig("sc_launch_count", u64)
    sig("sc_set_option", i32, vp, i32, i64)
    sig("sc_profile_read", i32, vp, C.POINTER(C.c_double))
    sig("sc_rx_frames_dev", i32, vp, vp, i64, i32, vp, i64, vp, vp)
    sig("sc_rx_frames_host", i32, vp, vp, i64, i32, vp, i64, vp)
    sig("sc_rx_frames_soft_dev", i32, vp, vp, i64, i32, vp, i64, vp, vp)
    sig("sc_rx_frames_soft_host", i32, vp, vp, i64, i32, vp, i64, vp)
    sig("sc_rx_packets_dev", i32, vp, vp, i64, i32, vp, i64, vp, i64, vp, vp)
    sig("sc_rx_packets_host", i32, vp, vp, i64, i32, vp, i64, vp, i64, C.POINTER(C.c_uint64))
    sig("sc_rx_packets_soft_dev", i32, vp, vp, i64, i32, vp, i64, vp, vp, i64, vp, vp, vp)
    sig("sc_rx_packets_soft_host", i32, vp, vp, i64, i32, vp, i64, vp, vp, i64, C.POINTER(C.c_uint64), vp)
    sig("sc_packet_keystream_word", u64, i32)
    sig("sc_unpack_bits", None, vp, i64, vp)
    sig("sc_tx_packets_dev", i32, vp, vp, vp, u64, i32, i32, vp, vp, i64, i64, vp)
    sig("sc_tx_channel_dev", i32, vp, vp, vp, u64, i32, i32, vp, C.POINTER(Channel), vp, i64, i64, vp)
    sig("sc_fir_batch_dev", i32, i32, i64, i32, vp, vp, i64, i32, vp)
    sig("sc_preamble_search_batch_dev", i32, i32, i64, vp, i64, vp, vp, vp)
    sig("sc_preamble_search_direct_batch_dev", i32, i32, i64, vp, i64, vp, vp, vp)
    sig("sc_preamble_search_fft_batch_dev", i32, i32, i64, vp, i64, vp, vp, vp)
    sig("sc_preamble_search_mma_batch_dev", i32, i32, i64, vp, i64, vp, vp, vp)
    sig("sc_preamble_search_tcgen05_batch_dev", i32, i32, i64, vp, i64, vp, vp, vp, vp)
    sig("sc_track_decide_batch_dev", i32, i32, i64, vp, i64, vp, vp, vp, u32, vp, vp, vp)
    sig("sc_fft_batch_dev", i32, i32, i64, i32, i32, vp, vp, vp)
    sig("sc_fftr_batch_dev", i32, i32, i64, i32, vp, vp, vp)
    sig("sc_fftri_batch_dev", i32, i32, i64, i32, vp, vp, vp)
    sig("sc_lock_stats_dev", i32, i32, vp, i64, i64, i32, vp, vp)
    sig("sc_selftest_rcp_dev", i32, i32, u32, u32, vp, vp)
    sig("sc_transfer_bytes", i32, vp, C.POINTER(C.c_uint64))
    sig("sc_release_caches", i32)
    sig("sc_state_size", i64, vp)
    sig("sc_state_export", i32, vp, vp, i64)
    sig("sc_state_import", i32, vp, vp, i64)
    sig("sc_ber_stats_dev", i32, i32, vp, i64, i64, i32, vp, i32, vp, i32, vp, i32, vp, vp)
    sig("sc_packet_ber_stats_dev", i32, i32, vp, i64, vp, vp, i64, i64, i32, vp, i32, vp, i32, vp, i32, vp, vp)
    sig("sc_reduce_stats", i32, vp, i32, vp, vp)
    sig("sc_comm_unique_id", i32, vp)
    sig("sc_comm_init_rank", i32, C.POINTER(vp), i32, i32, vp, i32)
    sig("sc_comm_init_all", i32, C.POINTER(vp), i32, C.POINTER(i32))
    sig("sc_comm_destroy", i32, vp)
    sig("sc_comm_group_start", i32)
    sig("sc_comm_group_end", i32)
    sig("sc_device_malloc", i32, i32, C.c_size_t, C.POINTER(vp))
    sig("sc_device_free", i32, i32, vp)
    sig("sc_device_copy", i32, i32, vp, vp, C.c_size_t, i32)
    sig("sc_device_synchronize", i32, i32)
    sig("sc_host_alloc", i32, C.POINTER(vp), C.c_size_t, i32, C.POINTER(i32))
    sig("sc_host_free", i32, vp)
    sig("sc_host_register", i32, vp, C.c_size_t)
    sig("sc_host_unregister", i32, vp)
    sig("sc_h2d_probe", i32, i32, C.c_size_t, C.c_size_t, C.c_size_t, C.c_double, i32, C.POINTER(C.c_double))
    sig("sc_nco_table_host", i32, vp, i32, u32, i32, vp)
    sig("sc_keystream_word", u64, u32)
    return lib


lib = _load()


def check(rc: int) -> None:
    if rc != SC_OK:
        raise SingleCarrierError(rc, lib.sc_last_error().decode(errors="replace"))
