/*
 * singlecarrier_b200.h -- C ABI of libsinglecarrier_b200.so (batched, handle based).
 *
 * The reference (srsampson/SingleCarrier) has no plugin/FFI layer: its boundary is its seven
 * headers and one global-state stream per process.  This library keeps those symbols as a
 * drop-in (see include/sc_compat/ *.h: fir.h, equalizer.h, kalman.h, scramble.h, fft.h,
 * qpsk_internal.h) and adds the batched layer below, which is what a caller binds to when it
 * has thousands of independent 8 kHz streams.  Plain pointers and sizes only; no torch types.
 *
 * A "modem bank" is N synchronized streams.  Every stream of a bank is at the same call index
 * n (number of qpsk_rx_frame() calls made so far), exactly like N copies of the reference
 * process fed in lock step.  Each entry point cites the reference interface it replaces.
 *
 * All functions return SC_OK (0) or a negative SC_E* code; sc_last_error() gives the text.
 * There is no CPU fallback: without a CUDA device every compute entry point fails with
 * SC_ECUDA.
 */
#ifndef SINGLECARRIER_B200_H
#define SINGLECARRIER_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SC_FRAME_SIZE        1880   /* samples per qpsk_rx_frame() call, qpsk_internal.h:47 */
#define SC_SYMBOLS_PER_FRAME 376    /* FRAME_SIZE / CYCLES                                   */
#define SC_PREAMBLE_LENGTH   128    /* qpsk_internal.h:52                                    */
#define SC_DATA_SYMBOLS      31     /* qpsk_internal.h:40                                    */
#define SC_BITS_PER_CALL     62     /* decided bits per valid call (SURVEY F5)               */
#define SC_NTAPS             49     /* fir.h:16                                              */
#define SC_EQ_LENGTH         5      /* kalman.h:26                                           */
#define SC_PACKET_SYMBOLS    376    /* 128 preamble + 8 x 31 data                            */

#define SC_OK        0
#define SC_EINVAL   -1
#define SC_ECUDA    -2
#define SC_ENOMEM   -3
#define SC_ESTATE   -4

#define SC_FLAG_WIDE      0x1u      /* firwide=true: alpha=0.5 taps (qpsk.c:60)              */
#define SC_FLAG_DEBUG_EQ  0x2u      /* keep eq_coeff[5] of every call (parity tests)         */
#define SC_FLAG_PACKET    0x4u      /* packet mode (extension, see sc_rx_packets_*): TX scrambles,
                                       RX can decode all 8 x 31 data symbols of a packet     */

typedef struct sc_modem sc_modem;

/*
 * Result of one qpsk_rx_frame() call of one stream (32 bytes, one DRAM sector).
 *   bits      bit k = bits[k] of the reference's output row: bits[2i] = Q, bits[2i+1] = I of
 *             data symbol i, descrambled (qpsk.c:206-215).  Decided for invalid calls too
 *             (the reference computes and discards them, qpsk.c:225-229).
 *   cost      valid: the DEBUG2 "Mean" = magnitude() (qpsk.c:190); invalid: the summed
 *             data_eq() returns tested against EOF_COST_VALUE (qpsk.c:223-235).
 *   rx_timing the static rx_timing AFTER the call (qpsk.c:219).
 */
typedef struct {
    uint64_t bits;
    float    max_value;     /* correlate() maximum, qpsk.c:176-183 */
    float    cost;
    int16_t  max_index;
    int16_t  matches;       /* equalize() return, qpsk.c:188       */
    int16_t  rx_timing;
    uint8_t  valid;         /* qpsk_rx_frame() return value         */
    uint8_t  reserved0;
    uint32_t call_index;    /* n, counted from the bank's cold start */
    uint32_t reserved1;
} sc_frame_result;

/* ---- life cycle ------------------------------------------------------------------------ */

/* Replaces the start-up block of main(), qpsk.c:361-368,427-434: cold state for n_streams
 * streams on CUDA device `device`.  foffset_hz is the reference's FOFFSET macro (qpsk.c:67). */
int  sc_create(sc_modem **out, int device, int64_t n_streams, uint32_t flags, float foffset_hz);
void sc_destroy(sc_modem *m);
int  sc_reset(sc_modem *m);                       /* back to call index 0, cold state */
int64_t  sc_n_streams(const sc_modem *m);
uint32_t sc_call_index(const sc_modem *m);
const char *sc_last_error(void);
const char *sc_version(void);
int  sc_device_count(void);
/* number of kernel launches issued by this library since load (bench.py's gpu_launches) */
uint64_t sc_launch_count(void);

/* Options.  SC_OPT_SLAB_PARTS: split the bank into this many slabs of streams, issued round-robin
 * on the library's internal CUDA streams (0 = default).  SC_OPT_PROFILE: bracket every front-end
 * and tracking kernel launch with CUDA events on the stream it is launched on; sc_profile_read()
 * synchronizes and returns {front-end ms, front-end launches, tracking ms, tracking launches}
 * accumulated since the last read (use with SC_OPT_SLAB_PARTS = 1 so launches do not overlap). */
#define SC_OPT_SLAB_PARTS 1
#define SC_OPT_PROFILE    2
/* SC_OPT_H2D_MODE: how sc_rx_frames_host moves the samples to the device (default SC_H2D_COLUMNS; the
 * environment variable SC_H2D_MODE overrides the default at sc_create).  All modes give identical results. */
#define SC_OPT_H2D_MODE   3
#define SC_H2D_COLUMNS    0   /* per frame: one 2-D copy of sample columns 80..1703 (86 % of the bytes)         */
#define SC_H2D_ROWS       1   /* per block of frames: one 2-D copy, rows trimmed by 256 samples                 */
#define SC_H2D_FULL       2   /* whole frames: one 2-D copy per block, a plain 1-D copy when streams are dense  */
#define SC_H2D_COLUMNS_3D 3   /* the COLUMNS bytes as one 3-D copy per block (stream_stride % 1880 == 0)        */
/* SC_OPT_FE_SEARCH: how the fused front-end finds the preamble.  Identical results either way. */
#define SC_OPT_FE_SEARCH     4
#define SC_FE_SEARCH_DIRECT  0   /* all 128 lags with the exact sequential sums                                   */
#define SC_FE_SEARCH_MMA     1   /* proposed on the tensor cores, the candidates verified with the exact sums      */
#define SC_FE_SEARCH_TCGEN05 2   /* the same with tcgen05.mma / tensor memory, 8 stream-frames per CTA             */
/* SC_OPT_TRACKER: which kernel runs the per-stream equalizer loop.  Identical results either way: the lane-
 * cooperative kernel executes the same operations in the same order, 16 lanes per stream, and is what makes a
 * bank too small to fill the GPU with one thread per stream 3x faster per call. */
#define SC_OPT_TRACKER       5
#define SC_TRACKER_AUTO      0   /* cooperative up to SC_TRACKER_COOP_MAX streams per launch, else one thread each */
#define SC_TRACKER_THREAD    1
#define SC_TRACKER_COOP      2
#define SC_TRACKER_COOP_MAX  1024
/* SC_OPT_OVERLAP: how the calls of a batch are queued.  Identical results either way.  A call's 128 training steps
 * need only its symbol window; rx_timing (which the previous call may change) enters with the 31 data steps.  With
 * the tracker cut there, the even and the odd calls of a batch form two chains that run side by side on two CUDA
 * streams -- about twice the speed for a bank too small to fill the GPU, extra launches and traffic for a large one.
 * AUTO: overlapped up to SC_OVERLAP_MAX streams per bank. */
#define SC_OPT_OVERLAP       6
#define SC_OVERLAP_AUTO      0
#define SC_OVERLAP_OFF       1
#define SC_OVERLAP_ON        2
#define SC_OVERLAP_MAX       32768
int  sc_set_option(sc_modem *m, int option, int64_t value);
int  sc_profile_read(sc_modem *m, double out[4]);
/* bytes queued host->device (out[0]) and device->host (out[1]) by sc_rx_frames_host since sc_create */
int  sc_transfer_bytes(const sc_modem *m, uint64_t out[2]);
/* frees the process-wide device caches (FFT twiddle / permutation tables) */
int  sc_release_caches(void);

/* ---- checkpoint / resume (SURVEY section 5; the reference cannot even reset its statics, qpsk.c:34-53) --- */

/* Everything a bank needs to continue bit-exactly in another handle or process: per stream rx_timing, the
 * tracker window, the pending (max_index, max_value) and the last frame of samples; per bank the call
 * index, RXMemory (src/scramble.c:42), fbb_rx_phase (qpsk.c:50) and the last frame's phasor table.
 * sc_state_size() bytes are written to / read from HOST memory; import needs a bank created with the same
 * n_streams, flags and foffset_hz (SC_EINVAL otherwise) and also clears a failed-batch condition. */
int64_t sc_state_size(const sc_modem *m);
int  sc_state_export(sc_modem *m, void *buf, int64_t buf_bytes);
int  sc_state_import(sc_modem *m, const void *buf, int64_t buf_bytes);

/* ---- RX: replaces the while(1) loop of main() calling qpsk_rx_frame(), qpsk.c:436-458 --- */

/*
 * n_frames calls per stream.  Stream s, call j reads 1880 int16 at in + s*stream_stride +
 * j*1880 (stream_stride in samples, >= n_frames*1880).  results[s*result_stride + j] receives
 * the call's result (result_stride in records, >= n_frames).  eq_dbg (may be NULL; needs
 * SC_FLAG_DEBUG_EQ) receives eq_coeff[5] as 10 floats at (s*result_stride + j)*10.
 *
 * _dev: all pointers are device pointers on the bank's device; work is ordered after
 *       everything already queued on `stream` (a cudaStream_t) and `stream` waits for it.
 * _host: all pointers are host pointers (pinned gives asynchronous copies); host->device
 *        copies of the samples and device->host copies of the results are pipelined with the
 *        kernels in slabs of streams; returns after everything has landed.  Only samples
 *        80..1703 of each frame are transferred: no other sample can influence any output.
 */
int sc_rx_frames_dev(sc_modem *m, const int16_t *in, int64_t stream_stride, int n_frames,
                     sc_frame_result *results, int64_t result_stride, float *eq_dbg, void *stream);
int sc_rx_frames_host(sc_modem *m, const int16_t *in, int64_t stream_stride, int n_frames,
                      sc_frame_result *results, int64_t result_stride, float *eq_dbg);

/* ---- packet mode: an EXTENSION with no counterpart in the reference ----------------------------- */

/*
 * The reference decodes 31 of a packet's 8 x 31 data symbols, never scrambles on transmit and reads the late
 * symbols of a window from unfiltered samples (qpsk.c:206-215, 386, 397, 161 -- TODOs / commented out).  With
 * SC_FLAG_PACKET the library finishes them WITHOUT changing anything the reference computes: sc_rx_packets_*
 * produce exactly the results of sc_rx_frames_* and, in addition, one sc_packet_result per VALID call n >= 2:
 * kalman_reset, the 128 training steps, then data_eq over all 248 data symbols of the packet (equalizer state
 * carried through the 8 frames, descrambler seeded per packet), on symbols taken from the CONTINUOUS
 * matched-filter output at 1880 (n-2) + 5 (max_index + j) + T.  Specification: oracle/sc_oracle_ext.c.
 * The transmit side (sc_tx_*_dev of a SC_FLAG_PACKET bank) seeds the TX register after every preamble and
 * scrambles every data dibit (qpsk.c:386,397 un-commented); `bits` / `bits_out` are the payload.
 */
typedef struct {
    uint64_t bits[8];       /* frame f: bit 2i = Q, bit 2i+1 = I of data symbol i, descrambled */
    int32_t  stream;
    uint32_t call_index;    /* the valid call this packet belongs to */
    int16_t  max_index;
    int16_t  matches;       /* of the packet's own training pass (equals the call's) */
    float    cost;          /* sum of the 248 data_eq() returns */
    uint32_t reserved0, reserved1;
    uint64_t reserved2;
} sc_packet_result;         /* 96 bytes */

/* packets: capacity records, appended in no particular order; *n_packets receives the number of packets found
 * (it can exceed capacity: the surplus is dropped).  _dev: device pointers, n_packets a device uint64 that is
 * ACCUMULATED into; _host: host pointers, *n_packets is set. */
int sc_rx_packets_dev(sc_modem *m, const int16_t *in, int64_t stream_stride, int n_frames,
                      sc_frame_result *results, int64_t result_stride, sc_packet_result *packets,
                      int64_t capacity, uint64_t *n_packets, void *stream);
int sc_rx_packets_host(sc_modem *m, const int16_t *in, int64_t stream_stride, int n_frames,
                       sc_frame_result *results, int64_t result_stride, sc_packet_result *packets,
                       int64_t capacity, uint64_t *n_packets);

/* Host helper: unpack results into the reference's on-disk format (qpsk.c:455-457): for every
 * VALID call, 62 bytes (0/1) are written to rows + (s*n_frames + j)*62; other rows untouched. */
void sc_unpack_bits(const sc_frame_result *results, int64_t n_records, uint8_t *rows);

/* ---- TX: replaces preamble_modulate()/qpsk_modulate()/qpsk_tx_frame(), qpsk.c:278-342 ---- */

/*
 * Synthesize n_packets packets per stream exactly as main() does (qpsk.c:380-413): per packet
 * one 640-sample BPSK preamble at half amplitude, eight 155-sample QPSK data frames built from
 * bits (62 bytes of 0/1 per data frame: bits[2i] = Q, bits[2i+1] = I, qpsk.c:251-256), then
 * gap_samples zeros that do NOT pass through the filter or the NCO (qpsk.c:410-412; the
 * reference uses 903).  lead_in[s] zeros precede the first packet of stream s (NULL = 0).
 * tx_filter and fbb_tx_phase persist across frames and packets as in the reference.
 *   bits: device pointer, [n_streams][n_packets][8][62] bytes, or NULL to draw them from the
 *         counter-based generator seeded with `seed` (returned through bits_out if not NULL,
 *         same layout).
 *   out : device pointer, stream s at out + s*stream_stride; samples beyond the last packet
 *         up to samples_per_stream are zero filled.
 * The bank's TX state is cold at the start of the call (one call = one whole transmission).
 */
int sc_tx_packets_dev(sc_modem *m, const uint8_t *bits, uint8_t *bits_out, uint64_t seed,
                      int n_packets, int gap_samples, const int32_t *lead_in,
                      int16_t *out, int64_t stream_stride, int64_t samples_per_stream, void *stream);

/*
 * Channel for synthetic loop-back (BASELINE.json configs 2-5; no counterpart in the reference
 * beyond FOFFSET): same synthesis as sc_tx_packets_dev, then, in this order, on the analytic TX
 * signal z[p] of stream s (p = output sample index, 0 at the stream's first sample, lead-in
 * included; z = 0 in the lead-in, the dead air and the tail):
 *   1. 2-tap channel h = [1, a[s]*exp(j*theta[s])] at delay d[s] samples:
 *      e[p] = z[p] + a[s]*exp(j*theta[s])*z[p - d[s]];
 *   2. rotation by exp(j(2*pi*(df[s] + 0.5*drift[s]*t)*t + phi[s])), t = p / 8000 s, i.e. the
 *      offset is that of the receiver's oscillator and applies to both paths alike;
 *   3. real part + real AWGN of standard deviation sigma[s] (int16 LSB), drawn from a counter-based
 *      generator keyed by (seed, s, p), s counted over the whole bank;
 *   4. saturation to +-32767 and rounding to nearest (ties to even).
 * Any of the per-stream parameter arrays (device pointers) may be NULL: echo_delay then means 1,
 * every other array 0.
 */
typedef struct {
    const float   *df_hz;       /* frequency offset                  */
    const float   *phi_rad;     /* phase offset                      */
    const float   *drift_hz_s;  /* linear frequency drift            */
    const float   *sigma_lsb;   /* AWGN standard deviation, int16 LSB */
    const float   *echo_amp;    /* second path amplitude a           */
    const float   *echo_theta;  /* second path phase                 */
    const int32_t *echo_delay;  /* second path delay in samples (1..16) */
} sc_channel;

int sc_tx_channel_dev(sc_modem *m, const uint8_t *bits, uint8_t *bits_out, uint64_t seed,
                      int n_packets, int gap_samples, const int32_t *lead_in, const sc_channel *ch,
                      int16_t *out, int64_t stream_stride, int64_t samples_per_stream, void *stream);

/* ---- stage entry points (device pointers; batched forms of the reference's L1 functions) -- */

/* fir(), fir.h:19 / src/fir.c:22-44, for n_streams independent (memory, sample) pairs:
 * memory[s*49 .. +49), sample[s*sample_stride .. +length) complex float, both updated in place.
 * wide: bit 0 = the reference's `choice` (alpha=0.5 taps); bit 1 = SC_FIR_FAST, the explicitly named
 * tolerance mode: multiply-adds are contracted (FFMA), results agree with the reference to ~1e-6
 * relative instead of bit for bit, and the kernel becomes HBM-bound.  Never used by sc_rx_frames_*. */
#define SC_FIR_FAST 0x2
int sc_fir_batch_dev(int device, int64_t n_streams, int wide, float *memory, float *sample,
                     int64_t sample_stride, int length, void *stream);

/* correlate() + argmax, qpsk.c:88-96,172-183: symbols[s*symbol_stride .. +255) complex float
 * -> max_index[s], max_value[s].  Two kernels, identical results to the last bit:
 *   sc_preamble_search_batch_dev         all 128 correlations are PROPOSED on the tensor cores (bf16 split of the
 *                                        operands, fp32 accumulation, rigorous error bound), then only the lags that
 *                                        can be the maximum are evaluated with the reference's exact sequential sums;
 *   sc_preamble_search_fft_batch_dev     the same scheme with an FFT proposer: two 256-point transforms held in the
 *                                        registers of one warp (radix-4 butterflies, lane exchanges by warp shuffle),
 *                                        warp-reduced argmax, exact verification of the candidates;
 *   sc_preamble_search_direct_batch_dev  every lag with the exact sums (the form the RX chain fuses). */
int sc_preamble_search_batch_dev(int device, int64_t n_streams, const float *symbols,
                                 int64_t symbol_stride, int32_t *max_index, float *max_value,
                                 void *stream);
/* the two tensor-core forms by name: mma.sync (any window layout) and tcgen05 + tensor memory + TMA (symbol_stride
 * >= 256 and even, array 16-byte aligned; approx, optional, receives the proposed |correlation|^2 [n_streams][128]).
 * sc_preamble_search_batch_dev picks tcgen05 when the layout allows it. */
int sc_preamble_search_mma_batch_dev(int device, int64_t n_streams, const float *symbols,
                                     int64_t symbol_stride, int32_t *max_index, float *max_value,
                                     void *stream);
int sc_preamble_search_tcgen05_batch_dev(int device, int64_t n_streams, const float *symbols,
                                         int64_t symbol_stride, int32_t *max_index, float *max_value,
                                         float *approx, void *stream);
int sc_preamble_search_fft_batch_dev(int device, int64_t n_streams, const float *symbols,
                                     int64_t symbol_stride, int32_t *max_index, float *max_value,
                                     void *stream);
int sc_preamble_search_direct_batch_dev(int device, int64_t n_streams, const float *symbols,
                                        int64_t symbol_stride, int32_t *max_index, float *max_value,
                                        void *stream);

/* kalman_reset() + equalize() + the data_eq() loop, qpsk.c:186-236: the decision half of one
 * qpsk_rx_frame() call on an explicit symbol window.  symbols[s*symbol_stride .. +290) complex
 * float, max_index[s] from the search, rx_timing[s] at entry, keystream position = call_index.
 * results[s] as above, rx_timing[s] updated in place. */
int sc_track_decide_batch_dev(int device, int64_t n_streams, const float *symbols,
                              int64_t symbol_stride, const int32_t *max_index, const float *max_value,
                              int32_t *rx_timing, uint32_t call_index, sc_frame_result *results,
                              float *eq_dbg, void *stream);

/* fft(), fft.h:46 / src/fft.c:133: n_batches independent length-nfft complex FFTs (any nfft the
 * reference accepts: radix 4, 2, 3, 5 and generic stages), out of place, unnormalised inverse.
 * Same factorisation, butterfly arithmetic and twiddles as src/fft.c. */
int sc_fft_batch_dev(int device, int64_t n_batches, int nfft, int inverse, const float *in, float *out,
                     void *stream);
/* fftr()/fftri(), fft.h:51-52 (encode_fftr/encode_fftri in src/fft.c:139-186): real nfft (even)
 * -> nfft/2+1 complex bins, and back (unnormalised). */
int sc_fftr_batch_dev(int device, int64_t n_batches, int nfft, const float *in, float *out, void *stream);
int sc_fftri_batch_dev(int device, int64_t n_batches, int nfft, const float *in, float *out, void *stream);

/* ---- lock / bit statistics (SURVEY section 5; reduced across GPUs with one ncclAllReduce) ----- */

#define SC_N_COUNTERS 16
/* counters (device pointer, uint64[16], ACCUMULATED into): 0 calls, 1 valid calls, 2 sum matches,
 * 3 sum matches over valid calls, 4 sum max_index over valid calls, 5 popcount of bits over valid
 * calls, 6 sum of (lo32(bits) + hi32(bits)) over valid calls (a checksum), 7 sum rx_timing,
 * 8..15 histogram of matches in bins of 16.  All plain sums: ranks combine them by addition. */
int sc_lock_stats_dev(int device, const sc_frame_result *results, int64_t n_streams, int64_t result_stride,
                      int n_frames, uint64_t *counters, void *stream);

/* Self-test: number of float bit patterns in [lo_bits, hi_bits] (as IEEE binary32) for which the
 * tracking kernel's branch-free reciprocal differs from the correctly rounded one (expected 0 for
 * 2^-120 .. 2^120).  *mismatches: device uint64, accumulated into. */
int sc_selftest_rcp_dev(int device, uint32_t lo_bits, uint32_t hi_bits, uint64_t *mismatches, void *stream);

#define SC_N_BER_COUNTERS 8
/* Bit errors against the transmitted bits, on the device (BASELINE.json configs 3-5; the reference's only
 * counter is preamble_frames_detected, qpsk.c:70,193).  results must hold calls 0..n_frames-1 of a cold
 * started bank.  A valid call n >= 2 found its preamble at decimated index max_index of the window taken
 * from frame n-2 with the rx_timing in force after call n-2, i.e. at sample
 * pos = (n-2)*1880 + 5*max_index + rx_timing - 48 (two 24-sample RRC delays) of the stream; it is "aligned"
 * when pos - lead_in[s] (lead_in NULL = 0) lies within 10 samples (inclusive) of the start
 * j*(1880 + gap) of a transmitted packet j, 0 <= j < n_packets.  Its 62 decided bits are the first data
 * frame of packet j (SURVEY F5); TX does not scramble (qpsk.c:397) and RX descrambles, so the low 62 bits
 * of bits ^ keystream(n) ^ tx_bits are the error pattern.
 *   tx_bits : device, [n_streams][n_packets][8][62] bytes of 0/1 (sc_tx_*_dev's bits_out)
 *   group   : device int32[n_streams] or NULL (all streams in group 0), values 0..n_groups-1; a stream
 *             whose group lies outside that range is not counted at all
 *   counters: device uint64[n_groups][8], ACCUMULATED into: 0 calls (n >= 2), 1 valid, 2 aligned, 3 bits
 *             compared (62 per aligned call), 4 bit errors, 5..7 reserved (0).  Plain sums. */
int sc_ber_stats_dev(int device, const sc_frame_result *results, int64_t n_streams, int64_t result_stride,
                     int n_frames, const uint8_t *tx_bits, int n_packets, const int32_t *lead_in, int gap_samples,
                     const int32_t *group, int n_groups, uint64_t *counters, void *stream);

/* ---- multi-GPU reduction of the counters (SURVEY section 8e: the path's only collective) ------------------ */

/* ncclAllReduce(sum) of n_counters uint64 in place on `stream`; nccl_comm is a ncclComm_t created by the
 * caller (ncclCommInitRank / ncclCommInitAll) or by the helpers below.  NCCL is bound at run time from the
 * libnccl.so.2 already loaded in the process (e.g. PyTorch's), else from the system library. */
int sc_reduce_stats(uint64_t *counters, int n_counters, void *nccl_comm, void *stream);
#define SC_NCCL_UNIQUE_ID_BYTES 128
int sc_comm_unique_id(void *id128);                                 /* ncclGetUniqueId (rank 0; broadcast it) */
int sc_comm_init_rank(void **comm, int n_ranks, int rank, const void *id128, int device);
int sc_comm_init_all(void **comms, int n_devices, const int *devices);  /* one process, n GPUs */
int sc_comm_destroy(void *comm);
int sc_comm_group_start(void);          /* ncclGroupStart/End: one process issuing the reduce of several ranks */
int sc_comm_group_end(void);

/* ---- device memory for callers without a CUDA binding (plain C, cgo, Rust FFI) ------------------------------ */
int sc_device_malloc(int device, size_t bytes, void **ptr);        /* zero-filled */
int sc_device_free(int device, void *ptr);
#define SC_COPY_H2D 0
#define SC_COPY_D2H 1
#define SC_COPY_D2D 2
int sc_device_copy(int device, void *dst, const void *src, size_t bytes, int kind);   /* synchronous */
int sc_device_synchronize(int device);

/* ---- host memory and the PCIe ceiling -------------------------------------------------------------------- */

/* Page-locked host memory placed on the NUMA node of `device` (thread affinity is narrowed to that node's
 * CPUs while the pages are first touched).  numa_node (may be NULL) receives the node used, -1 if unknown. */
int sc_host_alloc(void **ptr, size_t bytes, int device, int *numa_node);
int sc_host_free(void *ptr);
/* Page-lock caller-owned memory in place (cudaHostRegister), so sc_rx_frames_host copies asynchronously. */
int sc_host_register(void *ptr, size_t bytes);
int sc_host_unregister(void *ptr);
/* Measures plain copies between pinned host memory and `device` for at least min_seconds (CUDA events):
 * row_bytes == 0: contiguous cudaMemcpyAsync of buffer_bytes; else cudaMemcpy2DAsync of rows of row_bytes
 * taken every src_pitch_bytes.  d2h != 0 reverses the direction.  Used by bench.py on all ranks at once to
 * establish the platform ceiling that sc_rx_frames_host is judged against. */
int sc_h2d_probe(int device, size_t buffer_bytes, size_t row_bytes, size_t src_pitch_bytes, double min_seconds,
                 int d2h, double *gbytes_per_s);

/* ---- small utilities used by host code and tests --------------------------------------- */

/* RX/TX NCO phasor table exactly as the reference's recurrences generate it (qpsk.c:138-147,
 * 301-306): out[f*1880 + i] = phasor used for sample i of call f (f = first_call ..). Host out. */
int sc_nco_table_host(sc_modem *m, int tx, uint32_t first_call, int n_calls, float *out);
/* descrambler keystream word of call n (62 bits), src/scramble.c:57-69 seeded at qpsk.c:434 */
uint64_t sc_keystream_word(uint32_t call_index);

#ifdef __cplusplus
}
#endif
#endif
