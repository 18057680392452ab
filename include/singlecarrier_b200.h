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
#define SC_FLAG_PACKET_DD 0x8u      /* with SC_FLAG_PACKET only (else sc_create: SC_EINVAL):
                                       packets decoded by a decision-directed equalizer and
                                       carrier loop instead of the reference's Kalman one    */
#define SC_FLAG_PACKET_ACQ 0x10u    /* with SC_FLAG_PACKET | SC_FLAG_PACKET_DD only (else
                                       sc_create: SC_EINVAL): packets found by acquisition on
                                       the samples, not by the reference's per-call detection */

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
/* bytes queued host->device (out[0]) and device->host (out[1]) by sc_rx_frames_host / sc_rx_frames_soft_host
 * since sc_create (sc_rx_packets_host / sc_rx_packets_soft_host: the same for their ordinary calls; packet records
 * and packet symbols are not counted) */
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

/*
 * Soft output: the same calls, and in addition the equalizer output of every data step -- the value each
 * decision is sliced from (data_eq(), equalizer.c:64-80), before slicing and descrambling.  Data step i
 * (0..SC_DATA_SYMBOLS-1) of a call reads the symbol at sync_pos + i in a valid call and at rx_timing + i in an
 * invalid one; it is written for invalid calls too.  It is computed by the same float32 operations as the decision,
 * so bit 2i of the raw decision is (Im < 0) and bit 2i+1 is (Re < 0), and results[].bits = raw decisions XOR
 * sc_keystream_word(call_index) (valid calls).
 *
 * symbols: SC_DATA_SYMBOLS complex floats (re, im interleaved) per record, record (s, j) at
 * (s*result_stride + j) * 2*SC_DATA_SYMBOLS floats -- the same record indexing as results.  Required (NULL:
 * SC_EINVAL); a device pointer aligned to 8 bytes for _dev, a host pointer for _host (pinned gives asynchronous
 * copies; sc_transfer_bytes counts the copied symbol bytes).  results and the bank's state afterwards are exactly
 * what sc_rx_frames_* would have produced, on the same schedules (SC_OPT_OVERLAP included), so soft and plain
 * batches may alternate on one handle.  There is no eq_dbg argument.  On SC_FLAG_PACKET banks these are ordinary
 * calls (no sc_packet_result); sc_rx_packets_soft_* below gives the soft output of the packets.
 */
int sc_rx_frames_soft_dev(sc_modem *m, const int16_t *in, int64_t stream_stride, int n_frames,
                          sc_frame_result *results, int64_t result_stride, float *symbols, void *stream);
int sc_rx_frames_soft_host(sc_modem *m, const int16_t *in, int64_t stream_stride, int n_frames,
                           sc_frame_result *results, int64_t result_stride, float *symbols);

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
 *
 * The reference's equalizer diverges (its bits are near chance).  SC_FLAG_PACKET_DD decodes the same records, on the
 * same symbol grid, with a 5-tap normalised LMS filter and a second-order carrier loop instead (DESIGN.md section 8):
 * trained on the 128 preamble symbols, then decision-directed over the 248 data symbols.  Fields then: bits as below;
 * matches is the call's; cost is the float32 sequential sum of |d - y|^2 over the 248 data steps (d the decision, y
 * the derotated equalizer output, the value the soft forms return).  Every other result is unchanged.
 *
 * SC_FLAG_PACKET_ACQ (with SC_FLAG_PACKET | SC_FLAG_PACKET_DD) replaces the per-call detection as the source of records
 * by acquisition on the samples (DESIGN.md section 8b): a differential preamble metric rho on the matched-filter output
 * at every symbol position, which a carrier offset does not change, at most one packet per 1880-sample frame.  The
 * batch that contains call n emits the packets whose grid starts in frame n-2.  The DD loop starts from the offset the
 * metric measures.  Fields then: grid_sample (authoritative), call_index = 2 + floor(grid_sample / 1880), max_index =
 * (grid_sample mod 1880) / 5, matches = training steps whose output agrees with the preamble, acq_metric, acq_freq_hz.
 * Per-call results, per-call soft output and the bank state are those of a SC_FLAG_PACKET_DD bank.
 */
typedef struct {
    uint64_t bits[8];       /* frame f: bit 2i = Q, bit 2i+1 = I of data symbol i, descrambled */
    int32_t  stream;
    uint32_t call_index;    /* the valid call this packet belongs to */
    int16_t  max_index;
    int16_t  matches;       /* of the packet's own training pass (equals the call's) */
    float    cost;          /* sum of the 248 data_eq() returns (SC_FLAG_PACKET_DD: of |d - y|^2) */
    float    acq_metric;    /* SC_FLAG_PACKET_ACQ: rho on the record's grid, else 0 */
    float    acq_freq_hz;   /* SC_FLAG_PACKET_ACQ: carrier offset estimate nu0 * 1600 / (2 pi), else 0 */
    int64_t  grid_sample;   /* SC_FLAG_PACKET_ACQ: g, the stream's matched-filter sample of the grid's first symbol,
                               counted from the cold start, else 0 */
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

/*
 * Packet mode with soft output: sc_rx_packets_* and, in addition, the equalizer output of each of the 248 data
 * steps of every packet record written -- the value its decision is sliced from, before slicing and descrambling.
 * results, packets, capacity and n_packets mean exactly what they mean for sc_rx_packets_*; the records, results and
 * the bank's state afterwards are the same, so soft and plain batches may alternate on one handle.  The records are
 * appended in another order than sc_rx_packets_* appends them.
 *
 * packet_symbols: 8 x SC_DATA_SYMBOLS = 248 complex floats (re, im interleaved) per record; the block of packets[k]
 *   starts at float k * 496, so record k and block k always belong to the same packet (for _dev also when
 *   *n_packets does not start at 0).  Blocks of dropped records (beyond capacity) are not written.  Required (NULL:
 *   SC_EINVAL before any work, the call index does not advance); for _dev a device pointer aligned to 8 bytes.
 * symbols: NULL, or the per-call soft output with the layout and meaning of sc_rx_frames_soft_* (for _dev aligned to
 *   8 bytes).
 * Bit mapping: in data frame f (0..7) of a packet, with sym = the record's block, bit 2i of the raw decision is
 * (Im(sym[31 f + i]) < 0) and bit 2i+1 is (Re(sym[31 f + i]) < 0), and packets[k].bits[f] = raw decision XOR
 * sc_packet_keystream_word(f).  packets[k].cost is the float32 sequential sum over the 248 steps of
 * (c - Re) * 0.1f, c = (Re < 0 ? -1 : 1), each operation rounded.  On a SC_FLAG_PACKET_DD bank sym is the derotated
 * equalizer output y, the bit mapping is the same and cost is the sum of |d - y|^2 (d = the sliced +-1 +-1j).
 * sc_transfer_bytes counts what _host moves for the ordinary calls (results and per-call symbols) as for
 * sc_rx_frames_soft_host; like sc_rx_packets_host it does not count packet records or packet symbols.
 */
int sc_rx_packets_soft_dev(sc_modem *m, const int16_t *in, int64_t stream_stride, int n_frames,
                           sc_frame_result *results, int64_t result_stride, float *symbols,
                           sc_packet_result *packets, int64_t capacity, uint64_t *n_packets,
                           float *packet_symbols, void *stream);
int sc_rx_packets_soft_host(sc_modem *m, const int16_t *in, int64_t stream_stride, int n_frames,
                            sc_frame_result *results, int64_t result_stride, float *symbols,
                            sc_packet_result *packets, int64_t capacity, uint64_t *n_packets,
                            float *packet_symbols);
/* descrambler keystream word of data frame `frame` (0..7) of every packet: the register is seeded with 0x4A80 per
 * packet and advanced 62 steps per frame (0 for any other frame) */
uint64_t sc_packet_keystream_word(int frame);

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

#define SC_N_PACKET_BER_COUNTERS 32
/* Bit errors of packet-mode records (SC_FLAG_PACKET) against the transmitted bits, on the device: the counter that
 * goes with sc_rx_packets_dev / sc_rx_packets_soft_dev, so that a caller can queue the batch, this call and
 * sc_reduce_stats on one CUDA stream without a host synchronisation.
 *   packets, capacity, n_found: the buffers sc_rx_packets_dev filled; n_found is a DEVICE pointer, read by the kernel,
 *             which counts records 0 .. min(*n_found, capacity) - 1 (records accumulated over several batches are all
 *             counted).
 *   results, n_streams, result_stride, n_frames, tx_bits, n_packets, lead_in, gap_samples, group, n_groups: as for
 *             sc_ber_stats_dev (results: calls 0..n_frames-1 of a cold-started bank).
 * Alignment, the rule of sc_ber_stats_dev applied to the record: with n = call_index and
 * pos = (n-2)*1880 + 5*max_index + results[stream][n-2].rx_timing - 48 - lead_in[stream] -- or, when the record's
 * grid_sample is not 0 (SC_FLAG_PACKET_ACQ banks), pos = grid_sample - 48 - lead_in[stream] -- the record is aligned to
 * transmitted packet j when |pos - j*(1880 + gap_samples)| <= 10 and 0 <= j < n_packets.  TX scrambles and RX
 * descrambles in packet mode, so the error pattern of data frame f (0..7) is (bits[f] ^ txword(f)) & (2^62 - 1), where
 * txword(f) packs tx_bits[stream][j][f][0..61] & 1 (no keystream term).
 * A record is not counted at all when its stream is outside 0..n_streams-1, its call_index outside 2..n_frames-1 or
 * its stream's group outside 0..n_groups-1.
 *   counters: device uint64[n_groups][32], ACCUMULATED into, plain sums: 0 records counted, 1 aligned records, 2 bits
 *             compared (496 per aligned record), 3 bit errors, 4..7 reserved (0), 8+f bit errors in data frame f,
 *             16+f aligned records with at least one error in data frame f, 24+b histogram of the bit errors of an
 *             aligned record: b = 0 for none, b = 1..6 for 2^(b-1) .. 2^b - 1, b = 7 for 64 or more.  The packet
 *             error rate is (counter 1 - counter 24) / counter 1.
 * SC_EINVAL before any CUDA call: packets, n_found, results, tx_bits or counters NULL; capacity, n_streams or n_frames
 * negative; result_stride < n_frames, n_packets < 1, gap_samples < 0 or n_groups < 1.  capacity == 0, n_streams == 0
 * and n_frames < 3 launch nothing. */
int sc_packet_ber_stats_dev(int device, const sc_packet_result *packets, int64_t capacity, const uint64_t *n_found,
                            const sc_frame_result *results, int64_t n_streams, int64_t result_stride, int n_frames,
                            const uint8_t *tx_bits, int n_packets, const int32_t *lead_in, int gap_samples,
                            const int32_t *group, int n_groups, uint64_t *counters, void *stream);

/* ---- coded payload of packet-mode packets (DESIGN.md section 8c) -------------------------------------------------
 *
 * A fixed code on top of the packet format: SC_PACKET_PAYLOAD_BYTES bytes of payload, a CRC-16, a K = 7 rate-1/2
 * convolutional code and a block interleaver fill the first SC_PACKET_CODED_BITS of a packet's SC_PACKET_BITS bits;
 * the rest (the last ten data symbols, which the transmitter emits only in part) carry 0 and are never read.
 *   crc      CRC-16/CCITT-FALSE over the payload (poly 0x1021, init 0xFFFF, MSB first, no reflection, no final XOR:
 *            "123456789" -> 0x29B1), appended high byte first
 *   info     u[0..231] = the 29 bytes MSB first, u[232..237] = 0 (the encoder ends in state 0)
 *   encoder  s_t = (u[t-1] .. u[t-6]) with u[t-1] at bit 5, s_0 = 0; r = (u[t] << 6) | s_t;
 *            c[2t] = parity(r & 0133), c[2t+1] = parity(r & 0171) (octal), s_{t+1} = r >> 1; t = 0..237
 *   layout   packet bit p = 62 f + j (data frame f, bit j: the layout of sc_tx_*_dev's bits and of
 *            sc_packet_result.bits): c[n] goes to p = 17 (n mod 28) + floor(n / 28); p = 476..495 carry 0
 * All three entry points take a device, not a bank; pointers are device pointers.  SC_EINVAL before any CUDA call
 * on a NULL pointer, n or capacity < 0, or a misaligned pointer. */
#define SC_PACKET_PAYLOAD_BYTES 27
#define SC_PACKET_CODED_BITS    476
#define SC_PACKET_BITS          496

typedef struct {
    uint8_t  data[27];      /* the decoder's maximum-likelihood payload, also when crc_ok is 0 */
    uint8_t  crc_ok;        /* 1 when the CRC of data equals the decoded CRC bits */
    uint16_t flipped;       /* coded bits 0..475 whose LLR sign (L < 0: bit 1) disagrees with the decoded codeword */
    uint16_t reserved;      /* 0 */
} sc_packet_payload;        /* 32 bytes */

/* payload [n][27] -> bits [n][8][62] of 0/1, the bits sc_tx_packets_dev / sc_tx_channel_dev take: payloads laid out
 * [n_streams][n_packets][27] feed the transmitter directly.  n == 0 launches nothing. */
int sc_packet_encode_dev(int device, const uint8_t *payload, int64_t n, uint8_t *bits, void *stream);

/* Log-likelihood ratios of the 496 bits of every packet record, L > 0 favouring bit 0, from the packet symbols of
 * sc_rx_packets_soft_*: for record k < min(*n_found, capacity), 496 floats at llr + k * 496 from the 248 complex
 * floats at packet_symbols + k * 496 (the indexing of packet_symbols).  n_found is a DEVICE pointer read by the
 * kernel, so the call queues behind sc_rx_packets_soft_dev without a host synchronisation; blocks at or beyond that
 * count are not touched.  With y the record's block and d_i = (y_i.r < 0 ? -1 : 1) + j (y_i.i < 0 ? -1 : 1):
 *   v = sum_i |y_i - d_i|^2 / 496 (float32, floored at 1e-6), a per-packet estimate of the noise variance per
 *       dimension;
 *   bit 2i of frame f: L = 2 Im(y[31 f + i]) / v, bit 2i+1: L = 2 Re(y[31 f + i]) / v, negated where bit 2i (2i+1)
 *       of sc_packet_keystream_word(f) is 1; a non-finite L is written as 0.
 * So bit == (L < 0) is the record's hard decision wherever L != 0.  The estimate v assumes the DD loop's output
 * (SC_FLAG_PACKET_DD / SC_FLAG_PACKET_ACQ banks).  On a plain SC_FLAG_PACKET bank the symbols are the reference
 * Kalman equalizer's and the LLRs are defined but useless.  The decoder below does not depend on their scale.
 * packet_symbols and llr must be aligned to 8 bytes.  capacity == 0 launches nothing. */
int sc_packet_llr_dev(int device, const float *packet_symbols, int64_t capacity, const uint64_t *n_found, float *llr,
                      void *stream);

/* Soft-decision Viterbi decoding of the packet code: for record k < min(*n_found, capacity) (n_found read on the
 * device, as for sc_packet_llr_dev), the 496 LLRs at llr + k * 496 -> out[k].  Correlation metric, maximised, in
 * float32 with adds and compares only: each LLR is first sanitised (non-finite -> 0, clamped to +-2^24); ties go to
 * the predecessor whose newest-dropped bit is 0; traceback from state 0.  data holds the maximum-likelihood payload
 * even when crc_ok is 0.  llr must be aligned to 8 bytes and out to 4.  capacity == 0 launches nothing. */
int sc_packet_decode_dev(int device, const float *llr, int64_t capacity, const uint64_t *n_found,
                         sc_packet_payload *out, void *stream);

/* ---- code rates of the coded payload (DESIGN.md section 8c, "Code rates") ----------------------------------------
 *
 * The same mother code, punctured per stream to rate 2/3 or 3/4 with the IEEE 802.11a patterns; the packet layout,
 * the interleaver and the LLRs (sc_packet_llr_dev) do not change.  Each stream has one code, set at both ends of its
 * link (a device uint8 table stream_code[n_streams], the same for the encoder and the decoder):
 *   code  payload B  steps T = 8 B + 22  mother bits kept per period  transmitted bits N  free distance
 *   0     27         238                 c0 c1                        476                 10  (today's code)
 *   1     36         310                 c0 c1 | c0                   465                 6
 *   2     41         350                 c0 c1 | c0 | c1              467                 5
 *   info      u = B payload bytes, their CRC-16 (as above, high byte first), MSB first: 8 B + 16 bits; then 6 zeros
 *   encoder   the rate-1/2 encoder above over t = 0..T-1 -> mother bits c[2t] (0133), c[2t+1] (0171)
 *   puncture  transmitted bit n < N is mother bit m(n): code 0: m = n; code 1: m = 4 floor(n/3) + (0, 1, 2)[n mod 3];
 *             code 2: m = 6 floor(n/4) + (0, 1, 2, 5)[n mod 4]
 *   layout    transmitted bit n goes to packet bit p = 17 (n mod 28) + floor(n / 28); every other p of the 496 is 0
 *   decoder   L'[m(n)] = the sanitised LLR at p(n) for n < N, L'[m] = 0 for every punctured m; then the recursion of
 *             sc_packet_decode_dev over T steps and the traceback from state 0
 * For code 0 this is exactly the code of sc_packet_encode_dev / sc_packet_decode_dev. */
#define SC_PACKET_CODE_R12 0
#define SC_PACKET_CODE_R23 1
#define SC_PACKET_CODE_R34 2
#define SC_PACKET_PAYLOAD_MAX 41
int sc_packet_payload_bytes(int code);          /* 27, 36, 41; 0 for any other value (host function) */

typedef struct {
    uint8_t  data[41];      /* the first sc_packet_payload_bytes(code) bytes: the maximum-likelihood payload; the rest 0 */
    uint8_t  code;          /* the code the record was decoded with, as read from stream_code (255: stream out of range) */
    uint8_t  crc_ok;        /* 1 when the CRC of the payload equals the decoded CRC bits */
    uint8_t  reserved0;     /* 0 */
    uint16_t flipped;       /* of the code's N transmitted bits, those whose LLR sign disagrees with the decoded codeword */
    uint16_t reserved1;     /* 0 */
} sc_packet_payload_ex;     /* 48 bytes */

/* payload [n_streams][n_packets][41] (bytes past the stream's B are ignored), stream_code device uint8[n_streams]
 *   -> bits [n_streams][n_packets][8][62], the layout sc_tx_packets_dev / sc_tx_channel_dev take.  A stream whose code
 *   is not 0..2 gets all-zero bits.  SC_EINVAL before any CUDA call on a NULL pointer, n_streams < 0 or
 *   n_packets < 1; n_streams == 0 launches nothing. */
int sc_packet_encode_ex_dev(int device, const uint8_t *payload, int64_t n_streams, int n_packets,
                            const uint8_t *stream_code, uint8_t *bits, void *stream);

/* Record k < min(*n_found, capacity) (n_found read on the device, as for sc_packet_decode_dev): its code is
 *   stream_code[packets[k].stream]; the 496 LLRs at llr + 496 k (sc_packet_llr_dev's output) -> out[k].  A stream
 *   outside 0..n_streams-1, or a code that is not 0..2: data 0, crc_ok 0, flipped 0, code as read (255 for the
 *   stream).  Records at or past that count are not touched.  SC_EINVAL before any CUDA call on a NULL pointer, a
 *   negative capacity or n_streams, llr not aligned to 8 bytes or out not to 4; capacity == 0 launches nothing. */
int sc_packet_decode_ex_dev(int device, const float *llr, const sc_packet_result *packets, int64_t capacity,
                            const uint64_t *n_found, const uint8_t *stream_code, int64_t n_streams,
                            sc_packet_payload_ex *out, void *stream);

/* Per-packet codes.  sc_packet_encode_ex_dev takes one code per packet when each packet is given as a stream of its
 * own: payload [n_streams * n_packets][1][41], n_streams * n_packets "streams" of n_packets = 1, and a code table
 * uint8[n_streams * n_packets] (packet j of stream s at s * n_packets + j).  The bits come out in exactly the
 * [n_streams][n_packets][8][62] layout the transmitter takes.
 *
 * Blind code detection (DESIGN.md section 8c, "Blind code detection"): the receiver needs no code table.  Record
 * k < min(*n_found, capacity) (n_found read on the device, as above) is decoded at every code c of code_mask (bit c
 * set, c = 0..2), each exactly as sc_packet_decode_ex_dev decodes it at c, and one of those records is returned
 * unchanged in out[k] (its code field says which):
 *   better(a, b)  flipped_a * N_b < flipped_b * N_a (N = 476, 465, 467); equal: the lower code
 *   choose        the best of the candidates whose CRC passes; when none passes, the best of all (crc_ok 0)
 * The CRC identifies the code (a record decoded at the wrong code passes with probability about 2^-16); flipped / N
 * only breaks ties.  A one-code mask 1 << c gives exactly the records of sc_packet_decode_ex_dev with every stream at c.
 * Records at or past the count are not touched.  SC_EINVAL before any CUDA call on a NULL pointer, a negative
 * capacity, code_mask 0 or with a bit above bit 2, llr not aligned to 8 bytes or out not to 4; capacity == 0 launches
 * nothing. */
int sc_packet_decode_blind_dev(int device, const float *llr, int64_t capacity, const uint64_t *n_found,
                               unsigned code_mask, sc_packet_payload_ex *out, void *stream);

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
