// sc_kernels.h -- launcher prototypes shared between the kernel translation units and sc_api.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <atomic>

#include "../../include/singlecarrier_b200.h"

namespace sc {

extern std::atomic<unsigned long long> g_launch_count;

// rx_timing at entry of call n where nobody has stored it yet: qpsk.c:219 applied to call n-1 by the reader.
struct TimingSrc {
    const float *matches = nullptr;   // call n-1's match count (int bits) at matches[s * mstride]; nullptr: T_n is stored
    long mstride = 0;
    const int *max_index = nullptr;   // the max_index call n-1 used
    const int *timing_prev = nullptr; // T_{n-1}
    int *timing_out = nullptr;        // where the reader leaves T_n (front-end only; may be nullptr)
};

// sc_rx_kernels.cu
enum { NCO_RX = 0, NCO_TX_PACKET = 1, NCO_SINGLE = 2 };      // run lengths between phasor renormalisations
cudaError_t launch_nco_table(float2 *phase_state, float2 rect, int pattern, int seg_single, int n_seg, float scale,
                             float2 *out, cudaStream_t st);
cudaError_t launch_frontend(bool wide, const int16_t *in, long stream_stride, const float2 *mix_table,
                            const int *timing_cur, const int *timing_next, float2 *win, int *max_index,
                            float *max_value, int n_streams, cudaStream_t st, const void *search_a_table = nullptr,
                            const TimingSrc *ts = nullptr);
// timing_next == nullptr: the tall window of the overlapped chains (WIN_ROWS_OV rows per tile, sc_common.cuh); with
// ts->matches set the kernel derives rx_timing itself instead of reading timing_cur
cudaError_t launch_track(bool debug_eq, const float2 *win, const int *max_index, const float *max_value,
                         const int *timing_cur, int *timing_next, sc_frame_result *results, long result_stride,
                         float *eq_dbg, float *state_dbg, uint32_t call_index, unsigned long long keystream,
                         int n_streams, cudaStream_t st, bool coop = false, float *sym = nullptr);
cudaError_t launch_track_train(const float2 *win_ov, float *state, long state_stride, int n_streams, cudaStream_t st,
                               bool coop);
cudaError_t launch_track_data(const float2 *win_ov, float *state, long state_stride, const int *max_index,
                              const float *max_value, const int *timing_cur, int *timing_next, sc_frame_result *results,
                              long result_stride, uint32_t call_index, unsigned long long keystream, int n_streams,
                              cudaStream_t st, bool coop, const TimingSrc *ts = nullptr, int *timing_cur_out = nullptr,
                              float *sym = nullptr);
// timing_next / timing_cur_out may be nullptr (nothing stored).  sym (launch_track, launch_track_data): nullptr, or
// the equalizer outputs of the call's 31 data steps as NDATA float2 per record, records indexed like results
constexpr int TRACK_STATE_FLOATS = 48;   // C[5], G[5], U[10] complex, D[5], KY, 2 pad: the drop-in shim's view

// sc_stage_kernels.cu
cudaError_t launch_fir_batch(bool wide, long n_streams, float2 *memory, float2 *sample, long sample_stride,
                             int length, cudaStream_t st, bool fast = false);
cudaError_t launch_search_batch(long n_streams, const float2 *symbols, long symbol_stride, int *max_index,
                                float *max_value, cudaStream_t st);
void search_mma_make_table(uint32_t *table /* [9][32][4] */);
cudaError_t launch_search_mma_batch(long n_streams, const float2 *symbols, long symbol_stride, const void *a_table,
                                    int *max_index, float *max_value, cudaStream_t st);
void search_fft_make_table(float *table /* [8][32][2] */);
cudaError_t launch_search_fft_batch(long n_streams, const float2 *symbols, long symbol_stride, const float2 *tw,
                                    const void *ptab, int *max_index, float *max_value, cudaStream_t st);
// sc_frontend_umma.cu: the fused front-end with the search proposed on tcgen05 (SC_FE_SEARCH_TCGEN05); non-overlapped
// chains and 4-byte aligned frames only (frontend_umma_eligible), bit-identical to launch_frontend
constexpr int SU_A_ROWS = 368;                       // master rows r = -240 .. 127 of M[r][k] = pre[k - r]
constexpr int SU_A_WORDS4 = 2 * ((SU_A_ROWS + 7) / 8) * 128 / 16;   // 16-byte words of the master (11,776 bytes)
void search_umma_make_master(uint16_t *table /* [SU_A_WORDS4 * 8] */);
bool frontend_umma_eligible(const int16_t *in, long stream_stride);
cudaError_t launch_frontend_umma(bool wide, const int16_t *in, long stream_stride, const float2 *mix_table,
                                 const int *timing_cur, const int *timing_next, float2 *win, int *max_index,
                                 float *max_value, int n_streams, cudaStream_t st, const void *a_master);
// sc_search_umma.cu: the same search with the proposer on tcgen05 / tensor memory and TMA bulk loads
bool search_umma_eligible(const float2 *symbols, long symbol_stride);
cudaError_t launch_search_umma_batch(long n_streams, const float2 *symbols, long symbol_stride,
                                     int *max_index, float *max_value, float *dbg_approx, cudaStream_t st);
cudaError_t launch_track_window_batch(long n_streams, const float2 *symbols, long symbol_stride,
                                      const int *max_index, const float *max_value, int *rx_timing,
                                      uint32_t call_index, unsigned long long keystream,
                                      sc_frame_result *results, float *eq_dbg, cudaStream_t st);

// sc_fft_kernels.cu
struct FftPlan {
    int n, inverse, n_stages;
    int p[32], m[32];   // kf_factor(): radix and remaining length per stage (src/fft.c:433-459)
};
constexpr int FFT_SCRATCH_CTAS = 64;
constexpr int FFT_SMEM_LIMIT = 64 * 1024;
inline bool fft_needs_scratch(int n) { return (size_t) 2 * n * sizeof(float2) > (size_t) FFT_SMEM_LIMIT; }
void fft_make_plan(int n, int inverse, FftPlan *plan);
void fft_make_permutation(const FftPlan &plan, int *perm);
void fft_make_twiddles(int n, int inverse, float2 *tw);
void fft_make_super_twiddles(int ncfft, int inverse, float2 *tw);
cudaError_t launch_fft(const FftPlan &plan, const float2 *tw, const float2 *super_tw, const int *perm, int mode,
                       const void *in, void *out, float2 *scratch, long n_batches, cudaStream_t st);

cudaError_t launch_selftest_rcp(unsigned lo, unsigned hi, unsigned long long *mismatches, cudaStream_t st);

// sc_stats_kernels.cu
cudaError_t launch_lock_stats(const sc_frame_result *results, long n_streams, long result_stride, int n_frames,
                              unsigned long long *counters, cudaStream_t st);

cudaError_t launch_ber_stats(const sc_frame_result *results, long n_streams, long result_stride, int n_frames,
                             const uint8_t *tx_bits, int n_packets, const int *lead_in, int gap, const int *group,
                             int n_groups, unsigned long long *counters, cudaStream_t st);
// capacity >= 1; n_found is read on the device
cudaError_t launch_packet_ber_stats(const sc_packet_result *packets, long capacity, const unsigned long long *n_found,
                                    const sc_frame_result *results, long n_streams, long result_stride, int n_frames,
                                    const uint8_t *tx_bits, int n_packets, const int *lead_in, int gap,
                                    const int *group, int n_groups, unsigned long long *counters, cudaStream_t st);

// sc_packet_kernels.cu -- packet mode (extension)
constexpr int PK_DATA = 8 * SC_DATA_SYMBOLS;                              // 248 data symbols per packet
constexpr int PK_SYMS = SC_PREAMBLE_LENGTH + PK_DATA + SC_EQ_LENGTH - 1;  // 380 symbols feed one packet decode
struct PacketKey {
    unsigned long long k[8];    // scrambler keystream of the 8 data frames, register seeded per packet
};
struct PacketSrc {              // one block of calls [call0, call0 + nf) of a slab of streams
    const sc_frame_result *results;
    long result_stride;
    const int16_t *in;          // block frames, stream s at in + s * stride
    long stride;
    const int16_t *hist1, *hist2;       // frames call0-1 and call0-2, [stream][1880]
    const float2 *mix0;         // phasor table of frame call0-1; frames call0.. follow
    const float2 *mix_hist2;    // phasor table of frame call0-2
    const int *timing_before_call0, *timing_at_call0;   // rx_timing at entry of calls call0-1 and call0
    uint32_t call0;
    int stream0;                // bank index of the slab's first stream
    bool wide;
};
cudaError_t launch_packet_pass(const PacketSrc &src, int n_streams, int j_lo, int j_hi, int cap, int2 *list, int *count,
                               float2 *sym, const PacketKey &key, sc_packet_result *packets, long packet_capacity,
                               unsigned long long *n_packets, float2 *packet_sym, bool dd, cudaStream_t st);
// packet_sym: nullptr, or the equalizer outputs of the 248 data steps of every packet, PK_DATA float2 per record slot
// (record packets[k] <-> packet_sym[k * PK_DATA ..]); slots beyond packet_capacity are not written.
// dd: decode with the decision-directed equalizer (SC_FLAG_PACKET_DD) instead of the reference's

// sc_tx_kernels.cu
struct TxArgs {
    const uint8_t *bits;        // [n][n_packets][8][62] or nullptr
    uint8_t *bits_out;          // same layout or nullptr
    unsigned long long seed;
    int n_packets;
    int gap_samples;
    const int *lead_in;         // [n] or nullptr
    const float2 *tx_table;     // [n_packets*1880] TX NCO phasors
    int16_t *out;
    long stream_stride;
    long samples_per_stream;
    long n_streams;
    bool wide;
    bool use_channel;
    bool scramble;              // packet mode: data bits go through scramble(tx), register seeded per packet
    PacketKey key;
    sc_channel ch;
};
cudaError_t launch_tx(const TxArgs &a, cudaStream_t st);

}  // namespace sc
