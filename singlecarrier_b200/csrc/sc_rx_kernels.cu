// sc_rx_kernels.cu -- the RX hot path as hand-written sm_100a kernels.
//
// One qpsk_rx_frame() call of the reference (src/qpsk.c:133-239) over a bank of N streams is two
// launches:
//   track_kernel     (one thread per stream)  kalman_reset -> 128 x train_eq -> 31 x data_eq ->
//                    slice -> descramble on the symbol window prepared by the previous call;
//   frontend_kernel  (one warp per stream)    int16 -> mix -> 49-tap RRC evaluated only at the
//                    <= 290 decimated instants the reference can ever read -> 128-lag preamble
//                    correlation + first-maximum argmax -> tracker window for the next call.
// plus two tiny table kernels (NCO phasors; data independent, shared by all streams).
#include "sc_common.cuh"
#include "sc_tables.cuh"
#include "sc_tracker.cuh"
#include "sc_search.cuh"
#include "sc_search_mma.cuh"
#include "sc_track_core.cuh"
#include "sc_tracker_coop.cuh"
#include "sc_frontend.cuh"
#include "sc_kernels.h"

#include <stdlib.h>

namespace sc {

// rx_timing at entry of a call: stored, or derived from the previous call's outcome (qpsk.c:196,219)
__device__ __forceinline__ int resolve_timing(const TimingSrc &ts, const int *__restrict__ timing_cur, long s) {
    if (ts.matches == nullptr) return timing_cur[s];
    const bool valid = __float_as_int(ts.matches[s * ts.mstride]) > MATCH_THRESHOLD;
    return valid ? ts.max_index[s] + PRE : ts.timing_prev[s];
}


// ------------------------------------------------------------------------------------------------
// NCO phasor table.  The reference advances one complex phasor per sample by a float recurrence
// and renormalises it after every frame (qpsk.c:138-147 RX, :301-306 TX).  The sequence does not
// depend on the data, so it is generated once per batch by a single thread running the identical
// recurrence and shared by every stream.  `pattern` gives the run lengths between renormalisations
// (RX: 1880 per call; TX: 640,155 x 8 per packet).  scale multiplies the stored value (a power of
// two, exact): the RX table is stored pre-multiplied by 1/16384 so the mixer is phasor*(float)in.
// ------------------------------------------------------------------------------------------------
__global__ void nco_table_kernel(float2 *__restrict__ phase_state, float2 rect, int pattern, int seg_single,
                                 int n_seg, float scale, float2 *__restrict__ out) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    c32 ph = from2(*phase_state);
    const c32 r = from2(rect);
    long k = 0;
    for (int s = 0; s < n_seg; s++) {
        // NCO_RX: one run per qpsk_rx_frame() call; NCO_TX_PACKET: 640, then 8 x 155 (qpsk.c:380-405);
        // NCO_SINGLE: the caller's run length (one qpsk_tx_frame() call of the drop-in shim)
        const int len = pattern == NCO_RX ? FRAME
                        : pattern == NCO_TX_PACKET ? ((s % 9) == 0 ? PRE * CYC : NDATA * CYC) : seg_single;
        for (int i = 0; i < len; i++, k++) {
            ph = cmul(ph, r);
            out[k] = make_float2(__fmul_rn(ph.r, scale), __fmul_rn(ph.i, scale));
        }
        ph = renorm(ph);
    }
    *phase_state = to2(ph);
}


// GENERIC = false: every frame pointer is 4-byte aligned (checked by the launcher), loads are
// coalesced 32-bit pairs.  GENERIC = true: any alignment, scalar 16-bit loads, same arithmetic.
// rx_timing is 128..255 whenever the front-end runs (DESIGN.md section 3), so the first sample
// needed (rx_timing - 48) is never before the frame; it is clamped to keep a corrupt state in bounds.
// MMA = true: the search is proposed on the tensor cores and verified exactly (sc_search_mma.cuh), one warp of
// every warp PAIR doing it for both windows while the other goes on to the barrier; false: all 128 lags exact.
template <bool WIDE, bool GENERIC, bool MMA, bool OV>
__global__ void __launch_bounds__(FE_WARPS * 32, 6)
frontend_kernel(const int16_t *__restrict__ in, long stream_stride, const float2 *__restrict__ mix_table,
                const int *__restrict__ timing_cur, const int *__restrict__ timing_next,
                float2 *__restrict__ win, int *__restrict__ max_index_out, float *__restrict__ max_value_out,
                int n_streams, const uint4 *__restrict__ a_table, TimingSrc ts) {
    // OV = false: window rows 163.. are the 35 symbols from the NEXT call's rx_timing (the serial call chain);
    // OV = true: rows 163.. are W[128 ..], every symbol an rx_timing of 128..255 can select, so that this kernel does
    // not have to wait for the tracker of the call in between (overlapped chains, timing_next unused)
    constexpr int win_rows = OV ? WIN_ROWS_OV : WIN_ROWS;
    __shared__ __align__(16) float2 smem[FE_WARPS][FE_BUF];
    __shared__ int s_maxidx[FE_WARPS];
    __shared__ int s_t2[FE_WARPS];

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long s = (long) blockIdx.x * FE_WARPS + warp;
    const bool active = s < n_streams;
    float2 *mix = smem[warp];

    u64 accA[FE_R], accB[FE_R];
#pragma unroll
    for (int r = 0; r < FE_R; r++) accA[r] = accB[r] = 0ull;

    // warp-uniform set-up
    int base = 0, shift = 0, base2 = 0;
    const int16_t *frame = in;
    const float2 *tab = mix_table;
    const uint32_t *fp = nullptr;
    uint32_t raw[FE_KN];
#pragma unroll
    for (int k = 0; k < FE_KN; k++) raw[k] = 0u;
    if (active) {
        const int T = OV ? resolve_timing(ts, timing_cur, s) : timing_cur[s];
        if (OV && ts.timing_out != nullptr && lane == 0) ts.timing_out[s] = T;
        base = max(min(T, 2 * PRE - 1) - (NTAPS - 1), 0);  // first sample needed: 80..207 for T in 128..255
        frame = in + s * stream_stride;
        if (!GENERIC) {
            // ---- stage 1: pass A's global loads (coalesced 4-byte loads, the kernel's only HBM reads) ----
            base2 = base & ~1;
            shift = base - base2;
            fp = reinterpret_cast<const uint32_t *>(frame + base2);
            tab = mix_table + base2;
            fe_load<FE_KA_LO>(raw, fp, lane, base2);
        }
    }

    // ---- two passes: A = outputs 0..144 (rel 0..768), B = outputs 145..289 (rel 725..1493)
#pragma unroll 1
    for (int h = 0; h < 2; h++) {
        const int h0 = h * CYC * FE_PASS_OUT;
        const int front = FE_FRONT + ((shift + h0) & 1);       // makes every staged pair 16-byte aligned
        if (active) {
            if (!GENERIC) {
                if (h == 0) {
                    fe_stage<FE_KA_LO>(mix, raw, tab, lane, front - shift - h0);
                    fe_load<FE_KB_LO>(raw, fp, lane, base2);       // pass B's loads fly during pass A's FIR
                } else {
                    fe_stage<FE_KB_LO>(mix, raw, tab, lane, front - shift - h0);
                }
            } else {
                for (int rel = lane; rel < FE_PASS_SAMP; rel += 32) {
                    const int t = base + h0 + rel;
                    const float x = (float) frame[t];
                    const float2 ph = __ldg(mix_table + t);
                    mix[front + rel] = make_float2(__fmul_rn(ph.x, x), __fmul_rn(ph.y, x));
                }
            }
        }
        __syncwarp();
        u64 acc[FE_R];
#pragma unroll
        for (int r = 0; r < FE_R; r++) acc[r] = 0ull;
        if (active && lane < FE_FIR_LANES) fe_fir<WIDE>(mix, front, lane, acc);
        __syncwarp();
#pragma unroll
        for (int r = 0; r < FE_R; r++) {
            if (h == 0) accA[r] = acc[r];
            else accB[r] = acc[r];
        }
    }

    float2 *W = mix;                                        // [290]
    if (!MMA) {
        float *DE = reinterpret_cast<float *>(mix + WIN);   // search operands, sc_search.cuh
        if (active && lane < FE_FIR_LANES) {
#pragma unroll
            for (int r = 0; r < FE_R; r++) {
                float yr, yi;
                unpk(accA[r], yr, yi);
                const float2 wa = make_float2(__fmul_rn(yr, FIR_GAIN), __fmul_rn(yi, FIR_GAIN));       // src/fir.c:42
                unpk(accB[r], yr, yi);
                const float2 wb = make_float2(__fmul_rn(yr, FIR_GAIN), __fmul_rn(yi, FIR_GAIN));
                const int xa = FE_R * lane + r, xb = FE_PASS_OUT + xa;
                W[xa] = wa;
                W[xb] = wb;
                // ---- stage 3 operands straight from the registers (qpsk.c:88-96, see sc_search.cuh)
                de_store(DE, xa, wa);
                if (xb < SEARCH_SYMS) de_store(DE, xb, wb);
            }
        }
        __syncwarp();

        if (active) {
            int best_idx;
            float best_val;
            search_warp(DE, lane, best_idx, best_val);
            if (lane == 0) {
                max_index_out[s] = best_idx;
                max_value_out[s] = best_val;
                s_maxidx[warp] = best_idx;
                s_t2[warp] = OV ? PRE : timing_next[s];
            }
        }
    } else {
        // the pair's structures live behind W in the two warps' buffers: B operand in the even warp's, d/e + lists
        // in the odd warp's
        const int pw = warp & 1;
        SearchMmaB &sb = *reinterpret_cast<SearchMmaB *>(smem[warp & ~1] + WIN);
        SearchMmaDE &sd = *reinterpret_cast<SearchMmaDE *>(smem[warp | 1] + WIN);
        // each warp is about to write into its partner's buffer: both must be done with their FIR passes first
        static_assert(FE_WARPS == 4, "two warp pairs per CTA");
        if (warp >> 1) asm volatile("bar.sync 2, 64;" ::: "memory");
        else asm volatile("bar.sync 1, 64;" ::: "memory");
        float part = 0.0f;
        if (lane < FE_FIR_LANES) {
#pragma unroll
            for (int r = 0; r < FE_R; r++) {
                float yr, yi;
                unpk(accA[r], yr, yi);
                const float2 wa = make_float2(__fmul_rn(yr, FIR_GAIN), __fmul_rn(yi, FIR_GAIN));       // src/fir.c:42
                unpk(accB[r], yr, yi);
                const float2 wb = make_float2(__fmul_rn(yr, FIR_GAIN), __fmul_rn(yi, FIR_GAIN));
                const int xa = FE_R * lane + r, xb = FE_PASS_OUT + xa;
                W[xa] = wa;
                W[xb] = wb;
                // d = s.r - s.i, e = s.i + s.r: the exact operands of correlate(), qpsk.c:88-96
                const float da = __fsub_rn(wa.x, wa.y), ea = __fadd_rn(wa.y, wa.x);
                sd.de[pw][0][xa] = da;
                sd.de[pw][1][xa] = ea;
                part = __fadd_rn(part, __fadd_rn(fabsf(da), fabsf(ea)));
                if (xb < SEARCH_SYMS) {
                    const float db = __fsub_rn(wb.x, wb.y), eb = __fadd_rn(wb.y, wb.x);
                    sd.de[pw][0][xb] = db;
                    sd.de[pw][1][xb] = eb;
                    part = __fadd_rn(part, __fadd_rn(fabsf(db), fabsf(eb)));
                }
            }
        } else if (lane == FE_FIR_LANES) {
            sd.de[pw][0][SEARCH_SYMS] = 0.0f;               // x = 255 pads the last bf16 pair
            sd.de[pw][1][SEARCH_SYMS] = 0.0f;
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) part = __fadd_rn(part, __shfl_xor_sync(0xffffffffu, part, off));
        if (lane == 0) sd.s_abs[pw] = part;
        __syncwarp();
#pragma unroll
        for (int k = 0; k < 4; k++) {                       // bf16 pieces, symbol pairs (x, x + 1)
            const int x = 2 * lane + 64 * k;
            const float2 dd = *reinterpret_cast<const float2 *>(&sd.de[pw][0][x]);
            const float2 ee = *reinterpret_cast<const float2 *>(&sd.de[pw][1][x]);
            search_mma_stage_pieces(sb, pw, x, dd.x, dd.y, ee.x, ee.y);
        }
        // second named barrier of the pair (0 is __syncthreads): the odd warp only signals, the even one waits
        if (pw == 1) {
            if (warp >> 1) asm volatile("bar.arrive 4, 64;" ::: "memory");
            else asm volatile("bar.arrive 3, 64;" ::: "memory");
        } else {
            if (warp >> 1) asm volatile("bar.sync 4, 64;" ::: "memory");
            else asm volatile("bar.sync 3, 64;" ::: "memory");
            int bi[2];
            float bv[2];
            search_mma_pair<true>(sb, sd, a_table, lane, bi, bv);
            if (lane < 2 && s + lane < n_streams) {
                const int idx = lane ? bi[1] : bi[0];
                max_index_out[s + lane] = idx;
                max_value_out[s + lane] = lane ? bv[1] : bv[0];
                s_maxidx[warp + lane] = idx;
                s_t2[warp + lane] = OV ? PRE : timing_next[s + lane];
            }
        }
    }
    __syncthreads();

    // ---- stage 4: hand the tracker its window, 32-byte sectors (4 adjacent streams per row) ----
    {
        const long s0 = (long) blockIdx.x * FE_WARPS;
        const int j = threadIdx.x & (FE_WARPS - 1);
        const long sj = s0 + j;
        if (sj < n_streams) {
            const int mi = s_maxidx[j], t2 = s_t2[j];
            const float2 *Wj = smem[j];
            float2 *dst = win + ((sj >> 5) * win_rows) * 32 + (sj & 31);
            for (int row = threadIdx.x / FE_WARPS; row < win_rows; row += (FE_WARPS * 32) / FE_WARPS) {
                int src = row < X_ROWS ? mi + row : t2 + (row - X_ROWS);
                float2 v = make_float2(0.f, 0.f);
                if (src >= 0 && src < WIN) v = Wj[src];
                dst[row * 32] = v;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// track_kernel: one thread per stream; the decision half of qpsk_rx_frame(), qpsk.c:186-238.
// ------------------------------------------------------------------------------------------------
constexpr int TK_THREADS = 128;

struct TileLoader {
    const float2 *X;      // this stream's column of its 32-stream tile
    __device__ __forceinline__ c32 x(int r) const { return from2(X[r * 32]); }
    __device__ __forceinline__ c32 y(int r) const { return from2(X[(X_ROWS + r) * 32]); }
};

// Overlapped chains (DESIGN.md section 5b): the window tile is WIN_ROWS_OV rows high, rows 163.. hold W[128 ..], and
// the call's data symbols for the invalid branch start at row 163 + rx_timing - 128.
struct TileLoaderOv {
    const float2 *X, *Y;
    __device__ __forceinline__ c32 x(int r) const { return from2(X[r * 32]); }
    __device__ __forceinline__ c32 y(int r) const { return from2(Y[r * 32]); }
};
__device__ __forceinline__ int ov_alt_row(int rx_timing) { return X_ROWS + min(max(rx_timing - PRE, 0), PRE - 1); }

// SOFT: the 31 equalizer outputs of the call also go to sym, NDATA per record, records indexed like results.
template <bool DEBUG_EQ, bool SOFT>
__global__ void __launch_bounds__(TK_THREADS)
track_kernel(const float2 *__restrict__ win, const int *__restrict__ max_index, const float *__restrict__ max_value,
             const int *__restrict__ timing_cur, int *__restrict__ timing_next, sc_frame_result *__restrict__ results,
             long result_stride, float *__restrict__ eq_dbg, float *__restrict__ state_dbg, uint32_t call_index,
             unsigned long long keystream, int n_streams, float2 *__restrict__ sym) {
    const long s = (long) blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_streams) return;

    TileLoader ld;
    ld.X = win + ((s >> 5) * WIN_ROWS) * 32 + (s & 31);
    TrackOut o;
    track_core<SOFT>(ld, o, SOFT ? sym + s * result_stride * NDATA : nullptr);

    const int t_in = timing_cur[s];
    const int mi = max_index[s];
    const int t_out = o.valid ? mi + PRE : t_in;                   // qpsk.c:219
    timing_next[s] = t_out;
    store_result(results + s * result_stride, o, keystream, max_value[s], mi, t_out, call_index);

    if (DEBUG_EQ && eq_dbg != nullptr) {
        float *e = eq_dbg + s * result_stride * 10;
#pragma unroll
        for (int i = 0; i < EQ; i++) {
            e[2 * i] = o.tk.C[i].r;
            e[2 * i + 1] = o.tk.C[i].i;
        }
    }
    // the whole equalizer / Kalman state the reference leaves in its globals after the call
    // (src/kalman.c:19-35): eq_coeff, kalman_gain, u (upper triangle), d, kalman_y -- drop-in shim only
    if (DEBUG_EQ && state_dbg != nullptr) {
        float *e = state_dbg + s * TRACK_STATE_FLOATS;
#pragma unroll
        for (int i = 0; i < EQ; i++) {
            e[2 * i] = o.tk.C[i].r;
            e[2 * i + 1] = o.tk.C[i].i;
            e[10 + 2 * i] = o.tk.G[i].r;
            e[10 + 2 * i + 1] = o.tk.G[i].i;
            e[40 + i] = o.tk.D[i];
        }
#pragma unroll
        for (int i = 0; i < 10; i++) {
            e[20 + 2 * i] = o.tk.U[i].r;
            e[20 + 2 * i + 1] = o.tk.U[i].i;
        }
        e[45] = o.tk.KY;
    }
}

// ------------------------------------------------------------------------------------------------
// track_train_kernel / track_data_kernel: track_kernel cut at qpsk.c:196.  The 128 training steps need only the
// window; rx_timing enters with the 31 data steps (the invalid branch reads from it, and the new rx_timing is either
// max_index + 128 or the old one).  Cut there, the training of call n+1 no longer waits for call n, and two chains of
// calls (even, odd) run side by side: what a bank too small to fill the GPU needs (sc_api.cu: run_slab_overlapped).
// The tracker (eq_coeff, u, d), the match count and magnitude() travel through `state`, [TRK_STATE_WORDS][stride].
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(TK_THREADS)
track_train_kernel(const float2 *__restrict__ win, float *__restrict__ state, long stride, int n_streams) {
    const long s = (long) blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_streams) return;
    TileLoaderOv ld;
    ld.X = ld.Y = win + ((s >> 5) * WIN_ROWS_OV) * 32 + (s & 31);
    Tracker tk;
    int matches;
    float mag;
    track_train(ld, tk, matches, mag);
    float *e = state + s;
#pragma unroll
    for (int i = 0; i < EQ; i++) {
        e[(2 * i) * stride] = tk.C[i].r;
        e[(2 * i + 1) * stride] = tk.C[i].i;
        e[(30 + i) * stride] = tk.D[i];
    }
#pragma unroll
    for (int i = 0; i < 10; i++) {
        e[(10 + 2 * i) * stride] = tk.U[i].r;
        e[(10 + 2 * i + 1) * stride] = tk.U[i].i;
    }
    e[35 * stride] = __int_as_float(matches);
    e[36 * stride] = mag;
}

template <bool SOFT>
__global__ void __launch_bounds__(TK_THREADS)
track_data_kernel(const float2 *__restrict__ win, const float *__restrict__ state, long stride,
                  const int *__restrict__ max_index, const float *__restrict__ max_value,
                  const int *__restrict__ timing_cur, int *__restrict__ timing_next, sc_frame_result *__restrict__ results,
                  long result_stride, uint32_t call_index, unsigned long long keystream, int n_streams, TimingSrc ts,
                  int *__restrict__ timing_cur_out, bool coop_state, float2 *__restrict__ sym) {
    const long s = (long) blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_streams) return;
    const int t_in = resolve_timing(ts, timing_cur, s);
    if (timing_cur_out != nullptr) timing_cur_out[s] = t_in;
    TileLoaderOv ld;
    ld.X = win + ((s >> 5) * WIN_ROWS_OV) * 32 + (s & 31);
    ld.Y = ld.X + ov_alt_row(t_in) * 32;
    TrackOut o;
    float mag;
#pragma unroll
    for (int i = 0; i < EQ; i++) o.tk.G[i] = mk(0.0f, 0.0f);       // G and KY are rebuilt by every step
    o.tk.KY = 0.0f;
    if (coop_state) {
        // left by track_coop_kernel<TRK_TRAIN>: [stream][TRK_STATE_WORDS], columns of u with their d, then eq_coeff
        const float *e = state + s * TRK_STATE_WORDS;
#pragma unroll
        for (int j = 0; j < EQ; j++) {
#pragma unroll
            for (int i = 0; i < j; i++) o.tk.U[j * (j - 1) / 2 + i] = mk(e[9 * j + 2 * i], e[9 * j + 2 * i + 1]);
            o.tk.D[j] = e[9 * j + 8];
            o.tk.C[j] = mk(e[45 + 2 * j], e[45 + 2 * j + 1]);
        }
        o.matches = __float_as_int(e[55]);
        mag = e[56];
    } else {
        const float *e = state + s;
#pragma unroll
        for (int i = 0; i < EQ; i++) {
            o.tk.C[i] = mk(e[(2 * i) * stride], e[(2 * i + 1) * stride]);
            o.tk.D[i] = e[(30 + i) * stride];
        }
#pragma unroll
        for (int i = 0; i < 10; i++) o.tk.U[i] = mk(e[(10 + 2 * i) * stride], e[(10 + 2 * i + 1) * stride]);
        o.matches = __float_as_int(e[35 * stride]);
        mag = e[36 * stride];
    }
    o.valid = o.matches > MATCH_THRESHOLD;                          // qpsk.c:196
    float cost;
    track_data<SOFT>(ld, o.tk, o.valid, o.word, cost, SOFT ? sym + s * result_stride * NDATA : nullptr);
    o.cost = o.valid ? mag : cost;

    const int mi = max_index[s];
    const int t_out = o.valid ? mi + PRE : t_in;                    // qpsk.c:219
    if (timing_next != nullptr) timing_next[s] = t_out;
    store_result(results + s * result_stride, o, keystream, max_value[s], mi, t_out, call_index);
}

// ------------------------------------------------------------------------------------------------
// track_coop_kernel: the same call, two warps per four streams (sc_tracker_coop.cuh) -- for banks too small
// to fill the GPU with one thread per stream, where the tracker's dependent chain is the whole cost of a call.
// ------------------------------------------------------------------------------------------------
constexpr int TC_THREADS = 64;
constexpr int TC_STREAMS = 32 / TC_LANES;                          // streams per CTA: one lane group each, per warp
enum { TRK_ALL = 0, TRK_TRAIN = 1 };                               // the whole call, or the part before qpsk.c:196
// what a cooperative TRK_TRAIN launch hands to track_data_kernel, per stream (TRK_STATE_WORDS floats):
//   [9 j + 2 i], [9 j + 2 i + 1] = U(i, j), [9 j + 8] = d[j]  (column lane j);  [45 + 2 i ..] = eq_coeff[i];
//   [55] = matches, [56] = magnitude()
// (the 31 data steps of a cut call are off the chain's critical path and run one thread per stream: a 16th of the warps)
static_assert(TRK_STATE_WORDS >= 57, "cooperative tracker state");

__device__ __forceinline__ void tc_barrier() { asm volatile("bar.sync 1, 64;" ::: "memory"); }

template <int PHASE, bool SOFT>
__global__ void __launch_bounds__(TC_THREADS)
track_coop_kernel(const float2 *__restrict__ win, const int *__restrict__ max_index, const float *__restrict__ max_value,
                  const int *__restrict__ timing_cur, int *__restrict__ timing_next,
                  sc_frame_result *__restrict__ results, long result_stride, uint32_t call_index,
                  unsigned long long keystream, int n_streams, float *__restrict__ state, float2 *__restrict__ sym) {
    // The window is rows of 8 bytes in L2 (the front-end has just written it), ~700 clocks away; a step is ~250.
    // All of it is fetched at once into shared memory, then read from there.
    constexpr int ROWS = PHASE == TRK_ALL ? WIN_ROWS : PRE + EQ;
    constexpr int TILE_ROWS = PHASE == TRK_ALL ? WIN_ROWS : WIN_ROWS_OV;
    __shared__ __align__(16) float2 s_win[TC_STREAMS][ROWS + 2];
    __shared__ ExchangeA s_xa[2][TC_STREAMS];                      // what step k leaves for the taps: buffer k & 1
    __shared__ ExchangeB s_xb[TC_STREAMS];
    __shared__ int s_valid[TC_STREAMS];

    const int lane = threadIdx.x & 31, g = lane & (TC_LANES - 1), qs = lane / TC_LANES;
    const bool warp_a = threadIdx.x < 32;
    const long s = min((long) blockIdx.x * TC_STREAMS + qs, (long) n_streams - 1);
    const bool store = g == 0 && (long) blockIdx.x * TC_STREAMS + qs < n_streams;
    float *st = state + s * TRK_STATE_WORDS;                       // TRK_TRAIN only
    if (warp_a) {
        s_xa[0][qs].init(g);
        s_xa[1][qs].init(g);
    }
    for (int q2 = 0; q2 < TC_STREAMS; q2++) {
        const long s2 = min((long) blockIdx.x * TC_STREAMS + q2, (long) n_streams - 1);
        const float2 *X = win + ((s2 >> 5) * TILE_ROWS) * 32 + (s2 & 31);
        for (int row = threadIdx.x; row < ROWS; row += TC_THREADS) s_win[q2][row] = __ldg(X + row * 32);
    }
    __syncthreads();
    const float2 *W = s_win[qs];

    if (warp_a) {
        // ---- warp A: the gain recursion, one step ahead of the taps ----
        KalmanColumn ka;
        ka.init(lane);
        ka.reset();                                                // qpsk.c:186
        const float2 *X0 = W, *Xj = W + ka.myj;
        c32 x[4];
#pragma unroll 2
        for (int k = 0; k < PRE; k++) {
#pragma unroll
            for (int i = 0; i < 4; i++) x[i] = from2(X0[k + i]);
            ka.step(x, from2(Xj[k]), &s_xa[k & 1][qs]);
            tc_barrier();
        }
        if (PHASE == TRK_TRAIN) {
            if (ka.live) {
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    st[9 * ka.myj + 2 * i] = ka.U[i].r;
                    st[9 * ka.myj + 2 * i + 1] = ka.U[i].i;
                }
                st[9 * ka.myj + 8] = ka.D;
            }
            return;
        }
        tc_barrier();                                              // warp B has counted the matches of step 127
        const int row0 = s_valid[qs] ? PRE : X_ROWS;               // qpsk.c:196
        X0 += row0;
        Xj += row0;
#pragma unroll 1
        for (int k = 0; k < NDATA; k++) {
#pragma unroll
            for (int i = 0; i < 4; i++) x[i] = from2(X0[k + i]);
            ka.step(x, from2(Xj[k]), &s_xa[k & 1][qs]);
            tc_barrier();
        }
        return;
    }

    // ---- warp B: the taps ----
    TapLanes tp;
    tp.init(lane, &s_xb[qs]);
    tp.reset();
    const float2 *Xi = W + tp.i;

    // equalize(), qpsk.c:111-123, and magnitude(), qpsk.c:101-109 (the sum over x[0] is the one lane 0 keeps)
    int matches = 0, bI, bQ;
    float mag = 0.0f;
    c32 xi = from2(Xi[0]), v;
#pragma unroll 2
    for (int k = 0; k < PRE; k++) {
        const c32 ni = from2(Xi[k + 1]);
        const float ref = ((c_pre_neg[k >> 5] >> (k & 31)) & 1u) ? -1.0f : 1.0f;
        mag = __fadd_rn(mag, __fadd_rn(__fmul_rn(xi.r, xi.r), __fmul_rn(xi.i, xi.i)));
        const c32 err = tp.error<false>(xi, ref, bI, bQ, v);
        if (__fmul_rn(err.r, ref) > 0.0f) matches++;
        tc_barrier();
        tp.update(err, &s_xa[k & 1][qs]);
        xi = ni;
    }
    if (PHASE == TRK_TRAIN) {
        if (g < EQ) {
            st[45 + 2 * tp.i] = tp.C.r;
            st[45 + 2 * tp.i + 1] = tp.C.i;
        }
        if (g == 0) {
            st[55] = __int_as_float(matches);
            st[56] = mag;
        }
        return;
    }
    const bool valid = matches > MATCH_THRESHOLD;                  // qpsk.c:196
    if (g == 0) s_valid[qs] = valid;
    tc_barrier();

    // valid: data symbols follow the preamble; invalid: they start at rx_timing
    Xi += valid ? PRE : X_ROWS;
    xi = from2(Xi[0]);
    unsigned long long word = 0ull;
    float cost = 0.0f;
    float2 *ssym = SOFT ? sym + s * result_stride * NDATA : nullptr;   // written by the storing lane only
#pragma unroll 1
    for (int k = 0; k < NDATA; k++) {
        const c32 ni = from2(Xi[k + 1]);                           // at most row 197 + 1: inside the padded array
        const c32 err = tp.error<true>(xi, 0.0f, bI, bQ, v);
        if (SOFT && store) ssym[k] = to2(v);
        cost = __fadd_rn(cost, err.r);                             // qpsk.c:228
        word |= ((unsigned long long) (unsigned) (bQ | (bI << 1))) << (2 * k);
        tc_barrier();
        tp.update(err, &s_xa[k & 1][qs]);
        xi = ni;
    }

    if (store) {
        TrackOut o;
        o.word = word;
        o.cost = valid ? mag : cost;
        o.matches = matches;
        o.valid = valid;
        const int t_in = timing_cur[s];
        const int mi = max_index[s];
        const int t_out = valid ? mi + PRE : t_in;                 // qpsk.c:219
        timing_next[s] = t_out;
        store_result(results + s * result_stride, o, keystream, max_value[s], mi, t_out, call_index);
    }
}

// ------------------------------------------------------------------------------------------------
// host-side launchers (called from sc_api.cu)
// ------------------------------------------------------------------------------------------------

// The kernels of the overlapped chains (a small bank's even and odd calls) run side by side on different CUDA streams.
// An SM only takes CTAs of kernels that agree on its shared-memory / L1 split, so the cut trackers (little shared
// memory) are given the split the front-end needs (6 x 27 KB); without it a front-end launched while a tracker kernel
// occupies every SM waits for that kernel to drain (measured: 50 us instead of 14 on a 1,024-stream bank).  The
// serial chain's kernels keep their defaults: on a bank that fills the GPU, co-residency costs 10 % (65,536 streams).
template <class K>
static cudaError_t prefer_shared(K kernel) {
    return cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int) cudaSharedmemCarveoutMaxShared);
}
static cudaError_t rx_kernel_attributes() {
    static std::atomic<unsigned long long> done{0};            // bit per device
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 64 && ((done.load() >> dev) & 1ull)) return cudaSuccess;
#define SC_PREF(k)                          \
    if ((e = prefer_shared(k)) != cudaSuccess) return e
    SC_PREF((frontend_kernel<false, false, false, true>));
    SC_PREF((frontend_kernel<false, true, false, true>));
    SC_PREF((frontend_kernel<true, false, false, true>));
    SC_PREF((frontend_kernel<true, true, false, true>));
    SC_PREF(track_train_kernel);
    SC_PREF(track_data_kernel<false>);
    SC_PREF(track_data_kernel<true>);
    SC_PREF((track_coop_kernel<TRK_ALL, false>));
    SC_PREF((track_coop_kernel<TRK_ALL, true>));
    SC_PREF((track_coop_kernel<TRK_TRAIN, false>));
#undef SC_PREF
    if (dev < 64) done.fetch_or(1ull << dev);
    return cudaSuccess;
}

cudaError_t launch_nco_table(float2 *phase_state, float2 rect, int pattern, int seg_single, int n_seg, float scale,
                             float2 *out, cudaStream_t st) {
    nco_table_kernel<<<1, 32, 0, st>>>(phase_state, rect, pattern, seg_single, n_seg, scale, out);
    g_launch_count++;
    return cudaGetLastError();
}

cudaError_t launch_frontend(bool wide, const int16_t *in, long stream_stride, const float2 *mix_table,
                            const int *timing_cur, const int *timing_next, float2 *win, int *max_index,
                            float *max_value, int n_streams, cudaStream_t st, const void *search_a_table,
                            const TimingSrc *tsp) {
    const TimingSrc ts = tsp ? *tsp : TimingSrc();
    cudaError_t ea = rx_kernel_attributes();
    if (ea != cudaSuccess) return ea;
    const int grid = (n_streams + FE_WARPS - 1) / FE_WARPS;
    const int thr = FE_WARPS * 32;
    // the fast kernel reads the samples as aligned 32-bit pairs: every frame must start on a 4-byte boundary
    const bool generic = ((((uintptr_t) in) & 3) != 0) || ((stream_stride & 1) != 0);
    const uint4 *at = (const uint4 *) search_a_table;
    const bool ov = timing_next == nullptr;                 // overlapped chains: the tall window, all-exact search only
#define SC_FE_LAUNCH(W, G, M, O)                                                                                      \
    frontend_kernel<W, G, M, O><<<grid, thr, 0, st>>>(in, stream_stride, mix_table, timing_cur, timing_next, win, max_index, \
                                                      max_value, n_streams, at, ts)
    if (ov) {
        if (wide) {
            if (generic) SC_FE_LAUNCH(true, true, false, true);
            else SC_FE_LAUNCH(true, false, false, true);
        } else {
            if (generic) SC_FE_LAUNCH(false, true, false, true);
            else SC_FE_LAUNCH(false, false, false, true);
        }
    } else if (wide) {
        if (generic) SC_FE_LAUNCH(true, true, false, false);
        else if (at) SC_FE_LAUNCH(true, false, true, false);
        else SC_FE_LAUNCH(true, false, false, false);
    } else {
        if (generic) SC_FE_LAUNCH(false, true, false, false);
        else if (at) SC_FE_LAUNCH(false, false, true, false);
        else SC_FE_LAUNCH(false, false, false, false);
    }
#undef SC_FE_LAUNCH
    g_launch_count++;
    return cudaGetLastError();
}

cudaError_t launch_track(bool debug_eq, const float2 *win, const int *max_index, const float *max_value,
                         const int *timing_cur, int *timing_next, sc_frame_result *results, long result_stride,
                         float *eq_dbg, float *state_dbg, uint32_t call_index, unsigned long long keystream,
                         int n_streams, cudaStream_t st, bool coop, float *sym) {
    cudaError_t ea = rx_kernel_attributes();
    if (ea != cudaSuccess) return ea;
    float2 *sym2 = reinterpret_cast<float2 *>(sym);
    if (coop && !debug_eq) {
        const int grid = (n_streams + TC_STREAMS - 1) / TC_STREAMS;
        if (sym)
            track_coop_kernel<TRK_ALL, true><<<grid, TC_THREADS, 0, st>>>(
                win, max_index, max_value, timing_cur, timing_next, results, result_stride, call_index, keystream,
                n_streams, nullptr, sym2);
        else
            track_coop_kernel<TRK_ALL, false><<<grid, TC_THREADS, 0, st>>>(
                win, max_index, max_value, timing_cur, timing_next, results, result_stride, call_index, keystream,
                n_streams, nullptr, nullptr);
        g_launch_count++;
        return cudaGetLastError();
    }
    const int thr = TK_THREADS;                 // 32 / 64 / 128 measured equal within 0.3 %
    const int grid = (n_streams + thr - 1) / thr;
    if (debug_eq)
        track_kernel<true, false><<<grid, thr, 0, st>>>(win, max_index, max_value, timing_cur, timing_next, results,
                                                        result_stride, eq_dbg, state_dbg, call_index, keystream, n_streams,
                                                        nullptr);
    else if (sym)
        track_kernel<false, true><<<grid, thr, 0, st>>>(win, max_index, max_value, timing_cur, timing_next, results,
                                                        result_stride, nullptr, nullptr, call_index, keystream, n_streams,
                                                        sym2);
    else
        track_kernel<false, false><<<grid, thr, 0, st>>>(win, max_index, max_value, timing_cur, timing_next, results,
                                                         result_stride, eq_dbg, state_dbg, call_index, keystream, n_streams,
                                                         nullptr);
    g_launch_count++;
    return cudaGetLastError();
}

// The two halves of a call for the overlapped chains.  `state` is the slab's hand-over area: coop = false,
// [TRK_STATE_WORDS][state_stride] with this slab's first stream at state[0]; coop = true, [n_streams][TRK_STATE_WORDS]
// (which kernel trained; the data steps always run one thread per stream).
cudaError_t launch_track_train(const float2 *win_ov, float *state, long state_stride, int n_streams, cudaStream_t st,
                               bool coop) {
    if (coop)
        track_coop_kernel<TRK_TRAIN, false><<<(n_streams + TC_STREAMS - 1) / TC_STREAMS, TC_THREADS, 0, st>>>(
            win_ov, nullptr, nullptr, nullptr, nullptr, nullptr, 0, 0u, 0ull, n_streams, state, nullptr);
    else
        track_train_kernel<<<(n_streams + TK_THREADS - 1) / TK_THREADS, TK_THREADS, 0, st>>>(win_ov, state, state_stride,
                                                                                            n_streams);
    g_launch_count++;
    return cudaGetLastError();
}

cudaError_t launch_track_data(const float2 *win_ov, float *state, long state_stride, const int *max_index,
                              const float *max_value, const int *timing_cur, int *timing_next, sc_frame_result *results,
                              long result_stride, uint32_t call_index, unsigned long long keystream, int n_streams,
                              cudaStream_t st, bool coop, const TimingSrc *tsp, int *timing_cur_out, float *sym) {
    const TimingSrc ts = tsp ? *tsp : TimingSrc();
    // off the chains' critical path and sharing the SMs with their kernels: spread thin on small banks
    const int thr = n_streams <= 148 * 32 ? 32 : n_streams <= 148 * 64 ? 64 : TK_THREADS;
    const int grid = (n_streams + thr - 1) / thr;
    if (sym)
        track_data_kernel<true><<<grid, thr, 0, st>>>(
            win_ov, state, state_stride, max_index, max_value, timing_cur, timing_next, results, result_stride, call_index,
            keystream, n_streams, ts, timing_cur_out, coop, reinterpret_cast<float2 *>(sym));
    else
        track_data_kernel<false><<<grid, thr, 0, st>>>(
            win_ov, state, state_stride, max_index, max_value, timing_cur, timing_next, results, result_stride, call_index,
            keystream, n_streams, ts, timing_cur_out, coop, nullptr);
    g_launch_count++;
    return cudaGetLastError();
}

}  // namespace sc
