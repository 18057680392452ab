// sc_track_core.cuh -- the decision half of qpsk_rx_frame() for one stream in one thread
// (src/qpsk.c:186-238): kalman_reset -> equalize() (128 x train_eq, match count) + magnitude() ->
// 31 x data_eq from sync_pos (valid) or from rx_timing (invalid) -> bits, cost, new rx_timing.
//
// The symbol source is a Loader with  x(r) = dec[max_index + r]  (r < 163) and
// y(r) = dec[rx_timing + r]  (r < 35); loads are issued one step ahead of their use.
#pragma once
#include "sc_common.cuh"
#include "sc_tables.cuh"
#include "sc_tracker.cuh"

namespace sc {

// bit b of word w set <=> preamblevalues[32w + b] == -1 (one copy per translation unit)
static __constant__ uint32_t c_pre_neg[4] = {pre_neg_word(0), pre_neg_word(1), pre_neg_word(2), pre_neg_word(3)};

struct TrackOut {
    unsigned long long word;   // decided dibits before descrambling: bit 2i = Q, bit 2i+1 = I
    float cost;
    int matches;
    bool valid;
    Tracker tk;
};

// equalize(), qpsk.c:111-123, and magnitude(), qpsk.c:101-109, in one pass from a freshly reset tracker
template <class Loader>
__device__ __forceinline__ void track_train(const Loader &ld, Tracker &tk, int &matches_out, float &mag_out) {
    tk.reset();                                                    // qpsk.c:186

    c32 x[EQ];
#pragma unroll
    for (int i = 0; i < EQ - 1; i++) x[i] = ld.x(i);

    int matches = 0;
    float mag = 0.0f;
    c32 nxt = ld.x(EQ - 1);
    // two steps per iteration: the tail of one step (tap update) overlaps the head of the next (F from U), which a
    // rolled loop cannot do; 4 costs registers and loses on large banks (measured: 0.297 / 0.287 / 0.298 ms for 1 / 2 / 4)
#pragma unroll 2
    for (int i = 0; i < PRE; i++) {
        x[EQ - 1] = nxt;
        nxt = ld.x(i + EQ);
        const float ref = ((c_pre_neg[i >> 5] >> (i & 31)) & 1u) ? -1.0f : 1.0f;
        mag = __fadd_rn(mag, __fadd_rn(__fmul_rn(x[0].r, x[0].r), __fmul_rn(x[0].i, x[0].i)));
        const float er = tk.train(x, ref);
        if (__fmul_rn(er, ref) > 0.0f) matches++;
#pragma unroll
        for (int k = 0; k < EQ - 1; k++) x[k] = x[k + 1];
    }
    matches_out = matches;
    mag_out = mag;
}

// the 31 data_eq() steps of qpsk.c:206-215 (valid) / :226-229 (invalid), continuing from the trained tracker.
// SOFT: the equalizer output of step i also goes to sym[i] (one 8-byte store per step).
template <bool SOFT = false, class Loader>
__device__ __forceinline__ void track_data(const Loader &ld, Tracker &tk, bool valid, unsigned long long &word_out,
                                           float &cost_out, float2 *sym = nullptr) {
    // valid: data symbols follow the preamble; invalid: they start at rx_timing
    c32 x[EQ];
#pragma unroll
    for (int i = 0; i < EQ - 1; i++) x[i] = valid ? ld.x(PRE + i) : ld.y(i);
    c32 nxt = valid ? ld.x(PRE + EQ - 1) : ld.y(EQ - 1);

    unsigned long long word = 0ull;
    float cost = 0.0f;
#pragma unroll 1
    for (int i = 0; i < NDATA; i++) {
        x[EQ - 1] = nxt;
        const int rn = min(i + EQ, Y_ROWS - 1);
        nxt = valid ? ld.x(PRE + rn) : ld.y(rn);
        int bI, bQ;
        c32 s;
        const float er = tk.data(x, bI, bQ, s);
        if (SOFT) sym[i] = to2(s);
        cost = __fadd_rn(cost, er);                                // qpsk.c:228
        word |= ((unsigned long long) (unsigned) (bQ | (bI << 1))) << (2 * i);   // bits[2i]=Q, bits[2i+1]=I
#pragma unroll
        for (int k = 0; k < EQ - 1; k++) x[k] = x[k + 1];
    }
    word_out = word;
    cost_out = cost;
}

template <bool SOFT = false, class Loader>
__device__ __forceinline__ void track_core(const Loader &ld, TrackOut &o, float2 *sym = nullptr) {
    int matches;
    float mag, cost;
    track_train(ld, o.tk, matches, mag);
    const bool valid = matches > MATCH_THRESHOLD;                  // qpsk.c:196
    track_data<SOFT>(ld, o.tk, valid, o.word, cost, sym);
    o.cost = valid ? mag : cost;
    o.matches = matches;
    o.valid = valid;
}

__device__ __forceinline__ void store_result(sc_frame_result *dst, const TrackOut &o, unsigned long long keystream,
                                             float max_value, int max_index, int t_out, uint32_t call_index) {
    sc_frame_result r;
    r.bits = o.word ^ keystream;                                   // scramble(bits, rx), equalizer.c:87
    r.max_value = max_value;
    r.cost = o.cost;
    r.max_index = (int16_t) max_index;
    r.matches = (int16_t) o.matches;
    r.rx_timing = (int16_t) t_out;
    r.valid = o.valid ? 1 : 0;
    r.reserved0 = 0;
    r.call_index = call_index;
    r.reserved1 = 0;
    uint4 *d = reinterpret_cast<uint4 *>(dst);
    const uint4 *sp = reinterpret_cast<const uint4 *>(&r);
    d[0] = sp[0];
    d[1] = sp[1];
}

}  // namespace sc
