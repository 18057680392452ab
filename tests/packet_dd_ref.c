/*
 * packet_dd_ref.c -- TEST INFRASTRUCTURE ONLY: specification (as code) of packet mode's decision-directed equalizer
 * (SC_FLAG_PACKET_DD, DESIGN.md section 8).
 *
 * Packet mode (oracle/sc_oracle_ext.c) decodes every valid call n >= 2 on the 380-symbol grid S of the continuous
 * matched-filter output with the reference's Kalman equalizer (train_eq / data_eq), which diverges (SURVEY F4).  With
 * SC_FLAG_PACKET_DD the same grid -- same detection, max_index, T and record list -- is decoded instead by
 * scd_dd_packet(): a 5-tap complex normalised LMS filter followed by a second-order carrier loop.  Nothing the
 * reference computes changes.
 *
 * State: taps w[0..4] = 0, carrier phasor p = 1 + 0j, loop frequency nu = 0.  Step i (i = 0..375) on the window
 * x[k] = S[i + k], k = 0..4:
 *   z   = sum_k conj(w[k]) x[k]                   sequential in k, from 0
 *   y   = z conj(p)                               derotated output; the soft output of data steps
 *   d   = training (i < 128): DD_TRAIN_AMP v_i (1 + j), v_i = preamble value (+-1)
 *         data: (y.r < 0 ? -1 : 1) + j (y.i < 0 ? -1 : 1)      (qpsk_demod)
 *   e   = d - y
 *   q   = y conj(d)
 *   pe  = Im(q) / (sqrtf(|q|^2) + DD_PEPS)        sin of the phase error, whatever the amplitudes (the taps start
 *                                                 at 0, so |y| grows during training); 0 for y = 0
 *   g   = DD_MU / (DD_EPS + sum_k |x[k]|^2)       sequential in k
 *   u   = conj(e p) g
 *   w[k] = w[k] + x[k] u                          (NLMS on the un-derotated error e p)
 *   nu  = nu + DD_BETA pe
 *   phi = DD_ALPHA pe + nu
 *   p   = p (1 + j phi), then p = p / sqrtf(|p|^2)               (rotation by atan(phi), renormalised)
 * Data step k = i - 128 (k = 0..247) gives bI = y.r < 0, bQ = y.i < 0, bits[2k] = bQ, bits[2k+1] = bI after the
 * per-packet descrambler (register seeded with 0x4A80, as sco_ext_run_stream), and cost = cost + |e|^2 (float32,
 * sequential over the 248 data steps).
 *
 * Training amplitude: qpsk_tx_frame() scales the preamble by 8192 and data by 16384 (qpsk.c:313-319) and both go
 * through the same filters, so a filter that maps the preamble's v (1 + j) to DD_TRAIN_AMP v (1 + j) maps clean data
 * symbols to +-1 +-1j when DD_TRAIN_AMP = 8192 / 16384 = 1/2.
 *
 * Arithmetic: one IEEE binary32 rounding per operation, in the order written out below, built with
 * -ffp-contract=off; the only function called is sqrtf (correctly rounded).  The GPU kernel
 * (packet_track_dd_kernel, csrc/sc_packet_kernels.cu) mirrors it with __fmul_rn / __fadd_rn / __fsub_rn /
 * __fdiv_rn / __fsqrt_rn and is bit-identical.
 *
 * The final four data symbols: the transmitter's RRC filter delays each symbol's pulse peak by 24 samples, so the
 * pulses of symbols 372..375 of a packet (data steps 244..247) peak after the packet's 1880 samples end; their
 * second halves leave the transmitter only with the next call's output.  When a packet is followed by silence those
 * symbols are received with part of their energy and their decisions are unreliable in any equalizer.
 *
 * Built by tests/packet_dd_ref.py with the oracle's flags against oracle/libsc_oracle.so.
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "sc_oracle.h"

#define DD_NS 8
#define DD_DATA (DD_NS * SCO_DATA_SYMBOLS)                                   /* 248 */
#define DD_SYMS (SCO_PREAMBLE_LENGTH + DD_DATA + SCO_EQ_LENGTH - 1)         /* 380 */
#define DD_SEED 0x4A80

#define DD_MU 0.03f
#define DD_ALPHA 0.05f
#define DD_BETA 0.002f
#define DD_EPS 1e-6f
#define DD_TRAIN_AMP 0.5f
#define DD_PEPS 1e-6f

static inline sco_c32 c32(float r, float i) { sco_c32 z = { r, i }; return z; }

static inline sco_c32 cmul(sco_c32 a, sco_c32 b) {
    float rr = a.r * b.r;
    float ii = a.i * b.i;
    float ri = a.r * b.i;
    float ir = a.i * b.r;
    return c32(rr - ii, ri + ir);
}

static inline sco_c32 cadd(sco_c32 a, sco_c32 b) { return c32(a.r + b.r, a.i + b.i); }
static inline sco_c32 cconj(sco_c32 a) { return c32(a.r, -a.i); }

/* the loop's constants, for the tests */
void scd_dd_params(float out[6]) {
    out[0] = DD_MU;
    out[1] = DD_ALPHA;
    out[2] = DD_BETA;
    out[3] = DD_EPS;
    out[4] = DD_TRAIN_AMP;
    out[5] = DD_PEPS;
}

/*
 * Decodes one packet's grid S[380].  bits[496]: descrambled bits, one per byte, in sco_ext_packet's order;
 * z[248] (or NULL): the derotated equalizer output y of every data step; returns the cost.
 */
float scd_dd_packet(const sco_c32 S[DD_SYMS], uint8_t bits[2 * DD_DATA], sco_c32 z[DD_DATA]) {
    sco_c32 w[SCO_EQ_LENGTH];
    for (int k = 0; k < SCO_EQ_LENGTH; k++) w[k] = c32(0.0f, 0.0f);
    sco_c32 p = c32(1.0f, 0.0f);
    float nu = 0.0f;
    float cost = 0.0f;
    uint16_t lfsr = DD_SEED;

    for (int i = 0; i < SCO_PREAMBLE_LENGTH + DD_DATA; i++) {
        const sco_c32 *x = S + i;
        sco_c32 zz = c32(0.0f, 0.0f);
        for (int k = 0; k < SCO_EQ_LENGTH; k++) zz = cadd(zz, cmul(x[k], cconj(w[k])));
        const sco_c32 y = cmul(zz, cconj(p));

        sco_c32 d;
        if (i < SCO_PREAMBLE_LENGTH) {
            float a = DD_TRAIN_AMP * (float) sco_preamblevalues[i];
            d = c32(a, a);
        } else {
            d = c32(y.r < 0.0f ? -1.0f : 1.0f, y.i < 0.0f ? -1.0f : 1.0f);
        }
        const sco_c32 e = c32(d.r - y.r, d.i - y.i);
        const sco_c32 q = cmul(y, cconj(d));
        const float qm = sqrtf(q.r * q.r + q.i * q.i);
        const float pe = q.i / (qm + DD_PEPS);                    /* ~ sin of the phase error */

        float n = DD_EPS;
        for (int k = 0; k < SCO_EQ_LENGTH; k++) {
            float m2 = x[k].r * x[k].r + x[k].i * x[k].i;
            n = n + m2;
        }
        const float g = DD_MU / n;
        const sco_c32 ep = cmul(e, p);
        const sco_c32 u = c32(ep.r * g, -(ep.i * g));
        for (int k = 0; k < SCO_EQ_LENGTH; k++) w[k] = cadd(w[k], cmul(x[k], u));

        nu = nu + DD_BETA * pe;
        const float phi = DD_ALPHA * pe + nu;
        p = c32(p.r - p.i * phi, p.i + p.r * phi);
        const float m = sqrtf(p.r * p.r + p.i * p.i);
        p = c32(p.r / m, p.i / m);

        if (i >= SCO_PREAMBLE_LENGTH) {
            const int k = i - SCO_PREAMBLE_LENGTH;
            const float e2 = e.r * e.r + e.i * e.i;
            cost = cost + e2;
            if (z) z[k] = y;
            uint8_t dibit = (uint8_t) (((y.r < 0.0f) << 1) | (y.i < 0.0f));
            sco_scramble2(&dibit, &lfsr);
            bits[2 * k + 1] = dibit >> 1;
            bits[2 * k] = dibit & 0x1;
        }
    }
    return cost;
}

/* The reference's equalizer on the same grid: the inner loop of sco_ext_run_stream (kalman_reset, 128 train_eq,
 * 248 data_eq, descrambler seeded per packet).  Returns the cost; bits as scd_dd_packet. */
float scd_kalman_packet(const sco_c32 S[DD_SYMS], uint8_t bits[2 * DD_DATA]) {
    sco_kalman k;
    sco_kalman_init(&k);
    for (int i = 0; i < SCO_PREAMBLE_LENGTH; i++) sco_train_eq(&k, S, i, (float) sco_preamblevalues[i]);
    uint16_t lfsr = DD_SEED;
    float cost = 0.0f;
    for (int i = 0; i < DD_DATA; i++) {
        uint8_t dibit;
        cost = cost + sco_data_eq(&k, &lfsr, &dibit, S, SCO_PREAMBLE_LENGTH + i);
        bits[2 * i + 1] = dibit >> 1;
        bits[2 * i] = dibit & 0x1;
    }
    return cost;
}

typedef struct {
    int32_t call, max_index, matches, timing;
    float cost;
    uint8_t bits[2 * DD_DATA];
} scd_ext_packet;                                               /* sco_ext_packet's layout */

/*
 * sco_ext_run_stream() with the packets decoded by scd_dd_packet(): the same calls, grids and record list; matches is
 * the call's.  psym (or NULL): 248 outputs per packet; grids (or NULL): the 380 grid symbols of every packet.
 */
int scd_ext_run_stream_dd(const int16_t in[], int n_frames, int wide, float foffset_hz, uint8_t bits[],
                          sco_frame_stats stats[], scd_ext_packet packets[], sco_c32 psym[], sco_c32 grids[],
                          int max_packets) {
    sco_state *s = malloc(sizeof *s);
    sco_c32 *filt = calloc((size_t) (n_frames + 1) * SCO_FRAME_SIZE, sizeof *filt);
    int *t_entry = calloc((size_t) n_frames + 1, sizeof *t_entry);
    int n_packets = 0;

    sco_init(s, wide, foffset_hz);
    for (int n = 0; n < n_frames; n++) {
        t_entry[n] = s->rx_timing;                                /* rx_timing at entry of call n */
        sco_frame_stats st;
        uint8_t row[SCO_BITS_PER_CALL];
        memset(row, 255, sizeof row);
        int valid = sco_rx_frame(s, in + (size_t) n * SCO_FRAME_SIZE, row, &st);
        if (bits) memcpy(bits + (size_t) n * SCO_BITS_PER_CALL, row, sizeof row);
        if (stats) stats[n] = st;
        if (n >= 1) memcpy(filt + (size_t) (n - 1) * SCO_FRAME_SIZE, s->input_frame, SCO_FRAME_SIZE * sizeof *filt);

        if (valid && n >= 2 && n_packets < max_packets) {
            scd_ext_packet *p = &packets[n_packets];
            sco_c32 S[DD_SYMS];
            const int T = t_entry[n - 1];
            for (int j = 0; j < DD_SYMS; j++)
                S[j] = filt[(size_t) (n - 2) * SCO_FRAME_SIZE + 5 * (st.max_index + j) + T];
            if (grids) memcpy(grids + (size_t) n_packets * DD_SYMS, S, sizeof S);
            p->cost = scd_dd_packet(S, p->bits, psym ? psym + (size_t) n_packets * DD_DATA : NULL);
            p->call = n;
            p->max_index = st.max_index;
            p->matches = st.matches;
            p->timing = T;
            n_packets++;
        }
    }
    free(t_entry);
    free(filt);
    free(s);
    return n_packets;
}
