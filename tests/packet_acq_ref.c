/*
 * packet_acq_ref.c -- TEST INFRASTRUCTURE ONLY: specification (as code) of packet-mode acquisition
 * (SC_FLAG_PACKET_ACQ, DESIGN.md section 8b).
 *
 * Without the flag a packet record exists only where the reference's per-call detection found a valid call.  With it,
 * packets are found by a differential preamble metric on the continuous matched-filter output, which a carrier offset
 * only rotates, and decoded by the decision-directed equalizer (packet_dd_ref.c) seeded with the offset it measures.
 *
 *   filt[q]  the continuous output of the receiver's mixer and 49-tap RRC at stream sample q (from the cold start),
 *            exactly as packet_fir_kernel computes it; 0 for q < 0.  Here: the older half of the oracle's input_frame
 *            after call n holds filt of frame n-1.
 *   Metric on the grid u[i] = filt[g0 + 5 i], i = 0..127:
 *     z[i]  = u[i] conj(u[i-1])           z.r = u[i].r u[i-1].r + u[i].i u[i-1].i,  z.i = u[i].i u[i-1].r - u[i].r u[i-1].i
 *     D     = sum_{i=1..127} b_i z[i]      b_i = pre[i] pre[i-1] (+-1), sequential from 0 + 0j
 *     E     = sum_{i=0..127} |u[i]|^2      |u|^2 = u.r u.r + u.i u.i, sequential from 0
 *     Elo   = E after its first 64 terms (i = 0..63)
 *     rho   = (D.r D.r + D.i D.i) / (E E); 0 when E E == 0 or when the window's energy is not spread over both halves:
 *             not (4 Elo >= E and 4 Elo <= 3 E).  A window that holds only the edge of a burst -- the last symbols of a
 *             packet before silence -- can correlate with the preamble's few first or last differences by chance;
 *             a preamble fills both halves.
 *   Stage 1, frame f: rho1(k) = max(rho on g0 = 5 k, rho on g0 = 5 k + 2) for k in [376 f, 376 f + 376) -- two
 *     grids, so that no symbol instant is more than one sample from a grid point (on one grid the worst sub-symbol
 *     phase, 2 samples off, loses most of rho to intersymbol interference); k* = the first maximum of rho1.  Accepted when
 *     rho1(k*) >= ACQ_TAU and, for every k with 0 < |k - k*| <= ACQ_W outside the frame, rho1(k) < rho1(k*) (k < k*)
 *     or rho1(k) <= rho1(k*) (k > k*): ties go to the earlier lag.
 *   Stage 2: rho on g0 = 5 k* + s, s in the order 0, -1, +1, -2, +2; the first maximum gives g = 5 k* + s*, its D and
 *     rho.  The packet's grid is S[j] = filt[g + 5 j], j < 380.
 *   nu0 = D.i / D.r when D.r > 0, else 0: the tangent of the per-symbol rotation, which is what the DD loop's
 *     p = p (1 + j (alpha pe + nu)) consumes.  The DD loop then runs on S from nu = nu0 (scd_dd_packet otherwise).
 *   matches = the training steps with (y.r + y.i) v_i > 0; freq_hz = nu0 * (1600 / 2 pi), one float32 multiply.
 *   Frame f is decided by call n = f + 2 (its filt reaches frame f + 2 through the grid and the neighbours); the
 *   record's call_index is 2 + floor(g / 1880) and its max_index (g mod 1880) / 5.
 *
 * Arithmetic: one IEEE binary32 rounding per operation in the order written, built with -ffp-contract=off; the only
 * function called is sqrtf (correctly rounded, in the DD loop).  acq_detect_kernel (csrc/sc_acq_kernels.cu) and the
 * ACQ forms of the packet kernels are bit-identical to it.
 *
 * Built by tests/packet_acq_ref.py with the oracle's flags against oracle/libsc_oracle.so.
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "sc_oracle.h"

#define ACQ_NS 8
#define ACQ_DATA (ACQ_NS * SCO_DATA_SYMBOLS)                                 /* 248 */
#define ACQ_SYMS (SCO_PREAMBLE_LENGTH + ACQ_DATA + SCO_EQ_LENGTH - 1)       /* 380 */
#define ACQ_SEED 0x4A80
#define ACQ_LAGS SCO_DEC_LEN                                                 /* 376 lags per frame */

#define ACQ_TAU 0.2f
#define ACQ_W 8
#define ACQ_PHASE 2                                                          /* stage 1's second grid */
#define ACQ_HZ_PER_RAD 254.64790894703253f                                   /* 1600 / (2 pi) */

/* packet_dd_ref.c's constants */
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

/* tau, W, hz_per_rad */
void scd_acq_params(float out[3]) {
    out[0] = ACQ_TAU;
    out[1] = (float) ACQ_W;
    out[2] = ACQ_HZ_PER_RAD;
}

/* filt[0 .. n_frames * 1880) of one stream */
void scd_acq_filt(const int16_t in[], int n_frames, int wide, float foffset_hz, sco_c32 filt[]) {
    sco_state *s = malloc(sizeof *s);
    static const int16_t zero[SCO_FRAME_SIZE];
    sco_init(s, wide, foffset_hz);
    for (int n = 0; n <= n_frames; n++) {
        uint8_t row[SCO_BITS_PER_CALL];
        sco_frame_stats st;
        sco_rx_frame(s, n < n_frames ? in + (size_t) n * SCO_FRAME_SIZE : zero, row, &st);
        if (n >= 1) memcpy(filt + (size_t) (n - 1) * SCO_FRAME_SIZE, s->input_frame, SCO_FRAME_SIZE * sizeof *filt);
    }
    free(s);
}

static inline sco_c32 at(const sco_c32 filt[], long len, long q) { return q >= 0 && q < len ? filt[q] : c32(0.0f, 0.0f); }

/* rho on the grid filt[g0 + 5 i]; D (or NULL) receives D */
float scd_acq_metric(const sco_c32 filt[], long len, long g0, sco_c32 *D_out) {
    sco_c32 D = c32(0.0f, 0.0f);
    float E = 0.0f, Elo = 0.0f;
    sco_c32 prev = at(filt, len, g0);
    E = E + (prev.r * prev.r + prev.i * prev.i);
    for (int i = 1; i < SCO_PREAMBLE_LENGTH; i++) {
        const sco_c32 u = at(filt, len, g0 + 5L * i);
        const float b = (float) (sco_preamblevalues[i] * sco_preamblevalues[i - 1]);
        const float zr = u.r * prev.r + u.i * prev.i;
        const float zi = u.i * prev.r - u.r * prev.i;
        D = c32(D.r + b * zr, D.i + b * zi);
        E = E + (u.r * u.r + u.i * u.i);
        if (i == SCO_PREAMBLE_LENGTH / 2 - 1) Elo = E;
        prev = u;
    }
    if (D_out) *D_out = D;
    const float num = D.r * D.r + D.i * D.i;
    const float den = E * E;
    if (den == 0.0f || !(Elo * 4.0f >= E) || !(Elo * 4.0f <= E * 3.0f)) return 0.0f;
    return num / den;
}

/* the stage-1 metric of lags k = k0 .. k0 + n - 1: the larger of rho on g0 = 5 k and on g0 = 5 k + ACQ_PHASE */
void scd_acq_rho_lags(const sco_c32 filt[], long len, long k0, int n, float rho[]) {
    for (int i = 0; i < n; i++) {
        const float a = scd_acq_metric(filt, len, 5 * (k0 + i), NULL);
        const float b = scd_acq_metric(filt, len, 5 * (k0 + i) + ACQ_PHASE, NULL);
        rho[i] = a > b ? a : b;
    }
}

/*
 * scd_dd_packet (packet_dd_ref.c) started from nu = nu0, also counting the training steps whose output agrees with the
 * preamble: with nu0 = 0 its bits, cost and outputs are scd_dd_packet's (tests/test_packet_acq_oracle.py).
 */
float scd_dd_packet_seeded(const sco_c32 S[ACQ_SYMS], float nu0, uint8_t bits[2 * ACQ_DATA], sco_c32 z[ACQ_DATA],
                           int32_t *matches) {
    sco_c32 w[SCO_EQ_LENGTH];
    for (int k = 0; k < SCO_EQ_LENGTH; k++) w[k] = c32(0.0f, 0.0f);
    sco_c32 p = c32(1.0f, 0.0f);
    float nu = nu0;
    float cost = 0.0f;
    uint16_t lfsr = ACQ_SEED;
    int32_t m = 0;

    for (int i = 0; i < SCO_PREAMBLE_LENGTH + ACQ_DATA; i++) {
        const sco_c32 *x = S + i;
        sco_c32 zz = c32(0.0f, 0.0f);
        for (int k = 0; k < SCO_EQ_LENGTH; k++) zz = cadd(zz, cmul(x[k], cconj(w[k])));
        const sco_c32 y = cmul(zz, cconj(p));

        sco_c32 d;
        if (i < SCO_PREAMBLE_LENGTH) {
            float a = DD_TRAIN_AMP * (float) sco_preamblevalues[i];
            d = c32(a, a);
            if ((y.r + y.i) * (float) sco_preamblevalues[i] > 0.0f) m++;
        } else {
            d = c32(y.r < 0.0f ? -1.0f : 1.0f, y.i < 0.0f ? -1.0f : 1.0f);
        }
        const sco_c32 e = c32(d.r - y.r, d.i - y.i);
        const sco_c32 q = cmul(y, cconj(d));
        const float qm = sqrtf(q.r * q.r + q.i * q.i);
        const float pe = q.i / (qm + DD_PEPS);

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
        const float mm = sqrtf(p.r * p.r + p.i * p.i);
        p = c32(p.r / mm, p.i / mm);

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
    if (matches) *matches = m;
    return cost;
}

typedef struct {
    int64_t grid_sample;
    int32_t call, max_index, matches, frame;
    float cost, metric, freq_hz, nu0;
    uint8_t bits[2 * ACQ_DATA];
} scd_acq_packet;

/*
 * Acquisition over one stream of n_frames frames: every frame f <= n_frames - 3 is searched (the later ones need
 * calls the stream does not have).  seed_nu = 0 runs the DD loop from nu = 0 instead of nu0.  psym, grids (or NULL):
 * 248 outputs / 380 grid symbols per packet.  Returns the number of packets (at most max_packets are written).
 */
int scd_acq_run_stream(const int16_t in[], int n_frames, int wide, float foffset_hz, int seed_nu,
                       scd_acq_packet packets[], sco_c32 psym[], sco_c32 grids[], int max_packets) {
    const long len = (long) n_frames * SCO_FRAME_SIZE;
    sco_c32 *filt = malloc((size_t) (len > 0 ? len : 1) * sizeof *filt);
    float rho[ACQ_LAGS + 2 * ACQ_W];
    int n_packets = 0;
    if (n_frames > 0) scd_acq_filt(in, n_frames, wide, foffset_hz, filt);

    for (int f = 0; f + 2 < n_frames && n_packets < max_packets; f++) {
        const long k0 = (long) ACQ_LAGS * f;
        scd_acq_rho_lags(filt, len, k0 - ACQ_W, ACQ_LAGS + 2 * ACQ_W, rho);
        int kb = 0;
        for (int k = 1; k < ACQ_LAGS; k++)
            if (rho[ACQ_W + k] > rho[ACQ_W + kb]) kb = k;
        const float best = rho[ACQ_W + kb];
        if (!(best >= ACQ_TAU)) continue;
        int ok = 1;
        for (int d = 1; d <= ACQ_W; d++) {
            if (kb - d < 0 && !(rho[ACQ_W + kb - d] < best)) ok = 0;
            if (kb + d >= ACQ_LAGS && !(rho[ACQ_W + kb + d] <= best)) ok = 0;
        }
        if (!ok) continue;

        static const int order[5] = { 0, -1, 1, -2, 2 };
        const long base = 5 * (k0 + kb);
        sco_c32 D, Db = c32(0.0f, 0.0f);
        float rb = -1.0f;
        long g = base;
        for (int t = 0; t < 5; t++) {
            const float r = scd_acq_metric(filt, len, base + order[t], &D);
            if (r > rb) {
                rb = r;
                Db = D;
                g = base + order[t];
            }
        }
        const float nu0 = Db.r > 0.0f ? Db.i / Db.r : 0.0f;
        sco_c32 S[ACQ_SYMS];
        for (int j = 0; j < ACQ_SYMS; j++) S[j] = at(filt, len, g + 5L * j);

        scd_acq_packet *p = &packets[n_packets];
        if (grids) memcpy(grids + (size_t) n_packets * ACQ_SYMS, S, sizeof S);
        p->cost = scd_dd_packet_seeded(S, seed_nu ? nu0 : 0.0f, p->bits,
                                       psym ? psym + (size_t) n_packets * ACQ_DATA : NULL, &p->matches);
        const long gf = g >= 0 ? g / SCO_FRAME_SIZE : -((-g + SCO_FRAME_SIZE - 1) / SCO_FRAME_SIZE);
        p->grid_sample = g;
        p->call = (int32_t) (2 + gf);
        p->max_index = (int32_t) ((g - gf * SCO_FRAME_SIZE) / 5);
        p->frame = f;
        p->metric = rb;
        p->nu0 = nu0;
        p->freq_hz = nu0 * ACQ_HZ_PER_RAD;
        n_packets++;
    }
    free(filt);
    return n_packets;
}
