/*
 * sc_oracle.c -- TEST INFRASTRUCTURE ONLY (see sc_oracle.h).
 *
 * CPU restatement of the reference modem, one explicit IEEE binary32 operation per line of
 * arithmetic, in the reference's evaluation order.  Build with -ffp-contract=off (oracle/Makefile)
 * so no multiply-add is ever contracted.  Re-entrant: all state lives in sco_state, where the
 * reference uses file-scope statics.  Each function cites the reference lines it restates.
 *
 * Conventions: cmul(a,b) = (a.r*b.r - a.i*b.i, a.r*b.i + a.i*b.r) is what gcc emits for a C99
 * complex product of finite operands; complex (op) real is componentwise; conj flips the sign
 * of .i exactly.
 */
#include <math.h>
#include <complex.h>
#include <string.h>

#include "sc_oracle.h"

#define SC_TABLE_PREAMBLE const int8_t sco_preamblevalues[SCO_PREAMBLE_LENGTH]
#define SC_TABLE_RRC35    const float sco_alpha35_root[SCO_NTAPS]
#define SC_TABLE_RRC50    const float sco_alpha50_root[SCO_NTAPS]
#include "../include/sc_tables.inc"

#define FIR_GAIN   2.2f      /* headers/fir.h:17            */
#define FS_HZ      8000.0f   /* headers/qpsk_internal.h:32  */
#define CENTER_HZ  1100.0f   /* headers/qpsk_internal.h:37  */
#define LFSR_SEED  0x4A80    /* headers/scramble.h:16       */

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

/* cmplx(x) of headers/qpsk_internal.h:67 with x = TAU * f / FS evaluated in double
 * (glibc's M_PI is a double, so TAU is; qpsk.c:376,428) and narrowed to float by the call */
void sco_nco_rect(float freq_hz, sco_c32 *rect) {
    double tau = 2.0f * M_PI;
    float x = (float) (tau * freq_hz / FS_HZ);
    rect->r = cosf(x);
    rect->i = sinf(x);
}

/* phase /= cabsf(phase): qpsk.c:147,306 */
static inline sco_c32 renorm(sco_c32 p) {
    float m = cabsf(p.r + p.i * I);
    return c32(p.r / m, p.i / m);
}

/* ------------------------------------------------------------------ src/fir.c:22-44 */
void sco_fir(sco_c32 memory[], int wide, sco_c32 sample[], int length) {
    const float *c = wide ? sco_alpha50_root : sco_alpha35_root;

    for (int j = 0; j < length; j++) {
        for (int i = 0; i < SCO_NTAPS - 1; i++) memory[i] = memory[i + 1];
        memory[SCO_NTAPS - 1] = sample[j];

        float yr = 0.0f, yi = 0.0f;
        for (int i = 0; i < SCO_NTAPS; i++) {
            float pr = memory[i].r * c[i];
            float pi = memory[i].i * c[i];
            yr = yr + pr;
            yi = yi + pi;
        }
        sample[j] = c32(yr * FIR_GAIN, yi * FIR_GAIN);
    }
}

/* --------------------------------------------------------------- src/kalman.c:42-65 */
void sco_kalman_reset(sco_kalman *k) {
    for (int i = 0; i < SCO_EQ_LENGTH; i++) {
        k->C[i] = k->G[i] = k->F[i] = k->H[i] = c32(0.0f, 0.0f);
        k->D[i] = 1.0f;
        for (int j = 0; j < SCO_EQ_LENGTH; j++) k->U[i][j] = c32(0.0f, 0.0f);
    }
}

void sco_kalman_init(sco_kalman *k) {
    memset(k, 0, sizeof *k);
    k->E = 0.1f;
    k->q = 0.08f;
    sco_kalman_reset(k);
}

/* -------------------------------------------------------------- src/kalman.c:85-141 */
void sco_kalman_calculate(sco_kalman *k, const sco_c32 x[], int index) {
    const sco_c32 *xi = x + index;
    const sco_c32 x0c = cconj(xi[0]);

    k->F[0] = x0c;                                                   /* :89  */
    for (int j = 1; j < SCO_EQ_LENGTH; j++) {                        /* :94-100 */
        sco_c32 f = cadd(cmul(k->U[0][j], x0c), cconj(xi[j]));
        for (int i = 1; i < j; i++) f = cadd(f, cmul(k->U[i][j], cconj(xi[i])));
        k->F[j] = f;
    }

    for (int j = 0; j < SCO_EQ_LENGTH; j++)                          /* :105-107 */
        k->G[j] = c32(k->F[j].r * k->D[j], k->F[j].i * k->D[j]);

    /* crealf(g * conjf(f)) = g.r*f.r - g.i*(-f.i)                      :109-113 */
    {
        float p0 = k->G[0].r * k->F[0].r;
        float p1 = k->G[0].i * (-k->F[0].i);
        k->A[0] = k->E + (p0 - p1);
    }
    for (int j = 1; j < SCO_EQ_LENGTH; j++) {
        float p0 = k->G[j].r * k->F[j].r;
        float p1 = k->G[j].i * (-k->F[j].i);
        k->A[j] = k->A[j - 1] + (p0 - p1);
    }

    k->hq = 1.0f + k->q;                                             /* :115 */
    k->ht = k->A[SCO_EQ_LENGTH - 1] * k->q;                          /* :117 */
    k->KY = 1.0f / (k->A[0] + k->ht);                                /* :119 */
    k->D[0] = k->D[0] * ((k->hq * (k->E + k->ht)) * k->KY);          /* :121 */

    for (int j = 1; j < SCO_EQ_LENGTH; j++) {                        /* :125-140 */
        float B = k->A[j - 1] + k->ht;
        k->H[j] = c32((-k->F[j].r) * k->KY, (-k->F[j].i) * k->KY);
        k->KY = 1.0f / (k->A[j] + k->ht);
        k->D[j] = k->D[j] * ((k->hq * B) * k->KY);

        for (int i = 0; i < j; i++) {
            sco_c32 B1 = k->U[i][j];
            k->U[i][j] = cadd(B1, cmul(k->H[j], cconj(k->G[i])));
            k->G[i] = cadd(k->G[i], cmul(k->G[j], cconj(B1)));
        }
    }
}

/* ----------------------------------------------------------- src/equalizer.c:25-40 */
static void update_eq(sco_kalman *k, const sco_c32 in[], int index, sco_c32 error) {
    sco_kalman_calculate(k, in, index);

    error = c32(error.r * k->KY, error.i * k->KY);
    for (int i = 0; i < SCO_EQ_LENGTH; i++) k->C[i] = cadd(k->C[i], cmul(error, cconj(k->G[i])));
}

/* ----------------------------------------------------------- src/equalizer.c:45-58 */
float sco_train_eq(sco_kalman *k, const sco_c32 in[], int index, float ref) {
    sco_c32 val = c32(0.0f, 0.0f);

    for (int i = 0; i < SCO_EQ_LENGTH; i++) val = cadd(val, cmul(in[index + i], k->C[i]));

    /* conjf(ref - val): real - complex = (ref - val.r, -val.i), conjugated */
    sco_c32 error = c32(ref - val.r, -(-val.i));

    update_eq(k, in, index, error);
    return error.r;
}

/* ---------------------------------------------------------- src/scramble.c:57-69 */
void sco_scramble2(uint8_t *dibit, uint16_t *lfsr) {
    for (int i = 0; i < 2; i++) {
        uint16_t out = (uint16_t) (((*lfsr & 0x2) >> 1) ^ (*lfsr & 0x1));
        uint16_t b = (uint16_t) (((*dibit >> i) & 0x1) ^ out);
        *dibit = (uint8_t) ((*dibit & ~(1 << i)) | (b << i));
        *lfsr = (uint16_t) ((*lfsr >> 1) | (out << 14));
    }
}

/* ----------------------------------------------------------- src/equalizer.c:64-90 */
float sco_data_eq(sco_kalman *k, uint16_t *lfsr, uint8_t *bits, const sco_c32 in[], int index) {
    sco_c32 sym = c32(0.0f, 0.0f);

    for (int i = 0; i < SCO_EQ_LENGTH; i++) sym = cadd(sym, cmul(in[index + i], cconj(k->C[i])));

    int bI = sym.r < 0.0f;                    /* qpsk_demod, src/qpsk.c:268-271 */
    int bQ = sym.i < 0.0f;
    float ci = bI ? -1.0f : 1.0f;
    float cq = bQ ? -1.0f : 1.0f;

    sco_c32 error = c32((ci - sym.r) * 0.1f, (cq - sym.i) * 0.1f);

    update_eq(k, in, index, error);

    *bits = (uint8_t) ((bI << 1) | bQ);
    sco_scramble2(bits, lfsr);
    return error.r;
}

/* --------------------------------------------------------------- src/qpsk.c:88-96 */
float sco_correlate(const sco_c32 symbol[], int lag) {
    sco_c32 out = c32(0.0f, 0.0f);

    for (int i = 0; i < SCO_PREAMBLE_LENGTH; i++) {
        float v = (float) sco_preamblevalues[i];
        out = cadd(out, cmul(c32(v, v), symbol[lag + i]));
    }
    return fabsf(out.r * out.r + out.i * out.i);
}

/* ------------------------------------------------------------- src/qpsk.c:172-183 */
void sco_search(const sco_c32 symbol[], int32_t *max_index, float *max_value) {
    float best = 0.0f;
    int idx = 0;

    for (int lag = 0; lag < SCO_PREAMBLE_LENGTH; lag++) {
        float t = sco_correlate(symbol, lag);
        if (t > best) {
            best = t;
            idx = lag;
        }
    }
    *max_index = idx;
    *max_value = best;
}

/* -------------------------------- main() start-up: src/qpsk.c:361-368,375-376,427-434 */
void sco_init(sco_state *s, int wide, float foffset_hz) {
    memset(s, 0, sizeof *s);
    sco_kalman_init(&s->k);
    s->lfsr_tx = LFSR_SEED;
    s->lfsr_rx = LFSR_SEED;
    s->tx_phase = c32(1.0f, 0.0f);                    /* cmplx(0.0f) */
    s->rx_phase = c32(1.0f, 0.0f);
    sco_nco_rect(CENTER_HZ, &s->tx_rect);
    sco_nco_rect(-CENTER_HZ + foffset_hz, &s->rx_rect);
    s->rx_timing = 3;                                 /* FINE_TIMING_OFFSET */
    s->wide = wide;
}

/* ------------------------------------------------------------- src/qpsk.c:133-239 */
int sco_rx_frame(sco_state *s, const int16_t in[SCO_FRAME_SIZE], uint8_t bits[SCO_BITS_PER_CALL],
                 sco_frame_stats *st) {
    /* mixer, :138-147 */
    for (int i = 0; i < SCO_FRAME_SIZE; i++) {
        s->rx_phase = cmul(s->rx_phase, s->rx_rect);
        float v = (float) in[i] / 16384.0f;
        s->input_frame[i] = s->input_frame[SCO_FRAME_SIZE + i];
        s->input_frame[SCO_FRAME_SIZE + i] = c32(s->rx_phase.r * v, s->rx_phase.i * v);
    }
    s->rx_phase = renorm(s->rx_phase);

    /* matched filter on the OLDER half, :152 */
    sco_fir(s->rx_filter, s->wide, s->input_frame, SCO_FRAME_SIZE);

    /* decimate, :157-162 */
    for (int i = 0; i < SCO_DEC_LEN; i++) {
        s->dec[i] = s->dec[SCO_DEC_LEN + i];
        s->dec[SCO_DEC_LEN + i] = s->input_frame[i * SCO_CYCLES + s->rx_timing];
    }

    int32_t max_index;
    float max_value;
    sco_search(s->dec, &max_index, &max_value);       /* :172-183 */

    sco_kalman_reset(&s->k);                          /* :186 */

    int matches = 0;                                  /* equalize(), :111-123 */
    for (int i = 0; i < SCO_PREAMBLE_LENGTH; i++) {
        float ref = (float) sco_preamblevalues[i];
        if (sco_train_eq(&s->k, s->dec, max_index + i, ref) * ref > 0.0f) matches++;
    }

    float cost = 0.0f;
    int valid;

    if (matches > SCO_PREAMBLE_LENGTH - 30) {         /* :196 */
        for (int i = max_index; i < SCO_PREAMBLE_LENGTH + max_index; i++)  /* magnitude(), :101-109 */
            cost = cost + (s->dec[i].r * s->dec[i].r + s->dec[i].i * s->dec[i].i);

        int sync_pos = max_index + SCO_PREAMBLE_LENGTH;
        for (int i = 0; i < SCO_DATA_SYMBOLS; i++) {  /* :206-215 */
            uint8_t dibit;
            sco_data_eq(&s->k, &s->lfsr_rx, &dibit, s->dec, sync_pos + i);
            bits[2 * i + 1] = dibit >> 1;
            bits[2 * i] = dibit & 0x1;
        }
        s->rx_timing = sync_pos;                      /* :219 */
        valid = 1;
    } else {
        for (int i = 0; i < SCO_DATA_SYMBOLS; i++) {  /* :225-229 */
            uint8_t dibit;
            cost = cost + sco_data_eq(&s->k, &s->lfsr_rx, &dibit, s->dec, s->rx_timing + i);
        }
        valid = 0;
    }

    if (st != NULL) {
        st->valid = valid;
        st->max_index = max_index;
        st->matches = matches;
        st->rx_timing = s->rx_timing;
        st->max_value = max_value;
        st->cost = cost;
        for (int i = 0; i < SCO_EQ_LENGTH; i++) {
            st->eq_coeff[2 * i] = s->k.C[i].r;
            st->eq_coeff[2 * i + 1] = s->k.C[i].i;
        }
    }
    s->calls++;
    return valid;
}

/* ------------------------------------------------------------- src/qpsk.c:278-322 */
/* The transmitter up to the scaled complex signal, before qpsk_tx_frame() takes the real part and truncates it:
 * out[i].r is exactly the float the reference converts to int16, out[i].i is the quadrature component. */
int sco_tx_frame_analytic(sco_state *s, sco_c32 out[], const sco_c32 symbol[], int length, int preamble) {
    int n = length * SCO_CYCLES;

    for (int i = 0; i < length; i++) {                /* zero-stuff, :285-291 */
        out[i * SCO_CYCLES] = symbol[i];
        for (int j = 1; j < SCO_CYCLES; j++) out[i * SCO_CYCLES + j] = c32(0.0f, 0.0f);
    }

    sco_fir(s->tx_filter, s->wide, out, n);           /* :296 */

    for (int i = 0; i < n; i++) {                     /* :301-304 */
        s->tx_phase = cmul(s->tx_phase, s->tx_rect);
        out[i] = cmul(out[i], s->tx_phase);
    }
    s->tx_phase = renorm(s->tx_phase);                /* :306 */

    float scale = preamble ? 8192.0f : 16384.0f;      /* :313-319 */
    for (int i = 0; i < n; i++) out[i] = c32(out[i].r * scale, out[i].i * scale);

    return n;
}

int sco_tx_frame(sco_state *s, int16_t samples[], const sco_c32 symbol[], int length, int preamble) {
    sco_c32 signal[length * SCO_CYCLES];
    int n = sco_tx_frame_analytic(s, signal, symbol, length, preamble);
    for (int i = 0; i < n; i++) samples[i] = (int16_t) signal[i].r;             /* :319 */
    return n;
}

static void preamble_symbols(sco_c32 table[SCO_PREAMBLE_LENGTH]) {               /* :361-365 */
    for (int i = 0; i < SCO_PREAMBLE_LENGTH; i++) {
        float v = (float) sco_preamblevalues[i];
        table[i] = c32(v, v);
    }
}

static void data_symbols(sco_c32 symbol[], const uint8_t bits[], int n_symbols) {   /* :251-256 */
    for (int i = 0; i < n_symbols; i++) {
        float vi = (bits[2 * i + 1] == 1) ? -1.0f : 1.0f;
        float vq = (bits[2 * i] == 1) ? -1.0f : 1.0f;
        symbol[i] = c32(vi, vq);
    }
}

int sco_tx_preamble(sco_state *s, int16_t samples[]) {                    /* :327-329 */
    sco_c32 table[SCO_PREAMBLE_LENGTH];
    preamble_symbols(table);
    return sco_tx_frame(s, samples, table, SCO_PREAMBLE_LENGTH, 1);
}

int sco_tx_data(sco_state *s, int16_t samples[], const uint8_t bits[], int n_symbols) {   /* :334-342 */
    sco_c32 symbol[n_symbols];
    data_symbols(symbol, bits, n_symbols);
    return sco_tx_frame(s, samples, symbol, n_symbols, 0);
}

int sco_tx_preamble_analytic(sco_state *s, sco_c32 out[]) {
    sco_c32 table[SCO_PREAMBLE_LENGTH];
    preamble_symbols(table);
    return sco_tx_frame_analytic(s, out, table, SCO_PREAMBLE_LENGTH, 1);
}

int sco_tx_data_analytic(sco_state *s, sco_c32 out[], const uint8_t bits[], int n_symbols) {
    sco_c32 symbol[n_symbols];
    data_symbols(symbol, bits, n_symbols);
    return sco_tx_frame_analytic(s, out, symbol, n_symbols, 0);
}

/* ------------------------------------------------------------- src/qpsk.c:436-458 */
void sco_run_stream(const int16_t in[], int n_frames, int wide, float foffset_hz,
                    uint8_t bits[], sco_frame_stats stats[]) {
    sco_state s;
    uint8_t b[SCO_BITS_PER_CALL];

    sco_init(&s, wide, foffset_hz);
    for (int n = 0; n < n_frames; n++) {
        int valid = sco_rx_frame(&s, in + (size_t) n * SCO_FRAME_SIZE, b, stats ? &stats[n] : NULL);
        if (valid && bits != NULL) memcpy(bits + (size_t) n * SCO_BITS_PER_CALL, b, SCO_BITS_PER_CALL);
    }
}

long sco_run_streams(const int16_t in[], long n_streams, long stride, int n_frames, int wide,
                     uint8_t bits[], int32_t valid[]) {
    sco_state s;
    uint8_t b[SCO_BITS_PER_CALL];
    long total = 0;

    for (long k = 0; k < n_streams; k++) {
        sco_init(&s, wide, 0.0f);
        for (int n = 0; n < n_frames; n++) {
            int v = sco_rx_frame(&s, in + k * stride + (size_t) n * SCO_FRAME_SIZE, b, NULL);
            total += v;
            if (valid != NULL) valid[k * n_frames + n] = v;
            if (v && bits != NULL) memcpy(bits + ((size_t) k * n_frames + n) * SCO_BITS_PER_CALL, b, SCO_BITS_PER_CALL);
        }
    }
    return total;
}

unsigned long sco_sizeof_state(void) { return sizeof (sco_state); }
