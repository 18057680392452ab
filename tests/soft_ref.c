/*
 * soft_ref.c -- TEST INFRASTRUCTURE ONLY: the restatement's frame layer with the equalized data symbols handed out.
 *
 * The reference's data_eq() (src/equalizer.c:64-90) slices its output `sym` and keeps it local, so
 * sco_rx_frame() cannot return it.  scs_rx_frame_soft() is sco_rx_frame() (oracle/sc_oracle.c, qpsk.c:133-239) written
 * again on the oracle's exported primitives -- sco_fir, sco_search, sco_kalman_reset, sco_train_eq, sco_data_eq --
 * and, before every data step, forms `sym` from the equalizer taps as they stand with the operations sco_data_eq
 * uses: sym = sum_{i<5} in[index+i] * conj(C[i]), sequentially, one rounding per operation.
 *
 * tests/test_soft_oracle.py checks that its bits and stats equal sco_run_stream's byte for byte.  Built with the
 * oracle's flags (-std=gnu11 -O2 -ffp-contract=off) against oracle/libsc_oracle.so by tests/soft_ref.py.
 */
#include <complex.h>
#include <string.h>

#include "sc_oracle.h"

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

static inline sco_c32 renorm(sco_c32 p) {                                  /* qpsk.c:147 */
    float m = cabsf(p.r + p.i * I);
    return c32(p.r / m, p.i / m);
}

/* the output of data_eq() at `index`, from the taps before that step */
static sco_c32 data_sym(const sco_kalman *k, const sco_c32 in[], int index) {
    sco_c32 sym = c32(0.0f, 0.0f);
    for (int i = 0; i < SCO_EQ_LENGTH; i++) sym = cadd(sym, cmul(in[index + i], cconj(k->C[i])));
    return sym;
}

int scs_rx_frame_soft(sco_state *s, const int16_t in[SCO_FRAME_SIZE], uint8_t bits[SCO_BITS_PER_CALL],
                      sco_frame_stats *st, sco_c32 sym[SCO_DATA_SYMBOLS]) {
    for (int i = 0; i < SCO_FRAME_SIZE; i++) {                            /* mixer, :138-147 */
        s->rx_phase = cmul(s->rx_phase, s->rx_rect);
        float v = (float) in[i] / 16384.0f;
        s->input_frame[i] = s->input_frame[SCO_FRAME_SIZE + i];
        s->input_frame[SCO_FRAME_SIZE + i] = c32(s->rx_phase.r * v, s->rx_phase.i * v);
    }
    s->rx_phase = renorm(s->rx_phase);

    sco_fir(s->rx_filter, s->wide, s->input_frame, SCO_FRAME_SIZE);      /* :152 */

    for (int i = 0; i < SCO_DEC_LEN; i++) {                               /* decimate, :157-162 */
        s->dec[i] = s->dec[SCO_DEC_LEN + i];
        s->dec[SCO_DEC_LEN + i] = s->input_frame[i * SCO_CYCLES + s->rx_timing];
    }

    int32_t max_index;
    float max_value;
    sco_search(s->dec, &max_index, &max_value);                           /* :172-183 */

    sco_kalman_reset(&s->k);                                              /* :186 */

    int matches = 0;                                                      /* equalize(), :111-123 */
    for (int i = 0; i < SCO_PREAMBLE_LENGTH; i++) {
        float ref = (float) sco_preamblevalues[i];
        if (sco_train_eq(&s->k, s->dec, max_index + i, ref) * ref > 0.0f) matches++;
    }

    float cost = 0.0f;
    int valid;

    if (matches > SCO_PREAMBLE_LENGTH - 30) {                             /* :196 */
        for (int i = max_index; i < SCO_PREAMBLE_LENGTH + max_index; i++)  /* magnitude(), :101-109 */
            cost = cost + (s->dec[i].r * s->dec[i].r + s->dec[i].i * s->dec[i].i);

        int sync_pos = max_index + SCO_PREAMBLE_LENGTH;
        for (int i = 0; i < SCO_DATA_SYMBOLS; i++) {                      /* :206-215 */
            uint8_t dibit;
            sym[i] = data_sym(&s->k, s->dec, sync_pos + i);
            sco_data_eq(&s->k, &s->lfsr_rx, &dibit, s->dec, sync_pos + i);
            bits[2 * i + 1] = dibit >> 1;
            bits[2 * i] = dibit & 0x1;
        }
        s->rx_timing = sync_pos;                                          /* :219 */
        valid = 1;
    } else {
        for (int i = 0; i < SCO_DATA_SYMBOLS; i++) {                      /* :225-229 */
            uint8_t dibit;
            sym[i] = data_sym(&s->k, s->dec, s->rx_timing + i);
            cost = cost + sco_data_eq(&s->k, &s->lfsr_rx, &dibit, s->dec, s->rx_timing + i);
        }
        valid = 0;
    }

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
    s->calls++;
    return valid;
}

/* sco_run_stream() with the symbols: sym[n * 31 + i] = data step i of call n, valid call or not */
void scs_run_stream_soft(const int16_t in[], int n_frames, int wide, float foffset_hz, uint8_t bits[],
                         sco_frame_stats stats[], sco_c32 sym[]) {
    sco_state s;
    uint8_t b[SCO_BITS_PER_CALL];

    sco_init(&s, wide, foffset_hz);
    for (int n = 0; n < n_frames; n++) {
        int valid = scs_rx_frame_soft(&s, in + (size_t) n * SCO_FRAME_SIZE, b, &stats[n],
                                      sym + (size_t) n * SCO_DATA_SYMBOLS);
        if (valid) memcpy(bits + (size_t) n * SCO_BITS_PER_CALL, b, SCO_BITS_PER_CALL);
    }
}
