/*
 * packet_soft_ref.c -- TEST INFRASTRUCTURE ONLY: the packet-mode specification with the equalized data symbols
 * handed out.
 *
 * sco_ext_run_stream() (oracle/sc_oracle_ext.c) keeps the output `sym` of each data_eq() step local, as the reference's
 * data_eq() (src/equalizer.c:64-90) does.  scs_ext_run_stream_soft() is sco_ext_run_stream() written again on the
 * oracle's exported primitives -- sco_rx_frame, sco_kalman_init, sco_train_eq, sco_data_eq -- and, before every one of
 * a packet's 248 data steps, forms `sym` from the equalizer taps as they stand with the operations sco_data_eq uses:
 * sym = sum_{i<5} in[index+i] * conj(C[i]), sequentially, one rounding per operation (as tests/soft_ref.c does for
 * the ordinary calls).
 *
 * tests/test_packet_soft_oracle.py checks that its packets equal sco_ext_run_stream's and its bits and stats
 * sco_run_stream's.  Built with the oracle's flags (-std=gnu11 -O2 -ffp-contract=off) against oracle/libsc_oracle.so
 * by tests/packet_soft_ref.py.
 */
#include <stdlib.h>
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

/* the output of data_eq() at `index`, from the taps before that step */
static sco_c32 data_sym(const sco_kalman *k, const sco_c32 in[], int index) {
    sco_c32 sym = c32(0.0f, 0.0f);
    for (int i = 0; i < SCO_EQ_LENGTH; i++) sym = cadd(sym, cmul(in[index + i], cconj(k->C[i])));
    return sym;
}

/*
 * sco_ext_run_stream() (oracle/sc_oracle_ext.c, packet mode) written again on sco_rx_frame, sco_kalman_init,
 * sco_train_eq and sco_data_eq, with the 248 equalizer outputs of every packet: psym[k * 248 + i] = data step i of
 * packet k, formed before that step by data_sym().  The packet records have sco_ext_packet's layout.
 */
#define SCS_EXT_DATA (8 * SCO_DATA_SYMBOLS)                                   /* 248 */
#define SCS_EXT_SYMS (SCO_PREAMBLE_LENGTH + SCS_EXT_DATA + SCO_EQ_LENGTH - 1)  /* 380 */

typedef struct {
    int32_t call, max_index, matches, timing;
    float cost;
    uint8_t bits[2 * SCS_EXT_DATA];
} scs_ext_packet;

int scs_ext_run_stream_soft(const int16_t in[], int n_frames, int wide, float foffset_hz, uint8_t bits[],
                            sco_frame_stats stats[], scs_ext_packet packets[], sco_c32 psym[], int max_packets) {
    sco_state *s = malloc(sizeof *s);
    sco_c32 *filt = calloc((size_t) (n_frames + 1) * SCO_FRAME_SIZE, sizeof *filt);
    int *t_entry = calloc((size_t) n_frames + 1, sizeof *t_entry);
    int n_packets = 0;

    sco_init(s, wide, foffset_hz);
    for (int n = 0; n < n_frames; n++) {
        t_entry[n] = s->rx_timing;                                        /* rx_timing at entry of call n */
        sco_frame_stats st;
        uint8_t row[SCO_BITS_PER_CALL];
        memset(row, 255, sizeof row);
        int valid = sco_rx_frame(s, in + (size_t) n * SCO_FRAME_SIZE, row, &st);
        memcpy(bits + (size_t) n * SCO_BITS_PER_CALL, row, sizeof row);
        stats[n] = st;
        if (n >= 1) memcpy(filt + (size_t) (n - 1) * SCO_FRAME_SIZE, s->input_frame, SCO_FRAME_SIZE * sizeof *filt);

        if (valid && n >= 2 && n_packets < max_packets) {
            scs_ext_packet *p = &packets[n_packets];
            sco_c32 *out = psym + (size_t) n_packets * SCS_EXT_DATA;
            n_packets++;
            sco_c32 S[SCS_EXT_SYMS];
            const int T = t_entry[n - 1];
            for (int j = 0; j < SCS_EXT_SYMS; j++)
                S[j] = filt[(size_t) (n - 2) * SCO_FRAME_SIZE + 5 * (st.max_index + j) + T];
            sco_kalman k;
            memset(&k, 0, sizeof k);
            sco_kalman_init(&k);
            int matches = 0;
            for (int i = 0; i < SCO_PREAMBLE_LENGTH; i++) {
                float ref = (float) sco_preamblevalues[i];
                if (sco_train_eq(&k, S, i, ref) * ref > 0.0f) matches++;
            }
            uint16_t lfsr = 0x4A80;                                       /* seeded per packet */
            float cost = 0.0f;
            for (int i = 0; i < SCS_EXT_DATA; i++) {
                uint8_t dibit;
                out[i] = data_sym(&k, S, SCO_PREAMBLE_LENGTH + i);
                cost = cost + sco_data_eq(&k, &lfsr, &dibit, S, SCO_PREAMBLE_LENGTH + i);
                p->bits[2 * i + 1] = dibit >> 1;
                p->bits[2 * i] = dibit & 0x1;
            }
            p->call = n;
            p->max_index = st.max_index;
            p->matches = matches;
            p->timing = T;
            p->cost = cost;
        }
    }
    free(t_entry);
    free(filt);
    free(s);
    return n_packets;
}
