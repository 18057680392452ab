/*
 * sc_oracle.h -- TEST INFRASTRUCTURE ONLY.
 *
 * CPU restatement ("oracle") of the 1600-baud QPSK modem chain of srsampson/SingleCarrier,
 * written as explicit IEEE binary32 operations in the order the reference performs them
 * (SURVEY.md appendix A).  It exists so the CUDA path can be checked bit-for-bit on any
 * box, including the GPU box where /root/reference does not exist.
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference leg
 * may load this library.  The product (singlecarrier_b200/) never does.
 *
 * Parity pin: this restatement is itself checked against the reference's own object code
 * (oracle/_ref/libsc_ref.so, built from /root/reference/src by oracle/Makefile) in
 * tests/test_oracle_vs_ref.py, and against the committed golden vectors in tests/golden/
 * (generated from that reference build by tools/make_golden.py).
 */
#ifndef SC_ORACLE_H
#define SC_ORACLE_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SCO_FRAME_SIZE       1880   /* headers/qpsk_internal.h:47  */
#define SCO_CYCLES           5      /* headers/qpsk_internal.h:35  */
#define SCO_PREAMBLE_LENGTH  128    /* headers/qpsk_internal.h:52  */
#define SCO_DATA_SYMBOLS     31     /* headers/qpsk_internal.h:40  */
#define SCO_NTAPS            49     /* headers/fir.h:16            */
#define SCO_EQ_LENGTH        5      /* headers/kalman.h:26         */
#define SCO_DEC_LEN          376    /* FRAME_SIZE / CYCLES         */
#define SCO_BITS_PER_CALL    62     /* 2 * DATA_SYMBOLS, SURVEY F5 */

typedef struct { float r, i; } sco_c32;

/* Hsu square-root Kalman state: src/kalman.c:19-35 */
typedef struct {
    sco_c32 C[SCO_EQ_LENGTH];                   /* eq_coeff      */
    sco_c32 G[SCO_EQ_LENGTH];                   /* kalman_gain   */
    sco_c32 U[SCO_EQ_LENGTH][SCO_EQ_LENGTH];
    sco_c32 F[SCO_EQ_LENGTH];
    sco_c32 H[SCO_EQ_LENGTH];
    float D[SCO_EQ_LENGTH];
    float A[SCO_EQ_LENGTH];
    float KY;                                   /* kalman_y      */
    float E, q, hq, ht;
} sco_kalman;

/* everything the reference keeps in file-scope statics (src/qpsk.c:34-60, src/scramble.c:41-42) */
typedef struct {
    sco_c32 input_frame[2 * SCO_FRAME_SIZE];
    sco_c32 dec[2 * SCO_DEC_LEN];               /* 752, not 562: SURVEY F3 */
    sco_c32 rx_filter[SCO_NTAPS];
    sco_c32 tx_filter[SCO_NTAPS];
    sco_c32 rx_phase, rx_rect, tx_phase, tx_rect;
    sco_kalman k;
    int32_t rx_timing;
    int32_t wide;
    uint16_t lfsr_tx, lfsr_rx;
    int32_t calls;
} sco_state;

typedef struct {
    int32_t valid;
    int32_t max_index;
    int32_t matches;
    int32_t rx_timing;      /* after the call */
    float   max_value;
    float   cost;           /* valid: magnitude() of the window ("Mean"); invalid: sum of data_eq() returns */
    float   eq_coeff[10];   /* after the call */
} sco_frame_stats;

extern const int8_t sco_preamblevalues[SCO_PREAMBLE_LENGTH];
extern const float  sco_alpha35_root[SCO_NTAPS];
extern const float  sco_alpha50_root[SCO_NTAPS];

/* stage primitives (same semantics as the reference's L1 functions, but re-entrant) */
void  sco_nco_rect(float freq_hz, sco_c32 *rect);                         /* cmplx(TAU*f/FS), qpsk.c:376,428 */
void  sco_fir(sco_c32 memory[], int wide, sco_c32 sample[], int length);  /* src/fir.c:22-44                 */
void  sco_kalman_init(sco_kalman *k);                                     /* src/kalman.c:60-65              */
void  sco_kalman_reset(sco_kalman *k);                                    /* src/kalman.c:42-55              */
void  sco_kalman_calculate(sco_kalman *k, const sco_c32 x[], int index);  /* src/kalman.c:85-141             */
float sco_train_eq(sco_kalman *k, const sco_c32 in[], int index, float ref);               /* equalizer.c:45-58 */
float sco_data_eq(sco_kalman *k, uint16_t *lfsr, uint8_t *bits, const sco_c32 in[], int index); /* equalizer.c:64-90 */
void  sco_scramble2(uint8_t *dibit, uint16_t *lfsr);                      /* src/scramble.c:57-69            */
float sco_correlate(const sco_c32 symbol[], int lag);                     /* src/qpsk.c:88-96                */
void  sco_search(const sco_c32 symbol[], int32_t *max_index, float *max_value);   /* src/qpsk.c:172-183    */

/* frame layer */
void sco_init(sco_state *s, int wide, float foffset_hz);                  /* main() start-up, qpsk.c:361-368,375-376,427-434 */
int  sco_rx_frame(sco_state *s, const int16_t in[SCO_FRAME_SIZE], uint8_t bits[SCO_BITS_PER_CALL],
                  sco_frame_stats *st);                                   /* src/qpsk.c:133-239              */
int  sco_tx_frame(sco_state *s, int16_t samples[], const sco_c32 symbol[], int length, int preamble); /* qpsk.c:278-322 */
int  sco_tx_preamble(sco_state *s, int16_t samples[]);                    /* src/qpsk.c:327-329              */
int  sco_tx_data(sco_state *s, int16_t samples[], const uint8_t bits[], int n_symbols);    /* qpsk.c:334-342 */
/* the same transmitter stopped before the real part is taken: the scaled complex signal (sco_tx_frame() truncates
 * its real part to int16, so these are pinned to the reference through the int16 outputs) */
int  sco_tx_frame_analytic(sco_state *s, sco_c32 out[], const sco_c32 symbol[], int length, int preamble);
int  sco_tx_preamble_analytic(sco_state *s, sco_c32 out[]);
int  sco_tx_data_analytic(sco_state *s, sco_c32 out[], const uint8_t bits[], int n_symbols);

/* whole-stream drivers (what main()'s loop does, qpsk.c:436-458) */
void sco_run_stream(const int16_t in[], int n_frames, int wide, float foffset_hz,
                    uint8_t bits[], sco_frame_stats stats[]);
long sco_run_streams(const int16_t in[], long n_streams, long stride, int n_frames, int wide,
                     uint8_t bits[], int32_t valid[]);

unsigned long sco_sizeof_state(void);

#ifdef __cplusplus
}
#endif
#endif
