/*
 * packet_fec_ref.c -- TEST INFRASTRUCTURE ONLY: specification (as code) of packet mode's coded payload (DESIGN.md
 * section 8c): the encoder behind sc_packet_encode_dev, the LLRs of sc_packet_llr_dev and the Viterbi decoder of
 * sc_packet_decode_dev.  The GPU kernels (csrc/sc_fec_kernels.cu) are bit-identical to it.
 *
 * payload  P[0..26]; crc = CRC-16/CCITT-FALSE over P (poly 0x1021, init 0xFFFF, MSB first, no reflection, no final
 *          XOR), appended high byte first -> 29 bytes
 * info     u[0..231] = the 29 bytes MSB first; u[232..237] = 0 (the encoder ends in state 0)
 * encoder  s_t = (u[t-1] .. u[t-6]), u[t-1] at bit 5, s_0 = 0; r = (u[t] << 6) | s_t;
 *          c[2t] = parity(r & 0133), c[2t+1] = parity(r & 0171), s_{t+1} = r >> 1, t = 0..237 -> c[0..475]
 * layout   packet bit position p = 62 f + j (data frame f, bit j): c[n] goes to p = 17 (n mod 28) + floor(n / 28);
 *          positions 476..495 carry 0
 *
 * LLRs (L > 0 favours bit 0) of one 248-symbol block y of sc_rx_packets_soft_*: d = the DD slicer's +-1 +-1j,
 * e2_i = er*er + ei*ei; S = the sum of e2 in the order written out in scf_llr; v = S / 496, floored at 1e-6 (NaN
 * too); bit 2i of frame f: (2 y[31f+i].i) / v, bit 2i+1: (2 y[31f+i].r) / v; negated where the packet keystream bit
 * is 1; non-finite -> 0.
 *
 * Viterbi: correlation metric, maximised, float32 with one rounding per add and no multiply.  L' = the LLR at
 * p = pi(n), non-finite -> 0, clamped to [-2^24, 2^24] (so no path metric can reach inf - inf).  b = 1 only when
 * cand_1 > cand_0.  Traceback from state 0.
 *
 * Built with -ffp-contract=off; each float operation is rounded once, in the order written.
 */
#include <math.h>
#include <stdint.h>
#include <string.h>

#define SCF_PAYLOAD 27
#define SCF_INFO 232                 /* 29 bytes */
#define SCF_STEPS 238                /* + 6 tail bits */
#define SCF_CODED 476
#define SCF_BITS 496
#define SCF_SYMS 248
#define SCF_CLAMP 16777216.0f        /* 2^24 */

typedef struct {
    uint8_t data[27];
    uint8_t crc_ok;
    uint16_t flipped;
    uint16_t reserved;
} scf_payload;                       /* sc_packet_payload */

uint16_t scf_crc16(const uint8_t *p, int n) {
    uint16_t c = 0xFFFF;
    for (int k = 0; k < n; k++) {
        c ^= (uint16_t) (p[k] << 8);
        for (int i = 0; i < 8; i++) c = (c & 0x8000) ? (uint16_t) ((c << 1) ^ 0x1021) : (uint16_t) (c << 1);
    }
    return c;
}

int scf_perm(int n) { return 17 * (n % 28) + n / 28; }

static int parity(unsigned x) { return __builtin_parity(x); }

/* info bits u[0..237] -> coded bits c[0..475] */
static void encode_info(const uint8_t *u, uint8_t *c) {
    unsigned s = 0;
    for (int t = 0; t < SCF_STEPS; t++) {
        const unsigned r = ((unsigned) u[t] << 6) | s;
        c[2 * t] = (uint8_t) parity(r & 0133);
        c[2 * t + 1] = (uint8_t) parity(r & 0171);
        s = r >> 1;
    }
}

/* payload[27] -> bits[496] (0/1, the layout of sc_tx_*_dev's bits) */
void scf_encode(const uint8_t *payload, uint8_t *bits) {
    uint8_t by[29], u[SCF_STEPS], c[SCF_CODED];
    memcpy(by, payload, SCF_PAYLOAD);
    const uint16_t crc = scf_crc16(payload, SCF_PAYLOAD);
    by[27] = (uint8_t) (crc >> 8);
    by[28] = (uint8_t) (crc & 0xff);
    for (int t = 0; t < SCF_INFO; t++) u[t] = (by[t / 8] >> (7 - t % 8)) & 1;
    for (int t = SCF_INFO; t < SCF_STEPS; t++) u[t] = 0;
    encode_info(u, c);
    memset(bits, 0, SCF_BITS);
    for (int n = 0; n < SCF_CODED; n++) bits[scf_perm(n)] = c[n];
}

/* the descrambler keystream words of data frames 0..7: register seeded with 0x4A80 per packet, 62 steps per frame */
void scf_keystream(uint64_t *ks) {
    unsigned m = 0x4A80u;
    for (int f = 0; f < 8; f++) {
        uint64_t w = 0;
        for (int j = 0; j < 62; j++) {
            const unsigned out = ((m >> 1) ^ m) & 1u;
            m = (m >> 1) | (out << 14);
            w |= (uint64_t) out << j;
        }
        ks[f] = w;
    }
}

/* one record's block y (248 complex, re/im interleaved) -> llr[496]; returns v */
float scf_llr(const float *y, float *llr) {
    float partial[32];
    for (int l = 0; l < 32; l++) {
        float acc = 0.0f;
        for (int i = l; i < SCF_SYMS; i += 32) {
            const float yr = y[2 * i], yi = y[2 * i + 1];
            const float er = yr - (yr < 0.0f ? -1.0f : 1.0f);
            const float ei = yi - (yi < 0.0f ? -1.0f : 1.0f);
            const float a = er * er;
            const float b = ei * ei;
            const float e2 = a + b;
            acc = acc + e2;
        }
        partial[l] = acc;
    }
    for (int off = 16; off >= 1; off >>= 1) {
        float nxt[32];
        for (int l = 0; l < 32; l++) nxt[l] = partial[l] + partial[l ^ off];
        memcpy(partial, nxt, sizeof(nxt));
    }
    const float S = partial[0];
    float v = S / 496.0f;
    if (!(v >= 1e-6f)) v = 1e-6f;
    uint64_t ks[8];
    scf_keystream(ks);
    for (int k = 0; k < SCF_SYMS; k++) {
        const int f = k / 31, i = k % 31;
        const float yr = y[2 * k], yi = y[2 * k + 1];
        float lq = (2.0f * yi) / v, li = (2.0f * yr) / v;
        if ((ks[f] >> (2 * i)) & 1) lq = -lq;
        if ((ks[f] >> (2 * i + 1)) & 1) li = -li;
        llr[2 * k] = isfinite(lq) ? lq : 0.0f;
        llr[2 * k + 1] = isfinite(li) ? li : 0.0f;
    }
    return v;
}

static float sanitise(float x) {
    if (!isfinite(x)) return 0.0f;
    if (x > SCF_CLAMP) return SCF_CLAMP;
    if (x < -SCF_CLAMP) return -SCF_CLAMP;
    return x;
}

/* llr[496] -> one payload record; the final path metrics of the 64 states go to pm_out and the decoded info bits
 * u[0..237] to u_out (either may be NULL) */
void scf_decode(const float *llr, scf_payload *out, float *pm_out, uint8_t *u_out) {
    float L[SCF_CODED];
    for (int n = 0; n < SCF_CODED; n++) L[n] = sanitise(llr[scf_perm(n)]);
    float pm[64], nx[64];
    uint8_t dec[SCF_STEPS][64];
    for (int s = 0; s < 64; s++) pm[s] = s ? -INFINITY : 0.0f;
    for (int t = 0; t < SCF_STEPS; t++) {
        const float l0 = L[2 * t], l1 = L[2 * t + 1];
        for (int s = 0; s < 64; s++) {
            const unsigned u = (unsigned) s >> 5;
            float cand[2];
            for (int b = 0; b < 2; b++) {
                const unsigned q = (((unsigned) s << 1) & 63u) | (unsigned) b;
                const unsigned r = (u << 6) | q;
                const float m = (parity(r & 0133) ? -l0 : l0) + (parity(r & 0171) ? -l1 : l1);
                cand[b] = pm[q] + m;
            }
            const int take1 = cand[1] > cand[0];
            dec[t][s] = (uint8_t) take1;
            nx[s] = take1 ? cand[1] : cand[0];
        }
        memcpy(pm, nx, sizeof(pm));
    }
    if (pm_out) memcpy(pm_out, pm, sizeof(pm));
    uint8_t u[SCF_STEPS], c[SCF_CODED];
    unsigned s = 0;
    for (int t = SCF_STEPS - 1; t >= 0; t--) {
        u[t] = (uint8_t) (s >> 5);
        s = ((s << 1) & 63u) | dec[t][s];
    }
    if (u_out) memcpy(u_out, u, SCF_STEPS);
    memset(out, 0, sizeof(*out));
    uint8_t by[29];
    for (int k = 0; k < 29; k++) {
        unsigned x = 0;
        for (int i = 0; i < 8; i++) x = (x << 1) | u[8 * k + i];
        by[k] = (uint8_t) x;
    }
    memcpy(out->data, by, SCF_PAYLOAD);
    out->crc_ok = scf_crc16(by, SCF_PAYLOAD) == (uint16_t) ((by[27] << 8) | by[28]);
    encode_info(u, c);
    unsigned flipped = 0;
    for (int n = 0; n < SCF_CODED; n++) flipped += (L[n] < 0.0f) != (c[n] != 0);
    out->flipped = (uint16_t) flipped;
}

/* n records: blocks y [n][496] -> llr [n][496]; llr [n][496] -> out [n] */
void scf_llr_batch(const float *y, long n, float *llr) {
    for (long k = 0; k < n; k++) scf_llr(y + k * SCF_BITS, llr + k * SCF_BITS);
}

void scf_decode_batch(const float *llr, long n, scf_payload *out, float *pm_out, uint8_t *u_out) {
    for (long k = 0; k < n; k++)
        scf_decode(llr + k * SCF_BITS, out + k, pm_out ? pm_out + 64 * k : NULL, u_out ? u_out + SCF_STEPS * k : NULL);
}

void scf_encode_batch(const uint8_t *payload, long n, uint8_t *bits) {
    for (long k = 0; k < n; k++) scf_encode(payload + k * SCF_PAYLOAD, bits + k * SCF_BITS);
}
