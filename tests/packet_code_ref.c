/*
 * packet_code_ref.c -- TEST INFRASTRUCTURE ONLY: specification (as code) of the code rates of packet mode's coded
 * payload (DESIGN.md section 8c, "Code rates"): the encoder behind sc_packet_encode_ex_dev and the Viterbi decoder of
 * sc_packet_decode_ex_dev.  The GPU kernels (csrc/sc_fec_kernels.cu: packet_code_encode_kernel,
 * packet_code_viterbi_kernel) are bit-identical to it.  It is built on the rate-1/2 specification, packet_fec_ref.c,
 * which it includes: the CRC, the interleaver, the parity and the LLR sanitising are that file's.
 *
 * code      payload B  steps T = 8 B + 22  mother bits kept per period  transmitted bits N
 * 0 (1/2)   27         238                 c0 c1                        476   (exactly scf_encode / scf_decode)
 * 1 (2/3)   36         310                 c0 c1 | c0                   465
 * 2 (3/4)   41         350                 c0 c1 | c0 | c1              467
 * info      u = B payload bytes, their CRC (high byte first), MSB first: 8 B + 16 bits; then 6 zeros
 * encoder   the rate-1/2 encoder of packet_fec_ref.c over t = 0..T-1 -> mother bits c[2t], c[2t+1]
 * puncture  transmitted bit n < N is mother bit m(n): code 0: m = n; code 1: m = 4 floor(n/3) + (0, 1, 2)[n mod 3];
 *           code 2: m = 6 floor(n/4) + (0, 1, 2, 5)[n mod 4]
 * layout    transmitted bit n goes to p = scf_perm(n); every other position of the 496 carries 0 and is never read
 * decoder   L'[m(n)] = sanitise(llr[scf_perm(n)]) for n < N, L'[m] = 0 for every punctured m; the recursion of
 *           scf_decode over T steps and the traceback from state 0
 * output    data = the first B bytes (the rest 0); crc_ok; flipped over the N transmitted bits; code as given
 * A code that is not 0..2 encodes to all-zero bits and decodes to data 0, crc_ok 0, flipped 0. */
#include "packet_fec_ref.c"

#define SCF_PAYLOAD_MAX 41
#define SCF_STEPS_MAX 350

typedef struct {
    uint8_t data[41];
    uint8_t code;
    uint8_t crc_ok;
    uint8_t reserved0;
    uint16_t flipped;
    uint16_t reserved1;
} scf_payload_ex;                    /* sc_packet_payload_ex */

int scf_code_bytes(int code) { return code == 0 ? 27 : code == 1 ? 36 : code == 2 ? 41 : 0; }
int scf_code_steps(int code) { return scf_code_bytes(code) ? 8 * scf_code_bytes(code) + 22 : 0; }
int scf_code_coded(int code) { return code == 0 ? 476 : code == 1 ? 465 : code == 2 ? 467 : 0; }

int scf_mother(int code, int n) {
    static const int p1[3] = {0, 1, 2}, p2[4] = {0, 1, 2, 5};
    if (code == 1) return 4 * (n / 3) + p1[n % 3];
    if (code == 2) return 6 * (n / 4) + p2[n % 4];
    return n;
}

/* info bits u[0..T-1] -> mother bits c[0..2T-1] */
static void encode_steps(const uint8_t *u, int steps, uint8_t *c) {
    unsigned s = 0;
    for (int t = 0; t < steps; t++) {
        const unsigned r = ((unsigned) u[t] << 6) | s;
        c[2 * t] = (uint8_t) parity(r & 0133);
        c[2 * t + 1] = (uint8_t) parity(r & 0171);
        s = r >> 1;
    }
}

/* payload[41] (bytes past B ignored) -> bits[496] */
void scf_encode_code(int code, const uint8_t *payload, uint8_t *bits) {
    memset(bits, 0, SCF_BITS);
    const int B = scf_code_bytes(code), T = scf_code_steps(code), N = scf_code_coded(code);
    if (!B) return;
    uint8_t by[SCF_PAYLOAD_MAX + 2], u[SCF_STEPS_MAX], c[2 * SCF_STEPS_MAX];
    memcpy(by, payload, (size_t) B);
    const uint16_t crc = scf_crc16(payload, B);
    by[B] = (uint8_t) (crc >> 8);
    by[B + 1] = (uint8_t) (crc & 0xff);
    for (int t = 0; t < 8 * B + 16; t++) u[t] = (by[t / 8] >> (7 - t % 8)) & 1;
    for (int t = 8 * B + 16; t < T; t++) u[t] = 0;
    encode_steps(u, T, c);
    for (int n = 0; n < N; n++) bits[scf_perm(n)] = c[scf_mother(code, n)];
}

/* llr[496] -> one record at code; the final path metrics go to pm_out[64] and the decoded info bits u[0..T-1] to
 * u_out (either may be NULL; neither is written for a code that is not 0..2) */
void scf_decode_code(int code, const float *llr, scf_payload_ex *out, float *pm_out, uint8_t *u_out) {
    memset(out, 0, sizeof(*out));
    out->code = (uint8_t) code;
    const int B = scf_code_bytes(code), T = scf_code_steps(code), N = scf_code_coded(code);
    if (!B) return;
    float L[2 * SCF_STEPS_MAX];
    for (int m = 0; m < 2 * T; m++) L[m] = 0.0f;
    for (int n = 0; n < N; n++) L[scf_mother(code, n)] = sanitise(llr[scf_perm(n)]);
    float pm[64], nx[64];
    uint8_t dec[SCF_STEPS_MAX][64];
    for (int s = 0; s < 64; s++) pm[s] = s ? -INFINITY : 0.0f;
    for (int t = 0; t < T; t++) {
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
    uint8_t u[SCF_STEPS_MAX], c[2 * SCF_STEPS_MAX];
    unsigned s = 0;
    for (int t = T - 1; t >= 0; t--) {
        u[t] = (uint8_t) (s >> 5);
        s = ((s << 1) & 63u) | dec[t][s];
    }
    if (u_out) memcpy(u_out, u, (size_t) T);
    uint8_t by[SCF_PAYLOAD_MAX + 2];
    for (int k = 0; k < B + 2; k++) {
        unsigned x = 0;
        for (int i = 0; i < 8; i++) x = (x << 1) | u[8 * k + i];
        by[k] = (uint8_t) x;
    }
    memcpy(out->data, by, (size_t) B);
    out->crc_ok = scf_crc16(by, B) == (uint16_t) ((by[B] << 8) | by[B + 1]);
    encode_steps(u, T, c);
    unsigned flipped = 0;
    for (int n = 0; n < N; n++) {
        const int m = scf_mother(code, n);
        flipped += (L[m] < 0.0f) != (c[m] != 0);
    }
    out->flipped = (uint16_t) flipped;
}

/* n records, code[k] each: payload [n][41] -> bits [n][496]; llr [n][496] -> out [n] (pm_out [n][64], u_out
 * [n][350] if not NULL) */
void scf_encode_code_batch(const uint8_t *code, const uint8_t *payload, long n, uint8_t *bits) {
    for (long k = 0; k < n; k++) scf_encode_code(code[k], payload + k * SCF_PAYLOAD_MAX, bits + k * SCF_BITS);
}

void scf_decode_code_batch(const uint8_t *code, const float *llr, long n, scf_payload_ex *out, float *pm_out,
                           uint8_t *u_out) {
    for (long k = 0; k < n; k++)
        scf_decode_code(code[k], llr + k * SCF_BITS, out + k, pm_out ? pm_out + 64 * k : NULL,
                        u_out ? u_out + SCF_STEPS_MAX * k : NULL);
}
