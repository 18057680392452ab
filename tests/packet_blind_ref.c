/*
 * packet_blind_ref.c -- TEST INFRASTRUCTURE ONLY: specification (as code) of blind code detection for packet mode's
 * coded payload (DESIGN.md section 8c, "Blind code detection"): the decoder behind sc_packet_decode_blind_dev.  The GPU
 * kernel (csrc/sc_fec_kernels.cu: packet_blind_decode_kernel) is bit-identical to it.  It is built on the code-rate
 * specification, packet_code_ref.c, which it includes: every candidate is that file's scf_decode_code, unchanged.
 *
 * candidates  codes c in {0, 1, 2} with bit c of mask set (mask 1..7)
 * decode      r_c = scf_decode_code(c, llr)
 * better(a,b) flipped_a * N_b < flipped_b * N_a  (integers; N = 476, 465, 467); equal -> the lower code
 * choose      if any r_c.crc_ok: the best r_c among those with crc_ok; else the best r_c among all candidates
 * output      the chosen r_c, unchanged (data, code = c, crc_ok, flipped, reserved 0)
 * A mask without a candidate gives the all-zero record. */
#include "packet_code_ref.c"

void scf_decode_blind(const float *llr, unsigned mask, scf_payload_ex *out) {
    memset(out, 0, sizeof(*out));
    int have = 0;
    for (int c = 0; c < 3; c++) {
        if (!((mask >> c) & 1u)) continue;
        scf_payload_ex r;
        scf_decode_code(c, llr, &r, NULL, NULL);
        const long n_c = scf_code_coded(c), n_b = have ? scf_code_coded(out->code) : 1;
        int take;
        if (!have) take = 1;
        else if (r.crc_ok != out->crc_ok) take = r.crc_ok > out->crc_ok;
        else take = (long) r.flipped * n_b < (long) out->flipped * n_c;
        if (take) *out = r;
        have = 1;
    }
}

/* n records: llr [n][496] -> out [n] */
void scf_decode_blind_batch(unsigned mask, const float *llr, long n, scf_payload_ex *out) {
    for (long k = 0; k < n; k++) scf_decode_blind(llr + k * SCF_BITS, mask, out + k);
}
