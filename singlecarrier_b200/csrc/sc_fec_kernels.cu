// sc_fec_kernels.cu -- the coded payload of packet-mode packets (DESIGN.md section 8c): encoder, LLRs and a
// soft-decision Viterbi decoder, at rate 1/2 and at a per-stream code rate (1/2, 2/3, 3/4).  The specification is
// tests/packet_fec_ref.c (the code rates: tests/packet_code_ref.c); every kernel here is bit-identical to it.  The
// decoder uses adds and compares only (one rounding per add, no multiply that could be contracted).
#include "sc_common.cuh"
#include "sc_kernels.h"

namespace sc {

constexpr int FEC_STEPS = 238;                      // 232 info bits + 6 tail bits
constexpr int FEC_CODED = SC_PACKET_CODED_BITS;     // 476
constexpr int FEC_BITS = SC_PACKET_BITS;            // 496 floats / bits per packet
constexpr int FEC_SYMS = FEC_BITS / 2;              // 248
constexpr int FEC_WARPS = 8;                        // records per 256-thread block of the LLR and Viterbi kernels
constexpr unsigned FEC_G0 = 0133, FEC_G1 = 0171;
constexpr float FEC_CLAMP = 16777216.0f;            // 2^24: 476 x 2^24 keeps every path metric far below FLT_MAX

// CRC-16/CCITT-FALSE byte table, built by the block in shared memory (no module-scope table: a new __constant__
// symbol would move the constant-bank offsets of every other kernel of the library)
__device__ __forceinline__ void fec_crc_table(unsigned *tab) {
    for (int b = threadIdx.x; b < 256; b += blockDim.x) {
        unsigned c = (unsigned) b << 8;
        for (int i = 0; i < 8; i++) c = (c & 0x8000u) ? ((c << 1) ^ 0x1021u) & 0xffffu : (c << 1) & 0xffffu;
        tab[b] = c;
    }
    __syncthreads();
}

__device__ __forceinline__ unsigned fec_crc_byte(const unsigned *tab, unsigned crc, unsigned byte) {
    return ((crc << 8) ^ tab[((crc >> 8) ^ byte) & 0xffu]) & 0xffffu;
}

// Info bits are held as words: bit t at bit t & 31 of word t >> 5.  Mother (rate-1/2) bit n reads the window
// u[t-6 .. t] (t = n / 2, u of negative index 0), which is r = (u[t] << 6) | s_t bit for bit.
__device__ __forceinline__ unsigned fec_code_bit(unsigned hi, unsigned lo, int n) {
    const int t = n >> 1;
    const unsigned long long x = ((unsigned long long) hi << 32) | lo;    // hi = word t >> 5, lo = the word before
    const unsigned r = (unsigned) (x >> (26 + (t & 31))) & 127u;
    return (unsigned) __popc(r & ((n & 1) ? FEC_G1 : FEC_G0)) & 1u;
}

// packet bit position p -> the coded bit n with pi(n) = p; the padding positions 476..495 map to themselves
__device__ __forceinline__ int fec_coded_index(int p) { return p < FEC_CODED ? 28 * (p % 17) + p / 17 : p; }

// 4 bytes, first at bits 0..7, MSB first -> the info-bit word (and back: the map is an involution)
__device__ __forceinline__ unsigned fec_bytes_to_bits(unsigned w) { return __brev(__byte_perm(w, 0, 0x0123)); }

// mother (rate-1/2) bit m of the info words word(0), word(1), ...: the parity window of step m / 2
template <class Words>
__device__ __forceinline__ unsigned fec_mother_bit(const Words &word, int m) {
    const int wt = m >> 6;                                                 // word of t = m / 2
    return fec_code_bit(word(wt), wt ? word(wt - 1) : 0u, m);
}

// 1 when the hard decision of L[m] (L < 0: bit 1) disagrees with mother bit m of the info words
template <class Words>
__device__ __forceinline__ unsigned fec_flip(const Words &word, const float *L, int m) {
    const unsigned c = fec_mother_bit(word, m);
    return (L[m] < 0.0f) != (c != 0u);
}

// Code rates (DESIGN.md section 8c): payload bytes B, trellis steps T = 8 B + 22, transmitted bits N, and the mother
// bit m(n) of transmitted bit n (the IEEE 802.11a puncturing patterns of this mother code).  The callers check code.
__device__ __forceinline__ int fec_code_bytes(int code) { return code == 0 ? 27 : code == 1 ? 36 : 41; }
__device__ __forceinline__ int fec_code_coded(int code) { return code == 0 ? 476 : code == 1 ? 465 : 467; }
__device__ __forceinline__ int fec_mother_index(int code, int n) {
    if (code == 1) return 4 * (n / 3) + n % 3;                             // c0 c1 | c0
    if (code == 2) {                                                       // c0 c1 | c0 | c1
        const int r = n & 3;
        return 6 * (n >> 2) + r + (r == 3 ? 2 : 0);
    }
    return n;
}

// payload bytes p[0 .. n_bytes-1], then their CRC high byte first -> info words u[0], u[stride], ... (MSB first)
__device__ __forceinline__ void fec_info_words(const unsigned *tab, const uint8_t *p, int n_bytes, unsigned *u,
                                               int stride) {
    unsigned crc = 0xffffu, w = 0u;
    for (int b = 0; b < n_bytes + 2; b++) {
        unsigned byte;
        if (b < n_bytes) {
            byte = __ldg(p + b);
            crc = fec_crc_byte(tab, crc, byte);
        } else {
            byte = b == n_bytes ? crc >> 8 : crc & 0xffu;
        }
        w |= byte << (8 * (b & 3));
        if ((b & 3) == 3 || b == n_bytes + 1) {
            u[(b >> 2) * stride] = fec_bytes_to_bits(w);
            w = 0u;
        }
    }
}

// CRC of the first n_bytes bytes of the info words u[0..]
__device__ __forceinline__ unsigned fec_crc_info(const unsigned *tab, const unsigned *u, int n_bytes) {
    const int nq = (n_bytes + 3) >> 2;
    unsigned crc = 0xffffu;
    for (int q = 0; q < nq; q++) {
        const unsigned by = fec_bytes_to_bits(u[q]);                       // bytes 4q .. 4q + 3
        const int nb = q < nq - 1 ? 4 : n_bytes - 4 * (nq - 1);
        for (int e = 0; e < nb; e++) crc = fec_crc_byte(tab, crc, (by >> (8 * e)) & 0xffu);
    }
    return crc;
}

// byte i of the info words u[0..]
__device__ __forceinline__ unsigned fec_info_byte(const unsigned *u, int i) {
    return (fec_bytes_to_bits(u[i >> 2]) >> (8 * (i & 3))) & 0xffu;
}

__device__ __forceinline__ long fec_records(long capacity, const unsigned long long *n_found) {
    const unsigned long long found = *n_found;
    return found < (unsigned long long) capacity ? (long) found : capacity;
}

// ------------------------------------------------------------------------------------------------
// Encoder: one thread per packet.  Its info words live in a shared-memory column of its own.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
packet_encode_kernel(const uint8_t *__restrict__ payload, long n, uint8_t *__restrict__ bits) {
    __shared__ unsigned sh_u[8][256];
    __shared__ unsigned sh_crc[256];
    fec_crc_table(sh_crc);
    const int tid = threadIdx.x;
    for (long k = (long) blockIdx.x * blockDim.x + tid; k < n; k += (long) gridDim.x * blockDim.x) {
        const auto word = [&](int i) { return sh_u[i][tid]; };
        fec_info_words(sh_crc, payload + k * SC_PACKET_PAYLOAD_BYTES, SC_PACKET_PAYLOAD_BYTES, &sh_u[0][tid], 256);
        uint8_t *out = bits + k * FEC_BITS;
        const bool vec = ((uintptr_t) out & 15) == 0;
        for (int q = 0; q < FEC_BITS / 16; q++) {
            unsigned v[4] = {0u, 0u, 0u, 0u};
#pragma unroll
            for (int e = 0; e < 16; e++) {
                const int pbit = 16 * q + e;
                if (pbit < FEC_CODED) {
                    v[e >> 2] |= fec_mother_bit(word, fec_coded_index(pbit)) << (8 * (e & 3));
                }
            }
            if (vec) {
                *reinterpret_cast<uint4 *>(out + 16 * q) = make_uint4(v[0], v[1], v[2], v[3]);
            } else {
#pragma unroll
                for (int e = 0; e < 16; e++) out[16 * q + e] = (uint8_t) (v[e >> 2] >> (8 * (e & 3)));
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// LLRs: one warp per record.  Lane l loads symbols l, l + 32, ... (coalesced float2) and sums their squared
// slicer errors in that order; an xor butterfly completes S in the order the specification writes out.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
packet_llr_kernel(const float2 *__restrict__ sym, long capacity, const unsigned long long *__restrict__ n_found,
                  float2 *__restrict__ llr, PacketKey key) {
    __shared__ unsigned long long sh_ks[8];
    if (threadIdx.x < 8) {                          // selects, not an index: the parameter stays out of local memory
        unsigned long long v = key.k[0];
#pragma unroll
        for (int f = 1; f < 8; f++) v = threadIdx.x == f ? key.k[f] : v;
        sh_ks[threadIdx.x] = v;
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const long n_rec = fec_records(capacity, n_found);
    for (long k = (long) blockIdx.x * FEC_WARPS + (threadIdx.x >> 5); k < n_rec; k += (long) gridDim.x * FEC_WARPS) {
        const float2 *y = sym + k * FEC_SYMS;
        float acc = 0.0f;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const int idx = lane + 32 * i;
            if (idx < FEC_SYMS) {
                const float2 v = __ldg(y + idx);
                const float er = __fsub_rn(v.x, v.x < 0.0f ? -1.0f : 1.0f);
                const float ei = __fsub_rn(v.y, v.y < 0.0f ? -1.0f : 1.0f);
                acc = __fadd_rn(acc, __fadd_rn(__fmul_rn(er, er), __fmul_rn(ei, ei)));
            }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) acc = __fadd_rn(acc, __shfl_xor_sync(0xffffffffu, acc, off));
        float var = __fdiv_rn(acc, 496.0f);
        if (!(var >= 1e-6f)) var = 1e-6f;
        float2 *out = llr + k * FEC_SYMS;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const int idx = lane + 32 * i;
            if (idx < FEC_SYMS) {
                const int f = idx / SC_DATA_SYMBOLS, j = 2 * (idx - f * SC_DATA_SYMBOLS);
                const unsigned long long w = sh_ks[f] >> j;
                // loaded again (an L1 hit) rather than kept: live across the divide's out-of-line slow path, the
                // block would be saved to the stack
                const float2 v = __ldg(y + idx);
                float lq = __fdiv_rn(__fmul_rn(2.0f, v.y), var), li = __fdiv_rn(__fmul_rn(2.0f, v.x), var);
                if (w & 1ull) lq = -lq;
                if (w & 2ull) li = -li;
                out[idx] = make_float2(isfinite(lq) ? lq : 0.0f, isfinite(li) ? li : 0.0f);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Viterbi: one warp per record, lane l owns states l and l + 32.  Both of its new states have the predecessors
// 2l and 2l + 1, and the two generators share their first and last taps, so one metric M serves all four
// branches: +M for (l <- 2l), (l + 32 <- 2l + 1), -M for the other two.  Two shuffles bring pm[2l], pm[2l + 1]:
// even lanes offer (pm_l, pm_{l+32}), odd lanes the swapped pair.  Decisions go to shared memory by two ballots.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float fec_sanitise(float x) {
    return isfinite(x) ? fminf(fmaxf(x, -FEC_CLAMP), FEC_CLAMP) : 0.0f;
}

// what lane l needs for its states l and l + 32: the two shuffle sources and the branch signs
struct FecLane {
    bool hi, odd, neg0, neg1;
    int src_a, src_b;
};

__device__ __forceinline__ FecLane fec_lane(int lane) {
    FecLane q;
    q.hi = lane >= 16;
    q.odd = lane & 1;
    q.src_a = (2 * lane + (q.hi ? 1 : 0)) & 31;
    q.src_b = (2 * lane + (q.hi ? 0 : 1)) & 31;
    q.neg0 = __popc((2u * lane) & FEC_G0) & 1;
    q.neg1 = __popc((2u * lane) & FEC_G1) & 1;
    return q;
}

// one trellis step on the mother bits' L' pair l: the lane's two path metrics in place -> the warp's decisions
// (bit l of .x: state l took predecessor 2l + 1; .y: the same for state l + 32)
__device__ __forceinline__ uint2 fec_acs(const FecLane &q, float2 l, float &pm0, float &pm1) {
    const float m = __fadd_rn(q.neg0 ? -l.x : l.x, q.neg1 ? -l.y : l.y);
    const float a = __shfl_sync(0xffffffffu, q.odd ? pm1 : pm0, q.src_a);
    const float b = __shfl_sync(0xffffffffu, q.odd ? pm0 : pm1, q.src_b);
    const float p0 = q.hi ? b : a, p1 = q.hi ? a : b;                     // pm[2l], pm[2l + 1]
    const float c00 = __fadd_rn(p0, m), c01 = __fadd_rn(p1, -m);
    const float c10 = __fadd_rn(p0, -m), c11 = __fadd_rn(p1, m);
    const bool t0 = c01 > c00, t1 = c11 > c10;
    pm0 = t0 ? c01 : c00;
    pm1 = t1 ? c11 : c10;
    return make_uint2(__ballot_sync(0xffffffffu, t0), __ballot_sync(0xffffffffu, t1));
}

// traceback from state 0 over steps T-1 .. 0, uniform over the warp: bit t of the decoded info goes to bit t & 31 of
// word t >> 5 (lane 0 writes the words)
__device__ __forceinline__ void fec_traceback(const uint2 *dec, int steps, unsigned *u, int lane) {
    unsigned s = 0u, word = 0u;
    for (int t = steps - 1; t >= 0; t--) {
        word = (word << 1) | (s >> 5);
        if ((t & 31) == 0 && lane == 0) u[t >> 5] = word;
        const uint2 d = dec[t];
        s = ((s << 1) & 63u) | (((s & 32u) ? d.y : d.x) >> (s & 31u) & 1u);
    }
}

__global__ void __launch_bounds__(256)
packet_viterbi_kernel(const float2 *__restrict__ llr, long capacity, const unsigned long long *__restrict__ n_found,
                      sc_packet_payload *__restrict__ out) {
    __shared__ __align__(8) float sh_l[FEC_WARPS][FEC_BITS];    // L'[pi(n)] at n: step t reads one float2
    __shared__ uint2 sh_dec[FEC_WARPS][FEC_STEPS];
    __shared__ unsigned sh_u[FEC_WARPS][8];
    __shared__ unsigned sh_crc[256];
    fec_crc_table(sh_crc);
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const FecLane q = fec_lane(lane);
    float *L = sh_l[w];
    const long n_rec = fec_records(capacity, n_found);
    for (long k = (long) blockIdx.x * FEC_WARPS + w; k < n_rec; k += (long) gridDim.x * FEC_WARPS) {
        const float2 *src = llr + k * FEC_SYMS;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const int idx = lane + 32 * i;
            if (idx < FEC_SYMS) {
                const float2 x = __ldg(src + idx);
                L[fec_coded_index(2 * idx)] = fec_sanitise(x.x);
                L[fec_coded_index(2 * idx + 1)] = fec_sanitise(x.y);
            }
        }
        __syncwarp();
        float pm0 = lane == 0 ? 0.0f : -INFINITY, pm1 = -INFINITY;
        for (int t = 0; t < FEC_STEPS; t++) {
            const uint2 d = fec_acs(q, reinterpret_cast<const float2 *>(L)[t], pm0, pm1);
            if (lane == (t & 31)) sh_dec[w][t] = d;
        }
        __syncwarp();
        fec_traceback(sh_dec[w], FEC_STEPS, sh_u[w], lane);
        __syncwarp();
        const auto words = [&](int i) { return sh_u[w][i]; };
        unsigned flipped = 0u;
        for (int n = lane; n < FEC_CODED; n += 32) flipped += fec_flip(words, L, n);
        flipped = __reduce_add_sync(0xffffffffu, flipped);
        const unsigned crc = fec_crc_info(sh_crc, sh_u[w], SC_PACKET_PAYLOAD_BYTES);
        const unsigned rx_crc = (fec_info_byte(sh_u[w], 27) << 8) | fec_info_byte(sh_u[w], 28);
        const unsigned b6 = fec_bytes_to_bits(sh_u[w][6]);
        if (lane < 8) {
            unsigned v;
            if (lane < 6) v = fec_bytes_to_bits(sh_u[w][lane]);
            else if (lane == 6) v = (b6 & 0x00ffffffu) | ((crc == rx_crc ? 1u : 0u) << 24);
            else v = flipped;                                              // flipped, reserved = 0
            reinterpret_cast<unsigned *>(out + k)[lane] = v;
        }
        __syncwarp();                                                      // L and sh_u are reused by the next record
    }
}

// ------------------------------------------------------------------------------------------------
// Code rates (DESIGN.md section 8c, "Code rates"): the same mother code, punctured per stream.  Transmitted bit n is
// mother bit m(n); the decoder puts L'[pi(n)] at m(n) of a cleared mother-order buffer, so a punctured bit adds 0 to
// both branch terms and the step loop above runs unchanged over the code's T steps.
// ------------------------------------------------------------------------------------------------
constexpr int FEC_STEPS_MAX = 8 * SC_PACKET_PAYLOAD_MAX + 22;         // 350 (rate 3/4)
constexpr int FEC_WORDS_MAX = (FEC_STEPS_MAX + 31) / 32;              // 11
constexpr unsigned FEC_CODES = 3;

__global__ void __launch_bounds__(256)
packet_code_encode_kernel(const uint8_t *__restrict__ payload, long n_streams, int n_packets,
                          const uint8_t *__restrict__ stream_code, uint8_t *__restrict__ bits) {
    __shared__ unsigned sh_u[FEC_WORDS_MAX][256];
    __shared__ unsigned sh_crc[256];
    fec_crc_table(sh_crc);
    const int tid = threadIdx.x;
    const long n = n_streams * n_packets;
    const auto word = [&](int i) { return sh_u[i][tid]; };
    for (long k = (long) blockIdx.x * blockDim.x + tid; k < n; k += (long) gridDim.x * blockDim.x) {
        const unsigned code = __ldg(stream_code + k / n_packets);
        const int n_coded = code < FEC_CODES ? fec_code_coded(code) : 0;   // another code: all-zero bits
        if (n_coded)
            fec_info_words(sh_crc, payload + k * SC_PACKET_PAYLOAD_MAX, fec_code_bytes(code), &sh_u[0][tid], 256);
        uint8_t *out = bits + k * FEC_BITS;
        const bool vec = ((uintptr_t) out & 15) == 0;
        for (int q = 0; q < FEC_BITS / 16; q++) {
            unsigned v[4] = {0u, 0u, 0u, 0u};
#pragma unroll
            for (int e = 0; e < 16; e++) {
                const int nn = fec_coded_index(16 * q + e);                // >= 476 on the padding
                if (nn < n_coded) v[e >> 2] |= fec_mother_bit(word, fec_mother_index(code, nn)) << (8 * (e & 3));
            }
            if (vec) {
                *reinterpret_cast<uint4 *>(out + 16 * q) = make_uint4(v[0], v[1], v[2], v[3]);
            } else {
#pragma unroll
                for (int e = 0; e < 16; e++) out[16 * q + e] = (uint8_t) (v[e >> 2] >> (8 * (e & 3)));
            }
        }
    }
}

// One record's 496 LLRs at src decoded at code (0..2, uniform over the warp), with the warp's buffers L (2 T floats),
// dec (T steps) and u (the info words) -> word `lane` of its sc_packet_payload_ex record (lanes 0..11; 0 on the
// others), and crc_ok and flipped, uniform over the warp.  The caller syncs the warp before L or u is written again.
__device__ __forceinline__ unsigned fec_decode_code(const float2 *src, unsigned code, const FecLane &q, int lane, float *L,
                                                    uint2 *dec, unsigned *u, const unsigned *tab, bool &crc_ok,
                                                    unsigned &flipped) {
    const auto words = [&](int i) { return u[i]; };
    const int n_bytes = fec_code_bytes(code), steps = 8 * n_bytes + 22, n_coded = fec_code_coded(code);
    for (int m = lane; m < 2 * steps; m += 32) L[m] = 0.0f;
    __syncwarp();
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const int idx = lane + 32 * i;
        if (idx < FEC_SYMS) {
            const float2 x = __ldg(src + idx);
            const int n0 = fec_coded_index(2 * idx), n1 = fec_coded_index(2 * idx + 1);
            if (n0 < n_coded) L[fec_mother_index(code, n0)] = fec_sanitise(x.x);
            if (n1 < n_coded) L[fec_mother_index(code, n1)] = fec_sanitise(x.y);
        }
    }
    __syncwarp();
    float pm0 = lane == 0 ? 0.0f : -INFINITY, pm1 = -INFINITY;
    for (int t = 0; t < steps; t++) {
        const uint2 d = fec_acs(q, reinterpret_cast<const float2 *>(L)[t], pm0, pm1);
        if (lane == (t & 31)) dec[t] = d;
    }
    __syncwarp();
    fec_traceback(dec, steps, u, lane);
    __syncwarp();
    flipped = 0u;
    for (int n = lane; n < n_coded; n += 32) flipped += fec_flip(words, L, fec_mother_index(code, n));
    flipped = __reduce_add_sync(0xffffffffu, flipped);
    const unsigned crc = fec_crc_info(tab, u, n_bytes);
    const unsigned rx_crc = (fec_info_byte(u, n_bytes) << 8) | fec_info_byte(u, n_bytes + 1);
    crc_ok = crc == rx_crc;
    const int keep = n_bytes - 4 * lane;                                   // payload bytes in word lane of data
    unsigned v = 0u;
    if (lane < FEC_WORDS_MAX && keep > 0)
        v = fec_bytes_to_bits(u[lane]) & (keep >= 4 ? 0xffffffffu : (1u << (8 * keep)) - 1u);
    if (lane == 10) v |= (code << 8) | ((crc_ok ? 1u : 0u) << 16);        // data[40], code, crc_ok, 0
    if (lane == 11) v = flipped;                                           // flipped, reserved1 = 0
    return v;
}

// one warp per record, as packet_viterbi_kernel; the record's code is read once, so every branch on it is uniform
__global__ void __launch_bounds__(32 * FEC_WARPS, 4)
packet_code_viterbi_kernel(const float2 *__restrict__ llr, const sc_packet_result *__restrict__ packets, long capacity,
                           const unsigned long long *__restrict__ n_found, const uint8_t *__restrict__ stream_code,
                           long n_streams, sc_packet_payload_ex *__restrict__ out) {
    __shared__ __align__(8) float sh_l[FEC_WARPS][2 * FEC_STEPS_MAX];    // L'[m] in mother order; 0 where punctured
    __shared__ uint2 sh_dec[FEC_WARPS][FEC_STEPS_MAX];
    __shared__ unsigned sh_u[FEC_WARPS][FEC_WORDS_MAX];
    __shared__ unsigned sh_crc[256];
    fec_crc_table(sh_crc);
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const FecLane q = fec_lane(lane);
    const long n_rec = fec_records(capacity, n_found);
    for (long k = (long) blockIdx.x * FEC_WARPS + w; k < n_rec; k += (long) gridDim.x * FEC_WARPS) {
        const int s = __ldg(&packets[k].stream);
        const unsigned code = s >= 0 && s < n_streams ? __ldg(stream_code + s) : 255u;
        unsigned v = lane == 10 ? code << 8 : 0u;                         // the record not decoded: data 0, crc_ok 0
        if (code < FEC_CODES) {
            bool crc_ok;
            unsigned flipped;
            v = fec_decode_code(llr + k * FEC_SYMS, code, q, lane, sh_l[w], sh_dec[w], sh_u[w], sh_crc, crc_ok, flipped);
        }
        if (lane < 12) reinterpret_cast<unsigned *>(out + k)[lane] = v;
        __syncwarp();                                                      // L and sh_u are reused by the next record
    }
}

// ------------------------------------------------------------------------------------------------
// Blind code detection (DESIGN.md section 8c, "Blind code detection"): each record decoded at every code of the mask,
// in code order, through the same buffers.  A candidate replaces the kept one when it passes its CRC and the kept one
// does not, or when both agree on the CRC and its flipped / N is smaller (flipped_a N_b < flipped_b N_a, integers; a
// tie keeps the lower code).  Lanes 0..11 keep the kept record's words in a register; the record is written once.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32 * FEC_WARPS, 4)
packet_blind_decode_kernel(const float2 *__restrict__ llr, long capacity, const unsigned long long *__restrict__ n_found,
                           unsigned code_mask, sc_packet_payload_ex *__restrict__ out) {
    __shared__ __align__(8) float sh_l[FEC_WARPS][2 * FEC_STEPS_MAX];
    __shared__ uint2 sh_dec[FEC_WARPS][FEC_STEPS_MAX];
    __shared__ unsigned sh_u[FEC_WARPS][FEC_WORDS_MAX];
    __shared__ unsigned sh_crc[256];
    fec_crc_table(sh_crc);
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const FecLane q = fec_lane(lane);
    const long n_rec = fec_records(capacity, n_found);
    for (long k = (long) blockIdx.x * FEC_WARPS + w; k < n_rec; k += (long) gridDim.x * FEC_WARPS) {
        unsigned best_v = 0u, best_flipped = 0u, best_n = 0u;             // best_n 0: no candidate kept yet
        bool best_ok = false;
#pragma unroll 1
        for (unsigned code = 0; code < FEC_CODES; code++) {
            if (!((code_mask >> code) & 1u)) continue;
            bool crc_ok;
            unsigned flipped;
            const unsigned v = fec_decode_code(llr + k * FEC_SYMS, code, q, lane, sh_l[w], sh_dec[w], sh_u[w], sh_crc,
                                               crc_ok, flipped);
            const unsigned n = fec_code_coded(code);
            if (best_n == 0u || (crc_ok && !best_ok) || (crc_ok == best_ok && flipped * best_n < best_flipped * n)) {
                best_v = v;
                best_ok = crc_ok;
                best_flipped = flipped;
                best_n = n;
            }
            __syncwarp();                                                  // L and sh_u are reused by the next code
        }
        if (lane < 12) reinterpret_cast<unsigned *>(out + k)[lane] = best_v;
    }
}

// grid-stride loops: at most max_blocks CTAs (several per SM), each taking further records after its first
static int fec_grid(long work, int per_block, int max_blocks) {
    return (int) std::max<long>(1, std::min<long>((work + per_block - 1) / per_block, max_blocks));
}

cudaError_t launch_packet_encode(const uint8_t *payload, long n, uint8_t *bits, cudaStream_t st) {
    packet_encode_kernel<<<fec_grid(n, 256, 148 * 2), 256, 0, st>>>(payload, n, bits);
    g_launch_count++;
    return cudaGetLastError();
}

cudaError_t launch_packet_llr(const float *packet_symbols, long capacity, const unsigned long long *n_found, float *llr,
                              const PacketKey &key, cudaStream_t st) {
    packet_llr_kernel<<<fec_grid(capacity, FEC_WARPS, 148 * 16), 32 * FEC_WARPS, 0, st>>>(
        reinterpret_cast<const float2 *>(packet_symbols), capacity, n_found, reinterpret_cast<float2 *>(llr), key);
    g_launch_count++;
    return cudaGetLastError();
}

cudaError_t launch_packet_decode(const float *llr, long capacity, const unsigned long long *n_found,
                                 sc_packet_payload *out, cudaStream_t st) {
    packet_viterbi_kernel<<<fec_grid(capacity, FEC_WARPS, 148 * 16), 32 * FEC_WARPS, 0, st>>>(
        reinterpret_cast<const float2 *>(llr), capacity, n_found, out);
    g_launch_count++;
    return cudaGetLastError();
}

cudaError_t launch_packet_encode_ex(const uint8_t *payload, long n_streams, int n_packets, const uint8_t *stream_code,
                                    uint8_t *bits, cudaStream_t st) {
    packet_code_encode_kernel<<<fec_grid(n_streams * n_packets, 256, 148 * 2), 256, 0, st>>>(payload, n_streams,
                                                                                              n_packets, stream_code, bits);
    g_launch_count++;
    return cudaGetLastError();
}

cudaError_t launch_packet_decode_ex(const float *llr, const sc_packet_result *packets, long capacity,
                                    const unsigned long long *n_found, const uint8_t *stream_code, long n_streams,
                                    sc_packet_payload_ex *out, cudaStream_t st) {
    packet_code_viterbi_kernel<<<fec_grid(capacity, FEC_WARPS, 148 * 16), 32 * FEC_WARPS, 0, st>>>(
        reinterpret_cast<const float2 *>(llr), packets, capacity, n_found, stream_code, n_streams, out);
    g_launch_count++;
    return cudaGetLastError();
}

cudaError_t launch_packet_decode_blind(const float *llr, long capacity, const unsigned long long *n_found,
                                       unsigned code_mask, sc_packet_payload_ex *out, cudaStream_t st) {
    packet_blind_decode_kernel<<<fec_grid(capacity, FEC_WARPS, 148 * 16), 32 * FEC_WARPS, 0, st>>>(
        reinterpret_cast<const float2 *>(llr), capacity, n_found, code_mask, out);
    g_launch_count++;
    return cudaGetLastError();
}

}  // namespace sc
