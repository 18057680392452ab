// sc_stats_kernels.cu -- lock / bit statistics over a batch of results (SURVEY section 5: the
// reference only has the DEBUG2 printf and the preamble_frames_detected counter, qpsk.c:70,193,198).
// Counters are plain sums so that ranks can combine them with one ncclAllReduce(sum).
#include "sc_common.cuh"
#include "sc_kernels.h"

namespace sc {

__global__ void __launch_bounds__(256)
lock_stats_kernel(const sc_frame_result *__restrict__ results, long n_streams, long result_stride, int n_frames,
                  unsigned long long *__restrict__ counters) {
    __shared__ unsigned long long sh[SC_N_COUNTERS];
    if (threadIdx.x < SC_N_COUNTERS) sh[threadIdx.x] = 0ull;
    __syncthreads();
    unsigned long long c[SC_N_COUNTERS];
#pragma unroll
    for (int i = 0; i < SC_N_COUNTERS; i++) c[i] = 0ull;
    const long total = n_streams * (long) n_frames;
    for (long k = (long) blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (long) gridDim.x * blockDim.x) {
        const long s = k / n_frames, j = k - s * n_frames;
        const uint4 *p = reinterpret_cast<const uint4 *>(results + s * result_stride + j);
        const uint4 a = __ldg(p), b = __ldg(p + 1);
        const unsigned long long bits = ((unsigned long long) a.y << 32) | a.x;
        const int matches = (int) (short) (b.x >> 16);
        const int max_index = (int) (short) (b.x & 0xffffu);
        const int rx_timing = (int) (short) (b.y & 0xffffu);
        const bool valid = ((b.y >> 16) & 0xffu) != 0;
        c[0] += 1;
        c[2] += (unsigned long long) matches;
        c[7] += (unsigned long long) rx_timing;
        if (valid) {
            c[1] += 1;
            c[3] += (unsigned long long) matches;
            c[4] += (unsigned long long) max_index;
            c[5] += (unsigned long long) __popcll(bits);
            c[6] += (bits & 0xffffffffull) + (bits >> 32);
        }
        int bin = matches >> 4;
        bin = bin > 7 ? 7 : bin;
#pragma unroll
        for (int h = 0; h < 8; h++) c[8 + h] += (bin == h) ? 1ull : 0ull;
    }
#pragma unroll
    for (int i = 0; i < SC_N_COUNTERS; i++) {
        unsigned long long v = c[i];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
        if ((threadIdx.x & 31) == 0 && v) atomicAdd(&sh[i], v);
    }
    __syncthreads();
    if (threadIdx.x < SC_N_COUNTERS && sh[threadIdx.x]) atomicAdd(&counters[threadIdx.x], sh[threadIdx.x]);
}

cudaError_t launch_lock_stats(const sc_frame_result *results, long n_streams, long result_stride, int n_frames,
                              unsigned long long *counters, cudaStream_t st) {
    const long total = n_streams * (long) n_frames;
    int grid = (int) std::min<long>((total + 255) / 256, 148 * 8);
    if (grid < 1) grid = 1;
    lock_stats_kernel<<<grid, 256, 0, st>>>(results, n_streams, result_stride, n_frames, counters);
    g_launch_count++;
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Bit errors against the transmitted bits (sc_ber_stats_dev).  One thread per (stream, call).  The
// alignment rule is the one documented in include/singlecarrier_b200.h; the keystream words of calls
// 0..n_frames-1 are generated on the device by keystream_table_kernel (integer LFSR, src/scramble.c:57-69).
// ------------------------------------------------------------------------------------------------
__global__ void keystream_table_kernel(unsigned long long *__restrict__ ks, int n_frames) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    unsigned m = 0x4A80u;                                            // SEED, scramble.h:16
    for (int n = 0; n < n_frames; n++) {
        unsigned long long w = 0ull;
        for (int j = 0; j < SC_BITS_PER_CALL; j++) {
            const unsigned out = ((m >> 1) ^ m) & 1u;
            m = (m >> 1) | (out << 14);
            w |= (unsigned long long) out << j;
        }
        ks[n] = w;
    }
}

constexpr int BER_GROUP_DELAY = 48;                                  // TX RRC (24) + RX RRC (24) samples
constexpr int BER_ALIGN_TOL = 10;

__global__ void __launch_bounds__(256)
ber_stats_kernel(const sc_frame_result *__restrict__ results, long n_streams, long result_stride, int n_frames,
                 const uint8_t *__restrict__ tx_bits, int n_packets, const int *__restrict__ lead_in, int gap,
                 const int *__restrict__ group, int n_groups, const unsigned long long *__restrict__ ks,
                 unsigned long long *__restrict__ counters) {
    const long total = n_streams * (long) n_frames;
    const int period = FRAME + gap;
    for (long k = (long) blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (long) gridDim.x * blockDim.x) {
        const long s = k / n_frames;
        const int n = (int) (k - s * n_frames);
        if (n < 2) continue;
        const sc_frame_result *rec = results + s * result_stride;
        const uint4 *p = reinterpret_cast<const uint4 *>(rec + n);
        const uint4 a = __ldg(p), b = __ldg(p + 1);
        const bool valid = ((b.y >> 16) & 0xffu) != 0;
        int g = group ? group[s] : 0;
        if (g < 0 || g >= n_groups) continue;
        unsigned long long *c = counters + (long) g * SC_N_BER_COUNTERS;
        atomicAdd(&c[0], 1ull);
        if (!valid) continue;
        atomicAdd(&c[1], 1ull);
        const int max_index = (int) (short) (b.x & 0xffffu);
        // rx_timing in force when frame n-2 was decimated = its value after call n-2
        const int t_prev = (int) rec[n - 2].rx_timing;
        const long pos = (long) (n - 2) * FRAME + 5 * max_index + t_prev - BER_GROUP_DELAY - (lead_in ? lead_in[s] : 0);
        long pkt = pos + period / 2;
        pkt = pkt >= 0 ? pkt / period : -((-pkt + period - 1) / period);          // floor division
        if (pkt < 0 || pkt >= n_packets) continue;
        const long off = pos - pkt * period;
        if (off > BER_ALIGN_TOL || off < -BER_ALIGN_TOL) continue;
        const uint8_t *tb = tx_bits + ((s * n_packets + pkt) * 8) * (long) SC_BITS_PER_CALL;   // first data frame
        unsigned long long txw = 0ull;
        for (int j = 0; j < SC_BITS_PER_CALL; j++) txw |= (unsigned long long) (tb[j] & 1u) << j;
        const unsigned long long bits = ((unsigned long long) a.y << 32) | a.x;
        const unsigned long long diff = (bits ^ ks[n] ^ txw) & ((1ull << SC_BITS_PER_CALL) - 1ull);
        atomicAdd(&c[2], 1ull);
        atomicAdd(&c[3], (unsigned long long) SC_BITS_PER_CALL);
        atomicAdd(&c[4], (unsigned long long) __popcll(diff));
    }
}

cudaError_t launch_ber_stats(const sc_frame_result *results, long n_streams, long result_stride, int n_frames,
                             const uint8_t *tx_bits, int n_packets, const int *lead_in, int gap, const int *group,
                             int n_groups, unsigned long long *counters, cudaStream_t st) {
    unsigned long long *ks = nullptr;
    cudaError_t e = cudaMallocAsync((void **) &ks, (size_t) n_frames * sizeof(unsigned long long), st);
    if (e != cudaSuccess) return e;
    keystream_table_kernel<<<1, 32, 0, st>>>(ks, n_frames);
    g_launch_count++;
    const long total = n_streams * (long) n_frames;
    int grid = (int) std::min<long>((total + 255) / 256, 148 * 8);
    if (grid < 1) grid = 1;
    ber_stats_kernel<<<grid, 256, 0, st>>>(results, n_streams, result_stride, n_frames, tx_bits, n_packets, lead_in, gap,
                                           group, n_groups, ks, counters);
    g_launch_count++;
    e = cudaGetLastError();
    cudaFreeAsync(ks, st);
    return e;
}

// ------------------------------------------------------------------------------------------------
// Bit errors of packet-mode records (sc_packet_ber_stats_dev).  One thread per record; the alignment is
// ber_stats_kernel's, applied to the record's call and max_index.  TX scrambles and RX descrambles in packet
// mode, so the error pattern of data frame f is bits[f] ^ tx word, with no keystream term.
// ------------------------------------------------------------------------------------------------
constexpr int PBER_BYTES = 8 * SC_BITS_PER_CALL;                    // 496 transmitted bytes per packet
// Up to this many groups a block accumulates in shared memory and adds its sums to `counters` at the end: with
// every record's ~20 atomics going to the same few hundred global counters, contention is what the kernel costs.
constexpr int PBER_SHARED_GROUPS = 128;                              // 32 KB of counters

// bit 0 of each of the 8 bytes of x (little endian) -> bits 0..7: byte k lands alone at bit 56 + k
__device__ __forceinline__ unsigned long long pack8(unsigned long long x) {
    return ((x & 0x0101010101010101ull) * 0x0102040810204080ull) >> 56;
}

__device__ __forceinline__ uint4 load16(const uint8_t *p, bool vec) {
    if (vec) return __ldg(reinterpret_cast<const uint4 *>(p));
    unsigned u[4];
#pragma unroll
    for (int i = 0; i < 4; i++)
        u[i] = (unsigned) __ldg(p + 4 * i) | (unsigned) __ldg(p + 4 * i + 1) << 8 |
               (unsigned) __ldg(p + 4 * i + 2) << 16 | (unsigned) __ldg(p + 4 * i + 3) << 24;
    return make_uint4(u[0], u[1], u[2], u[3]);
}

__global__ void __launch_bounds__(256)
packet_ber_stats_kernel(const sc_packet_result *__restrict__ packets, long capacity,
                        const unsigned long long *__restrict__ n_found, const sc_frame_result *__restrict__ results,
                        long n_streams, long result_stride, int n_frames, const uint8_t *__restrict__ tx_bits,
                        int n_packets, const int *__restrict__ lead_in, int gap, const int *__restrict__ group,
                        int n_groups, bool shared, unsigned long long *__restrict__ counters) {
    extern __shared__ unsigned long long pber_sh[];
    unsigned long long *acc = counters;
    if (shared) {
        for (int i = threadIdx.x; i < n_groups * SC_N_PACKET_BER_COUNTERS; i += blockDim.x) pber_sh[i] = 0ull;
        __syncthreads();
        acc = pber_sh;
    }
    const unsigned long long found = *n_found;
    const long n_rec = found < (unsigned long long) capacity ? (long) found : capacity;
    const int period = FRAME + gap;
    const bool rec16 = ((uintptr_t) packets & 15) == 0;
    const bool tx16 = ((uintptr_t) tx_bits & 15) == 0;              // then every 496-byte packet block is aligned
    for (long k = (long) blockIdx.x * blockDim.x + threadIdx.x; k < n_rec; k += (long) gridDim.x * blockDim.x) {
        unsigned long long r[10];                                    // bits[8], stream | call, max_index | ...
        if (rec16) {
            const uint4 *p = reinterpret_cast<const uint4 *>(packets + k);
#pragma unroll
            for (int i = 0; i < 5; i++) {
                const uint4 v = __ldg(p + i);
                r[2 * i] = ((unsigned long long) v.y << 32) | v.x;
                r[2 * i + 1] = ((unsigned long long) v.w << 32) | v.z;
            }
        } else {
            const unsigned long long *p = reinterpret_cast<const unsigned long long *>(packets + k);
#pragma unroll
            for (int i = 0; i < 10; i++) r[i] = __ldg(p + i);
        }
        const long s = (long) (int) (r[8] & 0xffffffffull);
        const unsigned n = (unsigned) (r[8] >> 32);
        const int max_index = (int) (short) (r[9] & 0xffffull);
        if (s < 0 || s >= n_streams || n < 2u || n >= (unsigned) n_frames) continue;
        const int g = group ? group[s] : 0;
        if (g < 0 || g >= n_groups) continue;
        unsigned long long *c = acc + (long) g * SC_N_PACKET_BER_COUNTERS;
        atomicAdd(&c[0], 1ull);
        const int t_prev = (int) __ldg(&results[s * result_stride + n - 2].rx_timing);
        const long pos = (long) (n - 2) * FRAME + 5 * max_index + t_prev - BER_GROUP_DELAY - (lead_in ? lead_in[s] : 0);
        long pkt = pos + period / 2;
        pkt = pkt >= 0 ? pkt / period : -((-pkt + period - 1) / period);          // floor division
        if (pkt < 0 || pkt >= n_packets) continue;
        const long off = pos - pkt * period;
        if (off > BER_ALIGN_TOL || off < -BER_ALIGN_TOL) continue;
        atomicAdd(&c[1], 1ull);
        atomicAdd(&c[2], (unsigned long long) PBER_BYTES);
        // w[q] bit i = bit 0 of transmitted byte 64 q + i; data frame f is bits 62 f .. 62 f + 61 of w
        const uint8_t *tb = tx_bits + (s * n_packets + pkt) * (long) PBER_BYTES;
        unsigned long long w[8] = {0ull, 0ull, 0ull, 0ull, 0ull, 0ull, 0ull, 0ull};
#pragma unroll
        for (int q = 0; q < PBER_BYTES / 16; q++) {
            const uint4 v = load16(tb + 16 * q, tx16);
            const unsigned long long b = pack8(((unsigned long long) v.y << 32) | v.x) |
                                         pack8(((unsigned long long) v.w << 32) | v.z) << 8;
            w[q / 4] |= b << (16 * (q % 4));
        }
        int total = 0;
#pragma unroll
        for (int f = 0; f < 8; f++) {
            const int at = SC_BITS_PER_CALL * f, a = at / 64, o = at % 64;
            const unsigned long long tx = o ? (w[a] >> o) | (w[a + 1] << (64 - o)) : w[a];
            const int e = __popcll((r[f] ^ tx) & ((1ull << SC_BITS_PER_CALL) - 1ull));
            total += e;
            if (e) {
                atomicAdd(&c[8 + f], (unsigned long long) e);
                atomicAdd(&c[16 + f], 1ull);
            }
        }
        if (total) atomicAdd(&c[3], (unsigned long long) total);
        const int bin = total ? min(7, 32 - __clz(total)) : 0;      // 0 | 1 | 2..3 | ... | 32..63 | >= 64
        atomicAdd(&c[24 + bin], 1ull);
    }
    if (shared) {
        __syncthreads();
        for (int i = threadIdx.x; i < n_groups * SC_N_PACKET_BER_COUNTERS; i += blockDim.x)
            if (pber_sh[i]) atomicAdd(&counters[i], pber_sh[i]);
    }
}

cudaError_t launch_packet_ber_stats(const sc_packet_result *packets, long capacity, const unsigned long long *n_found,
                                    const sc_frame_result *results, long n_streams, long result_stride, int n_frames,
                                    const uint8_t *tx_bits, int n_packets, const int *lead_in, int gap,
                                    const int *group, int n_groups, unsigned long long *counters, cudaStream_t st) {
    const int grid = (int) std::min<long>((capacity + 255) / 256, 148 * 8);
    const bool shared = n_groups <= PBER_SHARED_GROUPS;
    const size_t smem = shared ? (size_t) n_groups * SC_N_PACKET_BER_COUNTERS * sizeof(unsigned long long) : 0;
    packet_ber_stats_kernel<<<grid, 256, smem, st>>>(packets, capacity, n_found, results, n_streams, result_stride,
                                                     n_frames, tx_bits, n_packets, lead_in, gap, group, n_groups,
                                                     shared, counters);
    g_launch_count++;
    return cudaGetLastError();
}

}  // namespace sc
