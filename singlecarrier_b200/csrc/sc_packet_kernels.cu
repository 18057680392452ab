// sc_packet_kernels.cu -- PACKET MODE (extension, off by default; no counterpart in the reference).
//
// The reference decodes 31 of a packet's 8 x 31 data symbols, never scrambles on transmit and takes the late
// symbols of a window from unfiltered samples (src/qpsk.c:206-215, 386, 397, 161: all TODOs).  Packet mode
// finishes them without touching anything the reference does compute: after the ordinary calls of a block have
// run, every VALID call n >= 2 gets a second, full decode --
//   S[j] = filt[1880 (n-2) + 5 (max_index + j) + T], j < 380, T = rx_timing at entry of call n-1, taken from the
//          continuous matched-filter output (frames n-2 and n-1);
//   kalman_reset, 128 x train_eq, then 248 x data_eq with the equalizer state carried through all 8 frames and the
//   descrambler re-seeded per packet.
// The specification is the CPU statement of exactly this in the test tree (DESIGN.md, packet mode), built from the
// pinned primitives; parity is against that statement only ("parity unpinned" in the sense of the reference).
//
//   packet_list_kernel    (one thread per stream x call)  valid calls of the block -> compact list
//   packet_fir_kernel     (one warp per listed packet)    int16 -> mix -> 49-tap RRC at the 380 symbol instants
//   packet_track_kernel   (one thread per listed packet)  the sequential loop, 128 + 248 steps
//   packet_track_dd_kernel                                 the same with the decision-directed equalizer (SC_FLAG_PACKET_DD)
//   packet_track_acq_kernel                                that equalizer on the grids acquisition found (SC_FLAG_PACKET_ACQ;
//                                                          the list then comes from sc_acq_kernels.cu)
#include "sc_common.cuh"
#include "sc_tables.cuh"
#include "sc_tracker.cuh"
#include "sc_kernels.h"
#include "sc_acq.cuh"

namespace sc {

static __constant__ uint32_t c_pk_pre_neg[4] = {pre_neg_word(0), pre_neg_word(1), pre_neg_word(2), pre_neg_word(3)};

__global__ void __launch_bounds__(256)
packet_list_kernel(const sc_frame_result *__restrict__ results, long result_stride, int n_streams, int j_lo, int j_hi,
                   uint32_t call0, int cap, int2 *__restrict__ list, int *__restrict__ count) {
    const int nj = j_hi - j_lo;
    const long total = (long) n_streams * nj;
    for (long k = (long) blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (long) gridDim.x * blockDim.x) {
        const int s = (int) (k / nj), j = j_lo + (int) (k - (long) s * nj);
        if (call0 + (uint32_t) j < 2u) continue;                     // frames n-2, n-1 must exist
        if (!results[s * result_stride + j].valid) continue;
        const int pos = atomicAdd(count, 1);
        if (pos < cap) list[pos] = make_int2(s, j);
    }
}

// ---- symbols of one packet ------------------------------------------------------------------------
constexpr int PK_NSAMP = NTAPS + CYC * (PK_SYMS - 1);                 // 1944 mixed samples
constexpr int PK_FIR_WARPS = 2;

// ACQ (SC_FLAG_PACKET_ACQ): the grid starts at g = 1880 (n-2) + info[e].x, which acquisition found; the samples
// reach from frame n-3 to frame n.
template <bool ACQ>
__global__ void __launch_bounds__(PK_FIR_WARPS * 32)
packet_fir_kernel(PacketSrc src, const int2 *__restrict__ list, const int *__restrict__ count, int cap,
                  float2 *__restrict__ sym, const int4 *__restrict__ info) {
    __shared__ __align__(16) float2 smem[PK_FIR_WARPS][PK_NSAMP + 4];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_list = min(*count, cap);
    float2 *mix = smem[warp];
    for (int e = blockIdx.x * PK_FIR_WARPS + warp; e < n_list; e += gridDim.x * PK_FIR_WARPS) {
        const int2 ent = list[e];
        const int s = ent.x, j = ent.y;
        int q0;                                                       // first raw sample, relative to frame n-2
        if constexpr (ACQ) {
            q0 = info[e].x - (NTAPS - 1);
        } else {
            const sc_frame_result *rec = src.results + (long) s * src.result_stride;
            const int mi = rec[j].max_index;
            int T;
            if (j >= 2) T = rec[j - 2].rx_timing;                     // rx_timing after call n-2 = at entry of call n-1
            else T = (j == 1 ? src.timing_at_call0 : src.timing_before_call0)[s];
            T = min(max(T, NTAPS - 1), 2 * PRE - 1);
            q0 = CYC * mi + T - (NTAPS - 1);                          // 0 .. 842: samples of frames n-2 and n-1 only
        }
        __syncwarp();
        // mixer, qpsk.c:138-145 (table = phasor / 16384)
        for (int i = lane; i < PK_NSAMP; i += 32) mix[i] = packet_mix(src, s, j, q0 + i);
        __syncwarp();
        float2 *out = sym + ((long) (e >> 5) * PK_SYMS) * 32 + (e & 31);
        for (int o = lane; o < PK_SYMS; o += 32) {                    // src/fir.c:36-42 at sample 5 o + 48 of the window
            const u64 *mp = reinterpret_cast<const u64 *>(mix) + CYC * o;
            u64 acc = 0ull;
            if (src.wide) {
#pragma unroll
                for (int k = 0; k < NTAPS; k++) acc = pk_add(acc, pk_mul_bcast_pz(mp[k], tap<true>(k)));
            } else {
#pragma unroll
                for (int k = 0; k < NTAPS; k++) acc = pk_add(acc, pk_mul_bcast_pz(mp[k], tap<false>(k)));
            }
            float yr, yi;
            unpk(acc, yr, yi);
            out[(long) o * 32] = make_float2(__fmul_rn(yr, FIR_GAIN), __fmul_rn(yi, FIR_GAIN));
        }
    }
}

// ---- the sequential loop over one packet ----------------------------------------------------------------
// SOFT: the equalizer output of data step i also goes to psym[pos * PK_DATA + i], pos = the packet's record slot.  The
// slot is claimed before the data loop (248 outputs cannot wait in registers), so a record and its symbol block always
// belong to the same packet; both are dropped beyond packet_capacity.
template <bool SOFT>
__global__ void __launch_bounds__(128)
packet_track_kernel(PacketSrc src, const int2 *__restrict__ list, const int *__restrict__ count, int cap,
                    const float2 *__restrict__ sym, PacketKey key, sc_packet_result *__restrict__ packets,
                    long packet_capacity, unsigned long long *__restrict__ n_packets, float2 *__restrict__ psym) {
    const int n_list = min(*count, cap);
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_list) return;
    const int2 ent = list[e];
    const float2 *X = sym + ((long) (e >> 5) * PK_SYMS) * 32 + (e & 31);

    Tracker tk;
    tk.reset();                                                       // qpsk.c:186
    c32 x[EQ];
#pragma unroll
    for (int i = 0; i < EQ - 1; i++) x[i] = from2(X[i * 32]);
    int matches = 0;
    c32 nxt = from2(X[(EQ - 1) * 32]);
#pragma unroll 1
    for (int i = 0; i < PRE; i++) {                                   // equalize(), qpsk.c:111-123
        x[EQ - 1] = nxt;
        nxt = from2(X[(i + EQ) * 32]);
        const float ref = ((c_pk_pre_neg[i >> 5] >> (i & 31)) & 1u) ? -1.0f : 1.0f;
        const float er = tk.train(x, ref);
        if (__fmul_rn(er, ref) > 0.0f) matches++;
#pragma unroll
        for (int k = 0; k < EQ - 1; k++) x[k] = x[k + 1];
    }
    sc_packet_result r;
    float cost = 0.0f;
    unsigned long long word = 0ull;
    unsigned long long pos = 0ull;
    float2 *out = nullptr;
    if (SOFT) {
        pos = atomicAdd(n_packets, 1ull);
        if ((long) pos < packet_capacity) out = psym + (long) pos * PK_DATA;
    }
#pragma unroll 1
    for (int i = 0; i < PK_DATA; i++) {                               // qpsk.c:206-215 over all NS x DATA_SYMBOLS symbols
        x[EQ - 1] = nxt;
        nxt = from2(X[min(PRE + i + EQ, PK_SYMS - 1) * 32]);
        int bI, bQ;
        float er;
        if (SOFT) {
            c32 s;
            er = tk.data(x, bI, bQ, s);
            if (out) out[i] = to2(s);
        } else {
            er = tk.data(x, bI, bQ);
        }
        cost = __fadd_rn(cost, er);
        const int f = i / NDATA, k = i - f * NDATA;
        word |= ((unsigned long long) (unsigned) (bQ | (bI << 1))) << (2 * k);
        if (k == NDATA - 1) {
            r.bits[f] = word ^ key.k[f];                              // scramble(bits, rx) from a register seeded per packet
            word = 0ull;
        }
#pragma unroll
        for (int kk = 0; kk < EQ - 1; kk++) x[kk] = x[kk + 1];
    }
    const sc_frame_result *rec = src.results + (long) ent.x * src.result_stride + ent.y;
    r.stream = src.stream0 + ent.x;
    r.call_index = src.call0 + (uint32_t) ent.y;
    r.max_index = rec->max_index;
    r.matches = (int16_t) matches;
    r.cost = cost;
    r.acq_metric = 0.0f;
    r.acq_freq_hz = 0.0f;
    r.grid_sample = 0;
    if (!SOFT) pos = atomicAdd(n_packets, 1ull);
    if ((long) pos < packet_capacity) packets[pos] = r;
}

// ---- SC_FLAG_PACKET_DD: the decision-directed equalizer over one packet ---------------------------------------------
// The same grid, list and record-slot protocol as packet_track_kernel; the loop is a 5-tap normalised LMS filter and a
// second-order carrier loop (DESIGN.md section 8; specification tests/packet_dd_ref.c, scd_dd_packet), written out
// operation for operation.  matches is the call's; cost is the sum of |d - y|^2 over the 248 data steps.
constexpr float DD_MU = 0.03f, DD_ALPHA = 0.05f, DD_BETA = 0.002f, DD_EPS = 1e-6f, DD_TRAIN_AMP = 0.5f,
                DD_PEPS = 1e-6f;

struct DdLoop {
    c32 w[EQ];
    c32 p;
    float nu;

    __device__ __forceinline__ void reset() {
#pragma unroll
        for (int k = 0; k < EQ; k++) w[k] = mk(0.0f, 0.0f);
        p = mk(1.0f, 0.0f);
        nu = 0.0f;
    }
    // the derotated output y of the window x
    __device__ __forceinline__ c32 output(const c32 (&x)[EQ]) const {
        c32 z = mk(0.0f, 0.0f);
#pragma unroll
        for (int k = 0; k < EQ; k++) z = cadd(z, cmulc(x[k], w[k]));
        return cmulc(z, p);
    }
    // one step towards the decision d; returns e = d - y
    __device__ __forceinline__ c32 step(const c32 (&x)[EQ], c32 y, c32 d) {
        const c32 e = mk(__fsub_rn(d.r, y.r), __fsub_rn(d.i, y.i));
        const c32 q = cmulc(y, d);
        const float qm = __fsqrt_rn(__fadd_rn(__fmul_rn(q.r, q.r), __fmul_rn(q.i, q.i)));
        const float pe = __fdiv_rn(q.i, __fadd_rn(qm, DD_PEPS));
        float n = DD_EPS;
#pragma unroll
        for (int k = 0; k < EQ; k++) n = __fadd_rn(n, __fadd_rn(__fmul_rn(x[k].r, x[k].r), __fmul_rn(x[k].i, x[k].i)));
        const float g = __fdiv_rn(DD_MU, n);
        const c32 ep = cmul(e, p);
        const c32 u = mk(__fmul_rn(ep.r, g), -__fmul_rn(ep.i, g));
#pragma unroll
        for (int k = 0; k < EQ; k++) w[k] = cadd(w[k], cmul(x[k], u));
        nu = __fadd_rn(nu, __fmul_rn(DD_BETA, pe));
        const float phi = __fadd_rn(__fmul_rn(DD_ALPHA, pe), nu);
        p = mk(__fsub_rn(p.r, __fmul_rn(p.i, phi)), __fadd_rn(p.i, __fmul_rn(p.r, phi)));
        const float m = __fsqrt_rn(__fadd_rn(__fmul_rn(p.r, p.r), __fmul_rn(p.i, p.i)));
        p = mk(__fdiv_rn(p.r, m), __fdiv_rn(p.i, m));
        return e;
    }
};

// ACQ (SC_FLAG_PACKET_ACQ, packet_track_acq_kernel): the loop starts from nu = nu0 of info[e], matches counts the
// training steps with (y.r + y.i) v_i > 0, and the record carries the grid's position, rho and the offset estimate.
template <bool SOFT, bool ACQ>
__device__ __forceinline__ void
track_dd(PacketSrc src, const int2 *__restrict__ list, const int *__restrict__ count, int cap,
         const float2 *__restrict__ sym, const PacketKey &key, sc_packet_result *__restrict__ packets,
         long packet_capacity, unsigned long long *__restrict__ n_packets, float2 *__restrict__ psym,
         const int4 *__restrict__ info) {
    const int n_list = min(*count, cap);
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_list) return;
    const int2 ent = list[e];
    const float2 *X = sym + ((long) (e >> 5) * PK_SYMS) * 32 + (e & 31);

    DdLoop dd;
    dd.reset();
    int4 acq = make_int4(0, 0, 0, 0);
    int acq_matches = 0;
    if constexpr (ACQ) {
        acq = info[e];
        dd.nu = __int_as_float(acq.z);
    }
    c32 x[EQ];
#pragma unroll
    for (int i = 0; i < EQ - 1; i++) x[i] = from2(X[i * 32]);
    c32 nxt = from2(X[(EQ - 1) * 32]);
#pragma unroll 1
    for (int i = 0; i < PRE; i++) {
        x[EQ - 1] = nxt;
        nxt = from2(X[(i + EQ) * 32]);
        const bool neg = (c_pk_pre_neg[i >> 5] >> (i & 31)) & 1u;
        const float a = neg ? -DD_TRAIN_AMP : DD_TRAIN_AMP;
        const c32 y = dd.output(x);
        if constexpr (ACQ)
            if (__fmul_rn(__fadd_rn(y.r, y.i), neg ? -1.0f : 1.0f) > 0.0f) acq_matches++;
        dd.step(x, y, mk(a, a));
#pragma unroll
        for (int k = 0; k < EQ - 1; k++) x[k] = x[k + 1];
    }
    sc_packet_result r;
    float cost = 0.0f;
    unsigned long long word = 0ull;
    unsigned long long pos = 0ull;
    float2 *out = nullptr;
    if (SOFT) {
        pos = atomicAdd(n_packets, 1ull);
        if ((long) pos < packet_capacity) out = psym + (long) pos * PK_DATA;
    }
#pragma unroll 1
    for (int i = 0; i < PK_DATA; i++) {
        x[EQ - 1] = nxt;
        nxt = from2(X[min(PRE + i + EQ, PK_SYMS - 1) * 32]);
        const c32 y = dd.output(x);
        const int bI = y.r < 0.0f, bQ = y.i < 0.0f;
        const c32 er = dd.step(x, y, mk(bI ? -1.0f : 1.0f, bQ ? -1.0f : 1.0f));
        cost = __fadd_rn(cost, __fadd_rn(__fmul_rn(er.r, er.r), __fmul_rn(er.i, er.i)));
        if (SOFT && out) out[i] = to2(y);
        const int f = i / NDATA, k = i - f * NDATA;
        word |= ((unsigned long long) (unsigned) (bQ | (bI << 1))) << (2 * k);
        if (k == NDATA - 1) {
            r.bits[f] = word ^ key.k[f];
            word = 0ull;
        }
#pragma unroll
        for (int kk = 0; kk < EQ - 1; kk++) x[kk] = x[kk + 1];
    }
    r.stream = src.stream0 + ent.x;
    r.cost = cost;
    if constexpr (ACQ) {
        const long long g = (long long) FRAME * ((long long) src.call0 + ent.y - 2) + acq.x;
        const long long f = g >= 0 ? g / FRAME : -((-g + FRAME - 1) / FRAME);
        r.call_index = (uint32_t) (2 + f);
        r.max_index = (int16_t) ((g - f * FRAME) / CYC);
        r.matches = (int16_t) acq_matches;
        r.acq_metric = __int_as_float(acq.y);
        r.acq_freq_hz = __fmul_rn(__int_as_float(acq.z), ACQ_HZ_PER_RAD);
        r.grid_sample = g;
    } else {
        const sc_frame_result *rec = src.results + (long) ent.x * src.result_stride + ent.y;
        r.call_index = src.call0 + (uint32_t) ent.y;
        r.max_index = rec->max_index;
        r.matches = rec->matches;
        r.acq_metric = 0.0f;
        r.acq_freq_hz = 0.0f;
        r.grid_sample = 0;
    }
    if (!SOFT) pos = atomicAdd(n_packets, 1ull);
    if ((long) pos < packet_capacity) packets[pos] = r;
}

template <bool SOFT>
__global__ void __launch_bounds__(128)
packet_track_dd_kernel(PacketSrc src, const int2 *__restrict__ list, const int *__restrict__ count, int cap,
                       const float2 *__restrict__ sym, PacketKey key, sc_packet_result *__restrict__ packets,
                       long packet_capacity, unsigned long long *__restrict__ n_packets, float2 *__restrict__ psym) {
    track_dd<SOFT, false>(src, list, count, cap, sym, key, packets, packet_capacity, n_packets, psym, nullptr);
}

template <bool SOFT>
__global__ void __launch_bounds__(128)
packet_track_acq_kernel(PacketSrc src, const int2 *__restrict__ list, const int *__restrict__ count, int cap,
                        const float2 *__restrict__ sym, PacketKey key, sc_packet_result *__restrict__ packets,
                        long packet_capacity, unsigned long long *__restrict__ n_packets, float2 *__restrict__ psym,
                        const int4 *__restrict__ info) {
    track_dd<SOFT, true>(src, list, count, cap, sym, key, packets, packet_capacity, n_packets, psym, info);
}

cudaError_t launch_packet_pass(const PacketSrc &src, int n_streams, int j_lo, int j_hi, int cap, int2 *list, int *count,
                               float2 *sym, const PacketKey &key, sc_packet_result *packets, long packet_capacity,
                               unsigned long long *n_packets, float2 *packet_sym, bool dd, const AcqScratch *acq,
                               cudaStream_t st) {
    cudaError_t e = cudaMemsetAsync(count, 0, sizeof(int), st);
    if (e != cudaSuccess) return e;
    const long total = (long) n_streams * (j_hi - j_lo);
    if (total <= 0) return cudaSuccess;
    if (acq) {
        e = launch_acq_pass(src, n_streams, j_lo, j_hi, cap, list, acq->info, count, st);
        if (e != cudaSuccess) return e;
    } else {
        const int g1 = (int) std::min<long>((total + 255) / 256, 148L * 8);
        packet_list_kernel<<<g1, 256, 0, st>>>(src.results, src.result_stride, n_streams, j_lo, j_hi, src.call0, cap, list,
                                               count);
    }
    // the list length is only known on the device: size the grids for the worst case (every call valid), capped;
    // blocks beyond the list return at once
    const long worst = std::min<long>(total, cap);
    const int g2 = (int) std::min<long>((worst + PK_FIR_WARPS - 1) / PK_FIR_WARPS, 148L * 16);
    if (acq)
        packet_fir_kernel<true><<<g2, PK_FIR_WARPS * 32, 0, st>>>(src, list, count, cap, sym, acq->info);
    else
        packet_fir_kernel<false><<<g2, PK_FIR_WARPS * 32, 0, st>>>(src, list, count, cap, sym, nullptr);
    const int g3 = (int) ((worst + 127) / 128);
    if (acq && packet_sym)
        packet_track_acq_kernel<true><<<g3, 128, 0, st>>>(src, list, count, cap, sym, key, packets, packet_capacity,
                                                          n_packets, packet_sym, acq->info);
    else if (acq)
        packet_track_acq_kernel<false><<<g3, 128, 0, st>>>(src, list, count, cap, sym, key, packets, packet_capacity,
                                                           n_packets, nullptr, acq->info);
    else if (dd && packet_sym)
        packet_track_dd_kernel<true><<<g3, 128, 0, st>>>(src, list, count, cap, sym, key, packets, packet_capacity,
                                                         n_packets, packet_sym);
    else if (dd)
        packet_track_dd_kernel<false><<<g3, 128, 0, st>>>(src, list, count, cap, sym, key, packets, packet_capacity,
                                                          n_packets, nullptr);
    else if (packet_sym)
        packet_track_kernel<true><<<g3, 128, 0, st>>>(src, list, count, cap, sym, key, packets, packet_capacity, n_packets,
                                                      packet_sym);
    else
        packet_track_kernel<false><<<g3, 128, 0, st>>>(src, list, count, cap, sym, key, packets, packet_capacity,
                                                       n_packets, nullptr);
    g_launch_count += acq ? 4 : 3;
    return cudaGetLastError();
}

}  // namespace sc
