// sc_acq_kernels.cu -- packet-mode acquisition (SC_FLAG_PACKET_ACQ, DESIGN.md section 8b).
//
// On ACQ banks these two kernels replace packet_list_kernel: packets are found from the samples themselves by the
// differential preamble metric rho of the specification (tests/packet_acq_ref.c), not taken from the reference's
// per-call detection.  Call n decides frame n-2.
//
//   acq_detect_kernel  (one CTA per stream-frame)  filt on the frame's grids 5 k and 5 k + 2 (376 lags, plus 127 + W
//                                                  after and W before), z, the sequential D and E of every lag and grid,
//                                                  the larger rho of the two grids, the first maximum, the neighbour
//                                                  test and the threshold; then, from the same samples in shared
//                                                  memory, rho on the 5 sub-sample grids around 5 k* -> g, rho, nu0
//                                                  -> compact list
//
// Every operation is a correctly rounded _rn intrinsic in the order of the specification; the FIR is
// packet_fir_kernel's inner loop, so filt is bit-identical to the value that kernel computes.
#include "sc_acq.cuh"
#include "sc_tables.cuh"

namespace sc {

constexpr int ACQ_NL = ACQ_LAGS + 2 * ACQ_W;                  // 392 lags evaluated per frame
constexpr int ACQ_NU = ACQ_NL + PRE - 1;                      // 519 grid samples u
constexpr int ACQ_Q0 = -CYC * ACQ_W - (NTAPS - 1);            // first raw sample, relative to frame n-2
constexpr int ACQ_NMIX = CYC * (ACQ_NU - 1) + NTAPS;          // 2639 mixed samples
constexpr int ACQ_R = 4;                                      // lags per thread
constexpr int ACQ_THREADS = 128;
static_assert(ACQ_NL <= ACQ_R * ACQ_THREADS, "lags per CTA");
// one float4 of padding per 8: the lanes of a warp read entries 4 apart, which then fall in distinct 16-byte slots of
// a 128-byte row (4 wavefronts per warp-wide 128-bit load, the minimum)
__host__ __device__ constexpr int acq_pad(int k) { return k + (k >> 3); }

// filt at mixed sample offset mp: the 49-tap RRC as packet_fir_kernel evaluates it
__device__ __forceinline__ float2 acq_fir(const float2 *mix, bool wide) {
    const u64 *mp = reinterpret_cast<const u64 *>(mix);
    u64 acc = 0ull;
    if (wide) {
#pragma unroll
        for (int k = 0; k < NTAPS; k++) acc = pk_add(acc, pk_mul_bcast_pz(mp[k], tap<true>(k)));
    } else {
#pragma unroll
        for (int k = 0; k < NTAPS; k++) acc = pk_add(acc, pk_mul_bcast_pz(mp[k], tap<false>(k)));
    }
    float yr, yi;
    unpk(acc, yr, yi);
    return make_float2(__fmul_rn(yr, FIR_GAIN), __fmul_rn(yi, FIR_GAIN));
}

// u[k] conj(u[k-1]) and |u|^2, as the specification writes them
__device__ __forceinline__ float2 acq_z(float2 u, float2 v) {
    return make_float2(__fadd_rn(__fmul_rn(u.x, v.x), __fmul_rn(u.y, v.y)),
                       __fsub_rn(__fmul_rn(u.y, v.x), __fmul_rn(u.x, v.y)));
}
__device__ __forceinline__ float acq_p(float2 u) { return __fadd_rn(__fmul_rn(u.x, u.x), __fmul_rn(u.y, u.y)); }

__device__ __forceinline__ float acq_rho(float dr, float di, float e, float elo) {
    const float num = __fadd_rn(__fmul_rn(dr, dr), __fmul_rn(di, di));
    const float den = __fmul_rn(e, e);
    if (den == 0.0f || !(__fmul_rn(elo, 4.0f) >= e) || !(__fmul_rn(elo, 4.0f) <= __fmul_rn(e, 3.0f))) return 0.0f;
    return __fdiv_rn(num, den);
}

__global__ void __launch_bounds__(ACQ_THREADS, 4)
acq_detect_kernel(PacketSrc src, int n_streams, int j_lo, int j_hi, int cap, int2 *__restrict__ list,
                  int4 *__restrict__ info, int *__restrict__ count) {
    __shared__ __align__(16) float2 mix[ACQ_NMIX + ACQ_PHASE];
    __shared__ float2 u[5 * PRE];                                  // the grid's u; then stage 2's five grids
    __shared__ float s_ref[3][5];                                  // stage 2: rho, D.r, D.i per grid
    __shared__ int s_kb;
    __shared__ float4 zp[acq_pad(ACQ_NU)];                          // (z, |u|^2, 0) of grid sample k at acq_pad(k)
    __shared__ float rho[ACQ_NL];
    __shared__ float wbest[ACQ_THREADS / 32];
    __shared__ int wk[ACQ_THREADS / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nj = j_hi - j_lo;
    const long total = (long) n_streams * nj;
    for (long e = blockIdx.x; e < total; e += gridDim.x) {
        const int s = (int) (e / nj), j = j_lo + (int) (e - (long) s * nj);
        if (src.call0 + (uint32_t) j < 2u) continue;                 // call n decides frame n-2
        __syncthreads();
        for (int i = tid; i < ACQ_NMIX + ACQ_PHASE; i += ACQ_THREADS) mix[i] = packet_mix(src, s, j, ACQ_Q0 + i);
#pragma unroll 1
        for (int ph = 0; ph <= ACQ_PHASE; ph += ACQ_PHASE) {          // the grids 5 k and 5 k + 2
            __syncthreads();
            for (int k = tid; k < ACQ_NU; k += ACQ_THREADS) u[k] = acq_fir(mix + ph + CYC * k, src.wide);
            __syncthreads();
            for (int k = tid; k < ACQ_NU; k += ACQ_THREADS) {
                const float2 zz = k > 0 ? acq_z(u[k], u[k - 1]) : make_float2(0.0f, 0.0f);
                zp[acq_pad(k)] = make_float4(zz.x, zz.y, acq_p(u[k]), 0.0f);
            }
            __syncthreads();
            if (tid * ACQ_R < ACQ_NL) {
                // lags l0 .. l0 + 3; w[r] holds grid sample l0 + r + i, one new entry loaded per step
                const int l0 = tid * ACQ_R;
                float dr[ACQ_R], di[ACQ_R], en[ACQ_R], elo[ACQ_R];
                float4 w[ACQ_R];
#pragma unroll
                for (int r = 0; r < ACQ_R; r++) {
                    w[r] = zp[acq_pad(l0 + r)];
                    dr[r] = 0.0f;
                    di[r] = 0.0f;
                    en[r] = __fadd_rn(0.0f, w[r].z);
                    elo[r] = 0.0f;
                }
#pragma unroll
                for (int i = 1; i < PRE; i++) {
                    const bool flip = pre_neg(i) != pre_neg(i - 1);  // b_i = -1
#pragma unroll
                    for (int r = 0; r < ACQ_R - 1; r++) w[r] = w[r + 1];
                    w[ACQ_R - 1] = zp[acq_pad(l0 + i + ACQ_R - 1)];    // <= 391 + 127
#pragma unroll
                    for (int r = 0; r < ACQ_R; r++) {
                        dr[r] = flip ? __fsub_rn(dr[r], w[r].x) : __fadd_rn(dr[r], w[r].x);
                        di[r] = flip ? __fsub_rn(di[r], w[r].y) : __fadd_rn(di[r], w[r].y);
                        en[r] = __fadd_rn(en[r], w[r].z);
                        if (i == PRE / 2 - 1) elo[r] = en[r];
                    }
                }
#pragma unroll
                for (int r = 0; r < ACQ_R; r++)
                    if (l0 + r < ACQ_NL) {
                        const float v = acq_rho(dr[r], di[r], en[r], elo[r]);
                        rho[l0 + r] = ph == 0 ? v : fmaxf(rho[l0 + r], v);
                    }
            }
        }
        __syncthreads();
        // first maximum over the frame's own lags W .. W + 375
        float best = -1.0f;
        int kb = 0;
        for (int k = tid; k < ACQ_LAGS; k += ACQ_THREADS) {
            const float v = rho[ACQ_W + k];
            if (v > best) { best = v; kb = k; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_down_sync(0xffffffffu, best, o);
            const int ok = __shfl_down_sync(0xffffffffu, kb, o);
            if (ov > best || (ov == best && ok < kb)) { best = ov; kb = ok; }
        }
        if (lane == 0) { wbest[warp] = best; wk[warp] = kb; }
        __syncthreads();
        if (tid == 0) {
            best = wbest[0];
            kb = wk[0];
            for (int w = 1; w < ACQ_THREADS / 32; w++)
                if (wbest[w] > best || (wbest[w] == best && wk[w] < kb)) { best = wbest[w]; kb = wk[w]; }
            bool ok = best >= ACQ_TAU;
            for (int d = 1; d <= ACQ_W; d++) {
                if (kb - d < 0 && !(rho[ACQ_W + kb - d] < best)) ok = false;
                if (kb + d >= ACQ_LAGS && !(rho[ACQ_W + kb + d] <= best)) ok = false;
            }
            s_kb = ok ? kb : -1;
        }
        __syncthreads();
        if (s_kb < 0) continue;                                     // uniform over the CTA
        // stage 2 on g0 = 5 k* + s, s = -2 .. 2: u of grid s + 2 at u[128 (s + 2) + i]; mixed sample index of filt
        // sample Q is Q + 40
        const int base = CYC * s_kb;
        for (int t = tid; t < 5 * PRE; t += ACQ_THREADS) {
            const int sg = t / PRE, i = t - sg * PRE;
            u[t] = acq_fir(mix + base + sg + 38 + CYC * i, src.wide);
        }
        __syncthreads();
        if (tid < 5) {                                              // thread c: the grid of order position c
            const int sv = (tid + 1) / 2 * ((tid & 1) ? -1 : 1);   // 0, -1, +1, -2, +2
            const float2 *uu = u + PRE * (sv + 2);
            float dr = 0.0f, di = 0.0f, en = __fadd_rn(0.0f, acq_p(uu[0])), elo = 0.0f;
            for (int i = 1; i < PRE; i++) {
                const float2 zz = acq_z(uu[i], uu[i - 1]);
                const bool flip = pre_neg(i) != pre_neg(i - 1);
                dr = flip ? __fsub_rn(dr, zz.x) : __fadd_rn(dr, zz.x);
                di = flip ? __fsub_rn(di, zz.y) : __fadd_rn(di, zz.y);
                en = __fadd_rn(en, acq_p(uu[i]));
                if (i == PRE / 2 - 1) elo = en;
            }
            s_ref[0][tid] = acq_rho(dr, di, en, elo);
            s_ref[1][tid] = dr;
            s_ref[2][tid] = di;
        }
        __syncthreads();
        if (tid == 0) {
            float rb = -1.0f, br = 0.0f, bi = 0.0f;
            int sb = 0;
            for (int c = 0; c < 5; c++)
                if (s_ref[0][c] > rb) {
                    rb = s_ref[0][c];
                    br = s_ref[1][c];
                    bi = s_ref[2][c];
                    sb = (c + 1) / 2 * ((c & 1) ? -1 : 1);
                }
            const float nu0 = br > 0.0f ? __fdiv_rn(bi, br) : 0.0f;
            const int pos = atomicAdd(count, 1);
            if (pos < cap) {
                list[pos] = make_int2(s, j);
                info[pos] = make_int4(base + sb, __float_as_int(rb), __float_as_int(nu0), 0);
            }
        }
    }
}

cudaError_t launch_acq_pass(const PacketSrc &src, int n_streams, int j_lo, int j_hi, int cap, int2 *list, int4 *info,
                            int *count, cudaStream_t st) {
    const long total = (long) n_streams * (j_hi - j_lo);
    const int g1 = (int) std::min<long>(total, 148L * 16);
    acq_detect_kernel<<<g1, ACQ_THREADS, 0, st>>>(src, n_streams, j_lo, j_hi, cap, list, info, count);
    return cudaGetLastError();
}

}  // namespace sc
