// sc_tracker_coop.cuh -- the per-stream sequential loop of sc_tracker.cuh spread over 5 + 5 lanes of two warps.
//
// One thread per stream (sc_tracker.cuh) is the right shape when there are enough streams to fill the GPU: the loop
// is a 63,000-operation dependent chain per call, and a lone warp per scheduler runs a step of ~400 instructions in
// ~940 clocks.  Small banks (fewer streams than the GPU has lanes) are bound by exactly that latency, so here one
// stream's step is cut along its data flow instead.
//
// The Kalman gain recursion (src/kalman.c:85-141) depends only on the received symbols, not on the equalizer's
// output; the taps (src/equalizer.c:25-85) consume its gain vector and kalman_y one step later.  So:
//
//   warp A, KalmanColumn -- lane j (of a group of 8) owns column j of the unit upper triangle U(0..j-1, j) and d[j]
//     (kalman.c:25,29).  F[j], G[j], the a[] term of the column, the column's part of 6.16 and the update 6.15 of
//     its own elements need nothing from other lanes but, once per step, the five a[] terms, the five G[] and the
//     products of 6.16 -- one exchange through shared memory per step (shuffles are slower: a lone warp issues one
//     SHFL every 4.4 clocks, tools/microbench_lat2.cu).
//   warp B, TapLanes -- lane i owns eq_coeff[i]: the final kalman_gain[i], equalizer output, decision, error, tap
//     update, match count, bits, cost.
//   One CTA barrier per step joins them (A is one step ahead; what it hands over is double-buffered).
//
// Every value is produced by the same operations in the same order as in the one-thread version (and therefore as in
// the reference); what changes is only which lane executes an operation, so the results are bit-identical by
// construction.  Sums that are shorter in some lanes than in others use predicated adds, or read -0 for the missing
// terms (x + (-0) == x for every x, including -0, in round-to-nearest).  tests/test_round2_gpu.py compares the two
// kernels on whole banks.
//
//   6.2   F[j] = conj(x[j]) + sum_{i<j} U(i,j) conj(x[i])        lane j
//   6.4   G[j] = F[j] d[j]                                        lane j
//   6.5-6 a[j] = a[j-1] + Re(G[j] conj(F[j]))                     terms exchanged; every lane runs the prefix
//   6.7.. ht, the denominators and their reciprocals              every lane, for its own column and the one before
//   6.13  d[j] *= hq (a[j-1] + ht) / (a[j] + ht)                  lane j
//   6.16  G[i] += G[j] conj(U(i,j))                               product P(i,j) on lane j, exchanged
//   6.15  U(i,j) += H[j] conj(G[i] as it stands before column j)  lane j: G[i] + P(i,i+1) + .. + P(i,j-1), in order
//   update_eq: eq_coeff[i] += (err kalman_y) conj(G[i])           warp B: G[i] + P(i,i+1) + .. + P(i,4), in order
//   train_eq / data_eq: sum_i x[i] eq_coeff[i]                    warp B: products exchanged, summed by every lane
#pragma once
#include "sc_common.cuh"

namespace sc {

constexpr int TC_LANES = 8;              // lanes per stream in each of the two warps (5 used)

// What warp A's five column lanes exchange, and what warp B reads one step later.  Slots that are never written
// keep the -0 they are initialised with: they are the missing terms of the shorter row sums.
struct __align__(16) ExchangeA {
    float2 g[6];         // G[j] = F[j] d[j]
    float2 p[5][4];      // p[i][r] = P(i, i+1+r) = G[i+1+r] conj(U(i, i+1+r)); r > 3 - i: -0
    float t[6];          // Re(G[j] conj(F[j]))
    float den;           // a[4] + ht, whose reciprocal is kalman_y
    float dump;

    __device__ __forceinline__ void init(int g8) {             // called by the 8 lanes of the group
        float *w = reinterpret_cast<float *>(this);
        for (int k = g8; k < (int) (sizeof(ExchangeA) / sizeof(float)); k += TC_LANES) w[k] = -0.0f;
    }
};

struct __align__(16) ExchangeB {
    float2 v[6];         // x[i] eq_coeff[i], i < 5
};

__device__ __forceinline__ void lds128(const void *p, float2 &a, float2 &b) {
    const float4 v = *reinterpret_cast<const float4 *>(p);
    a = make_float2(v.x, v.y);
    b = make_float2(v.z, v.w);
}

struct KalmanColumn {
    int myj;             // column; lanes 5..7 of a group shadow column 4 and store nothing
    bool has[4];         // has[i]: element U(i, myj) exists (i < myj)
    bool live, first;    // lanes 0..4 store their column's terms; lane 0 also stores a[4] + ht
    c32 U[4];            // U(i, myj)
    float D;             // d[myj]

    __device__ __forceinline__ void init(int lane) {
        const int g = lane & (TC_LANES - 1);
        live = g < EQ;
        first = g == 0;
        myj = min(g, EQ - 1);
#pragma unroll
        for (int i = 0; i < 4; i++) has[i] = i < myj;
    }

    __device__ __forceinline__ void reset() {                  // kalman_reset(), src/kalman.c:42-55
#pragma unroll
        for (int i = 0; i < 4; i++) U[i] = mk(0.0f, 0.0f);
        D = 1.0f;
    }

    // kalman_calculate(), src/kalman.c:85-141, on the window x[0..4]; xj = x[myj].  Leaves G[], the products of
    // 6.16 and a[4] + ht in ex for warp B.
    __device__ __forceinline__ void step(const c32 (&x)[4], c32 xj, ExchangeA *ex) {
        const float E = 0.1f, q = 0.08f;                       // kalman_init(), src/kalman.c:61-62

        c32 F = cconj(xj);                                     // 6.2
        if (has[0]) F = cadd(cmul(U[0], cconj(x[0])), F);
#pragma unroll
        for (int i = 1; i < 4; i++)
            if (has[i]) F = cadd(F, cmul(U[i], cconj(x[i])));
        const c32 G = cscale(F, D);                            // 6.4
        const float t = __fsub_rn(__fmul_rn(G.r, F.r), __fmul_rn(G.i, -F.i));  // 6.5, 6.6
        if (live) {
            ex->t[myj] = t;
            ex->g[myj] = to2(G);
#pragma unroll
            for (int i = 0; i < 4; i++)
                if (has[i]) ex->p[i][myj - i - 1] = to2(cmulc(G, U[i]));       // 6.16, this column's terms
        }
        __syncwarp();

        const float4 t03 = *reinterpret_cast<const float4 *>(ex->t);
        const float t4 = ex->t[4];
        float2 g0, g1, g2, g3, p00, p01, p10, p11;
        lds128(&ex->g[0], g0, g1);
        lds128(&ex->g[2], g2, g3);
        lds128(&ex->p[0][0], p00, p01);
        lds128(&ex->p[1][0], p10, p11);
        const float2 p02 = ex->p[0][2], p20 = ex->p[2][0];

        float A[EQ];
        A[0] = __fadd_rn(E, t03.x);
        A[1] = __fadd_rn(A[0], t03.y);
        A[2] = __fadd_rn(A[1], t03.z);
        A[3] = __fadd_rn(A[2], t03.w);
        A[4] = __fadd_rn(A[3], t4);
        float a_prev = E, a_mine = A[0];                       // column 0: 6.20 uses E + ht
#pragma unroll
        for (int j = 1; j < EQ; j++)
            if (has[j - 1]) {
                a_prev = A[j - 1];
                a_mine = A[j];
            }
        const float hq = __fadd_rn(1.0f, q);                   // 6.7
        const float ht = __fmul_rn(A[EQ - 1], q);
        const float den_m = __fadd_rn(a_mine, ht);             // a[myj] + ht
        const float den_p = __fadd_rn(a_prev, ht);             // a[myj-1] + ht (6.21), or E + ht for column 0 (6.20)
        if (first) ex->den = __fadd_rn(A[EQ - 1], ht);
        float rc_m, rc_p;                                      // kalman_y after columns myj and myj - 1
        if (fminf(den_m, den_p) >= 0x1p-120f && fmaxf(den_m, den_p) <= 0x1p120f) {
            rc_m = rcp_rn_normal(den_m);
            rc_p = rcp_rn_normal(den_p);
        } else {                                               // never seen in practice; NaNs land here
            rc_m = __frcp_rn(den_m);
            rc_p = __frcp_rn(den_p);
        }
        D = __fmul_rn(D, __fmul_rn(__fmul_rn(hq, den_p), rc_m));               // 6.20 / 6.13
        const c32 H = mk(__fmul_rn(-F.r, rc_p), __fmul_rn(-F.i, rc_p));        // 6.11 (unused in column 0)

        // kalman_gain[i] as it stands when column myj is reached: G[i] + P(i,i+1) + .. + P(i,myj-1)
        c32 acc0 = from2(g0), acc1 = from2(g1), acc2 = from2(g2);
        const c32 acc3 = from2(g3);
        if (has[1]) acc0 = cadd(acc0, from2(p00));             // myj > 1
        if (has[2]) {                                          // myj > 2
            acc0 = cadd(acc0, from2(p01));
            acc1 = cadd(acc1, from2(p10));
        }
        if (has[3]) {                                          // myj > 3
            acc0 = cadd(acc0, from2(p02));
            acc1 = cadd(acc1, from2(p11));
            acc2 = cadd(acc2, from2(p20));
        }
        U[0] = cadd(U[0], cmulc(H, acc0));                     // 6.15 (elements that do not exist are never read)
        U[1] = cadd(U[1], cmulc(H, acc1));
        U[2] = cadd(U[2], cmulc(H, acc2));
        U[3] = cadd(U[3], cmulc(H, acc3));
    }
};

struct TapLanes {
    ExchangeB *ex;
    int i;               // tap; lanes 5..7 of a group shadow tap 4 and store into the spare slot
    int slot;
    c32 C;               // eq_coeff[i]

    __device__ __forceinline__ void init(int lane, ExchangeB *e) {
        ex = e;
        const int g = lane & (TC_LANES - 1);
        i = min(g, EQ - 1);
        slot = min(g, EQ);
    }
    __device__ __forceinline__ void reset() { C = mk(0.0f, 0.0f); }

    // head of train_eq() (DATA = false, src/equalizer.c:45-52) or data_eq() (DATA = true, :64-80): the equalizer's
    // output from the taps as they stand (v, every lane of the group), decision, error.  xi = x[i].
    template <bool DATA>
    __device__ __forceinline__ c32 error(c32 xi, float ref, int &bI, int &bQ, c32 &v) const {
        ex->v[slot] = to2(DATA ? cmulc(xi, C) : cmul(xi, C));
        __syncwarp();
        float2 p0, p1, p2, p3;
        lds128(&ex->v[0], p0, p1);
        lds128(&ex->v[2], p2, p3);
        const float2 p4 = ex->v[4];
        __syncwarp();
        v = mk(0.0f, 0.0f);
        v = cadd(v, from2(p0));
        v = cadd(v, from2(p1));
        v = cadd(v, from2(p2));
        v = cadd(v, from2(p3));
        v = cadd(v, from2(p4));
        if (DATA) {
            bI = v.r < 0.0f;
            bQ = v.i < 0.0f;
            const float ci = bI ? -1.0f : 1.0f;
            const float cq = bQ ? -1.0f : 1.0f;
            return mk(__fmul_rn(__fsub_rn(ci, v.r), 0.1f), __fmul_rn(__fsub_rn(cq, v.i), 0.1f));
        }
        return mk(__fsub_rn(ref, v.r), v.i);                   // conjf(ref - val)
    }

    // update_eq(), src/equalizer.c:25-40, with what warp A left for this step: kalman_gain[i] = G[i] + the products
    // of row i in order (6.16), kalman_y = 1 / (a[4] + ht)
    __device__ __forceinline__ void update(c32 err, const ExchangeA *xa) {
        float2 r0, r1, r2, r3;
        const float2 g = xa->g[i];
        lds128(&xa->p[i][0], r0, r1);
        lds128(&xa->p[i][2], r2, r3);
        const float den = xa->den;
        c32 gain = from2(g);
        gain = cadd(gain, from2(r0));
        gain = cadd(gain, from2(r1));
        gain = cadd(gain, from2(r2));
        gain = cadd(gain, from2(r3));
        const float ky = (den >= 0x1p-120f && den <= 0x1p120f) ? rcp_rn_normal(den) : __frcp_rn(den);
        const c32 e2 = cscale(err, ky);
        C = cadd(C, cmulc(e2, gain));
    }
};

}  // namespace sc
