// sc_tracker.cuh -- the per-stream sequential loop: Hsu square-root Kalman gain estimator driving
// a 5-tap adaptive equalizer, BPSK training step and decision-directed QPSK step.
//
// Replaces src/kalman.c:42-141 and src/equalizer.c:25-90 of the reference.  One thread owns one
// stream; all state lives in registers (every loop below has compile-time bounds and is fully
// unrolled, so the arrays never touch local memory).  Arithmetic order is the reference's, one
// IEEE rounding per operation (sc_exact.cuh).
#pragma once
#include "sc_common.cuh"

namespace sc {

struct Tracker {
    c32 C[EQ];        // eq_coeff      (src/kalman.c:19)
    c32 G[EQ];        // kalman_gain   (src/kalman.c:20)
    c32 U[10];        // upper triangle of u[5][5]: (i,j), i<j at j*(j-1)/2 + i  (src/kalman.c:25)
    float D[EQ];      // d[]           (src/kalman.c:29)
    float KY;         // kalman_y      (src/kalman.c:21)

    // kalman_reset(), src/kalman.c:42-55 (f[], h[], a[] are per-call scratch here)
    __device__ __forceinline__ void reset() {
#pragma unroll
        for (int i = 0; i < EQ; i++) {
            C[i] = mk(0.0f, 0.0f);
            G[i] = mk(0.0f, 0.0f);
            D[i] = 1.0f;
        }
#pragma unroll
        for (int i = 0; i < 10; i++) U[i] = mk(0.0f, 0.0f);
        KY = 0.0f;
    }

    // kalman_calculate(x, index), src/kalman.c:85-141, with x[] = in[index .. index+4]
    __device__ __forceinline__ void kalman(const c32 (&x)[EQ]) {
        const float E = 0.1f, q = 0.08f;                 // kalman_init(), src/kalman.c:61-62
        c32 F[EQ];
        float A[EQ];

        const c32 x0c = cconj(x[0]);
        F[0] = x0c;                                       // 6.2
#pragma unroll
        for (int j = 1; j < EQ; j++) {
            c32 f = cadd(cmul(U[j * (j - 1) / 2], x0c), cconj(x[j]));
#pragma unroll
            for (int i = 1; i < j; i++) f = cadd(f, cmul(U[j * (j - 1) / 2 + i], cconj(x[i])));
            F[j] = f;
        }
#pragma unroll
        for (int j = 0; j < EQ; j++) G[j] = cscale(F[j], D[j]);       // 6.4

        // crealf(g * conjf(f)) = g.r*f.r - g.i*(-f.i)                  6.5, 6.6
        A[0] = __fadd_rn(E, __fsub_rn(__fmul_rn(G[0].r, F[0].r), __fmul_rn(G[0].i, -F[0].i)));
#pragma unroll
        for (int j = 1; j < EQ; j++)
            A[j] = __fadd_rn(A[j - 1], __fsub_rn(__fmul_rn(G[j].r, F[j].r), __fmul_rn(G[j].i, -F[j].i)));

        const float hq = __fadd_rn(1.0f, q);                          // 6.7
        const float ht = __fmul_rn(A[EQ - 1], q);

        // kalman_y takes the values 1/(a[j] + ht), j = 0..4 (6.19, 6.22).  All five denominators
        // are known here, so the reciprocals are taken together (off the serial chain) behind one
        // range test instead of five: a[] is non-decreasing (d[] > 0), so den[0] and den[4] bound them.
        float den[EQ], rc[EQ];
#pragma unroll
        for (int j = 0; j < EQ; j++) den[j] = __fadd_rn(A[j], ht);
        if (den[0] >= 0x1p-120f && den[EQ - 1] <= 0x1p120f) {
#pragma unroll
            for (int j = 0; j < EQ; j++) rc[j] = rcp_rn_normal(den[j]);
        } else {                                                      // never seen in practice; NaNs land here
#pragma unroll
            for (int j = 0; j < EQ; j++) rc[j] = __frcp_rn(den[j]);
        }

        KY = rc[0];                                                   // 6.19
        D[0] = __fmul_rn(D[0], __fmul_rn(__fmul_rn(hq, __fadd_rn(E, ht)), KY));   // 6.20

#pragma unroll
        for (int j = 1; j < EQ; j++) {                                // 6.10 - 6.16
            const float B = den[j - 1];                               // 6.21: a[j-1] + ht
            const c32 H = mk(__fmul_rn(-F[j].r, KY), __fmul_rn(-F[j].i, KY));      // 6.11
            KY = rc[j];                                               // 6.22
            D[j] = __fmul_rn(D[j], __fmul_rn(__fmul_rn(hq, B), KY));  // 6.13
#pragma unroll
            for (int i = 0; i < j; i++) {
                const c32 B1 = U[j * (j - 1) / 2 + i];
                U[j * (j - 1) / 2 + i] = cadd(B1, cmulc(H, G[i]));    // 6.15
                G[i] = cadd(G[i], cmulc(G[j], B1));                   // 6.16
            }
        }
    }

    // update_eq(), src/equalizer.c:25-40
    __device__ __forceinline__ void update(const c32 (&x)[EQ], c32 err) {
        kalman(x);
        err = cscale(err, KY);
#pragma unroll
        for (int i = 0; i < EQ; i++) C[i] = cadd(C[i], cmulc(err, G[i]));
    }

    // train_eq(in, index, ref), src/equalizer.c:45-58; returns crealf(error)
    __device__ __forceinline__ float train(const c32 (&x)[EQ], float ref) {
        c32 v = mk(0.0f, 0.0f);
#pragma unroll
        for (int i = 0; i < EQ; i++) v = cadd(v, cmul(x[i], C[i]));
        const c32 err = mk(__fsub_rn(ref, v.r), v.i);     // conjf(ref - val)
        update(x, err);
        return err.r;
    }

    // data_eq(&dibit, in, index) without the descrambler, src/equalizer.c:64-85 and
    // qpsk_demod(), src/qpsk.c:268-271.  Returns crealf(error); bI/bQ are the raw decisions, s the equalizer output
    // they are sliced from (`sym` of data_eq()).
    __device__ __forceinline__ float data(const c32 (&x)[EQ], int &bI, int &bQ, c32 &s) {
        s = mk(0.0f, 0.0f);
#pragma unroll
        for (int i = 0; i < EQ; i++) s = cadd(s, cmulc(x[i], C[i]));
        bI = s.r < 0.0f;
        bQ = s.i < 0.0f;
        const float ci = bI ? -1.0f : 1.0f;
        const float cq = bQ ? -1.0f : 1.0f;
        const c32 err = mk(__fmul_rn(__fsub_rn(ci, s.r), 0.1f), __fmul_rn(__fsub_rn(cq, s.i), 0.1f));
        update(x, err);
        return err.r;
    }
    __device__ __forceinline__ float data(const c32 (&x)[EQ], int &bI, int &bQ) {
        c32 s;
        return data(x, bI, bQ, s);
    }
};

}  // namespace sc
