// sc_acq.cuh -- packet-mode acquisition (SC_FLAG_PACKET_ACQ): constants shared by sc_acq_kernels.cu and the ACQ forms
// of the packet kernels, and the mixed-sample fetch of every packet FIR.  Specification: tests/packet_acq_ref.c
// (DESIGN.md 8b).
#pragma once
#include "sc_common.cuh"
#include "sc_kernels.h"

namespace sc {

constexpr float ACQ_TAU = 0.2f;                    // acceptance threshold on rho
constexpr int ACQ_PHASE = 2;                       // stage 1's second grid: 5 k + 2
constexpr int ACQ_W = 8;                           // neighbour lags compared across a frame boundary
constexpr int ACQ_LAGS = FRAME / CYC;              // 376 phase-0 lags per frame
constexpr float ACQ_HZ_PER_RAD = 254.64790894703253f;   // 1600 / (2 pi)

// The mixed sample (phasor / 16384) * in at raw sample q, counted from the first sample of block frame j - 2
// (-1880 <= q < 3 * 1880: frames j-3 .. j; those before the block from the history).  Frames before the stream's
// first one are zero.
__device__ __forceinline__ float2 packet_mix(const PacketSrc &src, int s, int j, int q) {
    const int fi = q >= 2 * FRAME ? 2 : q >= FRAME ? 1 : q >= 0 ? 0 : -1;
    const int fj = j - 2 + fi;
    if ((long) src.call0 + fj < 0) return make_float2(0.0f, 0.0f);
    const int qq = q - fi * FRAME;
    const int16_t *fr = fj >= 0 ? src.in + (long) s * src.stride + (long) fj * FRAME
                                : src.hist + (long) (fj + 1) * src.hist_pitch + (long) s * FRAME;
    const float2 *tb = src.mix0 + (long) (fj + 1) * FRAME;
    const float v = (float) fr[qq];
    const float2 ph = __ldg(tb + qq);
    return make_float2(__fmul_rn(ph.x, v), __fmul_rn(ph.y, v));
}

}  // namespace sc
