// Pieces of the fused resynthesis kernel (pv_fused.cu: k_synth_ola).
#pragma once
#include "pv_fft.cuh"
#include "pv_kernels.cuh"

namespace pvgpu {

template <int N> struct FusedShape {
    static constexpr int NC = N / 2;
    static constexpr int T = FftShape<NC>::kThreads;         // threads per frame
    static constexpr int kThreads = T > 256 ? T : 256;
    static constexpr int G = kThreads / T;                   // frames in flight per CTA
    static constexpr int UT = T < 32 ? 32 : T;               // threads of a token unit (whole warps)
    static constexpr int U = kThreads / UT;                  // token units
    static constexpr int FU = UT / T;                        // frames per unit (2 for N = 512: two half-warp frames)
};

__device__ __forceinline__ void named_sync(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ void named_arrive(int id, int count) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory"); }
constexpr int kTokenBarrier0 = 8;   // token barriers 8..15 (frame_sync uses 1..G, G <= 4 for the sizes with T > 32)

// ifftshift + synthesis window (impl.h:183-198, :1052-1056) + outAcc += frame (:1057-1064, product rounded first): complex
// output o of the inverse FFT holds samples 2o, 2o+1 of the un-shifted block; they land at (2o + N/2) mod N of the frame, i.e.
// at ring position off + that.  Even offsets take 64-bit read-modify-writes, odd ones two 32-bit ones.
template <int N>
__device__ __forceinline__ void fused_add_frame(const float2 (&v)[16], float *s_acc, int mask, int off, int ob, const float2 *__restrict__ w2) {
    constexpr int NC = N / 2;
    const float2 *__restrict__ wb = w2 + ob;
    const int base = off + 2 * ob;
    if ((off & 1) == 0) {
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const int oc = fft_out_const<NC>(i) ^ (NC / 2);
            const float2 w = __ldg(&wb[oc]);
            float2 *ap = (float2 *)(s_acc + ((base + 2 * oc) & mask));
            float2 s = *ap;
            s.x = __fadd_rn(s.x, __fmul_rn(v[i].x, w.x));
            s.y = __fadd_rn(s.y, __fmul_rn(v[i].y, w.y));
            *ap = s;
        }
    } else {
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const int oc = fft_out_const<NC>(i) ^ (NC / 2);
            const float2 w = __ldg(&wb[oc]);
            const int i0 = (base + 2 * oc) & mask, i1 = (base + 2 * oc + 1) & mask;
            s_acc[i0] = __fadd_rn(s_acc[i0], __fmul_rn(v[i].x, w.x));
            s_acc[i1] = __fadd_rn(s_acc[i1], __fmul_rn(v[i].y, w.y));
        }
    }
}

}  // namespace pvgpu
