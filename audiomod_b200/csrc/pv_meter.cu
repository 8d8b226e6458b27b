// Loudness meters on the output rows of streaming instances and live batches: momentary (400 ms) and short-term (3 s) loudness of
// ITU-R BS.1770-4 / EBU Tech 3341 without gating, every channel weighted 1.0, and the sample peak.  Specified by the published
// standard, not by the reference's own meter objects (src/meter/loudnessmeter.cc, src/envelope/envelope.cc), which are not restated.
//
// The K-weighting filter (a high-frequency shelf, then a high-pass) is a recursion serial in time, so the parallelism is across
// rows as in pv_post.cu: one thread per row, a warp takes 32 rows and moves 32 x 32 sample tiles through shared memory so that
// every global read is a coalesced row segment.  The rows of an instance advance in lock-step, so the position inside the open
// sub-block and the ring slot of the next completed one are the same in every row: the host tracks them and passes them in, the
// kernel keeps no per-row counters and its control flow is warp-uniform.  Everything after the sample load is double precision,
// every product and sum rounded on its own (no contraction).
#include <cmath>

#include "../../include/pvgpu.h"
#include "pv_kernels.cuh"

namespace pvgpu {

// x1, x2, y1, y2 of one direct-form-I section; returns y = b0 x + b1 x1 + b2 x2 - a1 y1 - a2 y2, left to right
__device__ __forceinline__ double kw_section(double x, double b0, double b1, double b2, double a1, double a2, double *s) {
    double acc = __dmul_rn(b0, x);
    acc = __dadd_rn(acc, __dmul_rn(b1, s[0]));
    acc = __dadd_rn(acc, __dmul_rn(b2, s[1]));
    acc = __dsub_rn(acc, __dmul_rn(a1, s[2]));
    acc = __dsub_rn(acc, __dmul_rn(a2, s[3]));
    s[1] = s[0]; s[0] = x; s[3] = s[2]; s[2] = acc;
    return acc;
}

// Columns [0, n) of rows [0, rows) of x (row r at x + r * pitch; T = float, or short measured as s / 32768).  state: [kMeterState][rows]
// doubles (shelf x1 x2 y1 y2, high-pass x1 x2 y1 y2, energy of the open sub-block); ring: [kMeterRing][rows] energies of the last
// completed sub-blocks.  pos: samples already in the open sub-block, L: samples per sub-block, ri: slot of the next completed
// sub-block.  peak[r] = max |x| over the n samples.
template <typename T>
__global__ void __launch_bounds__(32) k_meter_rows(const T *__restrict__ x, int64_t pitch, int n, int rows, const KWeighting kw,
                                                   double *__restrict__ state, double *__restrict__ ring, int pos, int L, int ri,
                                                   float *__restrict__ peak) {
    constexpr bool S16 = sizeof(T) == 2;
    __shared__ float tile[32][33];
    const int lane = threadIdx.x, row_base = blockIdx.x * 32, row = row_base + lane;
    const bool have_row = row < rows;
    double s[kMeterState];
#pragma unroll
    for (int k = 0; k < kMeterState; ++k) s[k] = have_row ? state[(int64_t)k * rows + row] : 0.0;
    float pk = 0.f;
    for (int c = 0; c < n; c += 32) {
        for (int r = 0; r < 32; ++r) {
            const int rr = row_base + r;
            float v = 0.f;
            if (rr < rows && c + lane < n) v = (float)x[(int64_t)rr * pitch + c + lane];
            tile[r][lane] = v;
        }
        __syncwarp();
        const int m = min(32, n - c);
        for (int j = 0; j < m; ++j) {
            const float v = tile[lane][j];
            pk = fmaxf(pk, S16 ? fabsf(v) * (1.f / 32768.f) : fabsf(v));   // s / 32768 is exact in float
            const double xd = S16 ? __dmul_rn((double)v, 1.0 / 32768.0) : (double)v;
            double z = kw_section(xd, kw.c[0], kw.c[1], kw.c[2], kw.c[3], kw.c[4], s);
            z = kw_section(z, 1.0, -2.0, 1.0, kw.c[5], kw.c[6], s + 4);
            s[8] = __dadd_rn(s[8], __dmul_rn(z, z));
            if (++pos == L) {   // the same in every lane
                if (have_row) ring[(int64_t)ri * rows + row] = s[8];
                s[8] = 0.0;
                pos = 0;
                ri = ri + 1 == kMeterRing ? 0 : ri + 1;
            }
        }
        __syncwarp();
    }
    if (have_row) {
#pragma unroll
        for (int k = 0; k < kMeterState; ++k) state[(int64_t)k * rows + row] = s[k];
        peak[row] = pk;
    }
}

// One thread per stream: out[j] = momentary, out[streams + j] = short-term loudness of stream j from the last 4 / 30 completed
// sub-blocks (ri = slot of the next one, so the oldest of the ring), summed oldest to newest per channel, then over the channels.
__global__ void k_meter_streams(const double *__restrict__ ring, int rows, int streams, int channels, int ri, int L, float *__restrict__ out) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= streams) return;
    double em = 0.0, es = 0.0;
    for (int c = 0; c < channels; ++c) {
        const int row = j * channels + c;
        double cm = 0.0, cs = 0.0;
        for (int w = 0; w < kMeterRing; ++w) {
            const int slot = ri + w < kMeterRing ? ri + w : ri + w - kMeterRing;
            const double e = ring[(int64_t)slot * rows + row];
            cs = __dadd_rn(cs, e);
            if (w >= kMeterRing - 4) cm = __dadd_rn(cm, e);
        }
        em = __dadd_rn(em, cm);
        es = __dadd_rn(es, cs);
    }
    out[j] = (float)__dadd_rn(-0.691, __dmul_rn(10.0, log10(__ddiv_rn(em, 4.0 * L))));
    out[streams + j] = (float)__dadd_rn(-0.691, __dmul_rn(10.0, log10(__ddiv_rn(es, (double)kMeterRing * L))));
}

void launch_meters(const void *x, int fmt, int64_t pitch, int n, int streams, int channels, const KWeighting &kw, int L, double *state,
                   double *ring, float *out, int *pos, int *ri, cudaStream_t st) {
    if (n <= 0) return;
    const int rows = streams * channels, ctas = (rows + 31) / 32;
    float *peak = out + 2 * (int64_t)streams;
    if (fmt == PVGPU_S16) k_meter_rows<short><<<ctas, 32, 0, st>>>((const short *)x, pitch, n, rows, kw, state, ring, *pos, L, *ri, peak);
    else k_meter_rows<float><<<ctas, 32, 0, st>>>((const float *)x, pitch, n, rows, kw, state, ring, *pos, L, *ri, peak);
    const int64_t done = ((int64_t)*pos + n) / L;   // sub-blocks this launch completed
    *pos = (int)(((int64_t)*pos + n) % L);
    *ri = (int)((*ri + done) % kMeterRing);
    if (done > 0) k_meter_streams<<<(streams + 127) / 128, 128, 0, st>>>(ring, rows, streams, channels, *ri, L, out);
}

// libebur128's analog-prototype design of the two K-weighting sections, in double.  At 48 kHz these are BS.1770-4's tables.
void kweighting_design(int sample_rate, double *c) {
    const double pi = 3.14159265358979323846, sr = sample_rate;
    {
        const double f0 = 1681.974450955533, G = 3.999843853973347, Q = 0.7071752369554196;
        const double K = std::tan(pi * f0 / sr), Vh = std::pow(10.0, G / 20.0), Vb = std::pow(Vh, 0.4996667741545416);
        const double a0 = 1.0 + K / Q + K * K;
        c[0] = (Vh + Vb * K / Q + K * K) / a0;
        c[1] = 2.0 * (K * K - Vh) / a0;
        c[2] = (Vh - Vb * K / Q + K * K) / a0;
        c[3] = 2.0 * (K * K - 1.0) / a0;
        c[4] = (1.0 - K / Q + K * K) / a0;
    }
    {
        const double f0 = 38.13547087602444, Q = 0.5003270373238773;
        const double K = std::tan(pi * f0 / sr), a0 = 1.0 + K / Q + K * K;
        c[5] = 2.0 * (K * K - 1.0) / a0;
        c[6] = (1.0 - K / Q + K * K) / a0;
    }
}

}  // namespace pvgpu
