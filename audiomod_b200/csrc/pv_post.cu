// FFT-free effects as a post-chain on the batch's output rows (SURVEY 8(f) rank 4): gain (src/gain/gain.cc:27-36),
// compressor (src/dynamics/compressor.cc:54-77), limiter (src/dynamics/limiter.cc:45-64) and biquad sections
// (src/common/filters/biquadfilter.cc:53-60; eight of them in a fixed order are the equalizer, src/equalizer/equalizer.cc:613-647)
// -- the per-sample recursions of
// the reference's processBlock, run over the whole output stream of a row (they carry their state from block to block, so
// the block size is invisible).  The recursions are serial in time (the attack / release coefficient of a sample depends
// on the previous state), so the parallelism is across rows: one thread per row, a warp takes 32 rows and moves 32 x 32
// sample tiles through shared memory so that every global access is a coalesced 128-byte row segment.
// Arithmetic follows the reference's types expression by expression (float members, the double literals where it has them,
// no FMA contraction); log10f / pow are CUDA's, within an ulp or two of glibc's (tolerance path, like the resampler).
#include "../../include/pvgpu.h"
#include "pv_kernels.cuh"
#include "pv_synth.cuh"

namespace pvgpu {

// compressor: a = dbyL_prev; limiter: a = xPeak, b = gain, pos = delay-line position; biquad: a, b, c, d = x1, x2, y1, y2
struct FxRegs { float a, b, c, d; int pos; };

// biquadfilter::process (src/common/filters/biquadfilter.cc:53-60): direct form I, every product and sum rounded to float
__device__ __forceinline__ float fx_biquad(float x, const PostFx &f, FxRegs &s) {
    float acc = __fmul_rn(f.p[0], x);
    acc = __fadd_rn(acc, __fmul_rn(f.p[1], s.a));
    acc = __fadd_rn(acc, __fmul_rn(f.p[2], s.b));
    acc = __fsub_rn(acc, __fmul_rn(f.p[4], s.c));
    acc = __fsub_rn(acc, __fmul_rn(f.p[5], s.d));
    const float y = __fdiv_rn(acc, f.p[3]);
    s.b = s.a; s.d = s.c; s.a = x; s.c = y;
    return y;
}

__device__ __forceinline__ float fx_compressor(float x, const PostFx &f, FxRegs &s) {
    const float ax = fabsf(x);
    const float dbx_g = ((double)ax < 0.000001) ? -120.f : __fmul_rn(20.f, log10f(ax));
    const float thr = f.p[0];
    const float dby_g = dbx_g >= thr ? __fadd_rn(thr, __fdiv_rn(__fsub_rn(dbx_g, thr), f.p[1])) : dbx_g;
    const float dbx_l = __fsub_rn(dbx_g, dby_g);
    const float alpha = dbx_l > s.a ? f.p[3] : f.p[4];
    const float dby_l = __fadd_rn(__fmul_rn(alpha, s.a), __fmul_rn(__fsub_rn(1.f, alpha), dbx_l));
    const float c = (float)pow(10.0, (double)__fdiv_rn(__fsub_rn(f.p[2], dby_l), 20.f));
    s.a = dby_l;
    return __fmul_rn(x, c);
}

__device__ __forceinline__ float fx_limiter(float x, const PostFx &f, FxRegs &s, float *ring) {
    x = __fmul_rn(x, f.p[0]);
    float x_abs = fabsf(x);
    if ((double)x_abs < 0.000001) x_abs = (float)0.000001;
    float alpha = x_abs > s.a ? f.p[2] : f.p[3];
    s.a = (float)__dadd_rn((double)__fmul_rn(alpha, s.a), __dmul_rn(__dsub_rn(1.0, (double)alpha), (double)x_abs));
    const float gain = fminf(1.f, __fdiv_rn(f.p[1], s.a));
    alpha = gain < s.b ? f.p[2] : f.p[3];
    s.b = (float)__dadd_rn((double)__fmul_rn(alpha, s.b), __dmul_rn(__dsub_rn(1.0, (double)alpha), (double)gain));
    float y = __fmul_rn(ring[s.pos], s.b);       // buffers_.front() * gains_; pop_front(); push_back(x)
    ring[s.pos] = x;
    s.pos = s.pos + 1 == f.delay ? 0 : s.pos + 1;
    if (y > 1.f) y = 1.f;
    if (y < -1.f) y = -1.f;
    return y;
}

constexpr int kPostWarps = 4;   // the batch's shape: 4 warps of 32 rows per CTA

// Columns [col0, col1) of every row's float32 output in g.out; state: [rows][state_stride] floats (4 x 4 scalars, then the delay
// lines).  The chained samples go to dst, indexed like g.out ([rows][out_stride], element 0 is output position out_base): float32
// (DST_S16 false; dst == g.out, in place) or int16 quantised by pcm_store's rule (DST_S16 true: a streaming instance of int16 rows,
// whose resynthesis stored float32 into g.out).  WARPS warps of 32 rows each per CTA.  The one-warp shape may take all 255
// registers (without the bound ptxas stopped at 128 and spilled); the batch's shape keeps the plain bound (168 registers).
// PER_ROW: every stream has its own coefficients, coef = [streams][pc.n][6] floats (the p[] of pc.fx, row r is stream
// r / g.channels); the kinds, delays and n stay pc's, so control flow is warp-uniform.  Each warp stages its rows' coefficients
// in shared memory as [fx][param][lane] (one conflict-free access per lane and read); the uniform instantiations ignore coef.
template <int WARPS, bool DST_S16, bool PER_ROW>
__global__ void __launch_bounds__(32 * WARPS, WARPS == 1 ? 8 : 0) k_postchain(const DevRows g, const PostChain pc, float *__restrict__ state, int state_stride,
                                                          int64_t col0, int64_t col1, void *dst, const float *__restrict__ coef) {
    __shared__ float tile[WARPS][32][33];
    __shared__ float row_p[PER_ROW ? WARPS : 1][PER_ROW ? kMaxPostFx * 6 : 1][32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row_base = (blockIdx.x * WARPS + warp) * 32;
    if (row_base >= g.rows) return;
    const int row = row_base + lane;
    const bool have_row = row < g.rows;
    if (PER_ROW && have_row) {   // a lane without a row stages nothing and runs no sample
        const float *c = coef + (int64_t)(row / g.channels) * pc.n * 6;
        for (int i = 0; i < pc.n * 6; ++i) row_p[PER_ROW ? warp : 0][i][lane] = c[i];
    }
    const float *out = (const float *)g.out;
    float *st = state + (int64_t)(have_row ? row : row_base) * state_stride;
    FxRegs regs[kMaxPostFx];
    float *rings[kMaxPostFx];
    {
        int ring_off = 4 * kMaxPostFx;
#pragma unroll
        for (int k = 0; k < kMaxPostFx; ++k) {
            regs[k].a = st[4 * k]; regs[k].b = st[4 * k + 1]; regs[k].pos = __float_as_int(st[4 * k + 2]);
            regs[k].c = regs[k].d = 0.f;
            if (k < pc.n && pc.fx[k].kind == kFxBiquad) { regs[k].c = st[4 * k + 2]; regs[k].d = st[4 * k + 3]; regs[k].pos = 0; }
            rings[k] = st + ring_off;
            if (k < pc.n && pc.fx[k].kind == kFxLimiter) ring_off += pc.fx[k].delay;
        }
    }
    const int64_t my_end = have_row ? min(col1, g.n_out[row]) : 0;
    for (int64_t c = col0; c < col1; c += 32) {
        for (int r = 0; r < 32; ++r) {
            const int rr = row_base + r;
            const int64_t idx = c + lane;
            float v = 0.f;
            if (rr < g.rows && idx < col1 && idx < g.n_out[rr]) v = out[(int64_t)rr * g.out_stride - g.out_base + idx];
            tile[warp][r][lane] = v;
        }
        __syncwarp();
        const int n = (int)max((int64_t)0, min((int64_t)32, my_end - c));
        for (int j = 0; j < n; ++j) {
            float x = tile[warp][lane][j];
#pragma unroll
            for (int k = 0; k < kMaxPostFx; ++k) {
                if (k >= pc.n) break;
                PostFx rf;   // PER_ROW: this row's coefficients of effect k
                if (PER_ROW) {
                    rf.kind = pc.fx[k].kind; rf.delay = pc.fx[k].delay;
#pragma unroll
                    for (int i = 0; i < 6; ++i) rf.p[i] = row_p[PER_ROW ? warp : 0][6 * k + i][lane];
                }
                const PostFx &f = PER_ROW ? rf : pc.fx[k];
                if (f.kind == kFxGain) {
                    x = __fmul_rn(x, f.p[0]);
                    if (x > 1.f) x = 1.f;
                    if (x < -1.f) x = -1.f;
                } else if (f.kind == kFxCompressor) {
                    x = fx_compressor(x, f, regs[k]);
                } else if (f.kind == kFxBiquad) {
                    x = fx_biquad(x, f, regs[k]);
                } else {
                    x = fx_limiter(x, f, regs[k], rings[k]);
                }
            }
            tile[warp][lane][j] = x;
        }
        __syncwarp();
        for (int r = 0; r < 32; ++r) {
            const int rr = row_base + r;
            const int64_t idx = c + lane;
            if (rr < g.rows && idx < col1 && idx < g.n_out[rr]) {
                const int64_t o = (int64_t)rr * g.out_stride - g.out_base + idx;
                if (DST_S16) pcm_store(dst, PVGPU_S16, o, tile[warp][r][lane]);
                else ((float *)dst)[o] = tile[warp][r][lane];
            }
        }
        __syncwarp();
    }
    if (have_row) {
#pragma unroll
        for (int k = 0; k < kMaxPostFx; ++k) {
            const bool bq = k < pc.n && pc.fx[k].kind == kFxBiquad;
            st[4 * k] = regs[k].a; st[4 * k + 1] = regs[k].b; st[4 * k + 2] = bq ? regs[k].c : __int_as_float(regs[k].pos); st[4 * k + 3] = regs[k].d;
        }
    }
}

// initial state of every row (compressor.cc:36-40: all zero; limiter.cc:34-38: xPeak = 10^(-120/20), gain 1, empty delay line)
__global__ void k_postchain_reset(const PostChain pc, float *__restrict__ state, int state_stride, int rows) {
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= rows) return;
    float *st = state + (int64_t)row * state_stride;
    for (int i = 0; i < state_stride; ++i) st[i] = 0.f;
    for (int k = 0; k < pc.n; ++k)
        if (pc.fx[k].kind == kFxLimiter) { st[4 * k] = pc.fx[k].p[4]; st[4 * k + 1] = 1.f; }
}

int postchain_state_stride(const PostChain &pc) {
    int n = 4 * kMaxPostFx;
    for (int k = 0; k < pc.n; ++k) if (pc.fx[k].kind == kFxLimiter) n += pc.fx[k].delay;
    return n;
}

void launch_postchain_reset(const PostChain &pc, float *state, int rows, cudaStream_t st) {
    k_postchain_reset<<<(rows + 127) / 128, 128, 0, st>>>(pc, state, postchain_state_stride(pc), rows);
}

void launch_postchain(const DevRows &g, const PostChain &pc, float *state, int64_t col0, int64_t col1, cudaStream_t st) {
    if (pc.n == 0 || col1 <= col0) return;
    const int rows_per_cta = 32 * kPostWarps;
    k_postchain<kPostWarps, false, false><<<(g.rows + rows_per_cta - 1) / rows_per_cta, 32 * kPostWarps, 0, st>>>(g, pc, state, postchain_state_stride(pc), col0, col1, g.out, nullptr);
}

// Streaming instances: a call's few hundred columns per row are walked serially by one thread per row, so the rows are spread
// over as many SMs as possible -- one warp (32 rows) per CTA, 128 CTAs for 4096 rows instead of the batch's 32.  Measured faster
// at both sizes (compressor + limiter: 0.91 against 1.08 ms per call at 1024 rows, 1.68 against 2.08 ms at 4096; B200,
// profiles/r04_live_postchain_latency.jsonl), so there is one shape.  coef non-null: per-stream coefficients (k_postchain<1, *,
// true>, one warp per CTA: four warps of staged coefficients would not fit 48 KB).  The engine passes its table when some
// stream's parameters differ from the chain's, or always with PVGPU_POST_PER_ROW=1 (pv_engine.cu; for measuring the two
// kernels on identical parameters).
void launch_postchain_stream(const DevRows &g, const PostChain &pc, float *state, int64_t col0, int64_t col1, void *dst, int dst_fmt, const float *coef,
                             cudaStream_t st) {
    if (pc.n == 0 || col1 <= col0) return;
    const int stride = postchain_state_stride(pc), ctas = (g.rows + 31) / 32;
    if (coef) {
        if (dst_fmt == PVGPU_S16) k_postchain<1, true, true><<<ctas, 32, 0, st>>>(g, pc, state, stride, col0, col1, dst, coef);
        else k_postchain<1, false, true><<<ctas, 32, 0, st>>>(g, pc, state, stride, col0, col1, dst, coef);
    } else {
        if (dst_fmt == PVGPU_S16) k_postchain<1, true, false><<<ctas, 32, 0, st>>>(g, pc, state, stride, col0, col1, dst, nullptr);
        else k_postchain<1, false, false><<<ctas, 32, 0, st>>>(g, pc, state, stride, col0, col1, dst, nullptr);
    }
}

// Pending per-stream coefficient updates into the [streams][n6] table: upd holds k records of 1 + n6 floats, the stream index
// (int bits) and then its coefficients.  One thread per coefficient.
__global__ void k_postchain_coef_scatter(const float *__restrict__ upd, int k, int n6, float *__restrict__ table) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= k * n6) return;
    const float *r = upd + (int64_t)(i / n6) * (1 + n6);
    table[(int64_t)__float_as_int(r[0]) * n6 + i % n6] = r[1 + i % n6];
}

void launch_postchain_coef_scatter(const float *upd, int k, int n6, float *table, cudaStream_t st) {
    if (k <= 0 || n6 <= 0) return;
    k_postchain_coef_scatter<<<(k * n6 + 255) / 256, 256, 0, st>>>(upd, k, n6, table);
}

}  // namespace pvgpu
