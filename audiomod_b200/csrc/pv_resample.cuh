// Speex quality-4 windowed-sinc resampler from a shared-memory input window (speex/resample.c:352-403 direct table,
// :462-560 cubic-interpolated table) -- the second half of k_ola_resample and of the fused k_synth_ola.
//
// The host has bucketed the outputs of a run of slices by their table phase (`offset` in resample.c:470), padded every bucket
// to whole rows of 32 entries and cut it into steps of up to kResPerThread rows (ResampleRun + step list, pv_kernels.cuh).
// A warp step therefore works on one phase: the sinc "quad" (tab[e-2], tab[e-1], tab[e], tab[e+1]) of every tap is a single
// broadcast shared-memory access that feeds 4 FMAs (two packed FFMA2) per row, and the host orders the entries so that the 32 input windows of a
// row start on different banks.  (Buckets used to be padded to whole 128-entry steps: 13 % dead lanes at 16 slices per run,
// 50 % at the 8 slices per run the fused kernel prefers; now only the last row of a bucket has dead lanes.)
#pragma once
#include "pv_kernels.cuh"
#include "pv_synth.cuh"

namespace pvgpu {

// Two fp32 FMAs in one instruction (sm_100 FFMA2): acc.{x,y} = x * t.{x,y} + acc.{x,y}, each half rounded exactly like a scalar
// fma.rn.  ptxas folds the (x, x) pair into the instruction's scalar-broadcast operand form (FFMA2 Rd, Rx.F32, Rt.F32x2, Rd.F32x2),
// so a tap costs two issue slots per output instead of four.
__device__ __forceinline__ void ffma2_bcast(float2 &acc, float x, float tx, float ty) {
    unsigned long long a, b, c;
    asm("mov.b64 %0, {%1, %1};" : "=l"(a) : "f"(x));
    asm("mov.b64 %0, {%1, %2};" : "=l"(b) : "f"(tx), "f"(ty));
    asm("mov.b64 %0, {%1, %2};" : "=l"(c) : "f"(acc.x), "f"(acc.y));
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(c) : "l"(a), "l"(b));
    asm("mov.b64 {%0, %1}, %2;" : "=f"(acc.x), "=f"(acc.y) : "l"(c));
}

// One warp step: ROWS rows of 32 outputs of ONE table phase.  The quad of a tap is loaded once (a broadcast) and feeds
// 4 x ROWS FMAs; two taps per stage, two stages in flight: the loads of the next stage are issued before the FMAs of the
// current one (filt_len is a multiple of 4, resample.c:712).
template <int OV, int ROWS>
__device__ __forceinline__ void resample_step(const DevPlan &p, const DevRows &g, const float4 *s_quad, const float *s_x, int x_shift, int64_t orow, int64_t out_limit,
                                              const unsigned *__restrict__ ent_tab, const float *__restrict__ frac_tab, int first, int bucket, int L) {
    const int lane = threadIdx.x & 31;
    unsigned ent[ROWS];
    const float *xs[ROWS];
    bool live[ROWS];
#pragma unroll
    for (int u = 0; u < ROWS; ++u) {
        ent[u] = __ldg(&ent_tab[first + lane + 32 * u]);
        live[u] = ent[u] != 0xffffffffu && (int64_t)(ent[u] & 0xffffu) < out_limit;
        // tap 0; dead entries read (and discard) from a safe place
        xs[u] = live[u] ? s_x + ((int)(ent[u] >> 16) + x_shift) : s_x + (kResPad + x_shift);
    }
    if (OV == 0) {
#pragma unroll
        for (int u = 0; u < ROWS; ++u) {
            if (!live[u]) continue;
            float sum = 0.f;
            const float *__restrict__ tt = p.rs_table + (size_t)__float_as_uint(__ldg(&frac_tab[first + lane + 32 * u])) * L;
            for (int j = 0; j < L; ++j) sum += xs[u][j] * __ldg(&tt[j]);
            pcm_store(g.out, out_fmt(g), orow + (ent[u] & 0xffffu), sum);
        }
        return;
    }
    const int qoff = 4 + OV - bucket;
    auto quad_at = [&](int tap) -> float4 { return s_quad[qoff + tap * OV]; };   // warp-uniform: a broadcast load
    float2 acc[ROWS][2];   // (accum[0], accum[1]) and (accum[2], accum[3]) of resample.c:478-489, as FFMA2 register pairs
#pragma unroll
    for (int u = 0; u < ROWS; ++u) { acc[u][0] = make_float2(0.f, 0.f); acc[u][1] = make_float2(0.f, 0.f); }
    float4 tqa[2], tqb[2];
    float xa[2][ROWS], xb[2][ROWS];
    auto load2 = [&](int j, float4 (&tq)[2], float (&x)[2][ROWS]) {
#pragma unroll
        for (int jj = 0; jj < 2; ++jj) {
            tq[jj] = quad_at(j + jj);
#pragma unroll
            for (int u = 0; u < ROWS; ++u) x[jj][u] = xs[u][j + jj];
        }
    };
    auto fma2 = [&](const float4 (&tq)[2], const float (&x)[2][ROWS]) {
#pragma unroll
        for (int jj = 0; jj < 2; ++jj)
#pragma unroll
            for (int u = 0; u < ROWS; ++u) {
                ffma2_bcast(acc[u][0], x[jj][u], tq[jj].x, tq[jj].y);
                ffma2_bcast(acc[u][1], x[jj][u], tq[jj].z, tq[jj].w);
            }
    };
    load2(0, tqa, xa);
#pragma unroll 1
    for (int j = 0; j < L - 4; j += 4) {
        load2(j + 2, tqb, xb);
        fma2(tqa, xa);
        load2(j + 4, tqa, xa);
        fma2(tqb, xb);
    }
    // last four taps; the outputs' cubic coefficients are fetched under them (the registers of the look-ahead stage are free now).
    // cubic_coef (resample.c:339-351) of the entry's fraction is computed on the host with the reference's own float / double
    // operations (Pipeline::build_resample_runs): one 16-byte load instead of ~30 instructions incl. three FP64 adds per output
    load2(L - 2, tqb, xb);
    float4 ic[ROWS];
#pragma unroll
    for (int u = 0; u < ROWS; ++u) ic[u] = __ldg(reinterpret_cast<const float4 *>(frac_tab) + (first + lane + 32 * u));   // padding entries hold zeros
    fma2(tqa, xa);
    fma2(tqb, xb);
#pragma unroll
    for (int u = 0; u < ROWS; ++u) {
        if (!live[u]) continue;
        pcm_store(g.out, out_fmt(g), orow + (ent[u] & 0xffffu), (ic[u].x * acc[u][0].x) + (ic[u].y * acc[u][0].y) + (ic[u].z * acc[u][1].x) + (ic[u].w * acc[u][1].y));
    }
}

// s_x[i + x_shift] is the normalised-stream sample an entry's packed tap-0 position i refers to; out positions are relative
// to orow (element index of the run's first output in g.out); outputs at or beyond out_limit are not stored.  The `nwarp`
// warps that call this (warp = 0..nwarp-1) take the run's steps round-robin (the host lists the long steps first).
template <int OV>   // sinc-table oversampling of the interpolated mode; 0 = direct table
__device__ __forceinline__ void resample_run(const DevPlan &p, const DevRows &g, const ResampleRun &hdr, const float4 *s_quad, const float *s_x, int x_shift,
                                             int64_t orow, int64_t out_limit, const unsigned *__restrict__ rs_ent, const float *__restrict__ rs_frac,
                                             const unsigned *__restrict__ rs_steps, int L, int warp, int nwarp) {
    const unsigned *__restrict__ ent_tab = rs_ent + hdr.ent_off;
    // per entry: the four cubic coefficients (interpolated table) or the table phase as raw bits (direct table)
    const float *__restrict__ frac_tab = rs_frac + (size_t)hdr.ent_off * (OV ? 4 : 1);
    const unsigned *__restrict__ steps = rs_steps + hdr.step_off;
    for (int s = warp; s < hdr.n_steps; s += nwarp) {
        const unsigned desc = __ldg(&steps[s]);   // warp-uniform
        const int first = (int)(desc & 0xfffffu), rows = (int)((desc >> 20) & 7u) + 1, bucket = (int)(desc >> 24);
        if (rows == 4) resample_step<OV, 4>(p, g, s_quad, s_x, x_shift, orow, out_limit, ent_tab, frac_tab, first, bucket, L);
        else if (rows == 3) resample_step<OV, 3>(p, g, s_quad, s_x, x_shift, orow, out_limit, ent_tab, frac_tab, first, bucket, L);
        else if (rows == 2) resample_step<OV, 2>(p, g, s_quad, s_x, x_shift, orow, out_limit, ent_tab, frac_tab, first, bucket, L);
        else resample_step<OV, 1>(p, g, s_quad, s_x, x_shift, orow, out_limit, ent_tab, frac_tab, first, bucket, L);
    }
}

}  // namespace pvgpu
