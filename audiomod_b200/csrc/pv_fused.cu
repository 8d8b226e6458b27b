// k_synth_ola: inverse FFT + synthesis window + overlap-add + window-sum normalisation + Speex resampler in ONE kernel,
// with the overlap-add accumulator in shared memory (north_star "Resynthesis ... shared-memory accumulate").
//
// Reference arithmetic: synthesiseSlice (phasevocoderprocess.cc:1001-1075: 1/N, inversePolar -> kiss_fftri
// kiss_fftr.c:123-159, ifftshift + Hann impl.h:183-198, outAcc += frame), writeSlice (:1140-1194: outAcc / winAcc for the
// first shiftIncrement samples, resample, shift the accumulators) and the Speex resampler (resample.c:462-560).
//
// Why this shape (it has no counterpart in the reference, which does all of this per slice on one thread): the reference's
// accumulator is a sliding window of N samples that receives frame k at position ola_off_k and emits its first shift_k
// samples -- a strictly ordered chain along time, but only along time.  The split version (k_synthesise_t writing every
// windowed frame to a DRAM ring, k_ola_resample gathering the ~N/shift frames that cover each output sample) spent 16 KB of
// DRAM traffic and a 4-frame gather loop per frame on re-assembling that order.  Here one CTA owns one channel row for a
// whole chunk of frames: its N/32-thread groups run the inverse FFTs of G consecutive frames concurrently in registers,
// and add their windowed outputs into a shared-memory ring in FRAME ORDER (a token passed between the groups through named
// barriers, so position t receives its frames in exactly the reference's order and the sums are bit-identical to the
// split kernels').  After every `run` frames the finished part of the ring is normalised into the resampler's input window
// (which keeps filt_len + 8 samples of history), the resampler produces that run's outputs from shared memory, and the ring
// moves on.  Between launches a row carries N floats of unfinished accumulator and the resampler history in global memory.
// No frame ring, no halo tables, no limit on how many frames overlap (extreme stretch ratios just mean more adds per sample).
#include "pv_kernels.cuh"
#include "pv_fft.cuh"
#include "pv_synth.cuh"
#include "pv_resample.cuh"
#include "pv_fused.cuh"

namespace pvgpu {

// kPre: 0 = generic pre-pass (polar spectra / robotic / whisper / vocoder / constant), 1 = Cartesian phase-locked core,
// 2 = the same + formant / gender frequency warp.  kOV8: the interpolated resampler with oversampling 8 (every ratio within
// an octave); otherwise the resampler variant is chosen at run time (direct table, oversampling 1/2/4, or none).
template <int N, int kPre, bool kOV8>
__global__ void __launch_bounds__(FusedShape<N>::kThreads, N <= 2048 ? 3 : 2) k_synth_ola(const DevPlan p, const DevRows g, const FusedArgs a) {
    using FS = FusedShape<N>;
    constexpr int NC = N / 2;
    using S = FftShape<NC>;
    constexpr int T = FS::T, G = FS::G, U = FS::U, UT = FS::UT, FU = FS::FU, kThreads = FS::kThreads;
    extern __shared__ __align__(16) float4 smem4[];
    __shared__ ResampleRun s_hdr;
    const int row = blockIdx.x, tid = threadIdx.x;
    const int group = tid / T, t = tid % T, unit = tid / UT;
    const bool rs = p.rs_active != 0;
    const bool quad = rs && !p.rs_direct;
    const int L = rs ? (int)p.rs_filt_len : 0;
    const int HL = a.hist_len;
    float4 *s_quad = smem4;
    float *s_in = (float *)(smem4 + (quad ? p.rs_table_len : 0));
    float *s_acc = s_in + a.in_len;
    float2 *buf = (float2 *)(s_acc + a.acc_len) + group * S::kPadded;
    const int mask = a.acc_len - 1;
    const SliceRec *__restrict__ rr = a.recs - a.recs_base;
    const long k0 = a.k0;
    const int nf = a.nf, R = a.run;
    const int64_t ola_base = rr[k0].ola_off;

    // ---- state in: unfinished accumulator (N samples from ola_base on), resampler history, sinc quads ----
    float *__restrict__ tail = g.ola_tail + (int64_t)row * N;
    for (int i = tid; i < a.acc_len; i += kThreads) s_acc[i] = i < N ? tail[i] : 0.f;
    float *__restrict__ hist = rs ? g.res_hist + (int64_t)row * HL : nullptr;
    for (int i = tid; i < HL; i += kThreads) s_in[i] = hist[i];
    if (quad) {
        const float4 *__restrict__ tab4 = p.rs_quads;
        for (int e = tid; e < p.rs_table_len; e += kThreads) s_quad[e] = __ldg(&tab4[e]);
    }
    __syncthreads();

    const int64_t row_out = (int64_t)row * g.out_stride - g.out_base;
    const int64_t row_limit = g.n_out[row];
    const float2 *__restrict__ w2 = (const float2 *)p.window;
    const int ob = fft_out_base<NC>(t);
    const long total_slots = ((long)(nf / R) * (R / G) + ((nf % R) + G - 1) / G) * U;
    long slot = unit;   // token slots are numbered (sub-iteration * U + unit); slot s adds after slot s - 1

    for (int r0 = 0; r0 < nf; r0 += R) {
        const int nfr = min(R, nf - r0);
        const long ka = k0 + r0, kb = ka + nfr;
        if (rs && tid < (int)(sizeof(ResampleRun) / sizeof(int)))   // this run's work-list header (visible after the barrier below)
            ((int *)&s_hdr)[tid] = ((const int *)&a.runs[(ka - a.run_origin) / R])[tid];

        // ---- inverse FFTs of the run's frames, G at a time, added to the ring in frame order ----
        for (int j0 = 0; j0 < nfr; j0 += G, slot += U) {
            const bool active = j0 + group < nfr;
            const int f = r0 + j0 + group;
            const long k = k0 + f;
            if (active) {
                if (kPre == 0) synth_prepass_generic<N>(p, g, a.car_mag, a.car_phase, row, f, k, t, buf);
                else synth_prepass_lock<N, kPre == 2>(p, g, row, f, t, buf);
            }
            frame_sync<T>(group);
            float2 v[16];
            if (active) fft_frame<NC, true>(v, buf, t, group, p.tw_inv, p.tw2_inv, p.tw3_inv);
            else { if (NC > 256) { frame_sync<T>(group); } frame_sync<T>(group); }
            // the token: all threads of the unit are past their last read of `buf` once it completes, so the next pre-pass may
            // overwrite it; U == 1 (one frame per CTA) only needs that second property
            if (U > 1) named_sync(kTokenBarrier0 + unit, slot != 0 ? 2 * UT : UT);   // slot 0 has no predecessor: the unit alone
            else __syncthreads();
#pragma unroll
            for (int h = 0; h < FU; ++h) {
                if (active && (FU == 1 || (group & (FU - 1)) == h)) {
                    fused_add_frame<N>(v, s_acc, mask, (int)(rr[k].ola_off - ola_base), ob, w2);
                }
                if (FU > 1) __syncwarp();
            }
            if (U > 1 && slot != total_slots - 1) named_arrive(kTokenBarrier0 + (unit + 1) % U, 2 * UT);
        }
        __syncthreads();

        // ---- the run's finished samples: normalise (:1152), hand to the resampler window or store, clear the ring ----
        const int64_t res_base = rr[ka].res_off;      // normalised-stream position of s_in[HL]
        for (long k = ka; k < kb; ++k) {
            const SliceRec rc = rr[k];
            if (rc.flags & 1) continue;               // dropped slice (:337-364): its frame stays in the accumulator, nothing is emitted
            const int off = (int)(rc.ola_off - ola_base);
            const int rel = (int)(rc.res_off - res_base) + HL;
            const float *__restrict__ nrm = a.norm + (rc.ola_off - a.norm_base);
            int n_store = rc.n_write;
            if (rc.out_off + n_store > row_limit) n_store = (int)max((int64_t)0, row_limit - rc.out_off);
            for (int e = tid; e < rc.shift_inc; e += kThreads) {
                const int idx = (off + e) & mask;
                const float s = s_acc[idx];
                s_acc[idx] = 0.f;
                if (e < rc.consumed) {
                    const float v = s / nrm[e];
                    if (rs) s_in[rel + e] = v;
                    else if (e < n_store) pcm_store(g.out, out_fmt(g), row_out + rc.out_off + e, v);
                }
            }
        }
        if (!rs) { __syncthreads(); continue; }
        __syncthreads();

        // ---- resampler over the run's work list; s_in[i] is normalised-stream position res_base - HL + i ----
        {
            const int x_shift = (int)(s_hdr.u_lo - (res_base - HL)) - kResPad;
            const int64_t orow = row_out + s_hdr.out_first, out_limit = row_limit - s_hdr.out_first;
            if (kOV8) resample_run<8>(p, g, s_hdr, s_quad, s_in, x_shift, orow, out_limit, a.rs_ent, a.rs_frac, a.rs_steps, L, tid >> 5, kThreads >> 5);
            else if (!quad) resample_run<0>(p, g, s_hdr, s_quad, s_in, x_shift, orow, out_limit, a.rs_ent, a.rs_frac, a.rs_steps, L, tid >> 5, kThreads >> 5);
            else if (p.rs_oversample == 4) resample_run<4>(p, g, s_hdr, s_quad, s_in, x_shift, orow, out_limit, a.rs_ent, a.rs_frac, a.rs_steps, L, tid >> 5, kThreads >> 5);
            else if (p.rs_oversample == 2) resample_run<2>(p, g, s_hdr, s_quad, s_in, x_shift, orow, out_limit, a.rs_ent, a.rs_frac, a.rs_steps, L, tid >> 5, kThreads >> 5);
            else if (p.rs_oversample == 8) resample_run<8>(p, g, s_hdr, s_quad, s_in, x_shift, orow, out_limit, a.rs_ent, a.rs_frac, a.rs_steps, L, tid >> 5, kThreads >> 5);
            else resample_run<1>(p, g, s_hdr, s_quad, s_in, x_shift, orow, out_limit, a.rs_ent, a.rs_frac, a.rs_steps, L, tid >> 5, kThreads >> 5);
        }
        __syncthreads();
        // ---- keep the last HL normalised samples as the next run's history ----
        {
            const SliceRec &last = rr[kb - 1];
            const int used = (int)(last.res_off - res_base) + ((last.flags & 1) ? 0 : last.consumed);
            if (used > 0) {
                for (int c = 0; c < HL; c += kThreads) {
                    const int i = c + tid;
                    const float v = i < HL ? s_in[used + i] : 0.f;
                    __syncthreads();
                    if (i < HL) s_in[i] = v;
                }
                __syncthreads();
            }
        }
    }

    // ---- state out ----
    {
        const SliceRec &last = rr[k0 + nf - 1];
        const int off_end = (int)(last.ola_off - ola_base) + ((last.flags & 1) ? 0 : last.shift_inc);
        for (int i = tid; i < N; i += kThreads) tail[i] = s_acc[(off_end + i) & mask];
        for (int i = tid; i < HL; i += kThreads) hist[i] = s_in[i];
    }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
static int pow2_at_least(int v) { int r = 1; while (r < v) r <<= 1; return r; }

template <int N> static int frames_in_flight() { return FusedShape<N>::G; }

int fused_frames_in_flight(int N) {
    switch (N) {
        case 512: return frames_in_flight<512>();
        case 1024: return frames_in_flight<1024>();
        case 2048: return frames_in_flight<2048>();
        case 4096: return frames_in_flight<4096>();
        case 8192: return frames_in_flight<8192>();
        default: return 0;   // other sizes have no fused kernel
    }
}

static size_t fused_smem(const DevPlan &p, const FusedArgs &a) {
    const bool quad = p.rs_active && !p.rs_direct;
    const int NC = p.N / 2, padded = NC + NC / 16 + NC / 256 + 2;
    const int G = fused_frames_in_flight(p.N);
    return (quad ? sizeof(float4) * (size_t)p.rs_table_len : 0) + sizeof(float) * ((size_t)a.in_len + a.acc_len) + sizeof(float2) * (size_t)G * padded;
}

// Shape of the fused kernel for a schedule: frames per run (a multiple of the frames in flight that divides
// frames_per_chunk), ring length, resampler window.  Returns false when no run length fits the shared-memory budget.
bool fused_plan(const DevPlan &p, int frames_per_chunk, int max_shift, int max_consumed, int max_out, size_t smem_limit, FusedArgs *out) {
    const int G = fused_frames_in_flight(p.N);
    if (G == 0) return false;
    const int L = p.rs_active ? (int)p.rs_filt_len : 0;
    if (L > kResPad) return false;
    FusedArgs best{};
    bool found = false;
    // prefer runs of about 8 frames at N = 2048 (three CTAs per SM); longer runs amortise the per-run barriers and the
    // padding of the resampler's work lists, shorter ones keep the ring small
    for (int run = G; run <= 64; run += G) {
        if (frames_per_chunk % run) continue;
        FusedArgs a{};
        a.run = run;
        a.hist_len = p.rs_active ? L + 8 : 0;
        a.acc_len = pow2_at_least(p.N + (run - 1) * max_shift);
        a.in_len = p.rs_active ? ((a.hist_len + run * max_consumed + 8 + 3) & ~3) : 4;
        // the packed work-list entries hold 16-bit positions relative to the run (see build_resample_runs)
        if (p.rs_active && (run * max_consumed + L + 8 + kResPad >= 65536 || run * max_out >= 65535)) break;
        const size_t sm = fused_smem(p, a);
        if (sm > smem_limit) break;
        const int target = p.N <= 2048 ? 3 : 2;   // resident CTAs per SM the launch bounds aim for
        const size_t per_cta = ((size_t)227 * 1024) / target - 1024;
        if (found && sm > per_cta) break;     // do not trade a resident CTA for a longer run
        best = a;
        found = true;
    }
    if (found) *out = best;
    return found;
}

template <int N, int kPre, bool kOV8>
static cudaError_t launch_one(const DevPlan &p, const DevRows &g, const FusedArgs &a, cudaStream_t st) {
    const size_t sm = fused_smem(p, a);
    static bool configured[16] = {};   // per device: shared-memory opt-in done
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 16 && !configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(k_synth_ola<N, kPre, kOV8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(200 * 1024));
        if (e != cudaSuccess) return e;
        configured[dev] = true;
    }
    k_synth_ola<N, kPre, kOV8><<<g.rows, FusedShape<N>::kThreads, sm, st>>>(p, g, a);
    return cudaSuccess;
}

template <int N>
static cudaError_t launch_n(const DevPlan &p, const DevRows &g, const FusedArgs &a, cudaStream_t st) {
    const bool ov8 = p.rs_active && !p.rs_direct && p.rs_oversample == 8;
    const int pre = g.synth_kind == 4 ? (p.warp_tab != nullptr ? 2 : 1) : 0;
    if (pre == 1) return ov8 ? launch_one<N, 1, true>(p, g, a, st) : launch_one<N, 1, false>(p, g, a, st);
    if (pre == 2) return ov8 ? launch_one<N, 2, true>(p, g, a, st) : launch_one<N, 2, false>(p, g, a, st);
    return ov8 ? launch_one<N, 0, true>(p, g, a, st) : launch_one<N, 0, false>(p, g, a, st);
}

cudaError_t launch_synth_ola(const DevPlan &p, const DevRows &g, const FusedArgs &a, cudaStream_t st) {
    switch (p.N) {
        case 512: return launch_n<512>(p, g, a, st);
        case 1024: return launch_n<1024>(p, g, a, st);
        case 2048: return launch_n<2048>(p, g, a, st);
        case 4096: return launch_n<4096>(p, g, a, st);
        case 8192: return launch_n<8192>(p, g, a, st);
        default: return cudaErrorInvalidValue;
    }
}

}  // namespace pvgpu
