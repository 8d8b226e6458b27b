// Hand-written sm_100a kernels of the batched phase vocoder.
//
// Stage map (reference file:line relative to the reference tree):
//   k_analyse      frame gather + Hann + fftshift + KissFFT-order real FFT + polar
//                  (phasevocoderprocess.cc:492-503, phasevocoderimpl.h:167-181, kiss_fftr.c:67-121,
//                   kiss_fft.c:36-104,250-286, FFT.cc:2617-2631)
//   k_phase_core   peak picking / peak linking / phase locking, and the classic per-bin propagation
//                  (phasevocoderprocess.cc:574-706, 708-753)
//   k_int_ratio    coremode 2 (phasevocoderprocess.cc:558-572)
//   k_fixed_phase  robotic / whisper (phasevocoderprocess.cc:805-822)
//   k_synthesise   [freq-comp warp :842-923] [vocoder band modulation :755-776] 1/N scale, polar->cartesian,
//                  inverse real FFT (kiss_fftr.c:123-159), ifftshift + Hann (:1024-1056, impl.h:183-198)
//   k_overlap_add  overlap-add in frame order + window-sum normalisation (:1057-1073, 1152, 1185-1190)
//   k_resample     Speex quality-4 windowed-sinc resampler (speex/resample.c:352-403,462-560)
//
// Rounding discipline: everything that feeds a discrete decision of the reference (the forward FFT,
// magnitude, atan2f, and the phase arithmetic) uses __f*_rn / __d*_rn intrinsics, which nvcc never
// contracts into FMAs, in the reference's operation order.  The synthesis side (inverse FFT, OLA,
// resampler) is held to the 1e-4 / 90 dB tolerance and may use FMA.
#include <algorithm>

#include "pv_kernels.cuh"
#include "pv_fft.cuh"
#include "pv_math.cuh"
#include "pv_synth.cuh"
#include "pv_resample.cuh"

// out-of-line copy of the general atan2f for the rare arguments the fast path rejects (keeps the hot kernels small)
__device__ __noinline__ float pv_atan2f_rare(float y, float x) { return pv_atan2f(y, x); }

namespace pvgpu {

// All butterfly stages of the nc-point complex FFT, in place in shared memory (data already permuted).
template <bool kInverse>
__device__ __forceinline__ void fft_stages(const DevPlan &p, float2 *F) {
    const float2 *__restrict__ tw = kInverse ? p.tw_inv : p.tw_fwd;
    const int nc = p.nc;
    for (int s = 0; s < p.nstages; ++s) {
        const int m = p.span[s], rad = p.radix[s];
        const int fstride = nc / (m * rad);
        if (rad == 2) {
            for (int b = threadIdx.x; b < nc / 2; b += blockDim.x) {
                const int grp = b / m, k = b - grp * m;
                float2 *f = F + grp * 2 * m + k;
                const float2 t = cmul_rn(f[m], __ldg(&tw[k * fstride]));
                const float2 a = f[0];
                f[m] = csub_rn(a, t);
                f[0] = cadd_rn(a, t);
            }
        } else {
            for (int b = threadIdx.x; b < nc / 4; b += blockDim.x) {
                const int grp = b / m, k = b - grp * m;
                float2 *f = F + grp * 4 * m + k;
                float2 f0 = f[0], f1 = f[m], f2 = f[2 * m], f3 = f[3 * m];
                bfly4<kInverse>(f0, f1, f2, f3, __ldg(&tw[k * fstride]), __ldg(&tw[2 * k * fstride]), __ldg(&tw[3 * k * fstride]));
                f[0] = f0; f[m] = f1; f[2 * m] = f2; f[3 * m] = f3;
            }
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------
// k_analyse: one CTA per (frame, row)
// ------------------------------------------------------------------------------------------------
__global__ void k_analyse(const DevPlan p, const DevRows g, long k0) {
    extern __shared__ float smem[];
    float *s_t = smem;                       // N floats: windowed, fft-shifted frame
    float2 *s_f = (float2 *)(smem + p.N);    // nc complex
    const int row = blockIdx.y;
    const long k = k0 + blockIdx.x;
    const int N = p.N, nc = p.nc, hs = N / 2;
    const int64_t xoff = (int64_t)row * g.in_stride - g.in_base;
    const int64_t start = (int64_t)k * p.hop;
    const int64_t nvalid = g.n_in[row];
    for (int j = threadIdx.x; j < N; j += blockDim.x) {
        const int64_t gi = start + j;
        const float v = gi < nvalid ? pcm_load(g.in, g.fmt, xoff + gi) : 0.f;
        s_t[(j + hs) & (N - 1)] = __fmul_rn(v, __ldg(&p.window[j]));
    }
    __syncthreads();
    const float2 *s_tc = (const float2 *)s_t;
    for (int o = threadIdx.x; o < nc; o += blockDim.x) s_f[o] = s_tc[p.perm[o]];
    __syncthreads();
    fft_stages<false>(p, s_f);
    // real-FFT post-pass (kiss_fftr.c:67-121) + polar (FFT.cc:2617-2631)
    float *__restrict__ mag = g.mag + ((int64_t)row * g.F + blockIdx.x) * p.Hp;
    float *__restrict__ ph = g.phase + ((int64_t)row * g.F + blockIdx.x) * p.Hp;
    for (int kk = threadIdx.x; kk <= nc / 2; kk += blockDim.x) {
        if (kk == 0) {
            const float tr = s_f[0].x, ti = s_f[0].y;
            const float dc = __fadd_rn(tr, ti), ny = __fsub_rn(tr, ti);
            mag[0] = __fsqrt_rn(__fadd_rn(__fmul_rn(dc, dc), 0.f));
            ph[0] = pv_atan2f(0.f, dc);
            mag[nc] = __fsqrt_rn(__fadd_rn(__fmul_rn(ny, ny), 0.f));
            ph[nc] = pv_atan2f(0.f, ny);
        } else {
            const float2 fpk = s_f[kk];
            const float2 fq = s_f[nc - kk];
            const float2 fpnk = make_float2(fq.x, -fq.y);
            const float2 f1k = cadd_rn(fpk, fpnk), f2k = csub_rn(fpk, fpnk);
            const float2 tw = cmul_rn(f2k, __ldg(&p.stw_fwd[kk]));
            const float ar = __fmul_rn(__fadd_rn(f1k.x, tw.x), 0.5f), ai = __fmul_rn(__fadd_rn(f1k.y, tw.y), 0.5f);
            const float br = __fmul_rn(__fsub_rn(f1k.x, tw.x), 0.5f), bi = __fmul_rn(__fsub_rn(tw.y, f1k.y), 0.5f);
            if (kk != nc - kk) {  // bin nc/2 is written twice by the reference; the second write wins
                mag[kk] = __fsqrt_rn(__fadd_rn(__fmul_rn(ar, ar), __fmul_rn(ai, ai)));
                ph[kk] = pv_atan2f(ai, ar);
            }
            mag[nc - kk] = __fsqrt_rn(__fadd_rn(__fmul_rn(br, br), __fmul_rn(bi, bi)));
            ph[nc - kk] = pv_atan2f(bi, br);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// k_analyse_t<N>: register-tiled version for N = 512..8192 (pv_fft.cuh).  T = N/32 threads own a frame; a CTA of
// max(T, 256) threads handles 256/T consecutive frames of the chunk.
// ------------------------------------------------------------------------------------------------
template <int N, bool kS16, bool kCart>
__global__ void __launch_bounds__((N / 32 > 256 ? N / 32 : 256)) k_analyse_t(const DevPlan p, const DevRows g, long k0, int nf, int total) {
    constexpr int NC = N / 2;
    using S = FftShape<NC>;
    constexpr int T = S::kThreads;
    constexpr int G = (T >= 256) ? 1 : 256 / T;
    extern __shared__ __align__(16) float2 sbuf[];
    const int group = threadIdx.x / T, t = threadIdx.x % T;
    float2 *buf = sbuf + group * S::kPadded;
    const int fid = blockIdx.x * G + group;
    const bool active = fid < total;   // whole groups are active or not, so group barriers stay consistent
    const int row = active ? fid / nf : 0, f = active ? fid % nf : 0;
    if (active) {
        const long k = k0 + f;
        const int64_t start = (int64_t)k * p.hop;
        const int64_t xoff = (int64_t)row * g.in_stride + (start - g.in_base);
        const int64_t left = g.n_in[row] - start;
        const int valid = left < 0 ? 0 : (left > N ? N : (int)left);   // samples of this frame that exist; the rest are zeros
        const float2 *__restrict__ w2 = (const float2 *)p.window;
        // gather + Hann + fftshift + KissFFT input permutation, one complex (two consecutive samples) at a time.  Complex
        // cc = t + T*i lands (after the fftshift by NC/2) at slot perm(t) | perm((T*i + NC/2) mod NC): the permutation is a
        // bit permutation and the two parts have disjoint bits, and the padded position is additive in the two parts, so
        // every store is base + compile-time constant.
        const int base = fft_pad(fft_slot_of_input<NC>(t));
        float x0[16], x1[16];
        if (kS16) {
            const short *__restrict__ xp = (const short *)g.in + xoff + 2 * t;
            if (valid == N && ((reinterpret_cast<uintptr_t>(xp) & 3) == 0)) {   // even frame start: one 32-bit load per sample pair
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const short2 xx = *(const short2 *)(xp + 2 * T * i);
                    x0[i] = (float)xx.x * (1.0f / 32768.0f); x1[i] = (float)xx.y * (1.0f / 32768.0f);
                }
            } else if (valid == N) {   // whole frame inside the stream: no per-sample bounds
#pragma unroll
                for (int i = 0; i < 16; ++i) { x0[i] = (float)xp[2 * T * i] * (1.0f / 32768.0f); x1[i] = (float)xp[2 * T * i + 1] * (1.0f / 32768.0f); }
            } else {
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const int s0 = 2 * (t + T * i);
                    x0[i] = s0 < valid ? (float)xp[2 * T * i] * (1.0f / 32768.0f) : 0.f;
                    x1[i] = s0 + 1 < valid ? (float)xp[2 * T * i + 1] * (1.0f / 32768.0f) : 0.f;
                }
            }
        } else {
            const float *__restrict__ xp = (const float *)g.in + xoff + 2 * t;
            if (valid == N && ((reinterpret_cast<uintptr_t>(xp) & 7) == 0)) {   // even frame start: one 64-bit load per sample pair
#pragma unroll
                for (int i = 0; i < 16; ++i) { const float2 xx = *(const float2 *)(xp + 2 * T * i); x0[i] = xx.x; x1[i] = xx.y; }
            } else if (valid == N) {
#pragma unroll
                for (int i = 0; i < 16; ++i) { x0[i] = xp[2 * T * i]; x1[i] = xp[2 * T * i + 1]; }
            } else {
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const int s0 = 2 * (t + T * i);
                    x0[i] = s0 < valid ? xp[2 * T * i] : 0.f;
                    x1[i] = s0 + 1 < valid ? xp[2 * T * i + 1] : 0.f;
                }
            }
        }
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const float2 w = __ldg(&w2[t + T * i]);
            const int K = fft_pad(fft_slot_of_input<NC>((T * i + NC / 2) & (NC - 1)));
            buf[base + K] = make_float2(__fmul_rn(x0[i], w.x), __fmul_rn(x1[i], w.y));
        }
    }
    frame_sync<T>(group);
    float2 v[16];
    if (active) fft_frame<NC, false>(v, buf, t, group, p.tw_fwd, p.tw2_fwd, p.tw3_fwd);
    else { if (NC > 256) { frame_sync<T>(group); } frame_sync<T>(group); }
    frame_sync<T>(group);   // all reads of the last pass are done before the natural-order write-back
    if (active) {
        float2 *bo = buf + fft_pad(fft_out_base<NC>(t));
#pragma unroll
        for (int i = 0; i < 16; ++i) bo[fft_pad(fft_out_const<NC>(i))] = v[i];
    }
    frame_sync<T>(group);
    if (!active) return;
    // real-FFT post-pass (kiss_fftr.c:67-121) + polar (FFT.cc:2617-2631)
    float *__restrict__ mag = g.mag + ((int64_t)row * g.F + f) * p.Hp;
    float *__restrict__ ph = g.phase + ((int64_t)row * g.F + f) * p.Hp;
    const float2 *__restrict__ stw = p.stw_fwd;
    constexpr int Q = (NC / 2) / T;
    const int pa = fft_pad(t), pb = fft_pad((T - t) & (T - 1));   // padded positions are additive in (t, T*q)
    // rolled on purpose: the body holds two atan2f and two sqrtf expansions, and unrolling it 8x makes the kernel
    // several times larger than the instruction cache
#pragma unroll 1
    for (int q = 0; q < Q; ++q) {
        const int kk = t + T * q;
        const float2 fpk = buf[pa + fft_pad(T * q)];
        // NC - (t + T*q) = T*(15-q) + (T-t) for t > 0, T*(16-q) for t == 0 (q == 0 pairs DC with itself)
        const float2 fq = buf[pb + (t == 0 ? fft_pad((T * (16 - q)) & (NC - 1)) : fft_pad(T * (15 - q)))];
        float ar, ai, br, bi;
        if (kk == 0) {
            ar = __fadd_rn(fpk.x, fpk.y); ai = 0.f;   // DC
            br = __fsub_rn(fpk.x, fpk.y); bi = 0.f;   // Nyquist
        } else {
            const float2 fpnk = make_float2(fq.x, -fq.y);
            const float2 f1k = cadd_rn(fpk, fpnk), f2k = csub_rn(fpk, fpnk);
            const float2 tw = cmul_rn(f2k, __ldg(&stw[kk]));
            ar = __fmul_rn(__fadd_rn(f1k.x, tw.x), 0.5f); ai = __fmul_rn(__fadd_rn(f1k.y, tw.y), 0.5f);
            br = __fmul_rn(__fsub_rn(f1k.x, tw.x), 0.5f); bi = __fmul_rn(__fsub_rn(tw.y, f1k.y), 0.5f);
        }
        if (kCart) {   // Cartesian spectra for the modes that never look at the analysis phase
            mag[kk] = ar; ph[kk] = ai;
            mag[NC - kk] = br; ph[NC - kk] = bi;
        } else {
            mag[kk] = __fsqrt_rn(__fadd_rn(__fmul_rn(ar, ar), __fmul_rn(ai, ai)));
            ph[kk] = pv_atan2f_fast(ai, ar);
            mag[NC - kk] = __fsqrt_rn(__fadd_rn(__fmul_rn(br, br), __fmul_rn(bi, bi)));
            ph[NC - kk] = pv_atan2f_fast(bi, br);
        }
    }
    if (t == 0) {   // bin NC/2 pairs with itself; the reference writes it twice and the second write wins (kiss_fftr.c:116-119)
        const float2 fpk = buf[fft_pad(NC / 2)];
        const float2 fpnk = make_float2(fpk.x, -fpk.y);
        const float2 f1k = cadd_rn(fpk, fpnk), f2k = csub_rn(fpk, fpnk);
        const float2 tw = cmul_rn(f2k, __ldg(&stw[NC / 2]));
        const float br = __fmul_rn(__fsub_rn(f1k.x, tw.x), 0.5f), bi = __fmul_rn(__fsub_rn(tw.y, f1k.y), 0.5f);
        if (kCart) {
            mag[NC / 2] = br; ph[NC / 2] = bi;
        } else {
            mag[NC / 2] = __fsqrt_rn(__fadd_rn(__fmul_rn(br, br), __fmul_rn(bi, bi)));
            ph[NC / 2] = pv_atan2f_fast(bi, br);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// phase core
// ------------------------------------------------------------------------------------------------
// princarg, src/common/system/sys.h:84-91 (double overload): mod(a + pi, -2pi) + pi with
// mod(x, y) = x - y*floor(x/y)
__device__ __forceinline__ double princarg_rn(double a) {
    const double pi = 3.14159265358979323846, m2pi = -2.0 * 3.14159265358979323846;
    const double x = __dadd_rn(a, pi);
    const double q = floor(__ddiv_rn(x, m2pi));
    return __dadd_rn(__dsub_rn(x, __dmul_rn(m2pi, q)), pi);
}

// Same value, cheaper: floor(x / -2pi) is taken from x * fl(-1/2pi) whenever that product is safely away from an
// integer (the two differ by < 4e-16 |q|); otherwise the exact division decides.
__device__ __forceinline__ double princarg_fast(double a) {
    const double pi = 3.14159265358979323846, m2pi = -2.0 * 3.14159265358979323846;
    const double x = __dadd_rn(a, pi);
    const double qa = __dmul_rn(x, -0.15915494309189535);
    double n = floor(qa);
    const double fr = qa - n;
    if (!(fr > 1e-9 && fr < 1.0 - 1e-9 && fabs(qa) < 1e6)) n = floor(__ddiv_rn(x, m2pi));
    return __dadd_rn(__dsub_rn(x, __dmul_rn(m2pi, n)), pi);
}

__device__ __forceinline__ float sub3_rn(float a, float b, float c) { return __fsub_rn(__fsub_rn(a, b), c); }

// One CTA per stream; frames and channels are visited in the reference's order because the peak
// lists are shared by the channels of a stream (phasevocoderimpl.h:237-238) and "first entry" is a
// per-process flag (phasevocoderprocess.cc:602,716).
template <bool kLocked>
__global__ void k_phase_core(const DevPlan p, const DevRows g, const SliceRec *__restrict__ recs, long recs_base, long k0, int nframes) {
    extern __shared__ float smem[];
    const int half = p.half, C = g.channels, maxpk = g.maxpk;
    float *s_mag = smem;                        // Hp
    float *s_ph = s_mag + p.Hp;                 // Hp
    float *s_pp = s_ph + p.Hp;                  // C * half   previous analysis phase
    float *s_po = s_pp + C * half;              // C * half   previous output phase
    int *s_cur = (int *)(s_po + C * half);      // maxpk
    int *s_prev = s_cur + maxpk;                // maxpk
    int *s_start = s_prev + maxpk;              // maxpk + 1
    float *s_rot = (float *)(s_start + maxpk + 1);  // maxpk
    int *s_misc = (int *)(s_rot + maxpk);       // [0]=npk [1]=nprev [2]=first, [8..8+32) warp sums
    const int stream = blockIdx.x;
    const int tid = threadIdx.x, nthr = blockDim.x;
    const int lane = tid & 31, warp = tid >> 5, nwarp = nthr >> 5;

    for (int c = 0; c < C; ++c) {
        const int64_t row = (int64_t)stream * C + c;
        for (int i = tid; i < half; i += nthr) {
            s_pp[c * half + i] = g.prev_phase[row * half + i];
            s_po[c * half + i] = g.prev_out[row * half + i];
        }
    }
    int *gpk = g.peaks + (int64_t)stream * (1 + maxpk);
    if (tid == 0) { s_misc[1] = gpk[0]; s_misc[2] = g.started[stream] == 0; }
    __syncthreads();
    for (int i = tid; i < s_misc[1]; i += nthr) s_prev[i] = gpk[1 + i];
    __syncthreads();

    const int E = (half + nthr - 1) / nthr;  // contiguous bins per thread
    for (int f = 0; f < nframes; ++f) {
        const float phase_inc = (float)recs[k0 + f - recs_base].phase_inc;  // size_t -> float conversion of the reference
        const float hopf = (float)p.hop;
        for (int c = 0; c < C; ++c) {
            const int64_t row = (int64_t)stream * C + c;
            float *__restrict__ gph = g.phase + (row * g.F + f) * p.Hp;
            const float *__restrict__ gmag = g.mag + (row * g.F + f) * p.Hp;
            for (int i = tid; i < half; i += nthr) {
                s_ph[i] = gph[i];
                if (kLocked) s_mag[i] = gmag[i];
            }
            __syncthreads();
            float *pp = s_pp + c * half, *po = s_po + c * half;
            int npk = 0;
            if (kLocked) {
                // peak picking (:587-596): every strict +-2 local maximum with 2 <= b <= half-3, in order
                int cnt = 0;
                unsigned flags = 0;
                const int b0 = tid * E;
                for (int e = 0; e < E; ++e) {
                    const int b = b0 + e;
                    if (b >= 2 && b + 2 < half) {
                        const float m = s_mag[b];
                        if (m > s_mag[b - 1] && m > s_mag[b - 2] && m > s_mag[b + 1] && m > s_mag[b + 2]) { flags |= 1u << e; ++cnt; }
                    }
                }
                int incl = cnt;
                for (int d = 1; d < 32; d <<= 1) {
                    const int v = __shfl_up_sync(0xffffffffu, incl, d);
                    if (lane >= d) incl += v;
                }
                if (lane == 31) s_misc[8 + warp] = incl;
                __syncthreads();
                int base = 0;
                for (int w = 0; w < warp; ++w) base += s_misc[8 + w];
                int pos = base + incl - cnt;
                for (int e = 0; e < E; ++e)
                    if (flags & (1u << e)) s_cur[pos++] = b0 + e;
                if (tid == nthr - 1) s_misc[0] = base + incl;
                __syncthreads();
                npk = s_misc[0];
            }
            const int nprev = s_misc[1];
            const int first = s_misc[2];
            if (first) {
                // first call of the process: pass the analysis phase through and seed the state (:606-616)
                for (int i = tid; i < half; i += nthr) { const float tp = s_ph[i]; pp[i] = tp; po[i] = tp; }
            } else if (npk == 0 || nprev == 0) {
                // classic propagation (:617-636 / :731-748)
                for (int i = tid; i < half; i += nthr) {
                    const float omega = __ldg(&p.omega[i]);
                    const float phi = s_ph[i];
                    const float dphi = (float)__dadd_rn((double)omega, princarg_rn((double)sub3_rn(phi, pp[i], omega)));
                    const float adv = __fdiv_rn(__fmul_rn(dphi, phase_inc), hopf);
                    const float outp = (float)princarg_rn((double)__fadd_rn(po[i], adv));
                    pp[i] = phi;
                    po[i] = outp;
                    gph[i] = outp;
                }
            } else {
                // per-peak rotation (:641-667) and region start (:668-683)
                for (int pk = tid; pk < npk; pk += nthr) {
                    const int p2 = s_cur[pk];
                    int lo = 0, hi = nprev;  // first previous peak >= p2
                    while (lo < hi) { const int mid = (lo + hi) >> 1; if (s_prev[mid] < p2) lo = mid + 1; else hi = mid; }
                    int j;
                    if (lo == 0) j = 0;
                    else if (lo == nprev) j = nprev - 1;
                    else j = (s_prev[lo] - p2 < p2 - s_prev[lo - 1]) ? lo : lo - 1;  // ties keep the lower index (:644-652)
                    const int p1 = s_prev[j];
                    const float avg_p = (float)((double)(p1 + p2) * 0.5);
                    const float pomega = (float)__ddiv_rn(__dmul_rn(p.two_pi_hop, (double)__fsub_rn(avg_p, 1.0f)), (double)p.N);
                    const float dphi = (float)__dadd_rn((double)pomega, princarg_rn((double)sub3_rn(s_ph[p2], pp[p1], pomega)));
                    const float target = (float)princarg_rn((double)__fadd_rn(po[p1], __fdiv_rn(__fmul_rn(dphi, phase_inc), hopf)));
                    s_rot[pk] = (float)princarg_rn((double)__fsub_rn(target, s_ph[p2]));
                    s_start[pk] = pk == 0 ? 0 : (s_cur[pk - 1] + p2 + 1) >> 1;  // round((a+b)*0.5), half away from zero
                }
                if (tid == 0) s_start[npk] = half;
                __syncthreads();
                // lock every bin to its region's peak rotation (:685-699)
                const int b0 = tid * E;
                if (b0 < half) {
                    int lo = 0, hi = npk;  // last pk with start <= b0
                    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (s_start[mid] <= b0) lo = mid; else hi = mid; }
                    int pk = lo;
                    for (int e = 0; e < E; ++e) {
                        const int i = b0 + e;
                        if (i >= half) break;
                        while (s_start[pk + 1] <= i) ++pk;
                        const float phi = s_ph[i];
                        const float locked = (float)princarg_rn((double)__fadd_rn(phi, s_rot[pk]));
                        pp[i] = phi;
                        po[i] = locked;
                        gph[i] = locked;
                    }
                }
            }
            __syncthreads();
            if (kLocked) {
                for (int i = tid; i < npk; i += nthr) s_prev[i] = s_cur[i];
                if (tid == 0) s_misc[1] = npk;
            }
            if (tid == 0) s_misc[2] = 0;
            __syncthreads();
        }
    }
    for (int c = 0; c < C; ++c) {
        const int64_t row = (int64_t)stream * C + c;
        for (int i = tid; i < half; i += nthr) {
            g.prev_phase[row * half + i] = s_pp[c * half + i];
            g.prev_out[row * half + i] = s_po[c * half + i];
        }
    }
    const int nprev = s_misc[1];
    for (int i = tid; i < nprev; i += nthr) gpk[1 + i] = s_prev[i];
    if (tid == 0) { gpk[0] = nprev; g.started[stream] = s_misc[2] ? 0 : 1; }
}

// ------------------------------------------------------------------------------------------------
// k_phase_lock_t<E>: the phase-locked core (coremode 1) for the templated FFT sizes.  One CTA per stream, half/E
// threads, thread t owns the E contiguous bins [E*t, E*t+E).  Same arithmetic as k_phase_core<true>; differences are
// purely organisational:
//  * the next (frame, channel)'s magnitudes and phases are prefetched into registers with 128-bit loads while the
//    current one is processed (the kernel is serial in time, so global latency would otherwise be exposed every frame);
//  * a thread handles its own peaks (at most ceil(E/3): peaks are >= 3 bins apart), so the analysis phase of a peak is
//    already in its registers, and the region of a bin is one of the two peaks around the thread's first bin -- no search;
//  * current / previous peak lists ping-pong instead of being copied; four block barriers per (frame, channel).
// ------------------------------------------------------------------------------------------------
template <int E, int kMaxThreads, int kMinBlocks>
__global__ void __launch_bounds__(kMaxThreads, kMinBlocks) k_phase_lock_t(const DevPlan p, const DevRows g, const SliceRec *__restrict__ recs, long recs_base, long k0,
                                                      int nframes) {
    static_assert(E == 4 || E == 8, "bins per thread");
    constexpr int kMaxOwn = (E + 2) / 3;
    extern __shared__ float smem[];
    const int half = p.half, C = g.channels, maxpk = g.maxpk;
    float *s_mag = smem;                          // half + 8 (two guard bins each side are never peaks, but are read)
    float *s_ph = s_mag + half + 8;               // half       analysis phase of the current frame (peaks read each other's)
    float *s_pp = s_ph + half;                    // C * half   previous analysis phase
    float *s_po = s_pp + C * half;                // C * half   previous output phase
    int *s_pk0 = (int *)(s_po + C * half);        // maxpk      peak list A
    int *s_pk1 = s_pk0 + maxpk;                   // maxpk      peak list B
    int *s_start = s_pk1 + maxpk;                 // maxpk + 1
    float *s_rot = (float *)(s_start + maxpk + 1);  // maxpk
    int *s_wsum = (int *)(s_rot + maxpk);         // 32
    const int stream = blockIdx.x, tid = threadIdx.x, nthr = blockDim.x;
    const int lane = tid & 31, warp = tid >> 5, nwarp = nthr >> 5;
    const int b0 = tid * E;

    for (int c = 0; c < C; ++c) {
        const int64_t row = (int64_t)stream * C + c;
        for (int i = tid; i < half; i += nthr) {
            s_pp[c * half + i] = g.prev_phase[row * half + i];
            s_po[c * half + i] = g.prev_out[row * half + i];
        }
    }
    int *gpk = g.peaks + (int64_t)stream * (1 + maxpk);
    int nprev = gpk[0];
    bool first = g.started[stream] == 0;
    int *s_prev = s_pk0, *s_cur = s_pk1;
    for (int i = tid; i < nprev; i += nthr) s_prev[i] = gpk[1 + i];
    if (tid < 4) { s_mag[half + 4 + tid] = 0.f; }

    const int total = nframes * C;
    float mg[E], phv[E];
    // element offset of (frame f, channel c, bin b0) in the spectra: advanced incrementally, one (frame, channel) per step
    const int64_t ch_step = (int64_t)g.F * p.Hp;            // next channel, same frame
    const int64_t fr_step = (int64_t)p.Hp - (C - 1) * ch_step;   // channel C-1 of frame f -> channel 0 of frame f+1
    int64_t off_fetch = (int64_t)stream * C * ch_step + b0;
    int c_fetch = 0;
    auto fetch = [&]() {
        const int64_t base = off_fetch;
        if (++c_fetch == C) { c_fetch = 0; off_fetch += fr_step; } else off_fetch += ch_step;
#pragma unroll
        for (int e = 0; e < E; e += 4) {
            const float4 m4 = *(const float4 *)(g.mag + base + e);
            const float4 p4 = *(const float4 *)(g.phase + base + e);
            mg[e] = m4.x; mg[e + 1] = m4.y; mg[e + 2] = m4.z; mg[e + 3] = m4.w;
            phv[e] = p4.x; phv[e + 1] = p4.y; phv[e + 2] = p4.z; phv[e + 3] = p4.w;
        }
    };
    if (total > 0) fetch();
    int64_t off_cur = (int64_t)stream * C * ch_step + b0;
    int f = 0, c = 0;
    const float hopf = (float)p.hop;
    __syncthreads();

    const SliceRec *__restrict__ rec_f = recs + (k0 - recs_base);
    for (int it = 0; it < total; ++it) {
        const float phase_inc = (float)rec_f[f].phase_inc;
        float *pp = s_pp + c * half, *po = s_po + c * half;
        float ph[E], m[E];
#pragma unroll
        for (int e = 0; e < E; ++e) { ph[e] = phv[e]; m[e] = mg[e]; }
#pragma unroll
        for (int e = 0; e < E; e += 4) {
            *(float4 *)(s_mag + 4 + b0 + e) = make_float4(m[e], m[e + 1], m[e + 2], m[e + 3]);
            *(float4 *)(s_ph + b0 + e) = make_float4(ph[e], ph[e + 1], ph[e + 2], ph[e + 3]);
        }
        __syncthreads();   // (A) magnitudes and phases visible
        // peak picking (:587-596): strict +-2 local maxima with 2 <= b <= half-3
        float w[E + 4];
        w[0] = s_mag[4 + b0 - 2]; w[1] = s_mag[4 + b0 - 1];
#pragma unroll
        for (int e = 0; e < E; ++e) w[2 + e] = m[e];
        w[E + 2] = s_mag[4 + b0 + E]; w[E + 3] = s_mag[4 + b0 + E + 1];
        unsigned flags = 0;
        int cnt = 0;
#pragma unroll
        for (int e = 0; e < E; ++e) {
            const int b = b0 + e;
            const bool pk = b >= 2 && b + 2 < half && w[e + 2] > w[e + 1] && w[e + 2] > w[e] && w[e + 2] > w[e + 3] && w[e + 2] > w[e + 4];
            flags |= (unsigned)pk << e;
            cnt += pk;
        }
        int incl = cnt;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += v;
        }
        if (lane == 31) s_wsum[warp] = incl;
        if (it + 1 < total) fetch();   // prefetch the next (frame, channel) while this one is processed
        __syncthreads();   // (B)
        int base = 0, npk = 0;
        for (int wv = 0; wv < nwarp; ++wv) { const int v = s_wsum[wv]; npk += v; if (wv < warp) base += v; }
        base += incl - cnt;   // peaks before this thread's first bin
        {
            int r = base;
#pragma unroll
            for (int e = 0; e < E; ++e) if (flags & (1u << e)) s_cur[r++] = b0 + e;
        }
        float *__restrict__ gph = g.phase + off_cur;
        if (first) {
            // first call of the process: pass the analysis phase through and seed the state (:606-616)
#pragma unroll
            for (int e = 0; e < E; ++e) { pp[b0 + e] = ph[e]; po[b0 + e] = ph[e]; }
            __syncthreads();   // (C) peak list complete
        } else if (npk == 0 || nprev == 0) {
            // classic propagation (:617-636)
            float outv[E];
#pragma unroll
            for (int e = 0; e < E; ++e) {
                const int i = b0 + e;
                const float omega = __ldg(&p.omega[i]);
                const float dphi = (float)__dadd_rn((double)omega, princarg_fast((double)sub3_rn(ph[e], pp[i], omega)));
                const float adv = __fdiv_rn(__fmul_rn(dphi, phase_inc), hopf);
                outv[e] = (float)princarg_fast((double)__fadd_rn(po[i], adv));
                pp[i] = ph[e];
                po[i] = outv[e];
            }
#pragma unroll
            for (int e = 0; e < E; e += 4) *(float4 *)(gph + e) = make_float4(outv[e], outv[e + 1], outv[e + 2], outv[e + 3]);
            __syncthreads();   // (C)
        } else {
            __syncthreads();   // (C) peak list complete
            // one thread per peak of the compacted list: rotation (:641-667) and region start (:668-683)
            for (int r = tid; r < npk; r += nthr) {
                const int p2 = s_cur[r];
                int lo = 0, hi = nprev;  // first previous peak >= p2
                while (lo < hi) { const int mid = (lo + hi) >> 1; if (s_prev[mid] < p2) lo = mid + 1; else hi = mid; }
                int j;
                if (lo == 0) j = 0;
                else if (lo == nprev) j = nprev - 1;
                else j = (s_prev[lo] - p2 < p2 - s_prev[lo - 1]) ? lo : lo - 1;  // ties keep the lower index (:644-652)
                const int p1 = s_prev[j];
                const float php = s_ph[p2];
                const float avg_p = (float)((double)(p1 + p2) * 0.5);
                // (2*pi*hop*(avg_p-1)) / N: N is a power of two, so the division is an exact scaling
                const float pomega = (float)__dmul_rn(__dmul_rn(p.two_pi_hop, (double)__fsub_rn(avg_p, 1.0f)), (double)p.inv_n);
                const float dphi = (float)__dadd_rn((double)pomega, princarg_fast((double)sub3_rn(php, pp[p1], pomega)));
                const float target = (float)princarg_fast((double)__fadd_rn(po[p1], __fdiv_rn(__fmul_rn(dphi, phase_inc), hopf)));
                s_rot[r] = (float)princarg_fast((double)__fsub_rn(target, php));
                s_start[r] = r == 0 ? 0 : (s_cur[r - 1] + p2 + 1) >> 1;  // round((a+b)*0.5), half away from zero
            }
            if (tid == 0) s_start[npk] = half;
            __syncthreads();   // (D) rotations and region starts complete; all reads of the old state are done
            // lock every bin to its region's peak (:685-699); the region of bin b0 is that of the peak before b0 or of the
            // first peak at/after b0, and at most kMaxOwn more regions start inside the thread's bins
            int pk = base < npk ? base : npk - 1;
            if (pk > 0 && s_start[pk] > b0) --pk;
            float outv[E];
#pragma unroll
            for (int e = 0; e < E; ++e) {
                const int i = b0 + e;
                while (s_start[pk + 1] <= i) ++pk;
                outv[e] = (float)princarg_fast((double)__fadd_rn(ph[e], s_rot[pk]));
                pp[i] = ph[e];
                po[i] = outv[e];
            }
#pragma unroll
            for (int e = 0; e < E; e += 4) *(float4 *)(gph + e) = make_float4(outv[e], outv[e + 1], outv[e + 2], outv[e + 3]);
        }
        // the list just built becomes the previous one (shared by the channels of the stream)
        { int *tsw = s_prev; s_prev = s_cur; s_cur = tsw; }
        nprev = npk;
        first = false;
        if (++c == C) { c = 0; ++f; off_cur += fr_step; } else off_cur += ch_step;
        (void)kMaxOwn;
    }
    __syncthreads();
    for (int c = 0; c < C; ++c) {
        const int64_t row = (int64_t)stream * C + c;
        for (int i = tid; i < half; i += nthr) {
            g.prev_phase[row * half + i] = s_pp[c * half + i];
            g.prev_out[row * half + i] = s_po[c * half + i];
        }
    }
    for (int i = tid; i < nprev; i += nthr) gpk[1 + i] = s_prev[i];
    if (tid == 0) { gpk[0] = nprev; g.started[stream] = (total > 0 || !first) ? 1 : 0; }
}

#include "pv_lock.cuh"   // k_lock_peaks / k_lock_chain: the phase-locked core on Cartesian spectra

// coremode 2: phase *= phaseIncrement / hop (two float roundings, :558-572)
__global__ void k_int_ratio(const DevPlan p, const DevRows g, const SliceRec *__restrict__ recs, long recs_base, long k0) {
    const int row = blockIdx.y, f = blockIdx.x;
    float *__restrict__ gph = g.phase + ((int64_t)row * g.F + f) * p.Hp;
    const float phase_inc = (float)recs[k0 + f - recs_base].phase_inc, hopf = (float)p.hop;
    for (int i = threadIdx.x; i < p.half; i += blockDim.x) gph[i] = __fdiv_rn(__fmul_rn(gph[i], phase_inc), hopf);
}

// robotic (zeros) / whisper (table of 2*pi*rand()/RAND_MAX drawn slice-major, channel, bin): all H bins
__global__ void k_fixed_phase(const DevPlan p, const DevRows g, const float *__restrict__ table, long k0) {
    const int row = blockIdx.y, f = blockIdx.x;
    const int c = row % g.channels;
    float *__restrict__ gph = g.phase + ((int64_t)row * g.F + f) * p.Hp;
    const float *__restrict__ t = table ? table + ((int64_t)(k0 + f - g.aux_base) * g.channels + c) * p.H : nullptr;
    for (int i = threadIdx.x; i < p.H; i += blockDim.x) gph[i] = t ? t[i] : 0.f;
}

// ------------------------------------------------------------------------------------------------
// k_synthesise: one CTA per (frame, row)
// ------------------------------------------------------------------------------------------------
__global__ void k_synthesise(const DevPlan p, const DevRows g, const float *__restrict__ car_mag, const float *__restrict__ car_phase, long k0) {
    extern __shared__ float smem[];
    const int N = p.N, nc = p.nc, H = p.H, hs = N / 2;
    float *b0 = smem;                             // 2H floats: mag | phase, later nc complex (pre-pass output)
    float2 *b1 = (float2 *)(smem + 2 * H + 2);    // H complex: packed spectrum, later the FFT workspace
    const int row = blockIdx.y, f = blockIdx.x;
    const long k = k0 + f;
    const float *__restrict__ gmag = g.mag + ((int64_t)row * g.F + f) * p.Hp;
    const float *__restrict__ gph = g.phase + ((int64_t)row * g.F + f) * p.Hp;
    float *s_mag = b0, *s_ph = b0 + H;
    for (int i = threadIdx.x; i < H; i += blockDim.x) { s_mag[i] = gmag[i]; s_ph[i] = gph[i]; }
    __syncthreads();
    const bool vocoder = car_mag != nullptr;
    const int band_len = N / 1024;
    for (int i = threadIdx.x; i < H; i += blockDim.x) {
        float m, ph;
        if (vocoder) {
            // modifySliceVocoder (:755-776): carrier magnitude scaled by the band mean of the input
            m = car_mag[(int64_t)(k - g.aux_base) * p.Hp + i];
            ph = car_phase[(int64_t)(k - g.aux_base) * p.Hp + i];
            if (i == 0 || i == H - 1) {
                m = 0.f;
            } else if (band_len > 0) {
                const int bs = (i / band_len) * band_len;
                float mean = 0.f;
                for (int e = 0; e < band_len; ++e) mean = __fadd_rn(mean, s_mag[bs + e]);
                mean = __fdiv_rn(mean, (float)(band_len * 2));
                m = __fmul_rn(m, mean);
            }
        } else if (p.freq_comp != 0.f) {
            // freqCompSlice (:842-923): both in-place loop orders read only not-yet-overwritten sources,
            // so the warp is a gather from the unmodified spectrum
            if (p.freq_comp > 1.0f || i < hs) {
                const int src = __float2int_rn(__fmul_rn((float)i, p.freq_comp));
                if (src > hs) {
                    m = 0.f; ph = 0.f;
                } else {
                    const float dw = (float)__ddiv_rn(__dmul_rn(p.two_pi_hop, (double)(i - src)), (double)N);
                    m = s_mag[src];
                    ph = __fadd_rn(s_ph[src], dw);
                }
            } else {  // expand direction leaves the Nyquist bin alone
                m = s_mag[i]; ph = s_ph[i];
            }
            m = __fmul_rn(m, p.fixed_gain);
        } else {
            m = s_mag[i]; ph = s_ph[i];
        }
        m = __fmul_rn(m, p.inv_n);
        float sn, cs;
        sincosf(ph, &sn, &cs);
        b1[i] = make_float2(m * cs, m * sn);
    }
    __syncthreads();
    // inverse real-FFT pre-pass (kiss_fftr.c:123-159)
    float2 *tmp = (float2 *)b0;
    for (int kk = threadIdx.x; kk <= nc / 2; kk += blockDim.x) {
        if (kk == 0) {
            tmp[0] = make_float2(b1[0].x + b1[nc].x, b1[0].x - b1[nc].x);
        } else {
            const float2 fk = b1[kk];
            const float2 fq = b1[nc - kk];
            const float2 fnkc = make_float2(fq.x, -fq.y);
            const float2 fek = cadd_rn(fk, fnkc), t = csub_rn(fk, fnkc);
            const float2 fok = cmul_rn(t, __ldg(&p.stw_inv[kk]));
            const float2 a = cadd_rn(fek, fok);
            const float2 b = csub_rn(fek, fok);
            if (kk != nc - kk) tmp[kk] = a;
            tmp[nc - kk] = make_float2(b.x, -b.y);
        }
    }
    __syncthreads();
    for (int o = threadIdx.x; o < nc; o += blockDim.x) b1[o] = tmp[p.perm[o]];
    __syncthreads();
    fft_stages<true>(p, b1);
    // ifftshift + synthesis window (impl.h:183-198, :1052-1056)
    const float *time = (const float *)b1;
    float *__restrict__ out = g.frames + ((int64_t)row * g.Fr + (k % g.Fr)) * N;
    for (int i = threadIdx.x; i < N; i += blockDim.x) out[i] = time[(i + hs) & (N - 1)] * __ldg(&p.window[i]);
}

// ------------------------------------------------------------------------------------------------
// k_synthesise_t<N>: register-tiled version (pv_fft.cuh).  Each thread builds the two packed bins kk and NC-kk straight
// from global memory (the frequency warp and the vocoder modulation are gathers from the unmodified spectrum), writes
// the inverse pre-pass result at its permuted slot, runs the inverse FFT in registers and stores the windowed,
// ifft-shifted frame with 8-byte stores.
// ------------------------------------------------------------------------------------------------
// kLock: Cartesian spectra of the phase-locked core only (g.synth_kind == 4), no other mode's code; kWarp: + the formant /
// gender frequency warp (p.warp_tab)
template <int N, bool kLock, bool kWarp>
__global__ void __launch_bounds__((N / 32 > 256 ? N / 32 : 256), 4) k_synthesise_t(const DevPlan p, const DevRows g, const float *__restrict__ car_mag,
                                                                                 const float *__restrict__ car_phase, long k0, int nf, int total) {
    constexpr int NC = N / 2;
    using S = FftShape<NC>;
    constexpr int T = S::kThreads;
    constexpr int G = (T >= 256) ? 1 : 256 / T;
    extern __shared__ __align__(16) float2 sbuf[];
    const int group = threadIdx.x / T, t = threadIdx.x % T;
    float2 *buf = sbuf + group * S::kPadded;
    const int fid = blockIdx.x * G + group;
    const bool active = fid < total;
    const int row = active ? fid / nf : 0, f = active ? fid % nf : 0;
    const long k = k0 + f;
    if (active) {   // inverse real-FFT pre-pass into the frame's exchange buffer (pv_synth.cuh)
        if (kLock) synth_prepass_lock<N, kWarp>(p, g, row, f, t, buf);
        else synth_prepass_generic<N>(p, g, car_mag, car_phase, row, f, k, t, buf);
    }
    frame_sync<T>(group);
    float2 v[16];
    if (active) fft_frame<NC, true>(v, buf, t, group, p.tw_inv, p.tw2_inv, p.tw3_inv);
    else { if (NC > 256) { frame_sync<T>(group); } frame_sync<T>(group); }
    if (!active) return;
    // ifftshift + synthesis window (impl.h:183-198, :1052-1056): complex output o holds samples 2o, 2o+1 of the
    // un-shifted block; they land at (2o + N/2) mod N
    float *__restrict__ out = g.frames + ((int64_t)row * g.Fr + (k % g.Fr)) * N;
    const float2 *__restrict__ w2 = (const float2 *)p.window;
    // the thread part of the output index never has the NC/2 bit, so the shift by NC/2 only touches the compile-time part
    const int ob = fft_out_base<NC>(t);
    const float2 *__restrict__ wb = w2 + ob;
    float2 *__restrict__ outb = (float2 *)out + ob;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const int oc = fft_out_const<NC>(i) ^ (NC / 2);
        const float2 w = __ldg(&wb[oc]);
        outb[oc] = make_float2(v[i].x * w.x, v[i].y * w.y);
    }
}

// ------------------------------------------------------------------------------------------------
// k_ola_resample: overlap-add + window-sum normalisation (+ the Speex resampler for pitch modes), one CTA per
// (run of consecutive slices, row).
//
// The accumulator of the reference receives frames in slice order starting from zero (:1057-1073) and its first
// shift_k samples are final after slice k (:1152,1185-1190), so position t of the normalised stream is the sum, in slice
// order, of the frames covering t, divided by the data-independent window sum norm[t].  The CTA first builds that stream
// for the span its outputs need (the run's own samples plus the filt_len-1 samples of resampler history before it) in
// shared memory, then either stores it (no resampling) or runs the windowed-sinc interpolation from shared memory
// (resample.c:462-560: four accumulators over filt_len taps, cubic interpolation between table phases).  The sinc table
// is staged as "quads" q[e] = (tab[e-2], tab[e-1], tab[e], tab[e+1]) so one 128-bit shared load feeds the four FMAs.
// ------------------------------------------------------------------------------------------------
constexpr int kOlaMaxSlices = 48;   // run + history slices held in the CTA's tables
constexpr int kOlaMaxFrames = 96;   // frames overlapping them


struct OlaTables {
    int res_rel[kOlaMaxSlices + 1];       // start of each table slice in the normalised stream, relative to u_lo (+ end sentinel)
    int ola_rel[kOlaMaxSlices];           // its OLA position relative to ola_base
    int j0[kOlaMaxSlices];                // first overlapping frame, relative to jmin
    int out_rel[kOlaMaxSlices];           // run slices only: output position relative to the run's first, and how many
    int n_store[kOlaMaxSlices];           //   samples may be stored (n_write clipped by the row's n_out)
    int fr_off[kOlaMaxFrames];            // ola_off of frame (jmin + i) relative to ola_base
    int fr_pos[kOlaMaxFrames];            // slot * N of that frame in the ring
};

template <int OV>   // sinc-table oversampling of the interpolated resampler mode; 0 = direct table or no resampler
__global__ void __launch_bounds__(256, 4) k_ola_resample(const DevPlan p, const DevRows g, const SliceRec *__restrict__ recs, const float *__restrict__ norm,
                                                      int64_t norm_base, long recs_base, long k0, int nf, int run, int max_in, const ResampleRun *__restrict__ runs,
                                                      const unsigned *__restrict__ rs_ent, const float *__restrict__ rs_frac, const unsigned *__restrict__ rs_steps, long run_origin) {
    extern __shared__ float4 smem4[];
    __shared__ OlaTables T;
    __shared__ ResampleRun s_hdr;
    const int row = blockIdx.y;
    const long ka = k0 + (long)blockIdx.x * run;
    const long kb = min(ka + run, k0 + (long)nf);
    const int L = p.rs_active ? (int)p.rs_filt_len : 1;
    const bool quad = p.rs_active && !p.rs_direct;
    float4 *s_quad = smem4;
    // s_in[-L .. 0) stays zero: the resampler's history before the start of a stream (speex mem is zero-initialised)
    float *s_in = (float *)(smem4 + (quad ? p.rs_table_len : 0)) + (p.rs_active ? L : 0);
    const int tid = threadIdx.x;
    if (p.rs_active) for (int i = tid; i < L; i += blockDim.x) s_in[i - L] = 0.f;

    // slices whose normalised samples are needed: the run plus the resampler history before it (every thread walks the
    // few records back; the loads are uniform and cached)
    const int N = p.N;
    const SliceRec *__restrict__ rr = recs - recs_base;
    long kmin, jmin;
    int64_t ola_base, u_lo;
    if (p.rs_active) {   // the host has walked the records (ResampleRun): one load instead of a chain of four
        const ResampleRun *__restrict__ h = &runs[(ka - run_origin) / run];
        kmin = ka - __ldg(&h->back_slices);
        jmin = ka - __ldg(&h->back_frames);
        ola_base = __ldg((const long long *)&h->ola_base);
        u_lo = __ldg((const long long *)&h->u_lo);
    } else {
        const int64_t u_lo_raw = rr[ka].res_off;
        kmin = ka;
        while (kmin > recs_base && kmin > 0 && rr[kmin].res_off > u_lo_raw && ka - kmin < kOlaMaxSlices - run - 1) --kmin;
        jmin = rr[kmin].jlo;
        ola_base = rr[jmin].ola_off;
        u_lo = u_lo_raw < 0 ? 0 : u_lo_raw;
    }
    const int nsl = (int)(kb - kmin);
    const int nfr = min((int)(kb - jmin), kOlaMaxFrames);   // the host's halo check keeps kb - jmin within the table
    const int64_t u_hi = rr[kb - 1].res_off + ((rr[kb - 1].flags & 1) ? 0 : rr[kb - 1].consumed);
    const int span = (int)min(u_hi - u_lo, (int64_t)max_in);
    const int64_t out_first = rr[ka].out_off;
    const int64_t row_limit = g.n_out[row];
    for (int n = tid; n < nsl; n += blockDim.x) {
        const SliceRec &r = rr[kmin + n];
        T.res_rel[n] = (int)(r.res_off - u_lo);
        T.ola_rel[n] = (int)(r.ola_off - ola_base);
        T.j0[n] = (int)(r.jlo - jmin);
        int n_store = (r.flags & 1) ? 0 : r.n_write;
        if (r.out_off + n_store > row_limit) n_store = (int)max((int64_t)0, row_limit - r.out_off);
        T.out_rel[n] = (int)(r.out_off - out_first);
        T.n_store[n] = n_store;
    }
    if (tid == 0) T.res_rel[nsl] = span;
    for (int i = tid; i < nfr; i += blockDim.x) {
        const long j = jmin + i;
        T.fr_off[i] = (int)(rr[j].ola_off - ola_base);
        T.fr_pos[i] = (int)(j % g.Fr) * N;
    }
    if (p.rs_active && tid < (int)(sizeof(ResampleRun) / sizeof(int)))   // this run's work-list header, needed after the overlap-add
        ((int *)&s_hdr)[tid] = ((const int *)&runs[(ka - run_origin) / run])[tid];
    if (quad) {
        const float4 *__restrict__ tab4 = p.rs_quads;   // host-built (tab[e-2], tab[e-1], tab[e], tab[e+1])
        for (int e = tid; e < p.rs_table_len; e += blockDim.x) s_quad[e] = __ldg(&tab4[e]);
    }
    __syncthreads();

    // ---- normalised overlap-add stream for [u_lo, u_hi) ----
    const float *__restrict__ fr = g.frames + (int64_t)row * g.Fr * N;
    const float *__restrict__ nrm = norm + (ola_base - norm_base);
    const int64_t row_out = (int64_t)row * g.out_stride - g.out_base;
    const int first_run_slice = (int)(ka - kmin);
    {
        // One warp per (table slice, 128-sample chunk): the frames covering a slice and their offsets are the same for all of
        // its samples, so the inner loop over the covering frames is warp-uniform and each lane just adds four strided loads.
        const int lane = tid & 31;
        const int nchunk = (max_in / run + 127) >> 7;   // >= ceil(longest slice / 128)
        const int nitem = nsl * nchunk;
        for (int item = tid >> 5; item < nitem; item += blockDim.x >> 5) {
            const int sl = item / nchunk, eb0 = (item - sl * nchunk) << 7;
            const int r0 = T.res_rel[sl];
            const int e_lo = max(r0, 0) + eb0, e_hi = min(T.res_rel[sl + 1], span);   // dropped slices share an offset: empty
            if (e_lo >= e_hi) continue;
            const int rel0 = T.ola_rel[sl] - r0;      // OLA position (relative to ola_base) of normalised sample e is rel0 + e
            const int jb = (int)(kmin - jmin) + sl;
            const int e0 = e_lo + lane;
            float acc[4] = {0.f, 0.f, 0.f, 0.f};
            // the window sums of these samples: fetched now so that their latency hides behind the frame loads
            float nr[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) nr[u] = e0 + 32 * u < e_hi ? __ldg(&nrm[rel0 + e0 + 32 * u]) : 1.f;
            // frames in slice order = the reference's accumulator sequence; four frames' loads are issued together
            for (int j = T.j0[sl]; j <= jb; j += 4) {
                float v[4][4];
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) {
                    const int jc = min(j + jj, jb);
                    const int o = rel0 + e0 - T.fr_off[jc];   // offset of sample e0 inside the frame (never negative)
                    const float *__restrict__ src = fr + (T.fr_pos[jc] + o);
                    const int lim = j + jj <= jb ? N : 0;     // frames past the last one contribute nothing
#pragma unroll
                    for (int u = 0; u < 4; ++u) v[jj][u] = o + 32 * u < lim ? src[32 * u] : 0.f;
                }
#pragma unroll
                for (int jj = 0; jj < 4; ++jj)
#pragma unroll
                    for (int u = 0; u < 4; ++u) acc[u] += v[jj][u];
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int e = e0 + 32 * u;
                if (e >= e_hi) break;
                const float v = acc[u] / nr[u];
                if (p.rs_active) {
                    s_in[e] = v;
                } else if (sl >= first_run_slice && e - r0 < T.n_store[sl]) {
                    // no resampling: the normalised sample is the output sample (n_write / n_out clip)
                    pcm_store(g.out, out_fmt(g), row_out + out_first + T.out_rel[sl] + (e - r0), v);
                }
            }
        }
    }
    if (!p.rs_active) return;
    __syncthreads();

    // ---- resampler ----
    // The host has bucketed the outputs of this run by their table phase (`offset` in resample.c:470), in output order
    // inside a bucket and with buckets starting at multiples of 32 (ResampleRun, pv_kernels.cuh).  A warp therefore
    // works on one phase: the sinc quad of every tap is a single broadcast shared-memory access, and the lanes' input
    // windows are a constant few samples apart (bank-conflict free).
    const ResampleRun &hdr = s_hdr;   // fetched into shared memory at the start of the kernel
    const int64_t orow = row_out + hdr.out_first;
    const int64_t out_limit = g.n_out[row] - hdr.out_first;
    const int in_shift = (int)(hdr.u_lo - u_lo) - kResPad;   // hdr.u_lo == u_lo; entries are biased by kResPad
    (void)out_first;
    resample_run<OV>(p, g, hdr, s_quad, s_in, in_shift, orow, out_limit, rs_ent, rs_frac, rs_steps, L, threadIdx.x >> 5, blockDim.x >> 5);
}

// ------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------
static int fft_threads(const DevPlan &p) {
    int t = p.nc / 4;
    if (t < 64) t = 64;
    if (t > 1024) t = 1024;
    return t;
}

size_t smem_analyse(const DevPlan &p) { return sizeof(float) * 2 * (size_t)p.N; }
size_t smem_synthesise(const DevPlan &p) { return sizeof(float) * ((size_t)2 * p.H + 2 + (size_t)2 * p.H + 2); }
size_t smem_phase_core(const DevPlan &p, int channels, int maxpk) {
    return sizeof(float) * ((size_t)2 * p.Hp + (size_t)2 * channels * p.half + (size_t)4 * maxpk + 1 + 8 + 32 + 8);
}

cudaError_t configure_kernels() {
    cudaError_t e;
    const int big = 200 * 1024;
    if ((e = cudaFuncSetAttribute(k_analyse, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_synthesise, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_ola_resample<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_ola_resample<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_ola_resample<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_ola_resample<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_ola_resample<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_phase_lock_t<4, 256, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_phase_lock_t<4, 512, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_phase_lock_t<8, 512, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return e;
    // (per device: configure_kernels runs for every pipeline's device)
#define PV_LOCK_ATTR(NN) \
    if ((e = cudaFuncSetAttribute(k_lock_peaks<NN, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return e; \
    if ((e = cudaFuncSetAttribute(k_lock_peaks<NN, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return e; \
    if ((e = cudaFuncSetAttribute(k_lock_peaks<NN, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return e;
    PV_LOCK_ATTR(512) PV_LOCK_ATTR(1024) PV_LOCK_ATTR(2048) PV_LOCK_ATTR(4096) PV_LOCK_ATTR(8192)
#undef PV_LOCK_ATTR
    if ((e = cudaFuncSetAttribute(k_lock_chain<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_lock_chain<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_lock_chain<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_phase_core<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_phase_core<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return e;
    return cudaSuccess;
}

template <int N> static void launch_analyse_t(const DevPlan &p, const DevRows &g, long k0, int nframes, cudaStream_t st) {
    using S = FftShape<N / 2>;
    constexpr int T = S::kThreads, G = (T >= 256) ? 1 : 256 / T;
    const int total = nframes * g.rows;
    const int grid = (total + G - 1) / G, block = T >= 256 ? T : 256;
    const size_t sm = sizeof(float2) * G * S::kPadded;
    if (g.spec) {
        if (g.fmt) k_analyse_t<N, true, true><<<grid, block, sm, st>>>(p, g, k0, nframes, total);
        else k_analyse_t<N, false, true><<<grid, block, sm, st>>>(p, g, k0, nframes, total);
    } else {
        if (g.fmt) k_analyse_t<N, true, false><<<grid, block, sm, st>>>(p, g, k0, nframes, total);
        else k_analyse_t<N, false, false><<<grid, block, sm, st>>>(p, g, k0, nframes, total);
    }
}

void launch_analyse(const DevPlan &p, const DevRows &g, long k0, int nframes, cudaStream_t st) {
    switch (p.N) {
        case 512: return launch_analyse_t<512>(p, g, k0, nframes, st);
        case 1024: return launch_analyse_t<1024>(p, g, k0, nframes, st);
        case 2048: return launch_analyse_t<2048>(p, g, k0, nframes, st);
        case 4096: return launch_analyse_t<4096>(p, g, k0, nframes, st);
        case 8192: return launch_analyse_t<8192>(p, g, k0, nframes, st);
        default: break;
    }
    dim3 grid(nframes, g.rows);
    k_analyse<<<grid, fft_threads(p), smem_analyse(p), st>>>(p, g, k0);
}

void launch_phase_core(const DevPlan &p, const DevRows &g, int coremode, const SliceRec *recs, long recs_base, long k0, int nframes, cudaStream_t st) {
    if (coremode == 2) {
        dim3 grid(nframes, g.rows);
        k_int_ratio<<<grid, 256, 0, st>>>(p, g, recs, recs_base, k0);
        return;
    }
    const int streams = g.rows / g.channels;
    if (coremode == 1 && (p.N == 512 || p.N == 1024 || p.N == 2048 || p.N == 4096 || p.N == 8192)) {
        const int E = p.N == 8192 ? 8 : 4;
        const size_t sm = sizeof(float) * ((size_t)2 * p.half + 8 + (size_t)2 * g.channels * p.half + (size_t)4 * g.maxpk + 1 + 32 + 8);
        if (E == 8) k_phase_lock_t<8, 512, 2><<<streams, p.half / 8, sm, st>>>(p, g, recs, recs_base, k0, nframes);
        else if (p.half / 4 > 256) k_phase_lock_t<4, 512, 2><<<streams, p.half / 4, sm, st>>>(p, g, recs, recs_base, k0, nframes);
        else k_phase_lock_t<4, 256, 4><<<streams, p.half / 4, sm, st>>>(p, g, recs, recs_base, k0, nframes);
        return;
    }
    const size_t sm = smem_phase_core(p, g.channels, g.maxpk);
    int threads = p.half / 4;
    if (threads < 64) threads = 64;
    if (threads > 512) threads = 512;
    if (coremode == 1) k_phase_core<true><<<streams, threads, sm, st>>>(p, g, recs, recs_base, k0, nframes);
    else k_phase_core<false><<<streams, threads, sm, st>>>(p, g, recs, recs_base, k0, nframes);
}

size_t lock_smem_bytes(const DevPlan &p, int channels, int maxpk) {
    return std::max(lock_peaks_smem(p.half, channels, maxpk), lock_chain_smem(p.half, channels, maxpk));
}

int lock_rec_stride(const DevPlan &p, int maxpk) { return maxpk > p.half / 2 ? maxpk : p.half / 2; }

template <int N, int kC>
static void launch_lock_peaks_nc(const DevPlan &p, const DevRows &g, const SliceRec *recs, long recs_base, long k0, int nframes, cudaStream_t st) {
    const dim3 grid((nframes + kLockRun - 1) / kLockRun, g.rows / g.channels);
    k_lock_peaks<N, kC><<<grid, LockShape<N>::kThreads, lock_peaks_smem(p.half, g.channels, g.maxpk), st>>>(p, g, recs, recs_base, k0, nframes);
}

template <int N>
static void launch_lock_peaks_n(const DevPlan &p, const DevRows &g, const SliceRec *recs, long recs_base, long k0, int nframes, cudaStream_t st) {
    if (g.channels == 1) launch_lock_peaks_nc<N, 1>(p, g, recs, recs_base, k0, nframes, st);
    else if (g.channels == 2) launch_lock_peaks_nc<N, 2>(p, g, recs, recs_base, k0, nframes, st);
    else launch_lock_peaks_nc<N, 0>(p, g, recs, recs_base, k0, nframes, st);
}

void launch_lock_peaks(const DevPlan &p, const DevRows &g, const SliceRec *recs, long recs_base, long k0, int nframes, cudaStream_t st) {
    switch (p.N) {   // g.spec is only set for these sizes (Pipeline::cartesian)
        case 512: return launch_lock_peaks_n<512>(p, g, recs, recs_base, k0, nframes, st);
        case 1024: return launch_lock_peaks_n<1024>(p, g, recs, recs_base, k0, nframes, st);
        case 2048: return launch_lock_peaks_n<2048>(p, g, recs, recs_base, k0, nframes, st);
        case 4096: return launch_lock_peaks_n<4096>(p, g, recs, recs_base, k0, nframes, st);
        default: return launch_lock_peaks_n<8192>(p, g, recs, recs_base, k0, nframes, st);
    }
}

void launch_lock_chain(const DevPlan &p, const DevRows &g, int nframes, cudaStream_t st) {
    const int streams = g.rows / g.channels;
    const size_t sm = lock_chain_smem(p.half, g.channels, g.maxpk);
    if (g.channels == 1) k_lock_chain<1><<<streams, kChainThreads, sm, st>>>(p, g, nframes);
    else if (g.channels == 2) k_lock_chain<2><<<streams, kChainThreads, sm, st>>>(p, g, nframes);
    else k_lock_chain<0><<<streams, kChainThreads, sm, st>>>(p, g, nframes);
}

void launch_fixed_phase(const DevPlan &p, const DevRows &g, const float *table, long k0, int nframes, cudaStream_t st) {
    dim3 grid(nframes, g.rows);
    k_fixed_phase<<<grid, 256, 0, st>>>(p, g, table, k0);
}

template <int N>
static void launch_synthesise_t(const DevPlan &p, const DevRows &g, const float *car_mag, const float *car_phase, long k0, int nframes, cudaStream_t st) {
    using S = FftShape<N / 2>;
    constexpr int T = S::kThreads, G = (T >= 256) ? 1 : 256 / T;
    const int total = nframes * g.rows;
    const int grid = (total + G - 1) / G, block = T >= 256 ? T : 256;
    const size_t sm = sizeof(float2) * G * S::kPadded;
    if (g.synth_kind == 4 && p.warp_tab != nullptr) k_synthesise_t<N, true, true><<<grid, block, sm, st>>>(p, g, car_mag, car_phase, k0, nframes, total);
    else if (g.synth_kind == 4) k_synthesise_t<N, true, false><<<grid, block, sm, st>>>(p, g, car_mag, car_phase, k0, nframes, total);
    else k_synthesise_t<N, false, false><<<grid, block, sm, st>>>(p, g, car_mag, car_phase, k0, nframes, total);
}

void launch_synthesise(const DevPlan &p, const DevRows &g, const float *car_mag, const float *car_phase, long k0, int nframes, cudaStream_t st) {
    switch (p.N) {
        case 512: return launch_synthesise_t<512>(p, g, car_mag, car_phase, k0, nframes, st);
        case 1024: return launch_synthesise_t<1024>(p, g, car_mag, car_phase, k0, nframes, st);
        case 2048: return launch_synthesise_t<2048>(p, g, car_mag, car_phase, k0, nframes, st);
        case 4096: return launch_synthesise_t<4096>(p, g, car_mag, car_phase, k0, nframes, st);
        case 8192: return launch_synthesise_t<8192>(p, g, car_mag, car_phase, k0, nframes, st);
        default: break;
    }
    dim3 grid(nframes, g.rows);
    k_synthesise<<<grid, fft_threads(p), smem_synthesise(p), st>>>(p, g, car_mag, car_phase, k0);
}

// dst[r * dst_pitch + ((dst_off + i) & dst_mask)] = src[r * src_pitch + ((src_off + i) & src_mask)], i < width: row-wise copy
// with independent pitches and any element alignment; a mask of cap - 1 makes that side a ring of cap elements per row (the
// device-resident output FIFO of a streaming instance), -1 a plain row.  Places the packed new input of a live batch behind the
// rows' device-resident windows (a 2-D cudaMemcpy of 4096 such rows ran at 7 GB/s).  T = float or short (int16 instances).
template <typename T>
__global__ void k_place_rows(T *__restrict__ dst, int64_t dst_pitch, int64_t dst_off, int64_t dst_mask, const T *__restrict__ src, int64_t src_pitch,
                             int64_t src_off, int64_t src_mask, int width) {
    const int r = blockIdx.y;
    const T *__restrict__ s = src + (int64_t)r * src_pitch;
    T *__restrict__ d = dst + (int64_t)r * dst_pitch;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < width; i += gridDim.x * blockDim.x) d[(dst_off + i) & dst_mask] = s[(src_off + i) & src_mask];
}
template <typename T>
void launch_place_rows(T *dst, int64_t dst_pitch, const T *src, int64_t src_pitch, int width, int rows, cudaStream_t st) {
    launch_ring_rows(dst, dst_pitch, 0, -1, src, src_pitch, 0, -1, width, rows, st);
}
template <typename T>
void launch_ring_rows(T *dst, int64_t dst_pitch, int64_t dst_off, int64_t dst_mask, const T *src, int64_t src_pitch, int64_t src_off, int64_t src_mask,
                      int width, int rows, cudaStream_t st) {
    if (width <= 0 || rows <= 0) return;
    dim3 grid((unsigned)std::min(8, (width + 255) / 256), (unsigned)rows);
    k_place_rows<T><<<grid, 256, 0, st>>>(dst, dst_pitch, dst_off, dst_mask, src, src_pitch, src_off, src_mask, width);
}
template void launch_place_rows<float>(float *, int64_t, const float *, int64_t, int, int, cudaStream_t);
template void launch_place_rows<short>(short *, int64_t, const short *, int64_t, int, int, cudaStream_t);
template void launch_ring_rows<float>(float *, int64_t, int64_t, int64_t, const float *, int64_t, int64_t, int64_t, int, int, cudaStream_t);
template void launch_ring_rows<short>(short *, int64_t, int64_t, int64_t, const short *, int64_t, int64_t, int64_t, int, int, cudaStream_t);

int ola_max_table_slices() { return kOlaMaxSlices; }

int ola_run_limit(const DevPlan &p, int run, int max_consumed, int max_out) {
    if (run > kOlaMaxSlices - 16) run = kOlaMaxSlices - 16;
    if (run < 1) run = 1;
    const int L = p.rs_active ? (int)p.rs_filt_len : 1;
    // the packed per-output entry holds two 16-bit fields: keep the span and the output count of a run below 64k - pad;
    // the run's normalised samples (+ history + sinc quads) must fit the 200 KB shared-memory opt-in
    const size_t quad_bytes = (p.rs_active && !p.rs_direct) ? sizeof(float4) * (size_t)p.rs_table_len : 0;
    while (run > 1 && (run * max_consumed + L + 8 + kResPad >= 65536 || run * max_out >= 65535 ||
                       quad_bytes + sizeof(float) * ((size_t)run * max_consumed + 2 * L + 16) > (size_t)196 * 1024)) run /= 2;
    return run;
}

void launch_ola_resample(const DevPlan &p, const DevRows &g, const SliceRec *recs, const float *norm, int64_t norm_base, long recs_base,
                         long k0, int nframes, int run, int max_consumed, const ResampleRun *runs, const unsigned *rs_ent, const float *rs_frac,
                         const unsigned *rs_steps, long run_origin, cudaStream_t st) {
    const int L = p.rs_active ? (int)p.rs_filt_len : 1;
    const bool quad = p.rs_active && !p.rs_direct;
    const int max_in = ((run * max_consumed + L + 8) + 3) & ~3;
    const size_t sm = (quad ? sizeof(float4) * (size_t)p.rs_table_len : 0) + sizeof(float) * (size_t)(max_in + (p.rs_active ? L : 0));
    dim3 grid((nframes + run - 1) / run, g.rows);
#define PV_OLA(OVV) k_ola_resample<OVV><<<grid, 256, sm, st>>>(p, g, recs, norm, norm_base, recs_base, k0, nframes, run, max_in, runs, rs_ent, rs_frac, rs_steps, run_origin)
    if (!quad) PV_OLA(0);
    else if (p.rs_oversample == 8) PV_OLA(8);
    else if (p.rs_oversample == 4) PV_OLA(4);
    else if (p.rs_oversample == 2) PV_OLA(2);
    else PV_OLA(1);
#undef PV_OLA
}

}  // namespace pvgpu

// ------------------------------------------------------------------------------------------------
// unit-test kernels (pvgpu_test_* in include/pvgpu.h)
// ------------------------------------------------------------------------------------------------
namespace pvgpu {
__global__ void k_test_atan2f(int64_t n, const float *__restrict__ y, const float *__restrict__ x, float *__restrict__ out) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) out[i] = pv_atan2f(y[i], x[i]);
}
__global__ void k_test_princarg(int64_t n, const double *__restrict__ a, double *__restrict__ out) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) out[i] = (i & 1) ? princarg_rn(a[i]) : princarg_fast(a[i]);
}
void launch_test_atan2f(int64_t n, const float *y, const float *x, float *out, cudaStream_t st) { k_test_atan2f<<<592, 256, 0, st>>>(n, y, x, out); }
void launch_test_princarg(int64_t n, const double *a, double *out, cudaStream_t st) { k_test_princarg<<<592, 256, 0, st>>>(n, a, out); }
}  // namespace pvgpu
