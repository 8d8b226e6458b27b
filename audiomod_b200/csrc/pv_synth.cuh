// Device pieces shared by the synthesis kernels (k_synthesise_t in pv_kernels.cu, k_synth_ola in pv_fused.cu): PCM
// conversions at the batch boundary and the inverse real-FFT pre-pass that turns a frame's (modified) spectrum into the
// permuted complex input of the register-tiled inverse FFT (pv_fft.cuh).  Reference file:line as in pv_kernels.cu.
#pragma once
#include "pv_fft.cuh"
#include "pv_kernels.cuh"

namespace pvgpu {

// PCM sample formats at the batch boundary.  int16 follows the reference's WAV reader / writer: in = (float)(s * (1.0/32768))
// (main/wavfile.cc:733-752, exact in float), out = (short)(int)clamp(x * 32768.f, -32768, 32767), truncating toward zero
// (wavfile.cc:1294-1306, 1508-1526).
__device__ __forceinline__ float pcm_load(const void *base, int fmt, int64_t idx) {
    return fmt ? (float)((const short *)base)[idx] * (1.0f / 32768.0f) : ((const float *)base)[idx];
}
__device__ __forceinline__ void pcm_store(void *base, int fmt, int64_t idx, float v) {
    if (fmt) {
        float s = __fmul_rn(v, 32768.0f);
        s = s > 32767.0f ? 32767.0f : (s < -32768.0f ? -32768.0f : s);
        ((short *)base)[idx] = (short)(int)s;
    } else {
        ((float *)base)[idx] = v;
    }
}

// format of the samples the resynthesis stores into g.out
__device__ __forceinline__ int out_fmt(const DevRows &g) { return g.out_f32 ? 0 : g.fmt; }

// (magnitude, phase) -> packed bin of the polar pipelines and of the phase-free modes on Cartesian spectra
struct SynthBinLoader {
    const DevPlan &p;
    const float *__restrict__ gmag, *__restrict__ gph, *__restrict__ cmag, *__restrict__ cph;
    const float *__restrict__ wphase;   // whisper phases of this (slice, channel)
    int spec, kind;                     // DevRows::spec / DevRows::synth_kind

    // analysis magnitude of bin i (FFT.cc:2624); with Cartesian spectra it is formed here, with the same operations
    __device__ __forceinline__ float in_mag(int i) const {
        if (!spec) return gmag[i];
        const float r = gmag[i], q = gph[i];
        return __fsqrt_rn(__fadd_rn(__fmul_rn(r, r), __fmul_rn(q, q)));
    }
    // (magnitude before the 1/N scale, phase) of packed bin i after the mode's spectral modification; for the constant
    // mode on Cartesian spectra the pair is (re, im) and finish() only scales it
    __device__ __forceinline__ float2 load(int i) const {
        const int hs = p.half;
        float m, ph;
        if (cmag != nullptr) {  // modifySliceVocoder (:755-776)
            m = cmag[i];
            ph = cph[i];
            const int band_len = p.N / 1024;
            if (i == 0 || i == hs) {
                m = 0.f;
            } else if (band_len > 0) {
                const int bs = (i / band_len) * band_len;
                float mean = 0.f;
                for (int e = 0; e < band_len; ++e) mean = __fadd_rn(mean, in_mag(bs + e));
                m = __fmul_rn(m, __fdiv_rn(mean, (float)(band_len * 2)));
            }
        } else if (kind == 1) {         // roboticSlice (:805-812)
            m = in_mag(i); ph = 0.f;
        } else if (kind == 2) {         // whisperSlice (:814-822)
            m = in_mag(i); ph = wphase[i];
        } else if (kind == 3 && spec) { // constant mode: the spectrum goes back unchanged
            m = gmag[i]; ph = gph[i];
        } else if (p.freq_comp != 0.f) {  // freqCompSlice (:842-923) as a gather
            if (p.freq_comp > 1.0f || i < hs) {
                const int src = __float2int_rn(__fmul_rn((float)i, p.freq_comp));
                if (src > hs) {
                    m = 0.f; ph = 0.f;
                } else {
                    const float dw = (float)__ddiv_rn(__dmul_rn(p.two_pi_hop, (double)(i - src)), (double)p.N);
                    m = gmag[src];
                    ph = __fadd_rn(gph[src], dw);
                }
            } else {
                m = gmag[i]; ph = gph[i];
            }
            m = __fmul_rn(m, p.fixed_gain);
        } else {
            m = gmag[i]; ph = gph[i];
        }
        return make_float2(m, ph);
    }
    // 1/N scale (:1024) and polar -> cartesian (FFT.cc:2711-2721)
    __device__ __forceinline__ float2 finish(float2 mp) const {
        const float m = __fmul_rn(mp.x, p.inv_n);
        if (kind == 1 && cmag == nullptr) return make_float2(m, 0.f);                          // cosf(0) = 1, sinf(0) = 0
        if (kind == 3 && spec && cmag == nullptr) return make_float2(m, __fmul_rn(mp.y, p.inv_n));   // (re, im) / N
        float sn, cs;
        sincosf(mp.y, &sn, &cs);
        return make_float2(m * cs, m * sn);
    }
    __device__ __forceinline__ float2 operator()(int i) const { return finish(load(i)); }
};

// Pre-pass of the phase-locked core on Cartesian spectra (g.synth_kind == 4; kWarp: + the formant / gender frequency warp).
// Bin i of a locked frame is (re, im) * (cos, sin) of its region's rotation (pv_lock.cuh); first and classic frames, and the
// Nyquist bin, go back as they are.  1/N scale (:1024), then the inverse real-FFT pre-pass (kiss_fftr.c:123-159), written at
// the permuted slot of the frame's exchange buffer.  Thread t of the frame's N/32 threads; four pairs per step: all their
// loads are issued before the dependent (cos, sin) gathers.
template <int N, bool kWarp>
__device__ __forceinline__ void synth_prepass_lock(const DevPlan &p, const DevRows &g, int row, int f, int t, float2 *buf) {
    constexpr int NC = N / 2;
    constexpr int T = FftShape<NC>::kThreads;
    const int64_t slot = (int64_t)row * g.F + f;
    const float *__restrict__ gre = g.mag + slot * p.Hp, *__restrict__ gim = g.phase + slot * p.Hp;
    const bool locked = g.lock_hdr[slot].y == 2;
    const unsigned short *__restrict__ lmap = g.lock_map + slot * p.half;
    const float2 *__restrict__ lcsn = g.lock_csn + slot * g.maxpk;
    const float2 *__restrict__ stw = p.stw_inv;
    constexpr int Q = (NC / 2) / T;
    constexpr int U = Q >= 4 ? 4 : Q;
    const int sa = fft_pad(fft_slot_of_input<NC>(t)), sb = fft_pad(fft_slot_of_input<NC>((T - t) & (T - 1)));
    const float inv_n = p.inv_n;
    // formant / gender modes: freqCompSlice (:842-923) as a gather -- target bin i takes the locked bin src(i) turned by
    // 2*pi*hop*(i - src)/N and scaled by the fixed gain; the host tabulates (gain cos, gain sin, src) per target bin
    const float4 *__restrict__ wt = kWarp ? p.warp_tab : nullptr;
    // The loads of a frame form a chain -- frame header (locked or not), bin -> region (lock_map), region -> rotation (lock_csn)
    // -- and a thread has nothing else to do until they are back, so the chain is kept as short as it can be: the region and
    // rotation loads do not wait for the header (they are issued for every frame from clamped indices; a frame that is not
    // locked ignores them), and the region loads of the next group of bins are issued one group ahead.
    const unsigned pk_max = (unsigned)(g.maxpk - 1);
    unsigned ml_n[U], mh_n[U];   // region of this group's bins, loaded one group ahead
    auto src_bins = [&](int q0, int (&sl)[U], int (&sh)[U], float2 (&wl)[U], float2 (&wh)[U]) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int kk = t + T * (q0 + u);
            sl[u] = kk; sh[u] = NC - kk;
            if (kWarp) {
                const float4 a4 = __ldg(&wt[kk]), b4 = __ldg(&wt[NC - kk]);
                sl[u] = __float_as_int(a4.z); sh[u] = __float_as_int(b4.z);
                wl[u] = make_float2(a4.x, a4.y); wh[u] = make_float2(b4.x, b4.y);
            }
        }
    };
    {
        int sl[U], sh[U];
        float2 wl[U], wh[U];
        src_bins(0, sl, sh, wl, wh);
#pragma unroll
        for (int u = 0; u < U; ++u) { ml_n[u] = lmap[min(sl[u], NC - 1)]; mh_n[u] = lmap[min(sh[u], NC - 1)]; }
    }
#pragma unroll 1
    for (int q0 = 0; q0 < Q; q0 += U) {
        float2 lo[U], hi[U];
        int sl[U], sh[U];
        float2 wl[U], wh[U];
        src_bins(q0, sl, sh, wl, wh);
#pragma unroll
        for (int u = 0; u < U; ++u) {
            lo[u] = make_float2(gre[sl[u]], gim[sl[u]]);
            hi[u] = make_float2(gre[sh[u]], gim[sh[u]]);
        }
        {
            // Two dependent gathers per bin (bin -> region -> rotation).  All region loads are issued first, then all rotation
            // loads, unconditionally from clamped indices, and the exceptions are patched afterwards.  Left to itself ptxas may
            // issue each rotation load right behind its own region load to save registers, which serialises the chains
            // (measured after a refactoring that did not change a single instruction of this loop, only their order:
            // long-scoreboard stalls 5.9 -> 12.2 per issue, 50 -> 72 ms); the `tie` below takes that freedom away.  Bin NC (Nyquist) is not part of any region -- the reference leaves its phase alone;
            // without the warp table only the upper bin of kk == 0 is NC, with it a low target bin can have it as source too
            // (factor > 2).
            unsigned ml[U], mh[U], all = 0;
            float2 cl[U], ch[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                ml[u] = min(ml_n[u], pk_max);
                mh[u] = min(mh_n[u], pk_max);
                all |= ml[u] | mh[u];
            }
            // every rotation address depends on every region index (through a mask that is zero at run time, which the compiler
            // cannot know): the 2U region loads are all in flight before the first rotation load can issue
            const unsigned tie = all & (unsigned)g.zero_mask;
#pragma unroll
            for (int u = 0; u < U; ++u) {
                cl[u] = lcsn[ml[u] + tie];
                ch[u] = lcsn[mh[u] + tie];
            }
            if (q0 + U < Q) {   // the next group's regions, behind this group's rotation loads
                int sl2[U], sh2[U];
                float2 wl2[U], wh2[U];
                src_bins(q0 + U, sl2, sh2, wl2, wh2);
#pragma unroll
                for (int u = 0; u < U; ++u) { ml_n[u] = lmap[min(sl2[u], NC - 1)]; mh_n[u] = lmap[min(sh2[u], NC - 1)]; }
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (kWarp && sl[u] >= NC) cl[u] = make_float2(1.f, 0.f);
                if (sh[u] >= NC) ch[u] = make_float2(1.f, 0.f);
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {   // a frame that is not locked keeps its bins as they are (selected, not multiplied by one)
                const float2 rl = make_float2(lo[u].x * cl[u].x - lo[u].y * cl[u].y, lo[u].x * cl[u].y + lo[u].y * cl[u].x);
                const float2 rh = make_float2(hi[u].x * ch[u].x - hi[u].y * ch[u].y, hi[u].x * ch[u].y + hi[u].y * ch[u].x);
                lo[u] = locked ? rl : lo[u];
                hi[u] = locked ? rh : hi[u];
            }
        }
        if (kWarp) {
#pragma unroll
            for (int u = 0; u < U; ++u) {
                lo[u] = make_float2(lo[u].x * wl[u].x - lo[u].y * wl[u].y, lo[u].x * wl[u].y + lo[u].y * wl[u].x);
                hi[u] = make_float2(hi[u].x * wh[u].x - hi[u].y * wh[u].y, hi[u].x * wh[u].y + hi[u].y * wh[u].x);
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int q = q0 + u, kk = t + T * q;
            const float2 fk = make_float2(__fmul_rn(lo[u].x, inv_n), __fmul_rn(lo[u].y, inv_n));
            const float2 fq = make_float2(__fmul_rn(hi[u].x, inv_n), __fmul_rn(hi[u].y, inv_n));
            if (kk == 0) {
                buf[fft_pad(fft_slot_of_input<NC>(0))] = make_float2(fk.x + fq.x, fk.x - fq.x);
            } else {
                const float2 fnkc = make_float2(fq.x, -fq.y);
                const float2 fek = cadd_rn(fk, fnkc), d = csub_rn(fk, fnkc);
                const float2 fok = cmul_rn(d, __ldg(&stw[kk]));
                const float2 a = cadd_rn(fek, fok);
                const float2 b = csub_rn(fek, fok);
                buf[sa + fft_pad(fft_slot_of_input<NC>(T * q))] = a;
                buf[sb + (t == 0 ? fft_pad(fft_slot_of_input<NC>((T * (16 - q)) & (NC - 1))) : fft_pad(fft_slot_of_input<NC>(T * (15 - q))))] =
                    make_float2(b.x, -b.y);
            }
        }
    }
    if (t == 0) {   // kk == NC/2 pairs with itself; the reference's second write wins (kiss_fftr.c:150-155)
        int src = NC / 2;
        float2 w = make_float2(1.f, 0.f);
        if (kWarp) { const float4 a4 = __ldg(&wt[NC / 2]); src = __float_as_int(a4.z); w = make_float2(a4.x, a4.y); }
        float2 fk = make_float2(gre[src], gim[src]);
        if (locked && src < NC) {
            const float2 cs = lcsn[lmap[src]];
            fk = make_float2(fk.x * cs.x - fk.y * cs.y, fk.x * cs.y + fk.y * cs.x);
        }
        if (kWarp) fk = make_float2(fk.x * w.x - fk.y * w.y, fk.x * w.y + fk.y * w.x);
        fk = make_float2(__fmul_rn(fk.x, inv_n), __fmul_rn(fk.y, inv_n));
        const float2 fnkc = make_float2(fk.x, -fk.y);
        const float2 fek = cadd_rn(fk, fnkc), d = csub_rn(fk, fnkc);
        const float2 fok = cmul_rn(d, __ldg(&stw[NC / 2]));
        const float2 b = csub_rn(fek, fok);
        buf[fft_pad(fft_slot_of_input<NC>(NC / 2))] = make_float2(b.x, -b.y);
    }
}

// Pre-pass of every other mode (polar spectra from the phase kernels; robotic / whisper / vocoder / constant on Cartesian
// spectra): each thread builds the two packed bins kk and NC-kk straight from global memory (the frequency warp and the
// vocoder modulation are gathers from the unmodified spectrum).
template <int N>
__device__ __forceinline__ void synth_prepass_generic(const DevPlan &p, const DevRows &g, const float *__restrict__ car_mag, const float *__restrict__ car_phase,
                                                      int row, int f, long k, int t, float2 *buf) {
    constexpr int NC = N / 2;
    constexpr int T = FftShape<NC>::kThreads;
    const int64_t so = ((int64_t)row * g.F + f) * p.Hp;
    const int64_t co = (int64_t)(k - g.aux_base) * p.Hp;
    const float *wph = g.whisper ? g.whisper + ((int64_t)(k - g.aux_base) * g.channels + row % g.channels) * p.H : nullptr;
    const SynthBinLoader bin{p, g.mag + so, g.phase + so, car_mag ? car_mag + co : nullptr, car_mag ? car_phase + co : nullptr, wph, g.spec, g.synth_kind};
    const float2 *__restrict__ stw = p.stw_inv;
    // inverse real-FFT pre-pass (kiss_fftr.c:123-159).  All loads of the thread's bins are issued before any of the
    // (long) sincos evaluations so their latency overlaps.
    constexpr int Q = (NC / 2) / T;
    const int sa = fft_pad(fft_slot_of_input<NC>(t)), sb = fft_pad(fft_slot_of_input<NC>((T - t) & (T - 1)));
    // rolled in groups of two pairs: four independent loads in flight per step without unrolling the (large) sincos
    // expansion 16 times, which would not fit the instruction cache
#pragma unroll 1
    for (int q0 = 0; q0 < Q; q0 += 2) {
        float2 lo[2], hi[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            lo[u] = bin.load(t + T * (q0 + u));
            hi[u] = bin.load(NC - (t + T * (q0 + u)));
        }
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int q = q0 + u, kk = t + T * q;
            const float2 fk = bin.finish(lo[u]);
            const float2 fq = bin.finish(hi[u]);
            if (kk == 0) {
                buf[fft_pad(fft_slot_of_input<NC>(0))] = make_float2(fk.x + fq.x, fk.x - fq.x);
            } else {
                const float2 fnkc = make_float2(fq.x, -fq.y);
                const float2 fek = cadd_rn(fk, fnkc), d = csub_rn(fk, fnkc);
                const float2 fok = cmul_rn(d, __ldg(&stw[kk]));
                const float2 a = cadd_rn(fek, fok);
                const float2 b = csub_rn(fek, fok);
                // slot(t + T*q) = slot(t) | slot(T*q) and the padded position is additive (see k_analyse_t)
                buf[sa + fft_pad(fft_slot_of_input<NC>(T * q))] = a;
                buf[sb + (t == 0 ? fft_pad(fft_slot_of_input<NC>((T * (16 - q)) & (NC - 1))) : fft_pad(fft_slot_of_input<NC>(T * (15 - q))))] =
                    make_float2(b.x, -b.y);
            }
        }
    }
    if (t == 0) {   // kk == NC/2 pairs with itself; the reference's second write wins (kiss_fftr.c:150-155)
        const float2 fk = bin(NC / 2);
        const float2 fnkc = make_float2(fk.x, -fk.y);
        const float2 fek = cadd_rn(fk, fnkc), d = csub_rn(fk, fnkc);
        const float2 fok = cmul_rn(d, __ldg(&stw[NC / 2]));
        const float2 b = csub_rn(fek, fok);
        buf[fft_pad(fft_slot_of_input<NC>(NC / 2))] = make_float2(b.x, -b.y);
    }
}

}  // namespace pvgpu
