// Host engine + C ABI (include/pvgpu.h) over the kernels in pv_kernels.cu.
//
// The reference processes one stream, slice by slice, on one CPU thread
// (src/phasevocoder/phasevocoderimpl.cc:340-369 -> phasevocoderprocess.cc:236-376).  Here the
// data-independent part of that loop (pv_plan.cc) runs once on the host, and the data-dependent part runs as
// kernels over [rows x frames] tiles; only the phase recursion is serial in time.
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <condition_variable>
#include <exception>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <type_traits>
#include <vector>

#include "../../include/pvgpu.h"
#include "pv_internal.h"
#include "pv_kernels.cuh"
#include "pv_plan.h"

#ifndef M_PI
#define M_PI 3.14159265358979323846
#endif

namespace pvgpu {

static thread_local std::string g_err;
const std::string &last_error_string() { return g_err; }
int fail(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}
// No exception may cross the C ABI (std::vector / std::map growth can throw): entry points run their bodies through this.
template <class F> static int guarded(F f) {
    try {
        return f();
    } catch (const std::bad_alloc &) {
        return fail(PVGPU_ENOMEM, "out of host memory");
    } catch (const std::exception &e) {
        return fail(PVGPU_ESTATE, "unexpected failure: %s", e.what());
    }
}
#define CU(call)                                                                                      \
    do {                                                                                              \
        cudaError_t e_ = (call);                                                                      \
        if (e_ != cudaSuccess) return fail(e_ == cudaErrorMemoryAllocation ? PVGPU_ENOMEM : PVGPU_ECUDA, \
                                           "%s: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

// RAII device buffer
struct DevBuf {
    void *p = nullptr;
    size_t bytes = 0;
    ~DevBuf() { release(); }
    void release() { if (p) cudaFree(p); p = nullptr; bytes = 0; }
    cudaError_t ensure(size_t n) {
        if (n <= bytes) return cudaSuccess;
        release();
        cudaError_t e = cudaMalloc(&p, n);
        if (e == cudaSuccess) bytes = n;
        return e;
    }
    template <typename T> T *as() const { return (T *)p; }
};

// Page-locked staging area of a streaming instance: everything one pvgpu_process call uploads (new input, slice records,
// normalisers, resampler work lists) is copied here first so that the H2D copies are truly asynchronous and the call needs a
// single synchronisation, and the call's output comes back through it.  Bump allocation, reset once per call.
struct PinnedArena {
    char *base = nullptr;
    size_t cap = 0, used = 0;
    ~PinnedArena() { if (base) cudaFreeHost(base); }
    // only between calls (nothing in flight): make room for at least `bytes`
    void reserve(size_t bytes) {
        used = 0;
        if (bytes <= cap) return;
        if (base) cudaFreeHost(base);
        base = nullptr; cap = 0;
        const size_t want = bytes + bytes / 2 + 4096;
        if (cudaHostAlloc((void **)&base, want, cudaHostAllocDefault) == cudaSuccess) cap = want;
        else { cudaGetLastError(); base = nullptr; }
    }
    void *take(size_t bytes) {
        bytes = (bytes + 63) & ~(size_t)63;
        if (!base || used + bytes > cap) return nullptr;
        void *p = base + used;
        used += bytes;
        return p;
    }
};

static Config to_config(const pvgpu_config &c) {
    Config k;
    k.sample_rate = c.sample_rate; k.channels = c.channels; k.time_ratio = c.time_ratio; k.pitch_semitones = c.pitch_semitones;
    k.mode = c.mode; k.coremode = c.coremode; k.fftsize = c.fftsize; k.hopsize = c.hopsize;
    return k;
}

static int validate(const pvgpu_config *cfg) {
    if (!cfg) return fail(PVGPU_EINVAL, "null config");
    if (cfg->channels < 1 || cfg->channels > 16) return fail(PVGPU_EINVAL, "channels must be 1..16");
    if (cfg->sample_rate < 1000) return fail(PVGPU_EINVAL, "sample_rate too small");
    if (cfg->fftsize < 16 || cfg->fftsize > 16384) return fail(PVGPU_EINVAL, "fftsize must be 16..16384");
    return PVGPU_OK;
}

static void fill_info(const Derived &d, pvgpu_info *info) {
    info->fftsize = d.N; info->hop = d.hop; info->bins = d.H;
    info->pitch_scale = d.pitch_scale; info->hs_ratio = d.hs;
    info->resampler_active = d.rs.active ? 1 : 0;
    info->resampler_filt_len = (int)d.rs.filt_len;
    info->resampler_num = d.rs.num; info->resampler_den = d.rs.den;
    info->outbuf_capacity = d.outbuf_cap;
}

// ------------------------------------------------------------------------------------------------
// Pipeline: device tables + launch sequence for a range of frames
// ------------------------------------------------------------------------------------------------
struct Pipeline {
    Derived d;
    Tables t;
    DevPlan p{};
    int device = 0;
    DevBuf b_window, b_twf, b_twi, b_stwf, b_stwi, b_perm, b_omega, b_rstab, b_rsquad, b_warp, b_tw2f, b_tw2i, b_tw3f, b_tw3i;
    // schedule on the device
    DevBuf b_recs, b_norm, b_whisper, b_carmag, b_carph;
    long recs_base = 0, recs_count = 0;
    int64_t norm_base = 0;
    int max_consumed = 1;   // largest per-slice contribution to the normalised stream seen so far
    int max_out = 1;        // largest per-slice output count seen so far
    int ola_run = 16;       // slices per CTA of k_ola_resample (upper bound)
    // fused inverse FFT + overlap-add + resampler (pv_fused.cu) instead of k_synthesise_t -> frame ring -> k_ola_resample
    bool fused = false;
    // Which resynthesis back end: -1 automatic (the split kernels, which are the faster ones on B200 -- profiles/r02_summary.md --
    // unless the schedule overlaps more frames / history slices than their per-CTA tables hold, then the fused kernel, which
    // has no such limit), 0 split only, 1 fused wherever the FFT size has one.  PVGPU_FUSED=0/1 overrides for every instance.
    int fused_pref = -1;
    PostChain post{};           // FFT-free effects applied to the output columns a chunk completes (pv_post.cu); n == 0: none
    FusedArgs fa{};             // run / ring / window shape; per-launch fields are filled in run_synth_ola
    // host copy of the uploaded records + the resampler work lists built from them (ResampleRun, pv_kernels.cuh)
    std::vector<SliceRec> h_recs;
    DevBuf b_runs, b_rsent, b_rsfrac, b_rssteps;
    long run_origin = 0;
    int table_run = 1;
    int64_t launches = 0;
    // optional per-kernel timing with CUDA events on the launching stream
    bool profile = false;
    struct Span { int kind; cudaEvent_t a, b; };
    std::vector<Span> spans;
    size_t spans_used = 0;
    double kind_ms[8] = {0};
    int64_t kind_n[8] = {0};

    ~Pipeline() { for (auto &sp : spans) { cudaEventDestroy(sp.a); cudaEventDestroy(sp.b); } }

    Span *span_begin(int kind, cudaStream_t st) {
        if (!profile) return nullptr;
        if (spans_used == spans.size()) {
            Span sp{kind, nullptr, nullptr};
            if (cudaEventCreate(&sp.a) != cudaSuccess || cudaEventCreate(&sp.b) != cudaSuccess) return nullptr;
            spans.push_back(sp);
        }
        Span *sp = &spans[spans_used++];
        sp->kind = kind;
        cudaEventRecord(sp->a, st);
        return sp;
    }
    static void span_end(Span *sp, cudaStream_t st) { if (sp) cudaEventRecord(sp->b, st); }
    // after the stream has been synchronised: fold the recorded spans into kind_ms / kind_n
    void collect_spans() {
        for (size_t i = 0; i < spans_used; ++i) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, spans[i].a, spans[i].b) == cudaSuccess) { kind_ms[spans[i].kind] += ms; kind_n[spans[i].kind] += 1; }
        }
        spans_used = 0;
    }

    int init(const pvgpu_config &cfg) {
        int ndev = 0;
        if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(PVGPU_ECUDA, "no CUDA device: the phase vocoder has no CPU fallback");
        if (cfg.device < 0 || cfg.device >= ndev) return fail(PVGPU_EINVAL, "device %d out of range (%d devices)", cfg.device, ndev);
        device = cfg.device;
        CU(cudaSetDevice(device));
        d = derive(to_config(cfg));
        if (d.hop < 1 || d.hop > d.N) return fail(PVGPU_EINVAL, "derived hop %d invalid for fft size %d", d.hop, d.N);
        t = make_tables(d.N, d.hop);
        if ((int)t.radix.size() > kMaxStages) return fail(PVGPU_EINVAL, "fft size too large");
        if (d.cepstral && !(d.N == 512 || d.N == 1024 || d.N == 2048 || d.N == 4096 || d.N == 8192))
            return fail(PVGPU_EINVAL, "the cepstral modes need an FFT size of 512..8192 (got %d)", d.N);
        CU(configure_kernels());
        p.N = d.N; p.H = d.H; p.half = d.N / 2; p.nc = d.N / 2; p.hop = d.hop;
        p.Hp = (d.H + 3) & ~3;
        p.nstages = (int)t.radix.size();
        for (int i = 0; i < p.nstages; ++i) { p.radix[i] = t.radix[i]; p.span[i] = t.span[i]; }
        p.inv_n = 1.f / d.N;
        p.two_pi_hop = 2 * M_PI * (size_t)d.hop;
        p.freq_comp = d.freq_comp;
        p.fixed_gain = d.fixed_gain;
        p.rs_active = (d.rs.active && !d.vocoder) ? 1 : 0;
        p.rs_direct = d.rs.direct ? 1 : 0;
        p.rs_num = d.rs.num; p.rs_den = d.rs.den; p.rs_filt_len = d.rs.filt_len; p.rs_oversample = d.rs.oversample;
        p.rs_int_adv = d.rs.int_adv; p.rs_frac_adv = d.rs.frac_adv;
        p.rs_table_len = (int)d.rs.table.size();
        if (!(d.robotic || d.whisper || d.vocoder || d.constant_mode) && d.cfg.coremode != 2 &&
            !(d.cfg.coremode == 1 && lock_smem_bytes(p, d.cfg.channels, max_peaks()) <= (size_t)200 * 1024) &&
            smem_phase_core(p, d.cfg.channels, max_peaks()) + 64 > (size_t)200 * 1024)
            return fail(PVGPU_EINVAL, "%d channels at FFT size %d need more shared memory per stream than the device has (the phase core keeps every channel's phase state on chip)",
                        d.cfg.channels, d.N);
        int rc;
        if ((rc = upload(b_window, t.window.data(), sizeof(float) * t.window.size()))) return rc;
        if ((rc = upload(b_twf, t.tw_fwd.data(), sizeof(float) * t.tw_fwd.size()))) return rc;
        if ((rc = upload(b_twi, t.tw_inv.data(), sizeof(float) * t.tw_inv.size()))) return rc;
        if ((rc = upload(b_stwf, t.stw_fwd.data(), sizeof(float) * t.stw_fwd.size()))) return rc;
        if ((rc = upload(b_stwi, t.stw_inv.data(), sizeof(float) * t.stw_inv.size()))) return rc;
        if ((rc = upload(b_perm, t.perm.data(), sizeof(uint16_t) * t.perm.size()))) return rc;
        if ((rc = upload(b_omega, t.omega.data(), sizeof(float) * t.omega.size()))) return rc;
        if (p.rs_active && (rc = upload(b_rstab, d.rs.table.data(), sizeof(float) * d.rs.table.size()))) return rc;
        p.window = b_window.as<float>();
        p.tw_fwd = b_twf.as<float2>(); p.tw_inv = b_twi.as<float2>();
        p.tw2_fwd = p.tw2_inv = p.tw3_fwd = p.tw3_inv = nullptr;
        {   // per-pass twiddle tables of the register-tiled FFT (pv_fft.cuh): the KissFFT twiddles in [entry][k] order
            const int nc = d.N / 2;
            if (nc == 256 || nc == 512 || nc == 1024 || nc == 2048 || nc == 4096) {
                const bool r2 = nc == 512 || nc == 2048;
                const int mid = r2 ? 8 : 16, last = mid * 16, T = nc / 16;
                auto pair_table = [&](const std::vector<float> &tw, int M) {
                    std::vector<float> out((size_t)2 * 15 * M);
                    const int Fa = nc / (4 * M), Fb = nc / (16 * M);
                    for (int k = 0; k < M; ++k) {
                        int idx[15] = {k * Fa, 2 * k * Fa, 3 * k * Fa};
                        for (int j1 = 0; j1 < 4; ++j1) { const int kk = k + j1 * M; idx[3 + 3 * j1] = kk * Fb; idx[4 + 3 * j1] = 2 * kk * Fb; idx[5 + 3 * j1] = 3 * kk * Fb; }
                        for (int e = 0; e < 15; ++e) { out[2 * ((size_t)e * M + k)] = tw[2 * idx[e]]; out[2 * ((size_t)e * M + k) + 1] = tw[2 * idx[e] + 1]; }
                    }
                    return out;
                };
                auto single_table = [&](const std::vector<float> &tw) {
                    std::vector<float> out((size_t)2 * 12 * T);
                    for (int t = 0; t < T; ++t)
                        for (int q = 0; q < 4; ++q)
                            for (int m = 1; m <= 3; ++m) {
                                const int idx = m * (t + T * q);
                                const size_t o = (size_t)(3 * q + m - 1) * T + t;
                                out[2 * o] = tw[2 * idx]; out[2 * o + 1] = tw[2 * idx + 1];
                            }
                    return out;
                };
                const std::vector<float> f2 = pair_table(t.tw_fwd, mid), i2 = pair_table(t.tw_inv, mid);
                if ((rc = upload(b_tw2f, f2.data(), sizeof(float) * f2.size()))) return rc;
                if ((rc = upload(b_tw2i, i2.data(), sizeof(float) * i2.size()))) return rc;
                p.tw2_fwd = b_tw2f.as<float2>(); p.tw2_inv = b_tw2i.as<float2>();
                if (nc / last == 16 || nc / last == 4) {
                    const std::vector<float> f3 = nc / last == 16 ? pair_table(t.tw_fwd, last) : single_table(t.tw_fwd);
                    const std::vector<float> i3 = nc / last == 16 ? pair_table(t.tw_inv, last) : single_table(t.tw_inv);
                    if ((rc = upload(b_tw3f, f3.data(), sizeof(float) * f3.size()))) return rc;
                    if ((rc = upload(b_tw3i, i3.data(), sizeof(float) * i3.size()))) return rc;
                    p.tw3_fwd = b_tw3f.as<float2>(); p.tw3_inv = b_tw3i.as<float2>();
                }
            }
        }
        p.stw_fwd = b_stwf.as<float2>(); p.stw_inv = b_stwi.as<float2>();
        p.perm = b_perm.as<uint16_t>();
        p.omega = b_omega.as<float>();
        p.rs_table = b_rstab.as<float>();
        if (p.rs_active && !d.rs.direct) {
            const std::vector<float> &tab = d.rs.table;
            const int n = (int)tab.size();
            std::vector<float> quads((size_t)4 * n);
            for (int e = 0; e < n; ++e) {
                quads[4 * e + 0] = e >= 2 ? tab[e - 2] : 0.f;
                quads[4 * e + 1] = e >= 1 ? tab[e - 1] : 0.f;
                quads[4 * e + 2] = tab[e];
                quads[4 * e + 3] = e + 1 < n ? tab[e + 1] : 0.f;
            }
            if ((rc = upload(b_rsquad, quads.data(), sizeof(float) * quads.size()))) return rc;
        }
        p.rs_quads = b_rsquad.as<float4>();
        p.warp_tab = nullptr;
        if (cartesian() && cartesian_lock() && d.freq_comp != 0.f) {
            // freqCompSlice (phasevocoderprocess.cc:842-923) for the Cartesian pipeline: target bin i = gain * locked bin src(i)
            // turned by delta_omega = 2*pi*hop*(i - src)/N (double expression narrowed to float like the reference's data_type)
            const int half = d.N / 2;
            std::vector<float> tab((size_t)4 * (half + 1));
            for (int i = 0; i <= half; ++i) {
                float wr = d.fixed_gain, wi = 0.f;
                int src = i;
                if (d.freq_comp > 1.0f || i < half) {   // the expanding direction leaves the Nyquist bin alone
                    src = (int)std::lrint((float)i * d.freq_comp);
                    if (src > half) { src = 0; wr = 0.f; wi = 0.f; }
                    else {
                        const float dw = (float)((2 * M_PI * (size_t)d.hop * (i - src)) / (double)d.N);
                        wr = (float)(d.fixed_gain * std::cos((double)dw)); wi = (float)(d.fixed_gain * std::sin((double)dw));
                    }
                }
                tab[4 * i] = wr; tab[4 * i + 1] = wi; std::memcpy(&tab[4 * i + 2], &src, sizeof src); tab[4 * i + 3] = 0.f;
            }
            if ((rc = upload(b_warp, tab.data(), sizeof(float) * tab.size()))) return rc;
            p.warp_tab = b_warp.as<float4>();
        }
        return PVGPU_OK;
    }

    // H2D on `st`: through the instance's pinned arena when there is one (asynchronous, the source may be a temporary),
    // else straight from the caller's memory -- then the caller must synchronise before the source goes away (staged_all)
    PinnedArena *arena = nullptr;
    bool staged_all = true;
    int h2d(void *dst, const void *src, size_t bytes, cudaStream_t st) {
        if (!bytes) return PVGPU_OK;
        void *pin = arena ? arena->take(bytes) : nullptr;
        if (pin) { std::memcpy(pin, src, bytes); src = pin; } else staged_all = false;
        CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st));
        return PVGPU_OK;
    }
    // work-list scratch of build_resample_runs (members so that a streaming instance does not allocate per call)
    struct RunScratch {
        std::vector<ResampleRun> runs;
        std::vector<unsigned> ent, steps, run_steps, be[kMaxBuckets], e2;
        std::vector<float> frac, coef, bf[kMaxBuckets], f2;
    } rsx;

    static int upload(DevBuf &b, const void *src, size_t bytes) {
        CU(b.ensure(bytes ? bytes : 4));
        if (bytes) CU(cudaMemcpy(b.p, src, bytes, cudaMemcpyHostToDevice));
        return PVGPU_OK;
    }

    int max_peaks() const { return p.half / 3 + 2; }

    // Modes that never use the analysis phase keep Cartesian spectra (no sqrtf / atan2f per bin in the analysis kernel); only
    // the templated FFT sizes have that variant.
    // The phase-locked core (coremode 1) of the shift / stretch / formant / gender modes also runs on Cartesian spectra
    // (pv_lock.cuh): locking a region is one rotation of its bins, and the analysis phase is only ever needed at the peaks.
    bool cartesian_lock() const {
        if (!(d.cfg.coremode == 1 && !(d.robotic || d.whisper || d.vocoder || d.constant_mode))) return false;
        // the split kernels keep per-channel spectra and maps of a stream in shared memory: with many channels at large FFT
        // sizes that exceeds the 200 KB opt-in, and the serial polar core (k_phase_lock_t) takes over
        return lock_smem_bytes(p, d.cfg.channels, max_peaks()) <= (size_t)200 * 1024;
    }
    bool cartesian() const {
        const bool templated = p.N == 512 || p.N == 1024 || p.N == 2048 || p.N == 4096 || p.N == 8192;
        return templated && (d.robotic || d.whisper || d.vocoder || d.constant_mode || cartesian_lock());
    }
    void apply_mode(DevRows &g) const {
        g.spec = cartesian() ? 1 : 0;
        g.synth_kind = d.vocoder ? 0 : d.robotic ? 1 : d.whisper ? 2 : d.constant_mode ? 3 : cartesian_lock() ? 4 : 0;
        g.whisper = (d.whisper && cartesian()) ? b_whisper.as<float>() : nullptr;
        if (!cartesian()) g.synth_kind = 0;   // polar spectra: k_fixed_phase has already written the phases
    }

    // Upload the slice records [first, first+count) and the normalisers from norm_first on.
    int upload_schedule(const Scheduler &s, cudaStream_t st) {
        const auto &recs = s.recs();
        const auto &norm = s.norm();
        CU(b_recs.ensure(sizeof(SliceRec) * std::max<size_t>(recs.size(), 1)));
        CU(b_norm.ensure(sizeof(float) * std::max<size_t>(norm.size(), 1)));
        int rc;
        if ((rc = h2d(b_recs.p, recs.data(), sizeof(SliceRec) * recs.size(), st))) return rc;
        if ((rc = h2d(b_norm.p, norm.data(), sizeof(float) * norm.size(), st))) return rc;
        recs_base = s.recs_base();
        recs_count = (long)recs.size();
        norm_base = s.norm_base();
        for (const SliceRec &r : recs) { max_consumed = std::max(max_consumed, std::max(r.consumed, r.shift_inc)); max_out = std::max(max_out, r.n_res); }
        h_recs = recs;
        return PVGPU_OK;
    }

    // Work lists of k_ola_resample for slices [origin, end) in runs of `run` slices (launches must start at
    // origin + multiple of run).  Output positions follow the reference's stepping (resample.c:548-554).
    int build_resample_runs(long origin, long end, int run, cudaStream_t st) {
        run_origin = origin;
        table_run = run;
        if (!p.rs_active) return PVGPU_OK;
        const int L = (int)p.rs_filt_len, ov = (int)p.rs_oversample, nb = p.rs_direct ? 1 : ov;
        if (L > kResPad) return fail(PVGPU_EINVAL, "resampler filter of %d taps is not supported (max %d)", L, kResPad);
        std::vector<ResampleRun> &runs = rsx.runs;
        std::vector<unsigned> &ent = rsx.ent, &steps = rsx.steps, &run_steps = rsx.run_steps;
        std::vector<float> &frac = rsx.frac;
        std::vector<unsigned> (&be)[kMaxBuckets] = rsx.be;
        std::vector<float> (&bf)[kMaxBuckets] = rsx.bf;
        runs.clear(); ent.clear(); frac.clear(); steps.clear(); run_steps.clear();
        for (long ka = origin; ka < end; ka += run) {
            const long kb = std::min<long>(ka + run, end);
            const SliceRec &ra = h_recs[ka - recs_base];
            ResampleRun hdr{};
            hdr.u_lo = std::max<int64_t>(0, ra.res_off + ra.rs_last - L + 1);
            hdr.out_first = ra.out_off;
            hdr.ent_off = (int)ent.size();
            {   // the walk k_ola_resample does over the records (same bounds), done once here
                const int64_t u_lo_raw = ra.res_off + ra.rs_last - L + 1;
                long kmin = ka;
                while (kmin > recs_base && kmin > 0 && h_recs[kmin - recs_base].res_off > u_lo_raw && ka - kmin < ola_max_table_slices() - run - 1) --kmin;
                const long jmin = h_recs[kmin - recs_base].jlo;
                hdr.back_slices = (int)(ka - kmin);
                hdr.back_frames = (int)(ka - jmin);
                hdr.ola_base = h_recs[jmin - recs_base].ola_off;
            }
            for (int q = 0; q < nb; ++q) { be[q].clear(); bf[q].clear(); }
            for (long k = ka; k < kb; ++k) {
                const SliceRec &r = h_recs[k - recs_base];
                if (r.flags & 1) continue;
                int last = r.rs_last;
                uint32_t fn = r.rs_frac;
                for (int i = 0; i < r.n_write; ++i) {
                    const int bucket = p.rs_direct ? 0 : (int)(fn * (uint32_t)ov / p.rs_den);
                    const int64_t rel = r.res_off + last - L + 1 - hdr.u_lo + kResPad;
                    const int64_t orel = r.out_off - hdr.out_first + i;
                    if (rel < 0 || rel > 65535 || orel > 65534) return fail(PVGPU_ESTATE, "resampler run does not fit its packed work list");
                    be[bucket].push_back(((unsigned)rel << 16) | (unsigned)orel);
                    float fv;
                    if (p.rs_direct) { std::memcpy(&fv, &fn, sizeof fv); }
                    else fv = ((float)((fn * (uint32_t)ov) % p.rs_den)) / p.rs_den;
                    bf[bucket].push_back(fv);
                    last += p.rs_int_adv;
                    fn += (uint32_t)p.rs_frac_adv;
                    if (fn >= p.rs_den) { fn -= p.rs_den; ++last; }
                }
            }
            int pos = 0;
            for (int q = 0; q < nb; ++q) {
                // A warp step takes kResBlock consecutive entries as kResPerThread rows of 32 lanes, and a row's 32 input windows are
                // read with one shared-memory load per tap: permute the entries (two blocks at a time) so that the windows of a row
                // start on different banks (start mod 32) as far as possible.  The order of the entries is otherwise free (each carries its
                // output position).  Measured before: 1.9 wavefronts per load instead of 1 (the starts advance by 3, 3, 2, ...).
                if (!p.rs_direct) {
                    std::vector<unsigned> &e = be[q];
                    std::vector<float> &f = bf[q];
                    // Entries permuted together: the whole bucket of the run when it fits (a row can only be conflict-free if every bank
                    // still has an entry left, so the pool must be large against the 32 banks: simulated for +7 st, wavefronts per load
                    // 1.60 / 1.27 / 1.13 for pools of 128 / 256 / 512 entries; ncu measured 1.32 at 256).  The stores of a row are
                    // scattered either way (same-phase outputs are ~8 samples apart) and merge in L2.
                    constexpr int kWin = 2048;
                    for (size_t b0 = 0; b0 < e.size(); b0 += kWin) {
                        const int n = (int)std::min<size_t>(kWin, e.size() - b0), nrow = (n + 31) / 32;
                        static thread_local int rows[kWin / 32][32], spill[kWin];
                        int cnt[kWin / 32] = {}, nspill = 0;
                        int seen[32] = {};   // the r-th entry of a bank goes to row r
                        for (int i = 0; i < n; ++i) {
                            const int r = seen[(e[b0 + i] >> 16) & 31u]++;
                            if (r < nrow && cnt[r] < 32) rows[r][cnt[r]++] = i; else spill[nspill++] = i;
                        }
                        int sp = 0;   // entries without a conflict-free row fill the rows that are not full, last row last
                        for (int r = 0; r < nrow; ++r) {
                            const int want = r + 1 < nrow ? 32 : n - 32 * (nrow - 1);
                            while (cnt[r] < want && sp < nspill) rows[r][cnt[r]++] = spill[sp++];
                            for (int r2 = nrow - 1; r2 > r && cnt[r] < want; --r2)
                                while (cnt[r] < want && cnt[r2] > 0) rows[r][cnt[r]++] = rows[r2][--cnt[r2]];
                        }
                        std::vector<unsigned> &e2 = rsx.e2;
                        std::vector<float> &f2 = rsx.f2;
                        e2.clear(); f2.clear();
                        for (int r = 0; r < nrow; ++r) for (int c = 0; c < cnt[r]; ++c) { e2.push_back(e[b0 + rows[r][c]]); f2.push_back(f[b0 + rows[r][c]]); }
                        for (int i = sp; i < nspill; ++i) { e2.push_back(e[b0 + spill[i]]); f2.push_back(f[b0 + spill[i]]); }
                        std::copy(e2.begin(), e2.end(), e.begin() + b0);
                        std::copy(f2.begin(), f2.end(), f.begin() + b0);
                    }
                }
                ent.insert(ent.end(), be[q].begin(), be[q].end());
                frac.insert(frac.end(), bf[q].begin(), bf[q].end());
                const int first = pos;
                pos += (int)be[q].size();
                while (pos % 32) { ent.push_back(0xffffffffu); frac.push_back(0.f); ++pos; }   // whole rows of 32 lanes
                // warp steps of this phase: up to kResPerThread rows each, a short one last
                for (int r0 = first / 32; r0 < pos / 32; r0 += kResPerThread) {
                    const int rows = std::min(kResPerThread, pos / 32 - r0);
                    if ((unsigned)(r0 * 32) > 0xfffffu) return fail(PVGPU_ESTATE, "resampler run does not fit its step list");
                    run_steps.push_back((unsigned)(r0 * 32) | ((unsigned)(rows - 1) << 20) | ((unsigned)q << 24));
                }
            }
            hdr.padded = pos;
            // long steps first: the CTA's warps take the steps round-robin
            std::stable_sort(run_steps.begin(), run_steps.end(), [](unsigned a, unsigned b) { return ((a >> 20) & 7u) > ((b >> 20) & 7u); });
            hdr.step_off = (int)steps.size();
            hdr.n_steps = (int)run_steps.size();
            steps.insert(steps.end(), run_steps.begin(), run_steps.end());
            run_steps.clear();
            runs.push_back(hdr);
        }
        CU(b_runs.ensure(sizeof(ResampleRun) * std::max<size_t>(runs.size(), 1)));
        CU(b_rsent.ensure(sizeof(unsigned) * std::max<size_t>(ent.size(), 1)));
        if (!p.rs_direct) {   // interpolated table: the four cubic coefficients of every entry (cubic_coef, resample.c:339-351)
            std::vector<float> &coef = rsx.coef;
            coef.resize(4 * frac.size());
            for (size_t i = 0; i < frac.size(); ++i) {
                const float fr = frac[i];
                float ip[4];
                ip[0] = -0.16667f * fr + 0.16667f * fr * fr * fr;
                ip[1] = fr + 0.5f * fr * fr - 0.5f * fr * fr * fr;
                ip[3] = -0.33333f * fr + 0.5f * fr * fr - 0.16667f * fr * fr * fr;
                ip[2] = (float)(1. - ip[0] - ip[1] - ip[3]);
                std::memcpy(&coef[4 * i], ip, sizeof ip);
            }
            frac.swap(coef);   // uploaded below in place of the fractions (the next call clears both)
        }
        CU(b_rsfrac.ensure(sizeof(float) * std::max<size_t>(frac.size(), 1)));
        CU(b_rssteps.ensure(sizeof(unsigned) * std::max<size_t>(steps.size(), 1)));
        int rc;
        if ((rc = h2d(b_runs.p, runs.data(), sizeof(ResampleRun) * runs.size(), st))) return rc;
        if ((rc = h2d(b_rsent.p, ent.data(), sizeof(unsigned) * ent.size(), st))) return rc;
        if ((rc = h2d(b_rsfrac.p, frac.data(), sizeof(float) * frac.size(), st))) return rc;
        if ((rc = h2d(b_rssteps.p, steps.data(), sizeof(unsigned) * steps.size(), st))) return rc;
        if (!staged_all) { CU(cudaStreamSynchronize(st)); staged_all = true; }   // sources that were not staged are reused by the next call
        return PVGPU_OK;
    }

    // whisper phases for slices [0, n_slices): 2*pi*rand()/RAND_MAX, slice-major, channel, bin (:814-822)
    int build_whisper(long n_slices) {
        const size_t n = (size_t)n_slices * d.cfg.channels * d.H;
        std::vector<int32_t> r(n);
        glibc_rand_fresh(r.data(), n);
        std::vector<float> ph(n);
        const float two_pi = 2 * M_PI;
        for (size_t i = 0; i < n; ++i) ph[i] = two_pi * (float)r[i] / (float)2147483647;
        return upload(b_whisper, ph.data(), sizeof(float) * n);
    }

    // Frames [k0, k0+nf) of the rows in g; the schedule for them must be on the device.  Three stages so that callers can
    // put them on different streams: analysis | phase modification + synthesis | overlap-add + resampler.
    void run_analyse(const DevRows &g, long k0, int nf, cudaStream_t st) {
        Span *sp = span_begin(0, st);
        launch_analyse(p, g, k0, nf, st);
        span_end(sp, st); ++launches;
    }
    int run_modify_synth(const DevRows &g, long k0, int nf, cudaStream_t st) {
        const SliceRec *recs = b_recs.as<SliceRec>();
        Span *sp;
        if (d.robotic || d.whisper) {
            if (g.spec) { /* phases are produced inside the synthesis kernel */ } else {
            sp = span_begin(5, st);
            launch_fixed_phase(p, g, d.whisper ? b_whisper.as<float>() : nullptr, k0, nf, st);
            span_end(sp, st); ++launches;
            }
        } else if (g.spec && cartesian_lock()) {
            // phase-locked core on Cartesian spectra: frame-parallel peak / link / advance records, then the serial chain
            sp = span_begin(6, st); launch_lock_peaks(p, g, recs, recs_base, k0, nf, st); span_end(sp, st); ++launches;
            // the chunk's last frame is what the next launch links to (before the chain touches classic frames in place)
            const size_t pitch = sizeof(float) * (size_t)g.F * p.Hp, w = sizeof(float) * (size_t)p.Hp;
            CU(cudaMemcpy2DAsync(g.lock_tail, 2 * w, g.mag + (size_t)(nf - 1) * p.Hp, pitch, w, g.rows, cudaMemcpyDeviceToDevice, st));
            CU(cudaMemcpy2DAsync(g.lock_tail + p.Hp, 2 * w, g.phase + (size_t)(nf - 1) * p.Hp, pitch, w, g.rows, cudaMemcpyDeviceToDevice, st));
            sp = span_begin(7, st); launch_lock_chain(p, g, nf, st); span_end(sp, st); ++launches;
        } else if (!d.vocoder && !d.constant_mode) {
            sp = span_begin(1, st); launch_phase_core(p, g, d.cfg.coremode, recs, recs_base, k0, nf, st); span_end(sp, st); ++launches;
        }
        if (d.cepstral) {   // optional modes 8 / 9: whiten by the cepstral envelope, put the warped envelope back (pv_cepstral.cu)
            sp = span_begin(5, st);
            if (!launch_cepstral(p, g, d.env_comp, nf, st)) return fail(PVGPU_EINVAL, "the cepstral modes need an FFT size of 512..8192");
            span_end(sp, st); ++launches;
        }
        if (fused) return PVGPU_OK;   // the inverse FFT is part of run_synth_ola
        sp = span_begin(2, st);
        launch_synthesise(p, g, d.vocoder ? b_carmag.as<float>() : nullptr, d.vocoder ? b_carph.as<float>() : nullptr, k0, nf, st);
        span_end(sp, st); ++launches;
        return PVGPU_OK;
    }
    // Decide whether launches of `frames_per_chunk` frames use the fused kernel, and its shape.  max_shift bounds the
    // per-slice accumulator advance (and so the resampler's per-slice input).
    // split_ok: the split kernels can run this schedule (their table limits hold)
    bool plan_fused(int frames_per_chunk, int max_shift, int max_out_bound, bool split_ok) {
        fused = false;
        const char *env = std::getenv("PVGPU_FUSED");
        const int pref = (env && (env[0] == '0' || env[0] == '1')) ? env[0] - '0' : fused_pref;
        if (pref == 0 || (pref < 0 && split_ok)) return false;
        if (fused_frames_in_flight(p.N) == 0) return false;
        FusedArgs a{};
        if (!fused_plan(p, frames_per_chunk, max_shift, max_shift, max_out_bound, (size_t)200 * 1024, &a)) return false;
        fa = a;
        fused = true;
        return true;
    }
    int run_synth_ola(const DevRows &g, long k0, int nf, cudaStream_t st) {
        FusedArgs a = fa;
        a.recs = b_recs.as<SliceRec>(); a.recs_base = recs_base;
        a.norm = b_norm.as<float>(); a.norm_base = norm_base;
        a.k0 = k0; a.nf = nf;
        a.runs = b_runs.as<ResampleRun>(); a.rs_ent = b_rsent.as<unsigned>(); a.rs_frac = b_rsfrac.as<float>(); a.rs_steps = b_rssteps.as<unsigned>(); a.run_origin = run_origin;
        a.car_mag = d.vocoder ? b_carmag.as<float>() : nullptr; a.car_phase = d.vocoder ? b_carph.as<float>() : nullptr;
        Span *sp = span_begin(4, st);
        CU(launch_synth_ola(p, g, a, st));
        span_end(sp, st); ++launches;
        return PVGPU_OK;
    }
    void run_ola(const DevRows &g, long k0, int nf, cudaStream_t st) {
        const SliceRec *recs = b_recs.as<SliceRec>();
        Span *sp = span_begin(3, st);
        launch_ola_resample(p, g, recs, b_norm.as<float>(), norm_base, recs_base, k0, nf, table_run, max_consumed, b_runs.as<ResampleRun>(),
                            b_rsent.as<unsigned>(), b_rsfrac.as<float>(), b_rssteps.as<unsigned>(), run_origin, st);
        span_end(sp, st); ++launches;
    }
    int run_frames(const DevRows &g, long k0, int nf, cudaStream_t st) {
        run_analyse(g, k0, nf, st);
        int rc = run_modify_synth(g, k0, nf, st);
        if (rc) return rc;
        if (fused) return run_synth_ola(g, k0, nf, st);
        run_ola(g, k0, nf, st);
        return PVGPU_OK;
    }
};

// Device workspace for a group of rows.
struct Workspace {
    DevBuf mag, phase, frames, prev_phase, prev_out, peaks, first, n_in, n_out;
    DevBuf lock_hdr, lock_rec, lock_map, lock_csn, lock_tail, lock_kind, lock_rot;   // phase-locked core on Cartesian spectra
    DevBuf ola_tail, res_hist;                                                       // fused kernel: per-row carry between launches
    DevBuf post_state;                                                               // post-chain: per-row effect state
    size_t lock_slots = 0;     // (row, frame) slots per lock buffer set; nbuf sets are allocated when the fused pipeline overlaps stages
    int rows = 0, F = 0, Fr = 0;

    // halo: frames before the current chunk that the overlap-add of the chunk (and of the resampler history before
    // it) still reads
    // nbuf spectra buffers / (nbuf*F + halo) ring slots: nbuf = 2 lets the analysis of chunk c+1 and the overlap-add of
    // chunk c-1 run while chunk c is in the phase / synthesis stage (see ChunkPipe)
    int nbuf = 1;
    size_t spec_stride = 0;   // floats between the spectra buffers
    int ensure(const Pipeline &pl, int rows_, int F_, int halo, int nbuf_ = 1) {
        const DevPlan &p = pl.p;
        rows = rows_; F = F_; nbuf = nbuf_; Fr = nbuf_ * F_ + halo;
        const int streams = rows / pl.d.cfg.channels;
        spec_stride = (size_t)rows * F * p.Hp;
        CU(mag.ensure(sizeof(float) * spec_stride * nbuf));
        CU(phase.ensure(sizeof(float) * spec_stride * nbuf));
        if (!pl.fused) CU(frames.ensure(sizeof(float) * (size_t)rows * Fr * p.N));   // the fused kernel keeps the overlap-add on chip
        else {
            CU(ola_tail.ensure(sizeof(float) * (size_t)rows * p.N));
            CU(res_hist.ensure(sizeof(float) * (size_t)rows * std::max(pl.fa.hist_len, 1)));
        }
        if (pl.post.n > 0) CU(post_state.ensure(sizeof(float) * (size_t)rows * postchain_state_stride(pl.post)));
        CU(prev_phase.ensure(sizeof(float) * (size_t)rows * p.half));
        CU(prev_out.ensure(sizeof(float) * (size_t)rows * p.half));
        CU(peaks.ensure(sizeof(int) * (size_t)streams * (1 + pl.max_peaks())));
        CU(first.ensure(sizeof(int) * (size_t)streams));
        if (pl.cartesian() && pl.cartesian_lock()) {
            // the fused pipeline reads a chunk's lock tables on the overlap-add stream while the next chunk's are being
            // written: one set per spectra buffer
            const size_t sets = pl.fused ? (size_t)nbuf : 1;
            const size_t slots = (size_t)rows * F * sets, mp = (size_t)pl.max_peaks();
            lock_slots = (size_t)rows * F;
            CU(lock_hdr.ensure(sizeof(int2) * slots));
            CU(lock_rec.ensure(sizeof(float4) * slots * lock_rec_stride(p, (int)mp) + sizeof(float4) * 256));
            CU(lock_map.ensure(sizeof(unsigned short) * slots * p.half));
            CU(lock_csn.ensure(sizeof(float2) * slots * mp));
            CU(lock_tail.ensure(sizeof(float) * (size_t)rows * 2 * p.Hp));
            CU(lock_kind.ensure(sizeof(int) * (size_t)rows));
            CU(lock_rot.ensure(sizeof(float) * (size_t)rows * mp));
        }
        return PVGPU_OK;
    }

    int reset_state(const Pipeline &pl, cudaStream_t st) {
        const DevPlan &p = pl.p;
        const int streams = rows / pl.d.cfg.channels;
        CU(cudaMemsetAsync(prev_phase.p, 0, sizeof(float) * (size_t)rows * p.half, st));
        CU(cudaMemsetAsync(prev_out.p, 0, sizeof(float) * (size_t)rows * p.half, st));
        CU(cudaMemsetAsync(peaks.p, 0, sizeof(int) * (size_t)streams * (1 + pl.max_peaks()), st));
        CU(cudaMemsetAsync(first.p, 0, sizeof(int) * (size_t)streams, st));
        if (lock_kind.p) {
            CU(cudaMemsetAsync(lock_kind.p, 0, sizeof(int) * (size_t)rows, st));
            CU(cudaMemsetAsync(lock_rot.p, 0, sizeof(float) * (size_t)rows * pl.max_peaks(), st));
        }
        if (pl.post.n > 0) launch_postchain_reset(pl.post, post_state.as<float>(), rows, st);
        if (pl.fused) {   // empty accumulator, zero history (speex mem is zero-initialised)
            CU(cudaMemsetAsync(ola_tail.p, 0, sizeof(float) * (size_t)rows * p.N, st));
            CU(cudaMemsetAsync(res_hist.p, 0, sizeof(float) * (size_t)rows * std::max(pl.fa.hist_len, 1), st));
        }
        return PVGPU_OK;
    }

    void bind(const Pipeline &pl, DevRows &g, int buf = 0) const {
        g.mag = mag.as<float>() + spec_stride * buf; g.phase = phase.as<float>() + spec_stride * buf; g.F = F;
        g.frames = frames.as<float>(); g.Fr = Fr;
        g.prev_phase = prev_phase.as<float>(); g.prev_out = prev_out.as<float>();
        g.peaks = peaks.as<int>(); g.maxpk = pl.max_peaks(); g.started = first.as<int>();
        const size_t ls = pl.fused ? lock_slots * (size_t)buf : 0;   // this chunk's set of lock tables
        g.rec_stride = lock_rec_stride(pl.p, pl.max_peaks());
        g.lock_hdr = lock_hdr.as<int2>() + ls; g.lock_rec = lock_rec.as<float4>() + ls * g.rec_stride;
        g.lock_map = lock_map.as<unsigned short>() + ls * pl.p.half; g.lock_csn = lock_csn.as<float2>() + ls * pl.max_peaks(); g.lock_tail = lock_tail.as<float>();
        g.ola_tail = ola_tail.as<float>(); g.res_hist = res_hist.as<float>();
        g.lock_kind = lock_kind.as<int>(); g.lock_rot = lock_rot.as<float>();
    }
};

// Frames before slice k that k_ola_resample reads when it produces slice k: the frames overlapping k (back to jlo) and,
// with a resampler, those overlapping the slices that hold its filt_len-1 samples of history.
static int halo_of(const std::vector<SliceRec> &recs, long recs_base, int hist_len) {
    long h = 1;
    for (size_t i = 0; i < recs.size(); ++i) {
        size_t kh = i;
        const int64_t u_lo = recs[i].res_off + recs[i].rs_last - hist_len + 1;
        while (kh > 0 && recs[kh].res_off > u_lo) --kh;
        h = std::max(h, recs_base + (long)i - recs[kh].jlo + 1);
    }
    return (int)h;
}

// Largest number of slices before slice k whose normalised samples the resampler's history (hist_len - 1 samples) reaches.
static int hist_slices_of(const std::vector<SliceRec> &recs, int hist_len) {
    long h = 0;
    for (size_t i = 0; i < recs.size(); ++i) {
        size_t kh = i;
        const int64_t u_lo = recs[i].res_off + recs[i].rs_last - hist_len + 1;
        while (kh > 0 && recs[kh].res_off > u_lo) --kh;
        h = std::max<long>(h, (long)(i - kh));
    }
    return (int)h;
}

}  // namespace pvgpu

using namespace pvgpu;

// ------------------------------------------------------------------------------------------------
// batch
// ------------------------------------------------------------------------------------------------
struct pvgpu_batch {
    pvgpu_config cfg{};
    Pipeline pl;
    int n_streams = 0;
    int64_t max_in = 0;
    bool planned = false;
    std::vector<int64_t> n_in, n_out;
    long n_slices = 0;
    int halo = 1;
    int64_t res_total = 0, out_total = 0;
    int frames_per_chunk = 64, rows_per_group = 0;
    // Groups of rows are processed round-robin on a few contexts (stream + workspace + staging buffers) so that the
    // serial-in-time phase kernel of one group overlaps the FFT kernels of another, and -- for host buffers -- H2D,
    // kernels and D2H of different groups overlap.
    struct Ctx {
        cudaStream_t st = nullptr;       // analysis (and everything, when the stages are not overlapped)
        cudaStream_t st_b = nullptr;     // phase modification + synthesis
        cudaStream_t st_c = nullptr;     // overlap-add + resampler
        cudaEvent_t done = nullptr;
        cudaEvent_t ev_an[4] = {}, ev_syn[4] = {}, ev_ola[4] = {};
        Workspace ws;
        DevBuf stage_in, stage_out;
    };
    static constexpr int kCtx = 4;
    int n_contexts = 3;
    Ctx ctx[kCtx];
    cudaEvent_t ev_fork = nullptr;
    DevBuf d_nin, d_nout;
    cudaStream_t stream = nullptr;
    cudaStream_t last_stream = cudaStreamLegacy;   // the caller's stream of the last pvgpu_batch_run_device
    int64_t h2d = 0, d2h = 0;
    ~pvgpu_batch() {
        for (auto &c : ctx) {
            if (c.st) cudaStreamDestroy(c.st);
            if (c.st_b) cudaStreamDestroy(c.st_b);
            if (c.st_c) cudaStreamDestroy(c.st_c);
            if (c.done) cudaEventDestroy(c.done);
            for (int i = 0; i < 4; ++i) { if (c.ev_an[i]) cudaEventDestroy(c.ev_an[i]); if (c.ev_syn[i]) cudaEventDestroy(c.ev_syn[i]); if (c.ev_ola[i]) cudaEventDestroy(c.ev_ola[i]); }
        }
        if (ev_fork) cudaEventDestroy(ev_fork);
        for (auto e : ev_pool) cudaEventDestroy(e);
        if (stream) cudaStreamDestroy(stream);
    }
    std::vector<cudaEvent_t> ev_pool;   // chunk events of the time-sliced host pipeline
    bool time_sliced = true;
    // stage overlap needs more than one context's worth of streams; contexts == 1 means strictly serial kernels (profiling)
    bool overlap_stages() const { return n_contexts > 1; }
    size_t max_ws_bytes = (size_t)24 << 30;   // largest workspace a single group may take: a third of the device's free memory at plan time
    size_t ws_bytes_per_row() const {
        size_t b = sizeof(float) * ((size_t)4 * frames_per_chunk * pl.p.Hp + 2 * (size_t)pl.p.half);
        b += pl.fused ? sizeof(float) * ((size_t)pl.p.N + pl.fa.hist_len) : sizeof(float) * (size_t)(2 * frames_per_chunk + halo) * pl.p.N;
        if (pl.cartesian() && pl.cartesian_lock())   // records, bin->region maps and rotations of k_lock_peaks / k_lock_chain
            b += (pl.fused ? 2 : 1) * (size_t)frames_per_chunk * (16 * (size_t)lock_rec_stride(pl.p, pl.max_peaks()) + 2 * (size_t)pl.p.half + 8 * (size_t)pl.max_peaks() + 8);
        return b;
    }
    int run_for_chunk = 0;   // frames_per_chunk the resampler work lists were built for
    int prepare_runs() {
        if (run_for_chunk == frames_per_chunk) return PVGPU_OK;
        // k_ola_resample's per-CTA tables bound the frames overlapping a run and the slices holding the resampler history
        const int hist_all = hist_slices_of(pl.h_recs, pl.p.rs_active ? (int)pl.p.rs_filt_len : 1);
        const bool split_ok = hist_all + 2 <= ola_max_table_slices() - 1 && halo + 1 <= 90;
        pl.plan_fused(frames_per_chunk, pl.max_consumed, pl.max_out, split_ok);   // fused kernel (and its shape) or the split kernels
        if (!pl.fused) {   // k_ola_resample's per-CTA tables: frames overlapping a run, slices holding the resampler history before it
            const int hist = hist_slices_of(pl.h_recs, pl.p.rs_active ? (int)pl.p.rs_filt_len : 1);
            if (hist + 2 > ola_max_table_slices() - 1)
                return fail(PVGPU_EINVAL, "the resampler history spans %d slices, more than the split kernels' tables hold (the fused kernel has no such limit)", hist);
            pl.ola_run = std::min(pl.ola_run, ola_max_table_slices() - hist - 1);
        }
        if (!pl.fused && halo + pl.ola_run > 90) pl.ola_run = std::max(1, 90 - halo);
        if (!pl.fused && halo + pl.ola_run > 90)
            return fail(PVGPU_EINVAL, "stretch/pitch ratio too extreme for the split kernels: %d overlapping frames (the fused kernel has no such limit)", halo);
        int run = pl.fused ? pl.fa.run : ola_run_limit(pl.p, pl.ola_run, pl.max_consumed, pl.max_out);
        while (run > 1 && frames_per_chunk % run) --run;   // chunks must start on run boundaries
        int rc = pl.build_resample_runs(0, n_slices, run, stream);
        if (rc) return rc;
        run_for_chunk = frames_per_chunk;
        return PVGPU_OK;
    }
    int group_rows() const {
        const int C = cfg.channels, total = n_streams * C;
        int group = rows_per_group;
        if (group <= 0) group = (size_t)total * ws_bytes_per_row() <= max_ws_bytes ? total : 1024;   // widest launches that fit
        group = std::min(group, 65535);   // several kernels put rows (or streams) on grid.y
        group = std::max(C, (group / C) * C);
        return std::min(group, total);
    }
};

// All frame chunks of one group.  With `overlap` the three stages of a chunk run on the context's three streams:
//   A  analysis of chunk c            (needs the spectra buffer c%2 free: synthesis of chunk c-2 done)
//   B  phase core + synthesis of c    (needs A(c); its ring slots free: overlap-add of chunk c-2 done)
//   C  overlap-add + resampler of c   (needs B(c))
// With the fused kernel B is the phase core alone and C is inverse FFT + overlap-add + resampler; the spectra and the lock
// tables of chunk c are then read by C(c), so A(c+2) and B(c+2) wait for C(c) (the wait on ev_ola below covers both).
// so the latency-bound, serial-in-time phase kernel shares the SMs with the FFT-heavy kernels of its neighbours.
// before(ci, k0, nf, stA) is called before the analysis of a chunk is enqueued on stA (e.g. to make it wait for an H2D
// copy), after(ci, k0, nf, stC) once the chunk's overlap-add has been enqueued on stC (e.g. to start a D2H copy).
// On return everything has been joined into ctx.st.
template <class Before, class After>
static int run_chunks(pvgpu_batch *b, pvgpu_batch::Ctx &ctx, DevRows g, bool overlap, Before before, After after) {
    Pipeline &pl = b->pl;
    const int F = ctx.ws.F;
    cudaStream_t sa = ctx.st, sb = overlap ? ctx.st_b : ctx.st, sc = overlap ? ctx.st_c : ctx.st;
    if (overlap) {   // fork: B and C start after what is already queued on A (state reset, earlier groups)
        CU(cudaEventRecord(ctx.done, sa));
        CU(cudaStreamWaitEvent(sb, ctx.done, 0));
        CU(cudaStreamWaitEvent(sc, ctx.done, 0));
    }
    long ci = 0;
    for (long k0 = 0; k0 < b->n_slices; k0 += F, ++ci) {
        const int nf = (int)std::min<long>(F, b->n_slices - k0);
        const int e = (int)(ci & 3), e2 = (int)((ci + 2) & 3);   // e2: the slot chunk ci-2 used
        ctx.ws.bind(pl, g, overlap ? (int)(ci & 1) : 0);
        int rc = before(ci, k0, nf, sa);
        if (rc) return rc;
        // the spectra buffer of chunk ci-2 is free once its inverse FFTs are done (split: stage B; fused: stage C)
        if (overlap && ci >= 2) CU(cudaStreamWaitEvent(sa, pl.fused ? ctx.ev_ola[e2] : ctx.ev_syn[e2], 0));
        pl.run_analyse(g, k0, nf, sa);
        if (overlap) {
            CU(cudaEventRecord(ctx.ev_an[e], sa));
            CU(cudaStreamWaitEvent(sb, ctx.ev_an[e], 0));
            if (ci >= 2) CU(cudaStreamWaitEvent(sb, ctx.ev_ola[e2], 0));
        }
        if ((rc = pl.run_modify_synth(g, k0, nf, sb))) return rc;
        if (overlap) {
            CU(cudaEventRecord(ctx.ev_syn[e], sb));
            CU(cudaStreamWaitEvent(sc, ctx.ev_syn[e], 0));
        }
        if (pl.fused) { if ((rc = pl.run_synth_ola(g, k0, nf, sc))) return rc; }
        else pl.run_ola(g, k0, nf, sc);
        if (pl.post.n > 0) {   // the output columns this chunk completed go through the effect chain before anything reads them
            const SliceRec &first = pl.h_recs[k0 - pl.recs_base], &last = pl.h_recs[k0 + nf - 1 - pl.recs_base];
            launch_postchain(g, pl.post, ctx.ws.post_state.as<float>(), first.out_off, last.out_off + ((last.flags & 1) ? 0 : last.n_write), sc);
            ++pl.launches;
        }
        if (overlap) CU(cudaEventRecord(ctx.ev_ola[e], sc));
        if ((rc = after(ci, k0, nf, sc))) return rc;
    }
    if (overlap) {   // join
        CU(cudaEventRecord(ctx.done, sb));
        CU(cudaStreamWaitEvent(sa, ctx.done, 0));
        CU(cudaEventRecord(ctx.done, sc));
        CU(cudaStreamWaitEvent(sa, ctx.done, 0));
    }
    CU(cudaGetLastError());
    return PVGPU_OK;
}

static DevRows group_rows_view(pvgpu_batch *b, const void *d_in, int64_t in_stride, void *d_out, int64_t out_stride, int row0, int rows, int fmt) {
    DevRows g{};
    g.rows = rows; g.channels = b->cfg.channels;
    g.in = d_in; g.in_stride = in_stride; g.in_base = 0; g.fmt = fmt;
    g.n_in = b->d_nin.as<int64_t>() + row0;
    g.n_out = b->d_nout.as<int64_t>() + row0;
    g.out = d_out; g.out_stride = out_stride; g.out_base = 0;
    b->pl.apply_mode(g);
    return g;
}

// One group of rows on one context; on return the group's completion is ordered on ctx.st.
static int batch_run_group(pvgpu_batch *b, pvgpu_batch::Ctx &ctx, const void *d_in, int64_t in_stride, void *d_out, int64_t out_stride,
                           int row0, int rows, int fmt) {
    int rc;
    ctx.ws.rows = rows;
    if ((rc = ctx.ws.reset_state(b->pl, ctx.st))) return rc;
    auto nop = [](long, long, int, cudaStream_t) { return (int)PVGPU_OK; };
    return run_chunks(b, ctx, group_rows_view(b, d_in, in_stride, d_out, out_stride, row0, rows, fmt), b->overlap_stages(), nop, nop);
}

extern "C" {

const char *pvgpu_last_error(void) { return g_err.c_str(); }
int pvgpu_version(void) { return 100; }

int pvgpu_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int pvgpu_describe(const pvgpu_config *cfg, pvgpu_info *info) {
    int rc = validate(cfg);
    if (rc) return rc;
    if (!info) return fail(PVGPU_EINVAL, "null info");
    fill_info(derive(to_config(*cfg)), info);
    return PVGPU_OK;
}

int pvgpu_plan_counts(const pvgpu_config *cfg, int64_t n_in, int block, int64_t *n_out, int64_t *n_slices, int64_t *n_dropped) {
    int rc = validate(cfg);
    if (rc) return rc;
    if (n_in < 0) return fail(PVGPU_EINVAL, "negative length");
    Scheduler sc(derive(to_config(*cfg)), false);
    const StreamPlan sp = plan_stream(sc, (long)n_in, block);
    if (n_out) *n_out = sp.n_out;
    if (n_slices) *n_slices = sp.n_slices;
    if (n_dropped) *n_dropped = sc.dropped();
    return PVGPU_OK;
}

static int pvgpu_batch_create_body(const pvgpu_config *cfg, int n_streams, int64_t max_in_samples, pvgpu_batch **out);
int pvgpu_batch_create(const pvgpu_config *cfg, int n_streams, int64_t max_in_samples, pvgpu_batch **out) {
    return guarded([&]() -> int { return pvgpu_batch_create_body(cfg, n_streams, max_in_samples, out); });
}
static int pvgpu_batch_create_body(const pvgpu_config *cfg, int n_streams, int64_t max_in_samples, pvgpu_batch **out) {
    int rc = validate(cfg);
    if (rc) return rc;
    if (!out || n_streams < 1 || max_in_samples < 0) return fail(PVGPU_EINVAL, "bad batch arguments");
    std::unique_ptr<pvgpu_batch> b(new (std::nothrow) pvgpu_batch);
    if (!b) return fail(PVGPU_ENOMEM, "out of host memory");
    b->cfg = *cfg;
    b->n_streams = n_streams;
    b->max_in = max_in_samples;
    if ((rc = b->pl.init(*cfg))) return rc;
    CU(cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking));
    CU(cudaEventCreateWithFlags(&b->ev_fork, cudaEventDisableTiming));
    for (auto &c : b->ctx) {
        CU(cudaStreamCreateWithFlags(&c.st, cudaStreamNonBlocking));
        {   // the phase + synthesis stage holds the latency-bound serial chain: its CTAs go first when SM slots free up
            int lo = 0, hi = 0;
            CU(cudaDeviceGetStreamPriorityRange(&lo, &hi));
            CU(cudaStreamCreateWithPriority(&c.st_b, cudaStreamNonBlocking, hi));
        }
        CU(cudaStreamCreateWithFlags(&c.st_c, cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(&c.done, cudaEventDisableTiming));
        for (int i = 0; i < 4; ++i) {
            CU(cudaEventCreateWithFlags(&c.ev_an[i], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&c.ev_syn[i], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&c.ev_ola[i], cudaEventDisableTiming));
        }
    }
    *out = b.release();
    return PVGPU_OK;
}

void pvgpu_batch_destroy(pvgpu_batch *b) {
    if (!b) return;
    cudaSetDevice(b->pl.device);
    delete b;
}

int pvgpu_batch_info(const pvgpu_batch *b, pvgpu_info *info) {
    if (!b || !info) return fail(PVGPU_EINVAL, "null argument");
    fill_info(b->pl.d, info);
    return PVGPU_OK;
}

int pvgpu_batch_tune(pvgpu_batch *b, int frames_per_chunk, int rows_per_group, int contexts) {
    if (!b) return fail(PVGPU_EINVAL, "null batch");
    if (frames_per_chunk > 0 && frames_per_chunk != b->frames_per_chunk) { b->frames_per_chunk = frames_per_chunk; b->run_for_chunk = 0; }
    if (rows_per_group > 0) { b->rows_per_group = rows_per_group; b->time_sliced = false; }   // explicit row groups pipeline across rows instead of time
    if (contexts > 0) b->n_contexts = std::min(contexts, (int)pvgpu_batch::kCtx);
    return PVGPU_OK;
}

// biquadfilter::computeCoeffs (src/common/filters/biquadfilter.cc:113-195: the RBJ audio-EQ-cookbook sections), with the
// reference's mix of float members and double libm calls; coeffs = {b0, b1, b2, a0, a1, a2} as it stores them (floats).
int pvgpu_biquad_design(int type, int sample_rate, float cutoff, float q, float db_gain, float *coeffs) {
    if (!coeffs || sample_rate <= 0 || !(q > 0.f) || type < 0 || type > 8) return fail(PVGPU_EINVAL, "bad biquad parameters");
    const float a = (float)std::pow(10.0, db_gain / 40.0);
    const float omega = (float)(2 * M_PI * cutoff / sample_rate);
    const float alpha = (float)(std::sin((double)omega) / 2.0 / q);
    const double cw = std::cos((double)omega), sw = std::sin((double)omega), sa = std::sqrt((double)a);
    float b0, b1, b2, a0, a1, a2;
    switch (type) {
        case 5:  b0 = b2 = (float)((1.0 - cw) / 2.0); b1 = (float)(1.0 - cw); a0 = (float)(1.0 + alpha); a1 = (float)(-2.0 * cw); a2 = 1 - alpha; break;   // lowPass
        case 0:  b0 = b2 = (float)((1.0 + cw) / 2.0); b1 = (float)(-(1.0 + cw)); a0 = (float)(1.0 + alpha); a1 = (float)(-2.0 * cw); a2 = 1 - alpha; break;  // highPass
        case 6:  b0 = (float)(sw / 2); b1 = 0; b2 = (float)(-sw / 2); a0 = 1 + alpha; a1 = (float)(-2 * cw); a2 = 1 - alpha; break;                            // bandpass, constant skirt
        case 7:  b0 = alpha; b1 = 0; b2 = -alpha; a0 = 1 + alpha; a1 = (float)(-2 * cw); a2 = 1 - alpha; break;                                                 // bandpass, constant 0 dB peak
        case 3:  b0 = 1; b1 = (float)(-2 * cw); b2 = 1; a0 = 1 + alpha; a1 = (float)(-2 * cw); a2 = 1 - alpha; break;                                           // notch
        case 8:  b0 = 1 - alpha; b1 = (float)(-2 * cw); b2 = 1 + alpha; a0 = 1 + alpha; a1 = (float)(-2 * cw); a2 = 1 - alpha; break;                           // allpass
        case 2:  b0 = 1 + alpha * a; b1 = (float)(-2 * cw); b2 = 1 - alpha * a; a0 = 1 + alpha / a; a1 = (float)(-2 * cw); a2 = 1 - alpha / a; break;           // peaking
        case 1:                                                                                                                                              // lowShelf
            b0 = (float)(a * (a + 1 - (a - 1) * cw + 2 * sa * alpha)); b1 = (float)(2 * a * (a - 1 - (a + 1) * cw)); b2 = (float)(a * (a + 1 - (a - 1) * cw - 2 * sa * alpha));
            a0 = (float)(a + 1 + (a - 1) * cw + 2 * sa * alpha); a1 = (float)(-2 * (a - 1 + (a + 1) * cw)); a2 = (float)(a + 1 + (a - 1) * cw - 2 * sa * alpha);
            break;
        default:                                                                                                                                             // highShelf (4)
            b0 = (float)(a * (a + 1 + (a - 1) * cw + 2 * sa * alpha)); b1 = (float)(-2 * a * (a - 1 + (a + 1) * cw)); b2 = (float)(a * (a + 1 + (a - 1) * cw - 2 * sa * alpha));
            a0 = (float)(a + 1 - (a - 1) * cw + 2 * sa * alpha); a1 = (float)(2 * (a - 1 - (a + 1) * cw)); a2 = (float)(a + 1 - (a - 1) * cw - 2 * sa * alpha);
            break;
    }
    coeffs[0] = b0; coeffs[1] = b1; coeffs[2] = b2; coeffs[3] = a0; coeffs[4] = a1; coeffs[5] = a2;
    return PVGPU_OK;
}

// equalizer::equalizer + processBlock (src/equalizer/equalizer.cc:19-146, 613-647): eight biquad sections in a fixed order
// (high-pass, low shelf, four peaking, high shelf, low-pass), each with {use flag, cutoff, Q, gain}; paramlist == NULL gives
// the reference's defaults (only the 200 Hz high-pass is on).  Writes the enabled sections as PVGPU_FX_BIQUAD entries.
int pvgpu_equalizer_chain(const float *paramlist, pvgpu_fx *chain, int *n_fx) {
    if (!chain || !n_fx) return fail(PVGPU_EINVAL, "null argument");
    static const float defaults[32] = {1, 200, 0.3f, 1.0f,  0, 400, 0.3f, -1.5f,  0, 1000, 0.3f, 1.5f,  0, 2000, 0.3f, 1.5f,
                                       0, 3000, 0.3f, 1.5f,  0, 4000, 0.3f, 1.5f,  0, 5000, 0.3f, -1.5f,  0, 6000, 0.3f, 1.0f};
    static const int types[8] = {0, 1, 2, 2, 2, 2, 4, 5};
    const float *pl = paramlist ? paramlist : defaults;
    int n = 0;
    for (int b = 0; b < 8; ++b) {
        if (!(pl[4 * b] > 0)) continue;
        chain[n].kind = PVGPU_FX_BIQUAD;
        chain[n].p[0] = (float)types[b]; chain[n].p[1] = pl[4 * b + 1]; chain[n].p[2] = pl[4 * b + 2]; chain[n].p[3] = pl[4 * b + 3];
        chain[n].p[4] = chain[n].p[5] = 0.f;
        ++n;
    }
    *n_fx = n;
    return PVGPU_OK;
}

}  // extern "C"

// pvgpu_fx entries -> the coefficients the kernels run with, as the reference's constructors compute them at sample rate sr; the
// conversion and the argument checks of pvgpu_batch_set_postchain and pvgpu_set_postchain.  *out is only written on success.
static int make_postchain(int sr, const pvgpu_fx *chain, int n_fx, PostChain *out) {
    if (n_fx < 0 || n_fx > kMaxPostFx || (n_fx > 0 && !chain)) return fail(PVGPU_EINVAL, "bad post-chain (at most %d effects)", kMaxPostFx);
    PostChain pc{};
    for (int i = 0; i < n_fx; ++i) {
        const pvgpu_fx &f = chain[i];
        PostFx &o = pc.fx[i];
        o.kind = f.kind;
        if (f.kind == PVGPU_FX_GAIN) {                    // gain::gain, src/gain/gain.cc:21-25
            o.p[0] = f.p[0];
        } else if (f.kind == PVGPU_FX_COMPRESSOR) {       // compressor::compressor, src/dynamics/compressor.cc:16-42
            const float tau_a = f.p[3], tau_r = f.p[4];
            o.p[0] = f.p[0]; o.p[1] = f.p[1]; o.p[2] = f.p[2];
            o.p[3] = (float)std::exp(-1 / (0.001 * sr * tau_a));
            o.p[4] = (float)std::exp(-1 / (0.001 * sr * tau_r));
            if (!(f.p[1] > 0.f)) return fail(PVGPU_EINVAL, "compressor ratio must be positive");
        } else if (f.kind == PVGPU_FX_LIMITER) {          // limiter::limiter, src/dynamics/limiter.cc:16-39 (LIMIT_OFFSET 0.01, ahead 6 ms)
            o.p[0] = (float)std::pow(10.0, f.p[1] / 20.0);
            o.p[1] = (float)std::pow(10.0, (f.p[0] - 0.01) / 20.0);
            o.p[2] = (float)std::exp(-1.0 / (sr * 0.001 * f.p[2]));
            o.p[3] = (float)std::exp(-1.0 / (sr * 0.001 * f.p[3]));
            o.p[4] = (float)std::pow(10.0, -120.0 / 20.0);
            o.delay = (int)(sr * 0.001 * 6.0f) + 1;
        } else if (f.kind == PVGPU_FX_BIQUAD) {           // biquadfilter::biquadfilter + computeCoeffs, src/common/filters/biquadfilter.cc:29-41,113-195
            float c[6];
            if (pvgpu_biquad_design((int)f.p[0], sr, f.p[1], f.p[2], f.p[3], c) != PVGPU_OK) return PVGPU_EINVAL;
            for (int j = 0; j < 6; ++j) o.p[j] = c[j];
        } else {
            return fail(PVGPU_EINVAL, "unknown effect kind %d", f.kind);
        }
    }
    pc.n = n_fx;
    *out = pc;
    return PVGPU_OK;
}

extern "C" {

int pvgpu_batch_set_postchain(pvgpu_batch *b, const pvgpu_fx *chain, int n_fx) {
    if (!b) return fail(PVGPU_EINVAL, "bad post-chain (at most %d effects)", kMaxPostFx);
    return make_postchain(b->cfg.sample_rate, chain, n_fx, &b->pl.post);
}

int pvgpu_batch_set_fused(pvgpu_batch *b, int enable) {
    if (!b) return fail(PVGPU_EINVAL, "null batch");
    b->pl.fused_pref = enable < 0 ? -1 : (enable == 1 ? 1 : 0);
    b->run_for_chunk = 0;   // re-plan the launches at the next run
    return PVGPU_OK;
}

static int pvgpu_batch_plan_body(pvgpu_batch *b, const int64_t *n_in, int block, int64_t *n_out);
int pvgpu_batch_plan(pvgpu_batch *b, const int64_t *n_in, int block, int64_t *n_out) {
    return guarded([&]() -> int { return pvgpu_batch_plan_body(b, n_in, block, n_out); });
}
static int pvgpu_batch_plan_body(pvgpu_batch *b, const int64_t *n_in, int block, int64_t *n_out) {
    if (!b || !n_in) return fail(PVGPU_EINVAL, "null argument");
    CU(cudaSetDevice(b->pl.device));
    Pipeline &pl = b->pl;
    const int C = b->cfg.channels;
    int64_t longest = 0;
    for (int s = 0; s < b->n_streams; ++s) {
        if (n_in[s] < 0 || n_in[s] > b->max_in) return fail(PVGPU_EINVAL, "stream %d: length %lld outside [0, %lld]", s, (long long)n_in[s], (long long)b->max_in);
        longest = std::max(longest, n_in[s]);
    }
    // one schedule (with normalisers) for the longest stream; every other length only needs its counts
    Scheduler main_sched(pl.d, true);
    const StreamPlan mp = plan_stream(main_sched, (long)longest, block);
    std::map<int64_t, StreamPlan> by_len;
    by_len[longest] = mp;
    b->n_in.assign(n_in, n_in + b->n_streams);
    b->n_out.resize(b->n_streams);
    for (int s = 0; s < b->n_streams; ++s) {
        auto it = by_len.find(n_in[s]);
        if (it == by_len.end()) {
            Scheduler cnt(pl.d, false);
            it = by_len.emplace(n_in[s], plan_stream(cnt, (long)n_in[s], block)).first;
        }
        b->n_out[s] = it->second.n_out;
        if (n_out) n_out[s] = it->second.n_out;
    }
    if (main_sched.dropped() != 0) return fail(PVGPU_ESTATE, "schedule dropped slices; use a smaller block");
    b->n_slices = mp.n_slices;
    b->res_total = main_sched.res_total();
    b->out_total = main_sched.total_out();
    b->halo = halo_of(main_sched.recs(), main_sched.recs_base(), pl.p.rs_active ? (int)pl.p.rs_filt_len : 1);
    int rc;
    if ((rc = pl.upload_schedule(main_sched, nullptr))) return rc;
    if (pl.d.whisper && (rc = pl.build_whisper(b->n_slices))) return rc;
    // per-row limits
    std::vector<int64_t> rin((size_t)b->n_streams * C), rout((size_t)b->n_streams * C);
    for (int s = 0; s < b->n_streams; ++s)
        for (int c = 0; c < C; ++c) { rin[(size_t)s * C + c] = b->n_in[s]; rout[(size_t)s * C + c] = b->n_out[s]; }
    if ((rc = Pipeline::upload(b->d_nin, rin.data(), sizeof(int64_t) * rin.size()))) return rc;
    if ((rc = Pipeline::upload(b->d_nout, rout.data(), sizeof(int64_t) * rout.size()))) return rc;
    if (pl.d.vocoder && b->n_slices > 0) {
        // the carrier pulse train is the same for every stream and channel: analyse it once
        const long n_car = mp.n_fed;
        std::vector<float> car((size_t)std::max<long>(n_car, 1));
        carrier_signal(b->cfg.sample_rate, b->cfg.mode == PVGPU_VOCODER_CHORD, car.data(), (size_t)n_car);
        DevBuf d_car, d_len;
        if ((rc = Pipeline::upload(d_car, car.data(), sizeof(float) * car.size()))) return rc;
        const int64_t len = n_car;
        if ((rc = Pipeline::upload(d_len, &len, sizeof len))) return rc;
        CU(pl.b_carmag.ensure(sizeof(float) * (size_t)b->n_slices * pl.p.Hp));
        CU(pl.b_carph.ensure(sizeof(float) * (size_t)b->n_slices * pl.p.Hp));
        DevRows g{};
        g.rows = 1; g.channels = 1;
        g.in = d_car.as<float>(); g.in_stride = 0; g.in_base = 0; g.n_in = d_len.as<int64_t>();
        g.mag = pl.b_carmag.as<float>(); g.phase = pl.b_carph.as<float>(); g.F = (int)b->n_slices;
        launch_analyse(pl.p, g, 0, (int)b->n_slices, nullptr);
        CU(cudaGetLastError());
        CU(cudaDeviceSynchronize());
    }
    CU(cudaDeviceSynchronize());
    {
        size_t free_b = 0, total_b = 0;
        if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) b->max_ws_bytes = std::max<size_t>((size_t)2 << 30, free_b / 3);
        else cudaGetLastError();
    }
    b->run_for_chunk = 0;
    if ((rc = b->prepare_runs())) return rc;
    b->planned = true;
    return PVGPU_OK;
}

// After a failed run: nothing of this batch may still be reading or writing the caller's buffers when the error is returned.
static int drain_after_error(pvgpu_batch *b, int rc) {
    if (rc != PVGPU_OK) {
        const std::string keep = g_err;
        cudaSetDevice(b->pl.device);
        cudaDeviceSynchronize();
        cudaGetLastError();
        g_err = keep;
    }
    return rc;
}

static int batch_run_device_impl(pvgpu_batch *b, const void *d_in, int64_t in_stride, void *d_out, int64_t out_stride, int fmt, cudaStream_t st) {
    const size_t esz = fmt == PVGPU_S16 ? sizeof(short) : sizeof(float);
    const int total_rows = b->n_streams * b->cfg.channels;
    int rc;
    if ((rc = b->prepare_runs())) return rc;   // also decides fused / split, which the workspace layout depends on
    const int group = b->group_rows();
    const int n_groups = (total_rows + group - 1) / group;
    const int n_ctx = std::min(n_groups, b->n_contexts);
    for (int i = 0; i < n_ctx; ++i)
        if ((rc = b->ctx[i].ws.ensure(b->pl, group, b->frames_per_chunk, b->halo, b->overlap_stages() ? 2 : 1))) return rc;
    b->pl.launches = 0;
    // fork: the contexts start after everything already queued on the caller's stream
    CU(cudaEventRecord(b->ev_fork, st));
    for (int i = 0; i < n_ctx; ++i) CU(cudaStreamWaitEvent(b->ctx[i].st, b->ev_fork, 0));
    for (int gi = 0; gi < n_groups; ++gi) {
        const int row0 = gi * group, rows = std::min(group, total_rows - row0);
        if ((rc = batch_run_group(b, b->ctx[gi % n_ctx], (const char *)d_in + (int64_t)row0 * in_stride * esz, in_stride,
                                  (char *)d_out + (int64_t)row0 * out_stride * esz, out_stride, row0, rows, fmt))) return rc;
    }
    // join
    for (int i = 0; i < n_ctx; ++i) {
        CU(cudaEventRecord(b->ctx[i].done, b->ctx[i].st));
        CU(cudaStreamWaitEvent(st, b->ctx[i].done, 0));
    }
    return PVGPU_OK;
}

// cuda_stream is the CALLER's stream, with CUDA's own convention that a null handle is the legacy default stream: the
// batch's internal (non-blocking) streams are forked from it and joined back into it with events, so the run is ordered
// after everything the caller queued on that stream before the call and before everything queued after it.  The call
// never blocks the host; pvgpu_batch_synchronize() does.
int pvgpu_batch_run_device(pvgpu_batch *b, const void *d_in, int64_t in_stride, void *d_out, int64_t out_stride, int fmt, void *cuda_stream) {
    if (!b || !d_in || !d_out) return fail(PVGPU_EINVAL, "null argument");
    if (!b->planned) return fail(PVGPU_ESTATE, "pvgpu_batch_plan has not been called");
    if (fmt != PVGPU_F32 && fmt != PVGPU_S16) return fail(PVGPU_EINVAL, "unknown sample format %d", fmt);
    if (fmt != PVGPU_F32 && b->pl.post.n > 0) return fail(PVGPU_EINVAL, "the post-chain works on float32 rows");
    CU(cudaSetDevice(b->pl.device));
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : cudaStreamLegacy;
    b->last_stream = st;
    return drain_after_error(b, guarded([&]() -> int { return batch_run_device_impl(b, d_in, in_stride, d_out, out_stride, fmt, st); }));
}

int pvgpu_batch_synchronize(pvgpu_batch *b) {
    if (!b) return fail(PVGPU_EINVAL, "null batch");
    CU(cudaSetDevice(b->pl.device));
    CU(cudaStreamSynchronize(b->last_stream));
    return PVGPU_OK;
}

// rows [r0, r0+rows) between host row pointers and a dense device block; one 2-D copy when the host rows are evenly
// spaced, one copy per row otherwise
static int copy_rows(void *dev, int64_t dev_stride, const void *const *host_rows, int r0, int rows, const int64_t *lens, int C, bool to_device,
                     size_t esz, cudaStream_t st, int64_t *bytes) {
    // the 2-D copy moves the same number of elements for every row, so it is only used when all rows of the block have the
    // same length (otherwise it would run past the end of the shorter host rows)
    bool regular = rows > 1;
    const ptrdiff_t pitch = rows > 1 ? (const char *)host_rows[r0 + 1] - (const char *)host_rows[r0] : 0;
    const int64_t maxlen = lens[r0 / C];
    for (int r = 0; r < rows; ++r) {
        if (lens[(r0 + r) / C] != maxlen) regular = false;
        if (r + 1 < rows && (const char *)host_rows[r0 + r + 1] - (const char *)host_rows[r0 + r] != pitch) regular = false;
    }
    if (regular && pitch >= (ptrdiff_t)(maxlen * esz) && maxlen > 0) {
        if (to_device) CU(cudaMemcpy2DAsync(dev, dev_stride * esz, host_rows[r0], (size_t)pitch, maxlen * esz, rows, cudaMemcpyHostToDevice, st));
        else CU(cudaMemcpy2DAsync((void *)host_rows[r0], (size_t)pitch, dev, dev_stride * esz, maxlen * esz, rows, cudaMemcpyDeviceToHost, st));
        for (int r = 0; r < rows; ++r) *bytes += esz * lens[(r0 + r) / C];
        return PVGPU_OK;
    }
    for (int r = 0; r < rows; ++r) {
        const int64_t n = lens[(r0 + r) / C];
        if (!n) continue;
        char *d = (char *)dev + (int64_t)r * dev_stride * esz;
        if (to_device) CU(cudaMemcpyAsync(d, host_rows[r0 + r], esz * n, cudaMemcpyHostToDevice, st));
        else CU(cudaMemcpyAsync((void *)host_rows[r0 + r], d, esz * n, cudaMemcpyDeviceToHost, st));
        *bytes += esz * n;
    }
    return PVGPU_OK;
}

// byte distance between consecutive host rows if it is the same for all of them (0 for a single row), else -1
static ptrdiff_t regular_pitch(const void *const *rows, int n) {
    if (n < 2) return 0;
    const ptrdiff_t pitch = (const char *)rows[1] - (const char *)rows[0];
    for (int r = 1; r + 1 < n; ++r)
        if ((const char *)rows[r + 1] - (const char *)rows[r] != pitch) return -1;
    return pitch;
}

// Host buffers, equal-length streams in evenly spaced host rows: the whole batch is one group (widest launches) and the
// pipeline runs along TIME instead -- frame chunk c only needs the input columns up to its last frame and completes the
// output columns of its slices, so H2D of later columns, the kernels of chunk c and D2H of earlier columns overlap on
// three streams with one 2-D copy per chunk and direction.
static int run_host_timesliced(pvgpu_batch *b, const void *const *in_rows, void *const *out_rows, int fmt, size_t esz, int64_t in_stride,
                               int64_t out_stride, ptrdiff_t in_pitch, ptrdiff_t out_pitch) {
    Pipeline &pl = b->pl;
    const int total_rows = b->n_streams * b->cfg.channels;
    pvgpu_batch::Ctx &c = b->ctx[0];
    cudaStream_t s_in = b->ctx[1].st, s_out = b->ctx[2].st;
    const bool overlap = b->overlap_stages();
    int rc;
    if ((rc = c.ws.ensure(pl, total_rows, b->frames_per_chunk, b->halo, overlap ? 2 : 1))) return rc;
    CU(c.stage_in.ensure(esz * (size_t)total_rows * in_stride));
    CU(c.stage_out.ensure(esz * (size_t)total_rows * out_stride));
    const int F = c.ws.F;
    const long n_chunks = (b->n_slices + F - 1) / F;
    while ((long)b->ev_pool.size() < 2 * n_chunks + 2) {
        cudaEvent_t e;
        CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        b->ev_pool.push_back(e);
    }
    c.ws.rows = total_rows;
    if ((rc = c.ws.reset_state(pl, c.st))) return rc;
    const int64_t n_in = b->n_in[0], n_out = b->n_out[0];
    int64_t in_done = 0, out_done = 0;
    const std::vector<SliceRec> &recs = pl.h_recs;
    auto before = [&](long ci, long k0, int nf, cudaStream_t sa) -> int {
        const int64_t need = std::min<int64_t>(n_in, (int64_t)(k0 + nf - 1) * pl.p.hop + pl.p.N);
        if (need > in_done) {
            CU(cudaMemcpy2DAsync((char *)c.stage_in.p + in_done * esz, in_stride * esz, (const char *)in_rows[0] + in_done * esz, (size_t)in_pitch,
                                 (size_t)(need - in_done) * esz, total_rows, cudaMemcpyHostToDevice, s_in));
            b->h2d += (int64_t)(need - in_done) * esz * total_rows;
            in_done = need;
            CU(cudaEventRecord(b->ev_pool[2 * ci], s_in));
            CU(cudaStreamWaitEvent(sa, b->ev_pool[2 * ci], 0));
        }
        return PVGPU_OK;
    };
    auto after = [&](long ci, long k0, int nf, cudaStream_t sc) -> int {
        const SliceRec &last = recs[k0 + nf - 1 - pl.recs_base];
        const int64_t avail = std::min<int64_t>(n_out, last.out_off + ((last.flags & 1) ? 0 : last.n_write));
        if (avail > out_done) {
            CU(cudaEventRecord(b->ev_pool[2 * ci + 1], sc));
            CU(cudaStreamWaitEvent(s_out, b->ev_pool[2 * ci + 1], 0));
            CU(cudaMemcpy2DAsync((char *)out_rows[0] + out_done * esz, (size_t)out_pitch, (const char *)c.stage_out.p + out_done * esz, out_stride * esz,
                                 (size_t)(avail - out_done) * esz, total_rows, cudaMemcpyDeviceToHost, s_out));
            b->d2h += (int64_t)(avail - out_done) * esz * total_rows;
            out_done = avail;
        }
        return PVGPU_OK;
    };
    if ((rc = run_chunks(b, c, group_rows_view(b, c.stage_in.p, in_stride, c.stage_out.p, out_stride, 0, total_rows, fmt), overlap, before, after)))
        return rc;
    CU(cudaStreamSynchronize(s_in));
    CU(cudaStreamSynchronize(c.st));
    CU(cudaStreamSynchronize(s_out));
    return PVGPU_OK;
}

static int batch_run_host_impl(pvgpu_batch *b, const void *const *in_rows, void *const *out_rows, int fmt) {
    const size_t esz = fmt == PVGPU_S16 ? sizeof(short) : sizeof(float);
    const int C = b->cfg.channels;
    const int total_rows = b->n_streams * C;
    int64_t in_stride = 0, out_stride = 0;
    for (int s = 0; s < b->n_streams; ++s) { in_stride = std::max(in_stride, b->n_in[s]); out_stride = std::max(out_stride, b->n_out[s]); }
    in_stride = std::max<int64_t>((in_stride + 3) & ~(int64_t)3, 4);
    out_stride = std::max<int64_t>((out_stride + 3) & ~(int64_t)3, 4);
    int rc;
    if ((rc = b->prepare_runs())) return rc;
    b->pl.launches = 0;
    b->h2d = b->d2h = 0;
    {
        bool uniform = b->n_slices > 0 && b->n_in[0] > 0 && b->n_out[0] > 0;
        for (int s = 1; s < b->n_streams && uniform; ++s) uniform = b->n_in[s] == b->n_in[0] && b->n_out[s] == b->n_out[0];
        const ptrdiff_t ip = regular_pitch(in_rows, total_rows), op = regular_pitch((const void *const *)out_rows, total_rows);
        const bool fits = (size_t)total_rows * b->ws_bytes_per_row() <= b->max_ws_bytes && total_rows <= 65535;
        if (uniform && fits && b->time_sliced && (total_rows == 1 || (ip >= (ptrdiff_t)(b->n_in[0] * esz) && op >= (ptrdiff_t)(b->n_out[0] * esz))))
            return run_host_timesliced(b, in_rows, out_rows, fmt, esz, in_stride, out_stride, ip, op);
    }
    const int group = b->group_rows();
    const int n_groups = (total_rows + group - 1) / group;
    const int n_ctx = std::min(n_groups, b->n_contexts);
    for (int i = 0; i < n_ctx; ++i) {
        pvgpu_batch::Ctx &c = b->ctx[i];
        if ((rc = c.ws.ensure(b->pl, group, b->frames_per_chunk, b->halo, b->overlap_stages() ? 2 : 1))) return rc;
        CU(c.stage_in.ensure(esz * (size_t)group * in_stride));
        CU(c.stage_out.ensure(esz * (size_t)group * out_stride));
    }
    // each context's stream carries H2D -> kernels -> D2H of its groups in order; the contexts run concurrently, so the
    // copies of one group overlap the kernels of the others
    for (int gi = 0; gi < n_groups; ++gi) {
        pvgpu_batch::Ctx &c = b->ctx[gi % n_ctx];
        const int row0 = gi * group, rows = std::min(group, total_rows - row0);
        if ((rc = copy_rows(c.stage_in.p, in_stride, in_rows, row0, rows, b->n_in.data(), C, true, esz, c.st, &b->h2d))) return rc;
        if ((rc = batch_run_group(b, c, c.stage_in.p, in_stride, c.stage_out.p, out_stride, row0, rows, fmt))) return rc;
        if ((rc = copy_rows(c.stage_out.p, out_stride, (const void *const *)out_rows, row0, rows, b->n_out.data(), C, false, esz, c.st, &b->d2h))) return rc;
    }
    for (int i = 0; i < n_ctx; ++i) CU(cudaStreamSynchronize(b->ctx[i].st));
    return PVGPU_OK;
}

int pvgpu_batch_run_host(pvgpu_batch *b, const void *const *in_rows, void *const *out_rows, int fmt) {
    if (!b || !in_rows || !out_rows) return fail(PVGPU_EINVAL, "null argument");
    if (!b->planned) return fail(PVGPU_ESTATE, "pvgpu_batch_plan has not been called");
    if (fmt != PVGPU_F32 && fmt != PVGPU_S16) return fail(PVGPU_EINVAL, "unknown sample format %d", fmt);
    if (fmt != PVGPU_F32 && b->pl.post.n > 0) return fail(PVGPU_EINVAL, "the post-chain works on float32 rows");
    CU(cudaSetDevice(b->pl.device));
    return drain_after_error(b, guarded([&]() -> int { return batch_run_host_impl(b, in_rows, out_rows, fmt); }));
}

int pvgpu_batch_profile(pvgpu_batch *b, int enable) {
    if (!b) return fail(PVGPU_EINVAL, "null batch");
    b->pl.profile = enable != 0;
    b->pl.spans_used = 0;
    for (int i = 0; i < 8; ++i) { b->pl.kind_ms[i] = 0; b->pl.kind_n[i] = 0; }
    return PVGPU_OK;
}

int pvgpu_batch_kernel_times(pvgpu_batch *b, double *ms, int64_t *count) {
    if (!b || !ms || !count) return fail(PVGPU_EINVAL, "null argument");
    CU(cudaSetDevice(b->pl.device));
    CU(cudaDeviceSynchronize());
    b->pl.collect_spans();
    for (int i = 0; i < 8; ++i) { ms[i] = b->pl.kind_ms[i]; count[i] = b->pl.kind_n[i]; }
    return PVGPU_OK;
}

int pvgpu_batch_stats(const pvgpu_batch *b, int64_t *kernel_launches, int64_t *slices, int64_t *h2d_bytes, int64_t *d2h_bytes) {
    if (!b) return fail(PVGPU_EINVAL, "null batch");
    if (kernel_launches) *kernel_launches = b->pl.launches;
    if (slices) *slices = b->n_slices;
    if (h2d_bytes) *h2d_bytes = b->h2d;
    if (d2h_bytes) *d2h_bytes = b->d2h;
    return PVGPU_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// stage hooks for the parity tests
// ------------------------------------------------------------------------------------------------
static int stage_pipeline(Pipeline &pl, int device, int fftsize) {
    pvgpu_config cfg{};
    cfg.sample_rate = 44100; cfg.channels = 1; cfg.time_ratio = 1.f; cfg.pitch_semitones = 0.f;
    cfg.mode = PVGPU_ROBOTIC; cfg.coremode = 1; cfg.fftsize = fftsize; cfg.hopsize = fftsize; cfg.device = device;
    int rc = validate(&cfg);
    if (rc) return rc;
    if (fftsize & (fftsize - 1)) return fail(PVGPU_EINVAL, "stage hooks need a power-of-two fft size");
    return pl.init(cfg);
}

extern "C" {

int pvgpu_test_forward_polar(int device, int fftsize, int n_frames, const float *frames, float *mag, float *phase) {
    if (!frames || !mag || !phase || n_frames < 1) return fail(PVGPU_EINVAL, "bad argument");
    Pipeline pl;
    int rc = stage_pipeline(pl, device, fftsize);
    if (rc) return rc;
    const int N = pl.p.N, H = pl.p.H, Hp = pl.p.Hp;
    DevBuf d_in, d_mag, d_ph, d_len;
    const int64_t len = (int64_t)n_frames * N;
    if ((rc = Pipeline::upload(d_in, frames, sizeof(float) * len))) return rc;
    if ((rc = Pipeline::upload(d_len, &len, sizeof len))) return rc;
    CU(d_mag.ensure(sizeof(float) * (size_t)n_frames * Hp));
    CU(d_ph.ensure(sizeof(float) * (size_t)n_frames * Hp));
    DevRows g{};
    g.rows = 1; g.channels = 1; g.in = d_in.as<float>(); g.in_stride = len; g.n_in = d_len.as<int64_t>();
    g.mag = d_mag.as<float>(); g.phase = d_ph.as<float>(); g.F = n_frames;
    launch_analyse(pl.p, g, 0, n_frames, nullptr);
    CU(cudaGetLastError());
    CU(cudaMemcpy2D(mag, sizeof(float) * H, d_mag.p, sizeof(float) * Hp, sizeof(float) * H, n_frames, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy2D(phase, sizeof(float) * H, d_ph.p, sizeof(float) * Hp, sizeof(float) * H, n_frames, cudaMemcpyDeviceToHost));
    return PVGPU_OK;
}

int pvgpu_test_inverse_polar(int device, int fftsize, int n_frames, const float *mag, const float *phase, float *frames) {
    if (!frames || !mag || !phase || n_frames < 1) return fail(PVGPU_EINVAL, "bad argument");
    Pipeline pl;
    int rc = stage_pipeline(pl, device, fftsize);
    if (rc) return rc;
    const int N = pl.p.N, H = pl.p.H, Hp = pl.p.Hp;
    DevBuf d_mag, d_ph, d_fr;
    CU(d_mag.ensure(sizeof(float) * (size_t)n_frames * Hp));
    CU(d_ph.ensure(sizeof(float) * (size_t)n_frames * Hp));
    CU(d_fr.ensure(sizeof(float) * (size_t)n_frames * N));
    CU(cudaMemcpy2D(d_mag.p, sizeof(float) * Hp, mag, sizeof(float) * H, sizeof(float) * H, n_frames, cudaMemcpyHostToDevice));
    CU(cudaMemcpy2D(d_ph.p, sizeof(float) * Hp, phase, sizeof(float) * H, sizeof(float) * H, n_frames, cudaMemcpyHostToDevice));
    DevRows g{};
    g.rows = 1; g.channels = 1;
    g.mag = d_mag.as<float>(); g.phase = d_ph.as<float>(); g.F = n_frames;
    g.frames = d_fr.as<float>(); g.Fr = n_frames;
    launch_synthesise(pl.p, g, nullptr, nullptr, 0, n_frames, nullptr);
    CU(cudaGetLastError());
    CU(cudaMemcpy(frames, d_fr.p, sizeof(float) * (size_t)n_frames * N, cudaMemcpyDeviceToHost));
    return PVGPU_OK;
}

int pvgpu_test_atan2f(int device, int64_t n, const float *y, const float *x, float *out) {
    if (!y || !x || !out || n < 1) return fail(PVGPU_EINVAL, "bad argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device >= ndev) return fail(PVGPU_ECUDA, "no CUDA device");
    CU(cudaSetDevice(device));
    DevBuf dy, dx, dout;
    int rc;
    if ((rc = Pipeline::upload(dy, y, sizeof(float) * n))) return rc;
    if ((rc = Pipeline::upload(dx, x, sizeof(float) * n))) return rc;
    CU(dout.ensure(sizeof(float) * n));
    launch_test_atan2f(n, dy.as<float>(), dx.as<float>(), dout.as<float>(), nullptr);
    CU(cudaGetLastError());
    CU(cudaMemcpy(out, dout.p, sizeof(float) * n, cudaMemcpyDeviceToHost));
    return PVGPU_OK;
}

int pvgpu_test_princarg(int device, int64_t n, const double *a, double *out) {
    if (!a || !out || n < 1) return fail(PVGPU_EINVAL, "bad argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device >= ndev) return fail(PVGPU_ECUDA, "no CUDA device");
    CU(cudaSetDevice(device));
    DevBuf da, dout;
    int rc;
    if ((rc = Pipeline::upload(da, a, sizeof(double) * n))) return rc;
    CU(dout.ensure(sizeof(double) * n));
    launch_test_princarg(n, da.as<double>(), dout.as<double>(), nullptr);
    CU(cudaGetLastError());
    CU(cudaMemcpy(out, dout.p, sizeof(double) * n, cudaMemcpyDeviceToHost));
    return PVGPU_OK;
}

int pvgpu_test_postchain(int device, int sample_rate, const pvgpu_fx *chain, int n_fx, int rows, int64_t n, float *samples) {
    if (rows < 1 || n < 0 || (n > 0 && !samples) || sample_rate < 1) return fail(PVGPU_EINVAL, "bad argument");
    PostChain pc{};
    int rc = make_postchain(sample_rate, chain, n_fx, &pc);
    if (rc) return rc;
    if (n == 0) return PVGPU_OK;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) return fail(PVGPU_ECUDA, "no CUDA device");
    CU(cudaSetDevice(device));
    const size_t bytes = sizeof(float) * (size_t)rows * n;
    DevBuf d_x, d_n, d_state;
    if ((rc = Pipeline::upload(d_x, samples, bytes))) return rc;
    const std::vector<int64_t> lim((size_t)rows, n);
    if ((rc = Pipeline::upload(d_n, lim.data(), sizeof(int64_t) * lim.size()))) return rc;
    CU(d_state.ensure(sizeof(float) * (size_t)rows * postchain_state_stride(pc)));
    DevRows g{};
    g.rows = rows; g.channels = 1;
    g.out = d_x.p; g.out_stride = n; g.out_base = 0; g.n_out = d_n.as<int64_t>();
    launch_postchain_reset(pc, d_state.as<float>(), rows, nullptr);
    launch_postchain(g, pc, d_state.as<float>(), 0, n, nullptr);   // the batch's launch, from fresh state
    CU(cudaGetLastError());
    CU(cudaMemcpy(samples, d_x.p, bytes, cudaMemcpyDeviceToHost));
    return PVGPU_OK;
}

int pvgpu_kweighting_design(int sample_rate, double *coeffs) {
    if (sample_rate <= 0 || !coeffs) return fail(PVGPU_EINVAL, "bad argument (sample_rate > 0, non-null coeffs)");
    kweighting_design(sample_rate, coeffs);
    return PVGPU_OK;
}

int pvgpu_test_loudness(int device, int sample_rate, int channels, int streams, int64_t n, int call, const float *samples, float *momentary,
                        float *short_term, float *peak) {
    if (sample_rate < 1 || channels < 1 || streams < 1 || (int64_t)channels * streams > 65535 || n < 0 || call < 1 || (n > 0 && !samples) ||
        !momentary || !short_term || !peak)
        return fail(PVGPU_EINVAL, "bad argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) return fail(PVGPU_ECUDA, "no CUDA device");
    CU(cudaSetDevice(device));
    const size_t R = (size_t)streams * channels, S = (size_t)streams;
    std::vector<float> out(2 * S + R, 0.f);
    std::fill(out.begin(), out.begin() + 2 * S, -INFINITY);
    DevBuf d_x, d_state, d_ring, d_out;
    int rc;
    if (n > 0 && (rc = Pipeline::upload(d_x, samples, sizeof(float) * R * n))) return rc;
    if ((rc = Pipeline::upload(d_out, out.data(), sizeof(float) * out.size()))) return rc;
    CU(d_state.ensure(sizeof(double) * kMeterState * R));
    CU(d_ring.ensure(sizeof(double) * kMeterRing * R));
    CU(cudaMemset(d_state.p, 0, sizeof(double) * kMeterState * R));
    CU(cudaMemset(d_ring.p, 0, sizeof(double) * kMeterRing * R));
    KWeighting kw{};
    kweighting_design(sample_rate, kw.c);
    int pos = 0, ri = 0;
    for (int64_t c0 = 0; c0 < n; c0 += call)   // the engine's launch, one piece after the other
        launch_meters(d_x.as<float>() + c0, PVGPU_F32, n, (int)std::min<int64_t>(call, n - c0), streams, channels, kw, (sample_rate + 5) / 10,
                      d_state.as<double>(), d_ring.as<double>(), d_out.as<float>(), &pos, &ri, nullptr);
    CU(cudaGetLastError());
    CU(cudaMemcpy(out.data(), d_out.p, sizeof(float) * out.size(), cudaMemcpyDeviceToHost));
    std::memcpy(momentary, out.data(), sizeof(float) * S);
    std::memcpy(short_term, out.data() + S, sizeof(float) * S);
    std::memcpy(peak, out.data() + 2 * S, sizeof(float) * R);
    return PVGPU_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// streaming instance: one audiomod::phasevocoder object.  Each process call appends the new input,
// lets the scheduler decide which slices that call runs (exactly the reference's block loop), runs
// those frames on the device and moves the produced samples into a host FIFO.
// ------------------------------------------------------------------------------------------------
// Small persistent pool for the per-row host copies of a live batch (thousands of rows per call: a single thread moves them at
// ~6 GB/s, which is what bounds the call).  run(n, samples_per_item, f) calls f(i) for i in [0, n) on the workers and the caller
// when the call moves at least 256 K samples (1 MB of float32), else on the caller alone.  The threshold counts samples, not
// bytes: 1024 rows of 480 int16 samples (983 KB) packed on one thread took 181 us per call against 64 us for the same rows of
// float32 on the pool (B200 at 1000 W, profiles/r03_live_s16_latency_byte_threshold.jsonl).
struct RowPool {
    std::vector<std::thread> workers;
    std::mutex m;
    std::condition_variable cv_go, cv_done;
    std::function<void(size_t)> fn;
    size_t n = 0, next = 0, chunk = 1, pending = 0;
    uint64_t gen = 0;
    bool stop = false;
    ~RowPool() {
        { std::lock_guard<std::mutex> l(m); stop = true; }
        cv_go.notify_all();
        for (auto &t : workers) t.join();
    }
    void start(int nthreads) {
        for (int i = 0; i < nthreads; ++i)
            workers.emplace_back([this]() {
                uint64_t seen = 0;
                std::unique_lock<std::mutex> l(m);
                for (;;) {
                    cv_go.wait(l, [&]() { return stop || gen != seen; });
                    if (stop) return;
                    seen = gen;
                    drain(l);
                    if (--pending == 0) cv_done.notify_one();
                }
            });
    }
    void drain(std::unique_lock<std::mutex> &l) {   // called with the lock held
        while (next < n) {
            const size_t a = next, b = std::min(n, a + chunk);
            next = b;
            l.unlock();
            for (size_t i = a; i < b; ++i) fn(i);
            l.lock();
        }
    }
    template <typename F> void run(size_t count, size_t samples_per_item, F &&f) {
        if (workers.empty() || count * samples_per_item < ((size_t)1 << 18)) { for (size_t i = 0; i < count; ++i) f(i); return; }
        std::unique_lock<std::mutex> l(m);
        fn = std::forward<F>(f);
        n = count; next = 0; chunk = std::max<size_t>(1, count / (4 * (workers.size() + 1)));
        pending = workers.size();
        ++gen;
        cv_go.notify_all();
        drain(l);
        cv_done.wait(l, [&]() { return pending == 0; });
    }
};

// Output FIFO of a streaming instance: every row holds the same number of samples (the rows advance in lock-step), so it is
// one [rows][cap] block with a common read position -- a ring (cap a power of two), no per-row containers, no compaction.
// The block is page-locked when it can be: the device-to-host copy of a call's output lands in the ring directly.  T is the
// instance's sample type (float, or int16_t for int16 rows).
template <typename T>
struct RowFifo {
    T *buf = nullptr;
    bool pinned = false;
    size_t rows = 0, cap = 0, rd = 0, count = 0;
    ~RowFifo() { release(); }
    void release() { if (buf) { if (pinned) cudaFreeHost(buf); else std::free(buf); } buf = nullptr; cap = 0; }
    void init(size_t rows_) { release(); rows = rows_; rd = count = 0; }
    static T *alloc(size_t bytes, bool *pinned) {
        void *p = nullptr;
        if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) == cudaSuccess) { *pinned = true; return (T *)p; }
        cudaGetLastError();
        *pinned = false;
        return (T *)std::malloc(bytes);
    }
    // only between calls (no copy in flight)
    bool reserve(size_t need) {
        if (need <= cap) return true;
        size_t ncap = cap ? cap : 4096;
        while (ncap < need) ncap *= 2;
        bool np = false;
        T *nb = alloc(sizeof(T) * rows * ncap, &np);
        if (!nb) return false;
        for (size_t r = 0; r < rows; ++r)
            for (size_t i = 0; i < count; ++i) nb[r * ncap + i] = buf[r * cap + ((rd + i) & (cap - 1))];
        release();
        buf = nb; pinned = np; cap = ncap; rd = 0;
        return true;
    }
    // where the next n samples of every row go: [w, w + first) and, if the ring wraps, [0, n - first); call after reserve
    void write_span(size_t n, size_t *w, size_t *first) const { *w = (rd + count) & (cap - 1); *first = std::min(n, cap - *w); }
    void commit(size_t n) { count += n; }
    // remove the oldest k samples of every row into out[r]
    void pop(T *const *out, size_t k, RowPool &pool) {
        if (k == 0) return;
        const size_t first = std::min(k, cap - rd);
        pool.run(rows, k, [&, first, k](size_t r) {
            std::memcpy(out[r], &buf[r * cap + rd], sizeof(T) * first);
            if (first < k) std::memcpy(out[r] + first, &buf[r * cap], sizeof(T) * (k - first));
        });
        rd = (rd + k) & (cap - 1);
        count -= k;
        if (count == 0) rd = 0;
    }
};

struct pvgpu_stream {
    pvgpu_config cfg{};
    int S = 1;                             // streams advancing in lock-step (pvgpu_create_multi); rows = S * channels, stream-major
    int R() const { return S * cfg.channels; }
    std::vector<int64_t> lim;              // per-row limits staged for every call
    Pipeline pl;
    std::unique_ptr<Scheduler> sched;
    std::unique_ptr<Carrier> carrier;
    GlibcRand rng;
    Workspace ws;
    // Kind of rows the instance is fed, fixed by its first data call: 0 not used yet, 1 host rows, 2 device rows (float32),
    // 3 host rows, 4 device rows (int16).  An int16 instance keeps int16 end to end: pending input, packed upload, device window,
    // output rings; the kernels convert as they load and quantise as they store (g.fmt = PVGPU_S16).
    int io_mode = 0;
    bool dev_rows() const { return io_mode == 2 || io_mode == 4; }
    size_t esz() const { return io_mode >= 3 ? sizeof(int16_t) : sizeof(float); }   // bytes per sample of the instance's rows
    // input fed by calls that completed no slice (not yet on the device): [rows][pend_cap] samples of the instance's type,
    // pend_len valid per row
    std::vector<unsigned char> pend;
    size_t pend_cap = 0, pend_len = 0;
    template <typename T> T *pend_row(size_t r) { return reinterpret_cast<T *>(pend.data()) + r * pend_cap; }
    template <typename T> void pend_append(const T *const *in, size_t n) {
        const size_t R_ = (size_t)R();
        if (pend_len + n > pend_cap) {
            size_t ncap = pend_cap ? pend_cap : 1024;
            while (ncap < pend_len + n) ncap *= 2;
            std::vector<unsigned char> nb(sizeof(T) * R_ * ncap);
            for (size_t r = 0; r < R_; ++r) std::memcpy(nb.data() + sizeof(T) * r * ncap, pend_row<T>(r), sizeof(T) * pend_len);
            pend.swap(nb);
            pend_cap = ncap;
        }
        for (size_t r = 0; r < R_; ++r) std::memcpy(pend_row<T>(r) + pend_len, in[r], sizeof(T) * n);
        pend_len += n;
    }
    // The input window [in_base, in_base + dev_len) lives on the device, in one of two buffers of in_cap samples per row: a call
    // uploads only the samples it was fed and compacts the still-needed part into the other buffer on the device.
    DevBuf d_inbuf[2];
    int cur_in = 0;
    int64_t in_cap = 0, dev_len = 0;
    std::vector<float> car_tail;
    int64_t in_base = 0;
    RowFifo<float> fifo;                   // output FIFO of all rows (the reference's outbuf ring)
    RowFifo<int16_t> fifo16;               // the same for int16 rows
    // Device-resident I/O (pvgpu_process_device / _retrieve_device): rows come from and go to device memory, everything is
    // enqueued on the caller's stream and no call waits for the device.  The output FIFO is a ring [rows][dfifo_cap] on the
    // device; what a call uploads is staged in one of four page-locked arenas, each guarded by an event.
    DevBuf d_fifo;
    size_t dfifo_cap = 0, dfifo_rd = 0, dfifo_count = 0;
    static constexpr int kDevArenas = 4;
    PinnedArena dev_arena[kDevArenas];
    cudaEvent_t dev_arena_ev[kDevArenas] = {};
    bool dev_arena_used[kDevArenas] = {};
    unsigned dev_arena_i = 0;
    RowPool pool;                          // host copies of a live batch's rows
    double tr_us[6] = {}, tr_dev[4] = {};  // PVGPU_STREAM_TRACE=1: accumulated microseconds per phase of a call (host) and per device phase
    cudaEvent_t tr_ev[7] = {};
    double tr_dev2[2] = {};
    long tr_calls = 0;
    int num_res = 0;
    DevBuf d_out, d_car, d_len, d_stage;
    // Post-chain (pvgpu_set_postchain): the effects are pl.post, their per-row state is ws.post_state ([R][postchain_state_stride]
    // floats), reset on the stream of the first call that runs the chain after a set (post_fresh).  int16 rows with a chain: the
    // resynthesis stores float32 into post_in ([R][out_stride]) and the chain quantises into d_out.
    DevBuf post_in;
    bool post_fresh = false;
    // Per-stream parameters of the chain (pvgpu_set_stream_postchain): post_coef is the host mirror [S][pl.post.n * 6] of every
    // stream's coefficients (the p[] of pl.post.fx), d_post_coef the device table the per-row kernel reads.  post_differs[j]: stream
    // j's coefficients are not pl.post's, post_n_differ counts them (> 0: the per-row kernel runs).  post_pending lists the streams
    // whose mirror rows the next call that runs the chain uploads, once each (post_is_pending), as records of 1 + 6n floats
    // (post_upd) scattered into the table from d_post_upd.  The setter of the chain sizes all of it.
    std::vector<float> post_coef, post_upd;
    std::vector<unsigned char> post_differs, post_is_pending;
    std::vector<int> post_pending;
    int post_n_differ = 0;
    bool post_force_per_row = false;   // PVGPU_POST_PER_ROW=1 when the instance was created: the per-row kernel for every chain (to
                                       // measure it against the uniform kernel on identical parameters)
    DevBuf d_post_coef, d_post_upd;
    // Loudness meters (pvgpu_set_meters): K-weighting state [kMeterState][R] and sub-block energies [kMeterRing][R] in doubles,
    // results d_meter = [momentary S][short-term S][peak R] floats.  Host rows: every producing call copies d_meter back with its
    // output, through the arena, into meter_host.  The rows advance in lock-step, so one set of counters serves them all: samples
    // measured, samples in the open sub-block of meter_L, ring slot of the next completed sub-block.
    bool meters = false;
    KWeighting kw{};
    int meter_L = 0, meter_pos = 0, meter_ri = 0;
    int64_t measured = 0;
    DevBuf d_meter_state, d_meter_ring, d_meter;
    std::vector<float> meter_host;
    std::vector<float> h_stage, scratch;
    std::vector<unsigned char> h_pack;
    PinnedArena arena;
    cudaStream_t st = nullptr;
    static constexpr int kF = 64;
    ~pvgpu_stream() {
        if (st) cudaStreamDestroy(st);
        for (auto e : tr_ev) if (e) cudaEventDestroy(e);
        for (auto e : dev_arena_ev) if (e) cudaEventDestroy(e);
    }
};

// Room for `len` samples per row in the instance's device-resident input window (rare: the window is bounded by the FFT size
// plus one call's input): grows both buffers, keeps the content.
static int stream_ensure_window(pvgpu_stream *s, int64_t len, cudaStream_t st) {
    if (len <= s->in_cap) return PVGPU_OK;
    const int R = s->R();
    const size_t es = s->esz();
    const int64_t cap = (std::max<int64_t>(2 * s->in_cap, len + 4096) + 3) & ~(int64_t)3;
    DevBuf grown;
    CU(grown.ensure(es * (size_t)R * cap));
    if (s->dev_len > 0)
        CU(cudaMemcpy2DAsync(grown.p, es * cap, s->d_inbuf[s->cur_in].p, es * s->in_cap, es * s->dev_len, R, cudaMemcpyDeviceToDevice, st));
    CU(cudaStreamSynchronize(st));
    std::swap(s->d_inbuf[s->cur_in].p, grown.p);
    std::swap(s->d_inbuf[s->cur_in].bytes, grown.bytes);
    s->d_inbuf[s->cur_in ^ 1].release();
    CU(s->d_inbuf[s->cur_in ^ 1].ensure(es * (size_t)R * cap));
    s->in_cap = cap;
    return PVGPU_OK;
}

template <typename T> static RowFifo<T> &host_fifo(pvgpu_stream *s) {
    if constexpr (std::is_same<T, float>::value) return s->fifo; else return s->fifo16;
}

// One pvgpu_process call that completed `added` new slices starting at slice k0.  Steady state: no heap allocation (the
// vectors keep their capacity), every upload goes through the page-locked arena, one stream synchronisation at the end.
// T is the sample type of the instance's rows (float or int16_t).
template <typename T>
static int stream_run_new(pvgpu_stream *s, long k0, int added, const T *const *in, int n_new, cudaStream_t user_st = nullptr) {
    static_assert(std::is_same<T, float>::value || std::is_same<T, int16_t>::value, "float32 or int16 rows");
    const bool dev = s->dev_rows();        // device rows: the input is already in the window, everything goes on the caller's stream
    cudaStream_t const st = dev ? user_st : s->st;
    Pipeline &pl = s->pl;
    Scheduler &sc = *s->sched;
    const DevPlan &p = pl.p;
    const int C = s->cfg.channels, R = s->R();
    CU(cudaSetDevice(pl.device));
    static const bool trace_env = []() { const char *v = std::getenv("PVGPU_STREAM_TRACE"); return v && v[0] == '1'; }();
    const bool trace = trace_env && !dev;
    auto now = []() { return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double t_start = trace ? now() : 0.0;
    double t_mark = t_start;
    auto mark = [&](int i) { if (trace) { const double t = now(); s->tr_us[i] += t - t_mark; t_mark = t; } };
    if (trace && !s->tr_ev[0]) for (auto &e : s->tr_ev) cudaEventCreate(&e);
    if (trace) cudaEventRecord(s->tr_ev[0], st);
    if (trace) cudaEventRecord(s->tr_ev[6], st);
    const int64_t pend = (int64_t)s->pend_len + n_new;   // earlier calls' samples that completed no slice + this call's
    const int64_t len = s->dev_len + pend;
    const SliceRec &first = sc.recs()[k0 - sc.recs_base()];
    const int64_t out_base = first.out_off;
    const int64_t new_out = sc.total_out() - out_base;
    const int64_t out_stride = std::max<int64_t>((new_out + 3) & ~(int64_t)3, 4);
    {   // room for everything this call stages (nothing is in flight between calls)
        const size_t lists = p.rs_active ? (size_t)(new_out + 8 * 32 * ((added + 3) / 4 + 1) + 64) * 24 + (size_t)added * sizeof(ResampleRun) : 0;
        const size_t need = sizeof(float) * ((size_t)R * (pend + 16) + s->car_tail.size() + sc.norm().size()) + sizeof(SliceRec) * sc.recs().size() +
                            lists + (pl.d.whisper ? sizeof(float) * (size_t)added * C * p.H : 0) + 64 * 16 + sizeof(int64_t) * (2 * R + 1) +
                            sizeof(float) * s->post_pending.size() * (1 + 6 * (size_t)pl.post.n) +
                            (s->meters && !dev ? sizeof(float) * s->meter_host.size() + 64 : 0);
        PinnedArena *ar = &s->arena;
        if (dev) {   // no call waits for the device: rotate the arenas, each is free again when the call that used it has run
            const unsigned i = s->dev_arena_i++ % pvgpu_stream::kDevArenas;
            if (!s->dev_arena_ev[i]) CU(cudaEventCreateWithFlags(&s->dev_arena_ev[i], cudaEventDisableTiming));
            if (s->dev_arena_used[i]) CU(cudaEventSynchronize(s->dev_arena_ev[i]));
            ar = &s->dev_arena[i];
        }
        ar->reserve(need);
        pl.arena = ar;
        pl.staged_all = true;
    }
    int rc;
    if ((rc = stream_ensure_window(s, len, st))) return rc;
    const int64_t in_stride = s->in_cap;
    T *d_in = s->d_inbuf[s->cur_in].as<T>();
    if (pend > 0) {
        // all rows' new samples straight from the caller's rows into one page-locked block, one copy (a live batch of thousands
        // of rows must not issue a copy per row); without page-locked memory the same block is pageable and the copy synchronous
        constexpr int64_t line = 64 / sizeof(T);
        const int64_t pp = (pend + line - 1) & ~(line - 1);   // packed row pitch: rows start on 64-byte lines
        T *pin = (T *)s->arena.take(sizeof(T) * (size_t)R * pp);
        const bool locked = pin != nullptr;
        if (!pin) { s->h_pack.resize(sizeof(T) * (size_t)R * pp); pin = (T *)s->h_pack.data(); }
        const size_t pl_ = s->pend_len;
        // non-temporal stores: the copy engine reads this block next, and lines left dirty in several cores' caches slow it 4-7x
        s->pool.run((size_t)R, (size_t)pend, [&, pl_, pin, pp, locked](size_t r) {
            if (locked) {
                if (pl_) copy_nt(pin + r * pp, s->pend_row<T>(r), pl_);
                if (n_new) copy_nt(pin + r * pp + pl_, in[r], (size_t)n_new);
                copy_nt_fence();
            } else {
                if (pl_) std::memcpy(pin + r * pp, s->pend_row<T>(r), sizeof(T) * pl_);
                if (n_new) std::memcpy(pin + r * pp + pl_, in[r], sizeof(T) * (size_t)n_new);
            }
        });
        mark(0);   // pack
        if (trace) cudaEventRecord(s->tr_ev[5], st);
        if (R >= 64) {
            // many short rows: one contiguous copy over PCIe, then the pitched placement on the device (a host-to-device 2-D copy
            // of 4096 rows of 1.9 KB to 4-byte-aligned destinations ran at 7 GB/s, and so did the device-to-device one)
            CU(s->d_stage.ensure(sizeof(T) * (size_t)R * pp));
            CU(cudaMemcpyAsync(s->d_stage.p, pin, sizeof(T) * (size_t)R * pp, cudaMemcpyHostToDevice, st));
            launch_place_rows(d_in + s->dev_len, in_stride, s->d_stage.as<T>(), pp, (int)pend, R, st);
        } else {
            CU(cudaMemcpy2DAsync(d_in + s->dev_len, sizeof(T) * in_stride, pin, sizeof(T) * pp, sizeof(T) * pend, R, cudaMemcpyHostToDevice, st));
        }
        if (trace) cudaEventRecord(s->tr_ev[6], st);   // input placed
    }
    // per-row limits: [0..R) valid input end, [R..2R) output limit, [2R] carrier length
    s->lim.resize(2 * (size_t)R + 1);
    for (int r = 0; r < R; ++r) { s->lim[r] = s->in_base + len; s->lim[R + r] = INT64_MAX; }
    s->lim[2 * R] = s->in_base + (int64_t)s->car_tail.size();
    CU(s->d_len.ensure(sizeof(int64_t) * (2 * (size_t)R + 1)));
    if ((rc = pl.h2d(s->d_len.p, s->lim.data(), sizeof(int64_t) * (2 * (size_t)R + 1), st))) return rc;
    if ((rc = pl.upload_schedule(sc, st))) return rc;
    if ((rc = pl.build_resample_runs(k0, k0 + added, pl.fused ? pl.fa.run : ola_run_limit(p, 8, pl.max_consumed, pl.max_out), st))) return rc;
    CU(s->d_out.ensure(sizeof(T) * (size_t)R * out_stride));
    const bool chain = pl.post.n > 0;
    const bool chain_s16 = chain && std::is_same<T, int16_t>::value;   // float32 staging between the resynthesis and the chain
    if (chain_s16) CU(s->post_in.ensure(sizeof(float) * (size_t)R * out_stride));
    if (!pl.fused && halo_of(sc.recs(), sc.recs_base(), p.rs_active ? (int)p.rs_filt_len : 1) > s->ws.Fr - s->ws.F) return fail(PVGPU_ESTATE, "too many overlapping (dropped) slices; retrieve output more often");
    DevRows g{};
    g.rows = R; g.channels = C;
    g.in = d_in; g.in_stride = in_stride; g.in_base = s->in_base;
    g.fmt = std::is_same<T, int16_t>::value ? PVGPU_S16 : PVGPU_F32;   // int16: the kernels convert on load and quantise on store
    g.n_in = s->d_len.as<int64_t>(); g.n_out = s->d_len.as<int64_t>() + R;
    g.out = chain_s16 ? s->post_in.p : s->d_out.p; g.out_stride = out_stride; g.out_base = out_base;
    g.out_f32 = chain_s16 ? 1 : 0;
    s->ws.bind(pl, g);
    g.aux_base = k0;
    if (pl.d.whisper) {   // whisperSlice draws rand() channel-major per slice (:814-822): the next added * C * H values of this instance's generator
        const size_t n = (size_t)added * C * p.H;
        s->scratch.resize(n);
        const float two_pi = 2 * M_PI;
        for (size_t i = 0; i < n; ++i) s->scratch[i] = two_pi * (float)s->rng.next() / (float)2147483647;
        CU(pl.b_whisper.ensure(sizeof(float) * n));
        if ((rc = pl.h2d(pl.b_whisper.p, s->scratch.data(), sizeof(float) * n, st))) return rc;
    }
    pl.apply_mode(g);   // after the whisper table has its final address
    if (pl.d.vocoder) {
        const int64_t clen = (int64_t)s->car_tail.size();
        CU(s->d_car.ensure(sizeof(float) * (size_t)std::max<int64_t>(clen, 1)));
        if ((rc = pl.h2d(s->d_car.p, s->car_tail.data(), sizeof(float) * clen, st))) return rc;
        CU(pl.b_carmag.ensure(sizeof(float) * (size_t)added * p.Hp));
        CU(pl.b_carph.ensure(sizeof(float) * (size_t)added * p.Hp));
        DevRows gc{};
        gc.rows = 1; gc.channels = 1;
        gc.in = s->d_car.as<float>(); gc.in_stride = 0; gc.in_base = s->in_base; gc.n_in = s->d_len.as<int64_t>() + 2 * R;
        gc.mag = pl.b_carmag.as<float>(); gc.phase = pl.b_carph.as<float>(); gc.F = added;
        launch_analyse(p, gc, k0, added, st);
    }
    if (trace) cudaEventRecord(s->tr_ev[1], st);   // uploads done
    for (long k = k0; k < k0 + added; k += s->ws.F)
        if ((rc = pl.run_frames(g, k, (int)std::min<long>(s->ws.F, k0 + added - k), st))) return rc;
    if (chain && new_out > 0) {   // every sample the call produced, once and in order, before it enters an output ring
        if (s->post_fresh) { launch_postchain_reset(pl.post, s->ws.post_state.as<float>(), R, st); s->post_fresh = false; }
        if (!s->post_pending.empty()) {   // per-stream parameters set since the last such call: only their rows move
            const size_t n6 = 6 * (size_t)pl.post.n, k = s->post_pending.size();
            s->post_upd.resize(k * (1 + n6));
            for (size_t i = 0; i < k; ++i) {
                const int j = s->post_pending[i];
                float *r = &s->post_upd[i * (1 + n6)];
                std::memcpy(r, &j, sizeof(int));
                std::memcpy(r + 1, &s->post_coef[(size_t)j * n6], sizeof(float) * n6);
                s->post_is_pending[j] = 0;
            }
            s->post_pending.clear();
            if ((rc = pl.h2d(s->d_post_upd.p, s->post_upd.data(), sizeof(float) * s->post_upd.size(), st))) return rc;
            if (!pl.staged_all) { CU(cudaStreamSynchronize(st)); pl.staged_all = true; }   // post_upd is rewritten by the next call
            launch_postchain_coef_scatter(s->d_post_upd.as<float>(), (int)k, (int)n6, s->d_post_coef.as<float>(), st);
        }
        const bool per_row = s->post_n_differ > 0 || s->post_force_per_row;   // the per-row kernel when some stream's coefficients are its own
        launch_postchain_stream(g, pl.post, s->ws.post_state.as<float>(), out_base, out_base + new_out, s->d_out.p, g.fmt,
                                per_row ? s->d_post_coef.as<float>() : nullptr, st);
        ++pl.launches;
    }
    float *meter_pin = nullptr;
    if (s->meters && new_out > 0) {   // the delivered samples, after the chain and before either ring
        launch_meters(s->d_out.p, g.fmt, out_stride, (int)new_out, s->S, C, s->kw, s->meter_L, s->d_meter_state.as<double>(),
                      s->d_meter_ring.as<double>(), s->d_meter.as<float>(), &s->meter_pos, &s->meter_ri, st);
        s->measured += new_out;
        if (!dev) {   // back with the output; without page-locked memory straight into the mirror
            const size_t bytes = sizeof(float) * s->meter_host.size();
            meter_pin = (float *)s->arena.take(bytes);
            CU(cudaMemcpyAsync(meter_pin ? (void *)meter_pin : (void *)s->meter_host.data(), s->d_meter.p, bytes, cudaMemcpyDeviceToHost, st));
        }
    }
    CU(cudaGetLastError());
    if (trace) cudaEventRecord(s->tr_ev[2], st);   // kernels done
    if (new_out > 0 && dev) {   // device rows: append to the device-resident ring
        if (s->dfifo_count + (size_t)new_out > s->dfifo_cap) {   // grow (rare): stop the world, re-lay the ring out
            size_t ncap = s->dfifo_cap ? s->dfifo_cap : 4096;
            while (ncap < s->dfifo_count + (size_t)new_out) ncap *= 2;
            DevBuf grown;
            CU(grown.ensure(sizeof(T) * (size_t)R * ncap));
            if (s->dfifo_count) launch_ring_rows(grown.as<T>(), (int64_t)ncap, 0, -1, s->d_fifo.as<T>(), (int64_t)s->dfifo_cap, (int64_t)s->dfifo_rd, (int64_t)s->dfifo_cap - 1, (int)s->dfifo_count, R, st);
            CU(cudaStreamSynchronize(st));
            std::swap(s->d_fifo.p, grown.p);
            std::swap(s->d_fifo.bytes, grown.bytes);
            s->dfifo_cap = ncap; s->dfifo_rd = 0;
        }
        launch_ring_rows(s->d_fifo.as<T>(), (int64_t)s->dfifo_cap, (int64_t)((s->dfifo_rd + s->dfifo_count) & (s->dfifo_cap - 1)), (int64_t)s->dfifo_cap - 1, s->d_out.as<T>(), out_stride, 0, -1,
                         (int)new_out, R, st);
        s->dfifo_count += (size_t)new_out;
    } else if (new_out > 0) {   // the output goes straight into the (page-locked) FIFO ring
        RowFifo<T> &fifo = host_fifo<T>(s);
        if (!fifo.reserve(fifo.count + (size_t)new_out)) return fail(PVGPU_ENOMEM, "out of host memory");
        size_t w, first;
        fifo.write_span((size_t)new_out, &w, &first);
        CU(cudaMemcpy2DAsync(fifo.buf + w, sizeof(T) * fifo.cap, s->d_out.p, sizeof(T) * out_stride, sizeof(T) * first, R, cudaMemcpyDeviceToHost, st));
        if (first < (size_t)new_out)
            CU(cudaMemcpy2DAsync(fifo.buf, sizeof(T) * fifo.cap, s->d_out.as<T>() + first, sizeof(T) * out_stride, sizeof(T) * ((size_t)new_out - first), R,
                                 cudaMemcpyDeviceToHost, st));
    }
    if (trace) cudaEventRecord(s->tr_ev[3], st);   // output copy done
    // forget the input no later slice can need: the rest of the window moves to the front of the other buffer, on the device
    const long k_next = k0 + added;
    const int64_t new_base = (int64_t)k_next * p.hop;
    const int64_t dropn = std::min<int64_t>(new_base - s->in_base, len);
    const int64_t keep = len - dropn;
    if (dropn > 0) {
        if (keep > 0)
            CU(cudaMemcpy2DAsync(s->d_inbuf[s->cur_in ^ 1].p, sizeof(T) * in_stride, d_in + dropn, sizeof(T) * in_stride, sizeof(T) * keep, R, cudaMemcpyDeviceToDevice, st));
        s->cur_in ^= 1;
    }
    if (trace) cudaEventRecord(s->tr_ev[4], st);   // window compaction done
    mark(1);   // enqueue: schedule upload, work lists, launches, copies
    if (dev) {
        const unsigned i = (s->dev_arena_i - 1) % pvgpu_stream::kDevArenas;
        CU(cudaEventRecord(s->dev_arena_ev[i], st));
        s->dev_arena_used[i] = true;
    } else {
        CU(cudaStreamSynchronize(st));   // the call's only synchronisation
    }
    mark(2);   // device
    if (trace) for (int i = 0; i < 4; ++i) { float ms = 0; cudaEventElapsedTime(&ms, s->tr_ev[i], s->tr_ev[i + 1]); s->tr_dev[i] += 1e3 * ms; }
    if (trace && pend > 0) { float ms = 0; cudaEventElapsedTime(&ms, s->tr_ev[0], s->tr_ev[5]); s->tr_dev2[0] += 1e3 * ms; cudaEventElapsedTime(&ms, s->tr_ev[5], s->tr_ev[6]); s->tr_dev2[1] += 1e3 * ms; }
    pl.staged_all = true;
    if (meter_pin) std::memcpy(s->meter_host.data(), meter_pin, sizeof(float) * s->meter_host.size());
    if (new_out > 0 && !dev) host_fifo<T>(s).commit((size_t)new_out);
    s->pend_len = 0;
    s->dev_len = keep;
    if (pl.d.vocoder) s->car_tail.erase(s->car_tail.begin(), s->car_tail.begin() + std::min<int64_t>(dropn, (int64_t)s->car_tail.size()));
    s->in_base += dropn;
    if (pl.fused) {
        // the fused kernel carries the unfinished accumulator and the resampler history on the device: the schedule and the
        // normalisers before the next slice are never needed again, so a call uploads only what it added
        sc.trim(k_next, sc.ola_total());
    } else {
        // keep every record / normaliser a later slice can still reach: the slices holding the last filt_len-1 samples of
        // the normalised stream (resampler history) and the frames overlapping them
        const auto &recs = sc.recs();
        const int64_t L = p.rs_active ? (int64_t)p.rs_filt_len : 1;
        size_t kh = recs.size() - 1;
        while (kh > 0 && recs[kh].res_off > sc.res_total() - L) --kh;
        sc.trim(recs[kh].jlo, recs[kh].ola_off);
    }
    mark(3);   // trim
    if (trace && ++s->tr_calls % 50 == 0) {
        std::fprintf(stderr, "[pvgpu stream trace] rows %d: pack %.1f us, enqueue %.1f, device wait %.1f, trim %.1f | device: uploads %.1f, kernels %.1f, output copy %.1f, window compaction %.1f per call (last 50)\n",
                     R, s->tr_us[0] / 50, s->tr_us[1] / 50, s->tr_us[2] / 50, s->tr_us[3] / 50, s->tr_dev[0] / 50, s->tr_dev[1] / 50, s->tr_dev[2] / 50, s->tr_dev[3] / 50);
        for (double &v : s->tr_us) v = 0;
        std::fprintf(stderr, "[pvgpu stream trace]   of the uploads: until the packed block is ready %.1f us, input copy + placement %.1f\n", s->tr_dev2[0] / 50, s->tr_dev2[1] / 50);
        s->tr_dev2[0] = s->tr_dev2[1] = 0;
        for (double &v : s->tr_dev) v = 0;
    }
    return PVGPU_OK;
}

// Ring FIFO of one sample type across wrap-arounds, growth and partial pops against a plain model.  Returns 0 or base + the
// number of the failed check (1 reserve, 2 popped samples, 3 a sample past the popped ones written, 4 count).
template <typename T> static int fifo_selftest(int base) {
    const size_t R = 7;
    RowFifo<T> f;
    f.init(R);
    RowPool none;
    std::vector<std::vector<T>> model(R);
    std::vector<T *> out(R);
    std::vector<std::vector<T>> got(R);
    unsigned seed = 12345;
    float next = 0.f;
    for (int it = 0; it < 400; ++it) {
        seed = seed * 1664525u + 1013904223u;
        const size_t n = (seed >> 16) % (it % 50 == 49 ? 9000 : 700);
        if (!f.reserve(f.count + n)) return base + 1;
        size_t w, first;
        f.write_span(n, &w, &first);
        for (size_t r = 0; r < R; ++r)
            for (size_t i = 0; i < n; ++i) {
                T v;
                if constexpr (std::is_same<T, float>::value) v = next + (float)r * 0.25f + (float)i;
                else v = (T)(uint16_t)((unsigned)it * 977u + (unsigned)r * 131u + (unsigned)i);   // every bit pattern, -1 included
                model[r].push_back(v);
                if (i < first) f.buf[r * f.cap + w + i] = v; else f.buf[r * f.cap + (i - first)] = v;
            }
        next += 1000.f;
        f.commit(n);
        seed = seed * 1664525u + 1013904223u;
        const size_t k = std::min<size_t>(f.count, (seed >> 16) % 900);
        for (size_t r = 0; r < R; ++r) { got[r].assign(k + 1, (T)-1); out[r] = got[r].data(); }
        f.pop(out.data(), k, none);
        for (size_t r = 0; r < R; ++r) {
            for (size_t i = 0; i < k; ++i) if (got[r][i] != model[r][i]) return base + 2;
            if (got[r][k] != (T)-1) return base + 3;
            model[r].erase(model[r].begin(), model[r].begin() + (long)k);
        }
        if (f.count != model[0].size()) return base + 4;
    }
    return 0;
}

// Host-only self-test of the live batch's containers (no device work): the ring FIFO across wrap-arounds and growth, the
// row-copy pool against a serial copy, non-temporal copies at every alignment; float32 rows (checks 1-6), int16 rows (7-11).
// Returns 0 or the number of the failed check.
static int host_structs_selftest() {
    int rc;
    if ((rc = fifo_selftest<float>(0))) return rc;
    {   // RowPool + copy_nt
        RowPool pool;
        pool.start(3);
        const size_t R = 600, n = 1031;
        std::vector<float> src(R * n), a(R * (n + 24), -2.f), b(R * (n + 24), -2.f);
        for (size_t i = 0; i < src.size(); ++i) src[i] = (float)(i % 9973) * 0.5f;
        for (int rep = 0; rep < 20; ++rep) {
            const size_t shift = (size_t)rep % 8;   // every destination alignment
            pool.run(R, n, [&](size_t r) { copy_nt(&a[r * (n + 24) + shift], &src[r * n], n); copy_nt_fence(); });
            for (size_t r = 0; r < R; ++r) std::memcpy(&b[r * (n + 24) + shift], &src[r * n], sizeof(float) * n);
            if (std::memcmp(a.data(), b.data(), sizeof(float) * a.size()) != 0) return 5;
        }
        size_t hits = 0;
        std::vector<unsigned char> seen(R, 0);
        pool.run(R, (size_t)1 << 18, [&](size_t r) { seen[r]++; });
        for (unsigned char c : seen) hits += c;
        if (hits != R) return 6;
    }
    if ((rc = fifo_selftest<int16_t>(6))) return rc;
    {   // 16-bit copy_nt at every 2-byte destination alignment of a 16-byte line, odd and even lengths, through the pool
        RowPool pool;
        pool.start(3);
        const size_t R = 600;
        for (size_t n : {(size_t)0, (size_t)1, (size_t)2, (size_t)3, (size_t)8, (size_t)9, (size_t)17, (size_t)1031}) {
            std::vector<int16_t> src(R * n), a(R * (n + 24), -2), b(R * (n + 24), -2);
            for (size_t i = 0; i < src.size(); ++i) src[i] = (int16_t)(uint16_t)(i * 40503u);
            for (size_t shift = 0; shift < 8; ++shift) {
                pool.run(R, n, [&](size_t r) { copy_nt(&a[r * (n + 24) + shift], &src[r * n], n); copy_nt_fence(); });
                for (size_t r = 0; r < R; ++r) std::memcpy(&b[r * (n + 24) + shift], &src[r * n], sizeof(int16_t) * n);
                if (std::memcmp(a.data(), b.data(), sizeof(int16_t) * a.size()) != 0) return 11;
            }
        }
    }
    return 0;
}

extern "C" {

int pvgpu_test_host_structs(void) {
    int rc = 0;
    const int g = guarded([&]() -> int { rc = host_structs_selftest(); return PVGPU_OK; });
    return g != PVGPU_OK ? -g : rc;
}

static int pvgpu_create_body(const pvgpu_config *cfg, int n_streams, pvgpu_stream **out);
int pvgpu_create(const pvgpu_config *cfg, pvgpu_stream **out) {
    return guarded([&]() -> int { return pvgpu_create_body(cfg, 1, out); });
}
int pvgpu_create_multi(const pvgpu_config *cfg, int n_streams, pvgpu_stream **out) {
    return guarded([&]() -> int { return pvgpu_create_body(cfg, n_streams, out); });
}
int pvgpu_stream_count(const pvgpu_stream *s) { return s ? s->S : 0; }
static int pvgpu_create_body(const pvgpu_config *cfg, int n_streams, pvgpu_stream **out) {
    int rc = validate(cfg);
    if (rc) return rc;
    if (!out) return fail(PVGPU_EINVAL, "null out pointer");
    if (n_streams < 1 || (long)n_streams * cfg->channels > 65535) return fail(PVGPU_EINVAL, "n_streams * channels must be 1..65535");
    std::unique_ptr<pvgpu_stream> s(new (std::nothrow) pvgpu_stream);
    if (!s) return fail(PVGPU_ENOMEM, "out of host memory");
    s->cfg = *cfg;
    s->S = n_streams;
    {
        const char *v = std::getenv("PVGPU_POST_PER_ROW");
        s->post_force_per_row = v && v[0] == '1';
    }
    if ((rc = s->pl.init(*cfg))) return rc;
    s->sched.reset(new Scheduler(s->pl.d, true));
    if (s->pl.d.vocoder) s->carrier.reset(new Carrier(cfg->sample_rate, cfg->mode == PVGPU_VOCODER_CHORD));
    s->fifo.init((size_t)s->R());
    s->fifo16.init((size_t)s->R());
    if (s->R() >= 256) s->pool.start((int)std::min(7u, std::max(1u, std::thread::hardware_concurrency() / 2)));   // live batch: parallel row copies
    CU(cudaStreamCreateWithFlags(&s->st, cudaStreamNonBlocking));
    const int halo = 80;
    s->pl.ola_run = 8;
    {   // fused kernel shape from bounds that hold for the whole stream: the increment is clamped to twice its nominal value
        // (phasevocoderprocess.cc:392-397); robotic / whisper / vocoder / constant / integer ratios advance by a fixed amount
        const Derived &d = s->pl.d;
        const bool fixed = d.robotic || d.whisper || d.vocoder || d.constant_mode || d.int_ratio;
        const int nominal = fixed ? (d.int_ratio && !(d.robotic || d.whisper || d.vocoder || d.constant_mode) ? (int)(size_t)(d.hop * d.hs) : d.hop)
                                  : (int)std::lrint(2.0 * d.hop * (double)d.hs) + 2;
        const int out_bound = (int)std::ceil(nominal * (double)(s->pl.p.rs_active ? d.rs.ratio : 1.f)) + 2;
        // split kernels: the instance's frame ring holds `halo` frames before a chunk; dozens of overlapping frames (extreme
        // stretch ratios) or a resampler history of many slices need the fused kernel
        const int min_shift = std::max(1, fixed ? nominal : (int)std::lrint(0.5 * d.hop * (double)d.hs));
        const int overlap = (d.N + min_shift - 1) / min_shift + (s->pl.p.rs_active ? ((int)d.rs.filt_len + min_shift - 1) / min_shift : 0) + 2;
        s->pl.plan_fused(pvgpu_stream::kF, std::max(nominal, 1), out_bound, overlap + 8 <= halo && overlap + 8 <= ola_max_table_slices() - 1);
    }
    if ((rc = s->ws.ensure(s->pl, s->R(), pvgpu_stream::kF, halo))) return rc;
    if ((rc = s->ws.reset_state(s->pl, s->st))) return rc;
    CU(cudaStreamSynchronize(s->st));   // device-row calls run on the caller's stream: the state must be in place before any of them
    *out = s.release();
    return PVGPU_OK;
}

void pvgpu_destroy(pvgpu_stream *s) {
    if (!s) return;
    cudaSetDevice(s->pl.device);
    delete s;
}

int pvgpu_stream_info(const pvgpu_stream *s, pvgpu_info *info) {
    if (!s || !info) return fail(PVGPU_EINVAL, "null argument");
    fill_info(s->pl.d, info);
    return PVGPU_OK;
}

// Earlier calls' kernels may still use the instance's device state (device-row calls do not wait): host-row calls ran on s->st,
// every device-row call recorded the event of its staging arena after its kernels.
static int stream_wait_idle(pvgpu_stream *s) {
    CU(cudaSetDevice(s->pl.device));
    CU(cudaStreamSynchronize(s->st));
    for (int i = 0; i < pvgpu_stream::kDevArenas; ++i)
        if (s->dev_arena_used[i]) CU(cudaEventSynchronize(s->dev_arena_ev[i]));
    return PVGPU_OK;
}

static int pvgpu_set_postchain_body(pvgpu_stream *s, const pvgpu_fx *chain, int n_fx) {
    if (!s) return fail(PVGPU_EINVAL, "bad post-chain (at most %d effects)", kMaxPostFx);
    PostChain pc{};
    int rc = make_postchain(s->cfg.sample_rate, chain, n_fx, &pc);
    if (rc) return rc;
    if (!s->pl.d.valid_mode) return PVGPU_OK;   // an instance of an unknown mode produces nothing (phasevocoder.cc:104-106)
    if ((rc = stream_wait_idle(s))) return rc;
    const size_t S = (size_t)s->S, n6 = 6 * (size_t)pc.n;
    if (pc.n > 0) {   // every stream starts with the chain's coefficients; the per-stream setter allocates nothing
        CU(s->ws.post_state.ensure(sizeof(float) * (size_t)s->R() * postchain_state_stride(pc)));
        CU(s->d_post_coef.ensure(sizeof(float) * S * n6));
        CU(s->d_post_upd.ensure(sizeof(float) * S * (1 + n6)));
        s->post_coef.resize(S * n6);
        for (size_t j = 0; j < S; ++j)
            for (int k = 0; k < pc.n; ++k) std::memcpy(&s->post_coef[(j * pc.n + k) * 6], pc.fx[k].p, sizeof(float) * 6);
        CU(cudaMemcpy(s->d_post_coef.p, s->post_coef.data(), sizeof(float) * S * n6, cudaMemcpyHostToDevice));
        s->post_upd.reserve(S * (1 + n6));
        s->post_pending.reserve(S);
    }
    s->post_differs.assign(S, 0);
    s->post_is_pending.assign(S, 0);
    s->post_pending.clear();
    s->post_n_differ = 0;
    s->pl.post = pc;
    s->post_fresh = pc.n > 0;   // fresh effect state, reset on the stream of the next call that runs the chain
    return PVGPU_OK;
}
int pvgpu_set_postchain(pvgpu_stream *s, const pvgpu_fx *chain, int n_fx) {
    return guarded([&]() -> int { return pvgpu_set_postchain_body(s, chain, n_fx); });
}

static const char *fx_name(int kind) {
    switch (kind) {
        case PVGPU_FX_GAIN: return "gain";
        case PVGPU_FX_COMPRESSOR: return "compressor";
        case PVGPU_FX_LIMITER: return "limiter";
        case PVGPU_FX_BIQUAD: return "biquad";
        default: return "unknown effect";
    }
}

// Host arithmetic and bookkeeping only: no device work, no allocation (the setter of the chain sized everything).
static int pvgpu_set_stream_postchain_body(pvgpu_stream *s, int stream, const pvgpu_fx *chain, int n_fx) {
    if (!s) return fail(PVGPU_EINVAL, "null instance");
    if (stream < 0 || stream >= s->S) return fail(PVGPU_EINVAL, "stream %d outside [0, %d)", stream, s->S);
    if (!chain) return fail(PVGPU_EINVAL, "null chain");
    PostChain pc{};
    int rc = make_postchain(s->cfg.sample_rate, chain, n_fx, &pc);
    if (rc) return rc;
    if (!s->pl.d.valid_mode) return PVGPU_OK;   // an instance of an unknown mode produces nothing (phasevocoder.cc:104-106)
    const PostChain &have = s->pl.post;
    if (have.n == 0) return fail(PVGPU_EINVAL, "this instance has no post-chain (pvgpu_set_postchain first)");
    if (pc.n != have.n) return fail(PVGPU_EINVAL, "chain of %d effects; this instance's chain has %d", pc.n, have.n);
    for (int k = 0; k < pc.n; ++k)
        if (pc.fx[k].kind != have.fx[k].kind)
            return fail(PVGPU_EINVAL, "effect %d is a %s; this instance's effect %d is a %s", k, fx_name(pc.fx[k].kind), k, fx_name(have.fx[k].kind));
    float *row = &s->post_coef[(size_t)stream * pc.n * 6];
    bool differs = false;
    for (int k = 0; k < pc.n; ++k) {
        std::memcpy(row + 6 * k, pc.fx[k].p, sizeof(float) * 6);
        differs = differs || std::memcmp(pc.fx[k].p, have.fx[k].p, sizeof(float) * 6) != 0;
    }
    s->post_n_differ += (int)differs - (int)s->post_differs[stream];
    s->post_differs[stream] = differs;
    if (!s->post_is_pending[stream]) { s->post_is_pending[stream] = 1; s->post_pending.push_back(stream); }
    return PVGPU_OK;
}
int pvgpu_set_stream_postchain(pvgpu_stream *s, int stream, const pvgpu_fx *chain, int n_fx) {
    return guarded([&]() -> int { return pvgpu_set_stream_postchain_body(s, stream, chain, n_fx); });
}

}  // extern "C"

// The kind of rows an instance takes is fixed by its first data call (pvgpu_stream::io_mode); a call of another kind is refused
// with the name of the call to use.
static const char *const kRowKind[5] = {"", "host", "device", "host int16", "device int16"};
static const char *const kProcessCall[5] = {"", "pvgpu_process", "pvgpu_process_device", "pvgpu_process_s16", "pvgpu_process_device_s16"};
static const char *const kRetrieveCall[5] = {"", "pvgpu_retrieve", "pvgpu_retrieve_device", "pvgpu_retrieve_s16", "pvgpu_retrieve_device_s16"};
static int lock_rows(pvgpu_stream *s, int mode) {
    const int have = s->io_mode;
    if (have && have != mode)
        return fail(PVGPU_ESTATE, "this instance is fed %s rows (%s); %s rows cannot be mixed", kRowKind[have], kProcessCall[have],
                    (have >= 3) != (mode >= 3) ? "float32 and int16" : "host and device");
    s->io_mode = mode;
    return PVGPU_OK;
}
static int check_retrieve_rows(const pvgpu_stream *s, int mode) {
    const int have = s->io_mode;
    if (have && have != mode) return fail(PVGPU_ESTATE, "this instance is fed %s rows; use %s", kRowKind[have], kRetrieveCall[have]);
    return PVGPU_OK;
}

template <typename T>
static int process_host(pvgpu_stream *s, const T *const *in, int n) {
    if (!s || n < 0 || (n > 0 && !in)) return fail(PVGPU_EINVAL, "bad argument");
    if (!s->pl.d.valid_mode) { s->num_res = 0; return PVGPU_OK; }  // phasevocoder.cc:104-106: unknown mode does nothing
    int rc;
    if ((rc = lock_rows(s, std::is_same<T, float>::value ? 1 : 3))) return rc;
    if (s->carrier) {
        const size_t at = s->car_tail.size();
        s->car_tail.resize(at + n);
        s->carrier->generate(s->car_tail.data() + at, (size_t)n);
    }
    const long k0 = s->sched->recs_base() + s->sched->slices();
    const int added = s->sched->feed(n);   // the schedule does not depend on the data
    if (added > 0) {
        if ((rc = stream_run_new<T>(s, k0, added, in, n))) return rc;
    } else if (n > 0) {
        s->pend_append<T>(in, (size_t)n);
    }
    s->num_res = (int)s->sched->available();
    return PVGPU_OK;
}

template <typename T>
static int retrieve_host(pvgpu_stream *s, T *const *out, int n) {
    if (!s || n < 0 || (n > 0 && !out)) return -fail(PVGPU_EINVAL, "bad argument");
    if (check_retrieve_rows(s, std::is_same<T, float>::value ? 1 : 3)) return -PVGPU_ESTATE;
    RowFifo<T> &fifo = host_fifo<T>(s);
    long k = std::min<long>(n, s->num_res);  // phasevocoder.cc:111-113
    k = std::min<long>(k, s->sched->available());
    k = std::min<long>(k, (long)fifo.count);
    fifo.pop(out, (size_t)k, s->pool);
    s->sched->drain(k);
    return (int)k;
}

template <typename T>
static int process_block_host(pvgpu_stream *s, T *const *buf, int n, int *ready) {
    if (!s || !ready) return fail(PVGPU_EINVAL, "bad argument");
    const int m = s->cfg.mode;
    if (m == PVGPU_NORMAL_STRETCH || m < -1 || m > PVGPU_FORMANT_CEPSTRAL) { *ready = 1; return PVGPU_OK; }  // processBlock routes neither (phasevocoder.cc:133-146)
    int rc = guarded([&]() -> int { return process_host<T>(s, buf, n); });
    if (rc) return rc;
    if (s->num_res >= n) {  // processBlockNormal, phasevocoder.cc:156-183
        const int saved = s->num_res;
        retrieve_host<T>(s, buf, n);
        s->num_res = saved;
        *ready = 1;
    } else {
        *ready = 0;
    }
    return PVGPU_OK;
}

template <typename T>
static int process_device(pvgpu_stream *s, const T *d_in, int64_t in_pitch, int n, cudaStream_t st) {
    if (!s || n < 0 || (n > 0 && !d_in) || in_pitch < n) return fail(PVGPU_EINVAL, "bad argument");
    if (!s->pl.d.valid_mode) { s->num_res = 0; return PVGPU_OK; }
    int rc;
    if ((rc = lock_rows(s, std::is_same<T, float>::value ? 2 : 4))) return rc;
    CU(cudaSetDevice(s->pl.device));
    if (s->carrier) {
        const size_t at = s->car_tail.size();
        s->car_tail.resize(at + n);
        s->carrier->generate(s->car_tail.data() + at, (size_t)n);
    }
    const long k0 = s->sched->recs_base() + s->sched->slices();
    const int added = s->sched->feed(n);   // the schedule does not depend on the data: no call has to wait for the device
    if (n > 0) {   // the new samples join the device-resident window right away
        if ((rc = stream_ensure_window(s, s->dev_len + n, st))) return rc;
        launch_place_rows(s->d_inbuf[s->cur_in].as<T>() + s->dev_len, s->in_cap, d_in, in_pitch, n, s->R(), st);
        s->dev_len += n;
    }
    if (added > 0 && (rc = stream_run_new<T>(s, k0, added, nullptr, 0, st))) return rc;
    s->num_res = (int)s->sched->available();
    return PVGPU_OK;
}

template <typename T>
static int retrieve_device(pvgpu_stream *s, T *d_out, int64_t out_pitch, int n, void *cuda_stream) {
    if (!s || n < 0 || (n > 0 && !d_out) || out_pitch < n) return -fail(PVGPU_EINVAL, "bad argument");
    if (check_retrieve_rows(s, std::is_same<T, float>::value ? 2 : 4)) return -PVGPU_ESTATE;
    long k = std::min<long>(n, s->num_res);
    k = std::min<long>(k, s->sched->available());
    k = std::min<long>(k, (long)s->dfifo_count);
    if (k > 0) {
        if (cudaSetDevice(s->pl.device) != cudaSuccess) return -fail(PVGPU_ECUDA, "cudaSetDevice failed");
        launch_ring_rows(d_out, out_pitch, 0, -1, s->d_fifo.as<T>(), (int64_t)s->dfifo_cap, (int64_t)s->dfifo_rd, (int64_t)s->dfifo_cap - 1, (int)k, s->R(),
                         cuda_stream ? (cudaStream_t)cuda_stream : cudaStreamLegacy);
        s->dfifo_rd = (s->dfifo_rd + (size_t)k) & (s->dfifo_cap - 1);
        s->dfifo_count -= (size_t)k;
        if (s->dfifo_count == 0) s->dfifo_rd = 0;
    }
    s->sched->drain(k);
    return (int)k;
}

template <typename T>
static int process_block_device(pvgpu_stream *s, T *d_buf, int64_t pitch, int n, void *cuda_stream, int *ready) {
    if (!s || !ready) return fail(PVGPU_EINVAL, "bad argument");
    const int m = s->cfg.mode;
    if (m == PVGPU_NORMAL_STRETCH || m < -1 || m > PVGPU_FORMANT_CEPSTRAL) { *ready = 1; return PVGPU_OK; }
    int rc = guarded([&]() -> int { return process_device<T>(s, d_buf, pitch, n, cuda_stream ? (cudaStream_t)cuda_stream : cudaStreamLegacy); });
    if (rc) return rc;
    if (s->num_res >= n) {
        const int saved = s->num_res;
        const int k = retrieve_device<T>(s, d_buf, pitch, n, cuda_stream);
        if (k < 0) return -k;
        s->num_res = saved;
        *ready = 1;
    } else {
        *ready = 0;
    }
    return PVGPU_OK;
}

extern "C" {

int pvgpu_process(pvgpu_stream *s, const float *const *in, int n) {
    return guarded([&]() -> int { return process_host<float>(s, in, n); });
}
int pvgpu_process_s16(pvgpu_stream *s, const int16_t *const *in, int n) {
    return guarded([&]() -> int { return process_host<int16_t>(s, in, n); });
}

int pvgpu_available(const pvgpu_stream *s) { return s ? s->num_res : 0; }

int pvgpu_retrieve(pvgpu_stream *s, float *const *out, int n) { return retrieve_host<float>(s, out, n); }
int pvgpu_retrieve_s16(pvgpu_stream *s, int16_t *const *out, int n) { return retrieve_host<int16_t>(s, out, n); }

int pvgpu_process_block(pvgpu_stream *s, float *const *buf, int n, int *ready) { return process_block_host<float>(s, buf, n, ready); }
int pvgpu_process_block_s16(pvgpu_stream *s, int16_t *const *buf, int n, int *ready) { return process_block_host<int16_t>(s, buf, n, ready); }

int pvgpu_process_device(pvgpu_stream *s, const float *d_in, int64_t in_pitch, int n, void *cuda_stream) {
    return guarded([&]() -> int { return process_device<float>(s, d_in, in_pitch, n, cuda_stream ? (cudaStream_t)cuda_stream : cudaStreamLegacy); });
}
int pvgpu_process_device_s16(pvgpu_stream *s, const int16_t *d_in, int64_t in_pitch, int n, void *cuda_stream) {
    return guarded([&]() -> int { return process_device<int16_t>(s, d_in, in_pitch, n, cuda_stream ? (cudaStream_t)cuda_stream : cudaStreamLegacy); });
}

int pvgpu_retrieve_device(pvgpu_stream *s, float *d_out, int64_t out_pitch, int n, void *cuda_stream) {
    return retrieve_device<float>(s, d_out, out_pitch, n, cuda_stream);
}
int pvgpu_retrieve_device_s16(pvgpu_stream *s, int16_t *d_out, int64_t out_pitch, int n, void *cuda_stream) {
    return retrieve_device<int16_t>(s, d_out, out_pitch, n, cuda_stream);
}

int pvgpu_process_block_device(pvgpu_stream *s, float *d_buf, int64_t pitch, int n, void *cuda_stream, int *ready) {
    return process_block_device<float>(s, d_buf, pitch, n, cuda_stream, ready);
}
int pvgpu_process_block_device_s16(pvgpu_stream *s, int16_t *d_buf, int64_t pitch, int n, void *cuda_stream, int *ready) {
    return process_block_device<int16_t>(s, d_buf, pitch, n, cuda_stream, ready);
}

static int pvgpu_set_meters_body(pvgpu_stream *s, int enable) {
    if (!s || (enable != 0 && enable != 1)) return fail(PVGPU_EINVAL, "bad argument (enable is 0 or 1)");
    int rc;
    if ((rc = stream_wait_idle(s))) return rc;   // earlier calls' kernels may still read or write the meter state
    s->meters = false;
    if (!enable) return PVGPU_OK;
    const size_t R = (size_t)s->R(), S = (size_t)s->S;
    CU(s->d_meter_state.ensure(sizeof(double) * kMeterState * R));
    CU(s->d_meter_ring.ensure(sizeof(double) * kMeterRing * R));   // sub-blocks before the first measured sample are silence
    CU(s->d_meter.ensure(sizeof(float) * (2 * S + R)));
    s->meter_host.assign(2 * S + R, 0.f);
    std::fill(s->meter_host.begin(), s->meter_host.begin() + 2 * S, -INFINITY);
    CU(cudaMemsetAsync(s->d_meter_state.p, 0, sizeof(double) * kMeterState * R, s->st));
    CU(cudaMemsetAsync(s->d_meter_ring.p, 0, sizeof(double) * kMeterRing * R, s->st));
    CU(cudaMemcpyAsync(s->d_meter.p, s->meter_host.data(), sizeof(float) * s->meter_host.size(), cudaMemcpyHostToDevice, s->st));
    CU(cudaStreamSynchronize(s->st));   // device-row calls run on the caller's stream: the fresh state must be in place first
    kweighting_design(s->cfg.sample_rate, s->kw.c);
    s->meter_L = (s->cfg.sample_rate + 5) / 10;
    s->meter_pos = s->meter_ri = 0;
    s->measured = 0;
    s->meters = true;
    return PVGPU_OK;
}
int pvgpu_set_meters(pvgpu_stream *s, int enable) {
    return guarded([&]() -> int { return pvgpu_set_meters_body(s, enable); });
}

// A getter of the other kind of rows is refused with the name of the one to use; before the first data call either works.
static int check_meters(const pvgpu_stream *s, bool device_getter) {
    if (!s->meters) return fail(PVGPU_ESTATE, "meters are off on this instance (pvgpu_set_meters)");
    if (s->io_mode && s->dev_rows() != device_getter)
        return fail(PVGPU_ESTATE, "this instance is fed %s rows; use %s", kRowKind[s->io_mode], s->dev_rows() ? "pvgpu_get_meters_device" : "pvgpu_get_meters");
    return PVGPU_OK;
}

int pvgpu_get_meters(const pvgpu_stream *s, float *momentary, float *short_term, float *peak, int64_t *measured) {
    if (!s) return fail(PVGPU_EINVAL, "null instance");
    int rc;
    if ((rc = check_meters(s, false))) return rc;
    const size_t S = (size_t)s->S;
    const float *h = s->meter_host.data();
    if (momentary) std::memcpy(momentary, h, sizeof(float) * S);
    if (short_term) std::memcpy(short_term, h + S, sizeof(float) * S);
    if (peak) std::memcpy(peak, h + 2 * S, sizeof(float) * (size_t)s->R());
    if (measured) *measured = s->measured;
    return PVGPU_OK;
}

int pvgpu_get_meters_device(pvgpu_stream *s, float *d_dst, void *cuda_stream, int64_t *measured) {
    if (!s || !d_dst) return fail(PVGPU_EINVAL, "null argument");
    int rc;
    if ((rc = check_meters(s, true))) return rc;
    CU(cudaSetDevice(s->pl.device));
    CU(cudaMemcpyAsync(d_dst, s->d_meter.p, sizeof(float) * s->meter_host.size(), cudaMemcpyDeviceToDevice,
                       cuda_stream ? (cudaStream_t)cuda_stream : cudaStreamLegacy));
    if (measured) *measured = s->measured;
    return PVGPU_OK;
}

}  // extern "C"
