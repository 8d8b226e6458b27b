/*
 * pv_oracle.c -- TEST INFRASTRUCTURE ONLY.  Never linked, imported or executed by the
 * product path (audiomod_b200/, include/, the C-ABI library).  Only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may use it.
 *
 * A scalar CPU restatement of tangkk/audiomod's phase-vocoder path for ONE stream with
 * fresh-process semantics (every piece of process-global state of the reference lives in
 * the per-stream struct here).  Each function cites the reference file:line it follows
 * (paths relative to /root/reference).  It is written to round exactly like the
 * reference's default build (x86-64 SSE2, -O3, no FMA contraction): compile with
 * -ffp-contract=off.  libm calls (atan2f, sinf, cosf, cos, sin, floor, lrint, round,
 * pow) go to the host glibc, like the reference's.
 *
 * Parity pin: the reference has no tests or golden vectors of its own (SURVEY.md s.4), so
 * this file is pinned against the UNMODIFIED reference compiled into oracle/_ref
 * (tests/test_oracle_vs_ref.py, bit-exact) and against fixtures generated from it
 * (tests/golden/, generator tests/golden/make_golden.py).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#ifndef M_PI
#define M_PI 3.14159265358979323846
#endif

/* mode constants: include/dafx/phasevocoder.h:22-30 */
enum { MODE_CONSTANT = -1, MODE_SHIFT = 0, MODE_GENDER = 1, MODE_FORMANT = 2, MODE_VOC_ROSEN = 3,
       MODE_VOC_CHORD = 4, MODE_STRETCH = 5, MODE_ROBOTIC = 6, MODE_WHISPER = 7 };

typedef struct { float r, i; } cpx;

/* ------------------------------------------------------------------------------------
 * Real FFT: restates the arithmetic of the vendored KissFFT as the reference uses it
 * (src/common/dsp/FFT.cc:2461-2741 -> src/common/kissfft/kiss_fftr.c, kiss_fft.c).
 * Iterative form of the recursive kf_work (kiss_fft.c:250-286): a digit permutation of
 * the input followed by the butterfly stages, innermost factor first.  Every butterfly
 * performs the same float operations in the same order as kf_bfly2/kf_bfly4.
 * ---------------------------------------------------------------------------------- */
typedef struct {
    int n, nc;               /* real length, complex length n/2 */
    int nstages;
    int radix[20], span[20]; /* execution order (innermost first); span = m of that stage */
    int *perm;               /* perm[o] = input index landing at output slot o */
    cpx *tw_f, *tw_i;        /* kiss_fft.c:341-347 */
    cpx *stw_f, *stw_i;      /* kiss_fftr.c:57-63 */
    cpx *tmp;
} fftplan;

static void make_cexp(cpx *dst, double phase) { /* _kiss_fft_guts.h:136-137,147-151 */
    dst->r = (float)cos(phase);
    dst->i = (float)sin(phase);
}

static fftplan *fft_new(int n) {
    fftplan *p = (fftplan *)calloc(1, sizeof(fftplan));
    int nc = n / 2, i, j;
    p->n = n; p->nc = nc;
    /* factorisation: kf_factor, kiss_fft.c:292-314 -- 4s first, then 2 (power-of-two sizes only here) */
    int fp[20], fm[20], nf = 0, rem = nc, q = 4;
    do {
        while (rem % q) q = 2;
        rem /= q;
        fp[nf] = q; fm[nf] = rem; nf++;
    } while (rem > 1);
    p->nstages = nf;
    for (i = 0; i < nf; i++) { p->radix[i] = fp[nf - 1 - i]; p->span[i] = fm[nf - 1 - i]; }
    /* permutation implied by the recursion (kiss_fft.c:265-275): input index
       j1 + p1*(j2 + p2*(...)) lands at j1*m1 + j2*m2 + ... */
    p->perm = (int *)malloc(sizeof(int) * nc);
    for (i = 0; i < nc; i++) {
        int in = 0, stride = 1, o = i;
        for (j = 0; j < nf; j++) {
            int d = o / fm[j];
            o -= d * fm[j];
            in += d * stride;
            stride *= fp[j];
        }
        p->perm[i] = in;
    }
    p->tw_f = (cpx *)malloc(sizeof(cpx) * nc); p->tw_i = (cpx *)malloc(sizeof(cpx) * nc);
    p->stw_f = (cpx *)malloc(sizeof(cpx) * nc); p->stw_i = (cpx *)malloc(sizeof(cpx) * nc);
    p->tmp = (cpx *)malloc(sizeof(cpx) * (nc + 1));
    for (i = 0; i < nc; i++) { /* kiss_fft.c:341-347 */
        const double pi = 3.141592653589793238462643383279502884197169399375105820974944;
        double phase = -2 * pi * i / nc;
        make_cexp(&p->tw_f[i], phase);
        phase *= -1;
        make_cexp(&p->tw_i[i], phase);
    }
    for (i = 0; i < nc; i++) { /* kiss_fftr.c:57-63 */
        double phase = -3.14159265358979323846264338327 * ((double)i / nc + .5);
        make_cexp(&p->stw_f[i], phase);
        phase *= -1;
        make_cexp(&p->stw_i[i], phase);
    }
    return p;
}

static void fft_free(fftplan *p) {
    if (!p) return;
    free(p->perm); free(p->tw_f); free(p->tw_i); free(p->stw_f); free(p->stw_i); free(p->tmp); free(p);
}

#define CMUL(m, a, b) do { (m).r = (a).r * (b).r - (a).i * (b).i; (m).i = (a).r * (b).i + (a).i * (b).r; } while (0)

/* complex FFT of length nc: kf_work + kf_bfly2 (kiss_fft.c:36-57) + kf_bfly4 (:59-104) */
static void cfft(const fftplan *p, const cpx *in, cpx *out, int inverse) {
    const int nc = p->nc;
    const cpx *tw = inverse ? p->tw_i : p->tw_f;
    int s, base, k;
    for (k = 0; k < nc; k++) out[k] = in[p->perm[k]];
    for (s = 0; s < p->nstages; s++) {
        const int m = p->span[s], rad = p->radix[s], len = m * rad, fstride = nc / len;
        for (base = 0; base < nc; base += len) {
            cpx *F = out + base;
            if (rad == 2) {
                for (k = 0; k < m; k++) {
                    cpx t;
                    CMUL(t, F[k + m], tw[k * fstride]);
                    F[k + m].r = F[k].r - t.r; F[k + m].i = F[k].i - t.i;
                    F[k].r += t.r; F[k].i += t.i;
                }
            } else {
                for (k = 0; k < m; k++) {
                    cpx s0, s1, s2, s3, s4, s5;
                    CMUL(s0, F[k + m], tw[k * fstride]);
                    CMUL(s1, F[k + 2 * m], tw[2 * k * fstride]);
                    CMUL(s2, F[k + 3 * m], tw[3 * k * fstride]);
                    s5.r = F[k].r - s1.r; s5.i = F[k].i - s1.i;
                    F[k].r += s1.r; F[k].i += s1.i;
                    s3.r = s0.r + s2.r; s3.i = s0.i + s2.i;
                    s4.r = s0.r - s2.r; s4.i = s0.i - s2.i;
                    F[k + 2 * m].r = F[k].r - s3.r; F[k + 2 * m].i = F[k].i - s3.i;
                    F[k].r += s3.r; F[k].i += s3.i;
                    if (inverse) {
                        F[k + m].r = s5.r - s4.i; F[k + m].i = s5.i + s4.r;
                        F[k + 3 * m].r = s5.r + s4.i; F[k + 3 * m].i = s5.i - s4.r;
                    } else {
                        F[k + m].r = s5.r + s4.i; F[k + m].i = s5.i - s4.r;
                        F[k + 3 * m].r = s5.r - s4.i; F[k + 3 * m].i = s5.i + s4.r;
                    }
                }
            }
        }
    }
}

/* kiss_fftr, kiss_fftr.c:67-121.  HALF_OF(x) is (x)*.5 with a double constant
   (_kiss_fft_guts.h:141), i.e. an exact halving. */
static void rfft_forward(fftplan *p, const float *time, cpx *freq) {
    const int nc = p->nc;
    int k;
    cfft(p, (const cpx *)time, p->tmp, 0);
    {
        float tr = p->tmp[0].r, ti = p->tmp[0].i;
        freq[0].r = tr + ti;
        freq[nc].r = tr - ti;
        freq[nc].i = freq[0].i = 0;
    }
    for (k = 1; k <= nc / 2; ++k) {
        cpx fpk = p->tmp[k], fpnk, f1k, f2k, tw;
        fpnk.r = p->tmp[nc - k].r;
        fpnk.i = -p->tmp[nc - k].i;
        f1k.r = fpk.r + fpnk.r; f1k.i = fpk.i + fpnk.i;
        f2k.r = fpk.r - fpnk.r; f2k.i = fpk.i - fpnk.i;
        CMUL(tw, f2k, p->stw_f[k]);
        freq[k].r = (float)((f1k.r + tw.r) * .5);
        freq[k].i = (float)((f1k.i + tw.i) * .5);
        freq[nc - k].r = (float)((f1k.r - tw.r) * .5);
        freq[nc - k].i = (float)((tw.i - f1k.i) * .5);
    }
}

/* kiss_fftri, kiss_fftr.c:123-159 */
static void rfft_inverse(fftplan *p, const cpx *freq, float *time) {
    const int nc = p->nc;
    int k;
    p->tmp[0].r = freq[0].r + freq[nc].r;
    p->tmp[0].i = freq[0].r - freq[nc].r;
    for (k = 1; k <= nc / 2; ++k) {
        cpx fk = freq[k], fnkc, fek, fok, t;
        fnkc.r = freq[nc - k].r;
        fnkc.i = -freq[nc - k].i;
        fek.r = fk.r + fnkc.r; fek.i = fk.i + fnkc.i;
        t.r = fk.r - fnkc.r; t.i = fk.i - fnkc.i;
        CMUL(fok, t, p->stw_i[k]);
        p->tmp[k].r = fek.r + fok.r; p->tmp[k].i = fek.i + fok.i;
        p->tmp[nc - k].r = fek.r - fok.r; p->tmp[nc - k].i = fek.i - fok.i;
        p->tmp[nc - k].i *= -1;
    }
    cfft(p, p->tmp, (cpx *)time, 1);
}

/* D_KISSFFT::forwardPolar, FFT.cc:2617-2631 */
static void fft_forward_polar(fftplan *p, cpx *packed, const float *in, float *mag, float *phase) {
    const int hs = p->n / 2;
    int i;
    rfft_forward(p, in, packed);
    for (i = 0; i <= hs; ++i) mag[i] = sqrtf(packed[i].r * packed[i].r + packed[i].i * packed[i].i);
    for (i = 0; i <= hs; ++i) phase[i] = atan2f(packed[i].i, packed[i].r);
}

/* D_KISSFFT::inversePolar, FFT.cc:2711-2721 */
static void fft_inverse_polar(fftplan *p, cpx *packed, const float *mag, const float *phase, float *out) {
    const int hs = p->n / 2;
    int i;
    for (i = 0; i <= hs; ++i) {
        packed[i].r = mag[i] * cosf(phase[i]);
        packed[i].i = mag[i] * sinf(phase[i]);
    }
    rfft_inverse(p, packed, out);
}

/* ------------------------------------------------------------------------------------
 * Hann window: windowfunc<float>(Hanning, n), src/common/dsp/windowfunc.h:101-169
 * ---------------------------------------------------------------------------------- */
static float make_hann(float *w, int n) {
    const float a0 = 0.50f, a1 = 0.50f, a2 = 0.0f, a3 = 0.0f;
    float area = 0;
    int i;
    for (i = 0; i < n; ++i) w[i] = 1.0f;
    for (i = 0; i < n; ++i) {
        w[i] *= (a0 - a1 * cos(2 * M_PI * i / n) + a2 * cos(4 * M_PI * i / n) - a3 * cos(6 * M_PI * i / n));
    }
    for (i = 0; i < n; ++i) area += w[i];
    area /= n;
    return area;
}

/* princarg, src/common/system/sys.h:84-91 (the double overload is the one called) */
static double pv_mod(double x, double y) { return x - (y * floor(x / y)); }
static double princarg(double a) { return pv_mod(a + M_PI, -2.0 * M_PI) + M_PI; }

/* ------------------------------------------------------------------------------------
 * glibc rand() in a fresh process (whisperSlice, phasevocoderprocess.cc:820 calls the
 * unseeded libc rand()).  glibc 2.39 (third-party, not in /root/reference): TYPE_3
 * additive-feedback generator, degree 31, separation 3, seed 1, 310 values discarded,
 * output = state word >> 1.  Checked against the host rand() in tests/test_oracle_units.py.
 * ---------------------------------------------------------------------------------- */
typedef struct { int32_t r[31]; int f, b; } grand_t;

static int32_t grand_next(grand_t *g) {
    uint32_t v = (uint32_t)g->r[g->f] + (uint32_t)g->r[g->b];
    g->r[g->f] = (int32_t)v;
    if (++g->f >= 31) g->f = 0;
    if (++g->b >= 31) g->b = 0;
    return (int32_t)(v >> 1);
}

static void grand_seed(grand_t *g, unsigned seed) {
    int i;
    int32_t word;
    if (seed == 0) seed = 1;
    g->r[0] = (int32_t)seed;
    word = (int32_t)seed;
    for (i = 1; i < 31; ++i) {
        long hi = word / 127773, lo = word % 127773;
        word = (int32_t)(16807 * lo - 2836 * hi);
        if (word < 0) word += 2147483647;
        g->r[i] = word;
    }
    g->f = 3; g->b = 0;
    for (i = 0; i < 310; ++i) (void)grand_next(g);
}

/* ------------------------------------------------------------------------------------
 * Speex resampler at quality 4 as wrapped by RS_Speex (src/common/dsp/resampler.cc:696-817)
 * over src/common/speex/resample.c.  Only the call sequence the phase vocoder produces is
 * restated: construct (1:1), reset, first doresample sets the real ratio while not yet
 * started, skip_zeros once, then fixed-ratio processing (no filter-length change, hence
 * no "magic samples").
 * ---------------------------------------------------------------------------------- */
static const double kaiser8_tab[36] = { /* resample.c:229-236 (numeric table of the Kaiser-8 window) */
    0.99635258, 1.00000000, 0.99635258, 0.98548012, 0.96759014, 0.94302200,
    0.91223751, 0.87580811, 0.83439927, 0.78875245, 0.73966538, 0.68797126,
    0.63451750, 0.58014482, 0.52566725, 0.47185369, 0.41941150, 0.36897272,
    0.32108304, 0.27619388, 0.23465776, 0.19672670, 0.16255380, 0.13219758,
    0.10562887, 0.08273982, 0.06335451, 0.04724088, 0.03412321, 0.02369490,
    0.01563093, 0.00959968, 0.00527363, 0.00233883, 0.00050000, 0.00000000};
#define KAISER8_OVERSAMPLE 32

typedef struct {
    uint32_t num, den;        /* in-rate : out-rate, reduced */
    uint32_t filt_len, oversample;
    int int_adv, frac_adv;
    float cutoff;
    int direct;               /* 1: per-phase table (den <= oversample), 0: interpolated table */
    float *table; int table_len;
    float *mem;               /* filt_len-1 history samples */
    int last_sample; uint32_t frac_num;
    float lastratio; int initial;
} rs_t;

static double rs_window(float x) { /* compute_func, resample.c:300-322 */
    float y, frac;
    double interp[4];
    int ind;
    y = x * KAISER8_OVERSAMPLE;
    ind = (int)floor(y);
    frac = (y - ind);
    interp[3] = -0.1666666667 * frac + 0.1666666667 * (frac * frac * frac);
    interp[2] = frac + 0.5 * (frac * frac) - 0.5 * (frac * frac * frac);
    interp[0] = -0.3333333333 * frac + 0.5 * (frac * frac) - 0.1666666667 * (frac * frac * frac);
    interp[1] = 1.f - interp[3] - interp[2] - interp[0];
    return interp[0] * kaiser8_tab[ind] + interp[1] * kaiser8_tab[ind + 1] +
           interp[2] * kaiser8_tab[ind + 2] + interp[3] * kaiser8_tab[ind + 3];
}

static float rs_sinc(float cutoff, float x, int N) { /* sinc, resample.c:325-337 */
    float xx = x * cutoff;
    if (fabsf(x) < 1e-6)
        return cutoff;
    else if (fabsf(x) > .5 * N)
        return 0;
    return cutoff * sin(M_PI * xx) / (M_PI * xx) * rs_window(fabs(2. * x / N));
}

static uint32_t gcd_u32(uint32_t a, uint32_t b) { while (b) { uint32_t t = b; b = a % b; a = t; } return a; }

/* RS_Speex::setratio (resampler.cc:740-770) -> speex_resampler_set_rate_frac
   (resample.c:1117-1158) -> update_filter (resample.c:661-779) with quality 4
   (quality_map[4] = {64, 8, 0.921f, 0.940f, KAISER8}, resample.c:286) */
static void rs_setratio(rs_t *rs, float ratio) {
    const unsigned int big = 272408136U;
    unsigned int denom = 1, num = 1;
    uint32_t g, i;
    if (ratio < 1.f) {
        denom = big;
        double dnum = (double)big * (double)ratio;
        num = (unsigned int)dnum;
    } else if (ratio > 1.f) {
        num = big;
        double ddenom = (double)big / (double)ratio;
        denom = (unsigned int)ddenom;
    }
    /* set_rate_frac(st, ratio_num = denom, ratio_den = num) */
    rs->num = denom; rs->den = num;
    g = gcd_u32(rs->num, rs->den);
    rs->num /= g; rs->den /= g;
    /* samp_frac_num rescale (resample.c:1141-1150): it is 0 before the first block */
    rs->frac_num = 0;

    rs->oversample = 8;
    rs->filt_len = 64;
    if (rs->num > rs->den) {
        rs->cutoff = 0.921f * rs->den / rs->num;
        rs->filt_len = (unsigned int)ceil(rs->filt_len * ((double)rs->num / (double)rs->den));
        rs->filt_len &= (~0x3);
        if (2 * rs->den < rs->num) rs->oversample >>= 1;
        if (4 * rs->den < rs->num) rs->oversample >>= 1;
        if (8 * rs->den < rs->num) rs->oversample >>= 1;
        if (16 * rs->den < rs->num) rs->oversample >>= 1;
        if (rs->oversample < 1) rs->oversample = 1;
    } else {
        rs->cutoff = 0.940f;
    }
    free(rs->table);
    if (rs->den <= rs->oversample) {
        rs->direct = 1;
        rs->table_len = (int)(rs->filt_len * rs->den);
        rs->table = (float *)malloc(sizeof(float) * rs->table_len);
        for (i = 0; i < rs->den; i++) {
            int j;
            for (j = 0; j < (int)rs->filt_len; j++)
                rs->table[i * rs->filt_len + j] =
                    rs_sinc(rs->cutoff, ((j - (int)rs->filt_len / 2 + 1) - ((float)i) / rs->den), rs->filt_len);
        }
    } else {
        int k;
        rs->direct = 0;
        rs->table_len = (int)(rs->filt_len * rs->oversample + 8);
        rs->table = (float *)malloc(sizeof(float) * rs->table_len);
        for (k = -4; k < (int)(rs->oversample * rs->filt_len + 4); k++)
            rs->table[k + 4] = rs_sinc(rs->cutoff, (k / (float)rs->oversample - rs->filt_len / 2), rs->filt_len);
    }
    rs->int_adv = rs->num / rs->den;
    rs->frac_adv = rs->num % rs->den;
    free(rs->mem);
    rs->mem = (float *)calloc(rs->filt_len - 1, sizeof(float)); /* !started: zeroed at the new length */
    rs->lastratio = ratio;
    if (rs->initial) { /* speex_resampler_skip_zeros, resample.c:1220-1229 */
        rs->last_sample = rs->filt_len / 2;
        rs->initial = 0;
    }
}

static void rs_init(rs_t *rs) { /* RS_Speex ctor + reset(), resampler.cc:696-731,819-825 */
    memset(rs, 0, sizeof(*rs));
    rs->lastratio = -1.0f;
    rs->initial = 1;
    rs->last_sample = 0;
    rs->frac_num = 0;
}

/* RS_Speex::doresample (resampler.cc:772-817), mono -> speex_resampler_process_native
   (resample.c:986-1059) -> resampler_basic_{interpolate,direct}_single (:352-403,462-560) */
static int rs_process(rs_t *rs, const float *in, int incount, float ratio, float *out) {
    if (ratio != rs->lastratio) rs_setratio(rs, ratio);
    unsigned int in_len = incount;
    unsigned int out_len = lrintf(ceilf(incount * ratio));
    const int N = rs->filt_len;
    int out_sample = 0, j;
    int last_sample = rs->last_sample;
    uint32_t frac_num = rs->frac_num;
    float *mem = rs->mem;

    while (!(last_sample >= (int)in_len || out_sample >= (int)out_len)) {
        float sum;
        if (rs->direct) {
            sum = 0;
            for (j = 0; j < N; j++) {
                int pos = last_sample - N + 1 + j;
                float x = pos < 0 ? mem[last_sample + j] : in[pos];
                sum += x * rs->table[frac_num * rs->filt_len + j];
            }
        } else {
            float accum[4] = {0.f, 0.f, 0.f, 0.f};
            float interp[4];
            int offset = frac_num * rs->oversample / rs->den;
            float frac = ((float)((frac_num * rs->oversample) % rs->den)) / rs->den;
            for (j = 0; j < N; j++) {
                int pos = last_sample - N + 1 + j;
                float x = pos < 0 ? mem[last_sample + j] : in[pos];
                const float *t = rs->table + 4 + (j + 1) * rs->oversample - offset;
                accum[0] += x * t[-2];
                accum[1] += x * t[-1];
                accum[2] += x * t[0];
                accum[3] += x * t[1];
            }
            /* cubic_coef, resample.c:339-351 */
            interp[0] = -0.16667f * frac + 0.16667f * frac * frac * frac;
            interp[1] = frac + 0.5f * frac * frac - 0.5f * frac * frac * frac;
            interp[3] = -0.33333f * frac + 0.5f * frac * frac - 0.16667f * frac * frac * frac;
            interp[2] = 1. - interp[0] - interp[1] - interp[3];
            sum = (interp[0] * accum[0]) + (interp[1] * accum[1]) + (interp[2] * accum[2]) + (interp[3] * accum[3]);
        }
        out[out_sample++] = sum;
        last_sample += rs->int_adv;
        frac_num += rs->frac_adv;
        if (frac_num >= rs->den) { frac_num -= rs->den; last_sample++; }
    }
    rs->frac_num = frac_num;
    /* resample.c:1040-1056: consumed count, position rebase, history update */
    if (last_sample < (int)in_len) in_len = last_sample;
    last_sample -= in_len;
    rs->last_sample = last_sample;
    for (j = 0; j < N - 1 - (int)in_len; j++) mem[j] = mem[j + in_len];
    for (; j < N - 1; j++) mem[j] = in[j + in_len - N + 1];
    return out_sample;
}

/* ------------------------------------------------------------------------------------
 * Rosenberg glottal pulse carriers: src/common/gen/rosenberg.cc:19-53, rosenbergchord.cc
 * ---------------------------------------------------------------------------------- */
typedef struct { int period, n1, n2, phase; float inv_n1, inv_2n2; } rosen_t;

static void rosen_init(rosen_t *g, float sample_rate, float freq, float alpha, float beta) {
    g->period = round(1.f / freq * sample_rate);
    g->phase = 0;
    g->n1 = round(alpha * g->period);
    g->inv_n1 = 1.f / (float)(g->n1);
    g->n2 = round(beta * g->period);
    g->inv_2n2 = 0.5 / (float)(g->n2);
}

static float rosen_next(rosen_t *g) {
    float res = 0;
    if (g->phase <= g->n1) {
        res = 0.5 * (1 - cosf(M_PI * g->phase * g->inv_n1));
    } else if (g->phase - g->n1 <= g->n2) {
        res = cosf(M_PI * (g->phase - g->n1) * g->inv_2n2);
    } else {
        res = 0;
    }
    if (++g->phase > g->period) g->phase = 0;
    return res;
}

/* ------------------------------------------------------------------------------------
 * Engine state: phasevocodercore::Impl (phasevocoderimpl.{h,cc}) + channelinfo
 * (channelinfo.{h,cc}) + the facade (phasevocoder.cc).
 * ---------------------------------------------------------------------------------- */
typedef struct {
    float *data; long cap, fill; /* circularqueue<float>(cap): usable capacity == cap (circularqueue.h:145-173) */
} fifo_t;

static void fifo_init(fifo_t *f, long cap) { f->data = (float *)malloc(sizeof(float) * (cap + 1)); f->cap = cap; f->fill = 0; }
static long fifo_space(const fifo_t *f) { return f->cap - f->fill; }
static long fifo_write(fifo_t *f, const float *src, long n) {
    if (n > fifo_space(f)) n = fifo_space(f);
    if (n > 0) { memcpy(f->data + f->fill, src, sizeof(float) * n); f->fill += n; }
    return n;
}
static void fifo_peek(const fifo_t *f, float *dst, long n) { memcpy(dst, f->data, sizeof(float) * n); }
static void fifo_drop(fifo_t *f, long n) {
    if (n > f->fill) n = f->fill;
    memmove(f->data, f->data + n, sizeof(float) * (f->fill - n));
    f->fill -= n;
}
static long fifo_read(fifo_t *f, float *dst, long n) {
    if (n > f->fill) n = f->fill;
    if (n > 0) { fifo_peek(f, dst, n); fifo_drop(f, n); }
    return n;
}

typedef struct { /* channelinfo, channelinfo.cc:26-115 */
    fifo_t inbuf, outbuf;
    float *iface, *internal;     /* interfacebuffer / internalbuffer */
    float *outacc, *winacc;
    float *mag, *phase, *prev_phase, *prev_outphase, *locked;
    cpx *packed;
    size_t prev_increment;
    rs_t res;
} chan_t;

typedef struct pvo {
    int sr, ch, mode, coremode;
    float time_ratio, pitch_scale;
    int N, hop;
    long outbuf_size;
    int opt_formant, opt_gender, opt_robotic, opt_whisper;
    fftplan *fft;
    float *win; float area;
    chan_t *chan, *carrier;
    float *resamplebuf;
    /* shared across channels: Impl::peak_loc / prev_peak_loc, phasevocoderimpl.h:237-238 */
    int *peak, npeak, *prev_peak, nprev;
    /* function-local statics of the reference, one set per fresh process */
    int first_locked, first_simple;            /* phasevocoderprocess.cc:602,716 */
    float recovery, divergence;                /* phasevocoderprocess.cc:380-384 */
    grand_t rng;
    rosen_t *rosen;                            /* one per channel */
    rosen_t *chord;                            /* three per channel */
    int num_res, outready;
    long slices, dropped;
    /* optional record of modify_locked (pvo_phase_core_frames): per peak its rotation and region [bin1, bin2); null = none */
    float *rec_rot;
    int *rec_bin1, *rec_bin2;
} pvo_t;

static void chan_init(chan_t *c, int N, long outbuf_size) {
    const int H = N / 2 + 1, buf = 2 * N;
    if (outbuf_size < buf) outbuf_size = buf;
    fifo_init(&c->inbuf, buf);
    fifo_init(&c->outbuf, outbuf_size);
    c->iface = (float *)calloc(buf, sizeof(float));
    c->internal = (float *)calloc(buf, sizeof(float));
    c->outacc = (float *)calloc(buf, sizeof(float));
    c->winacc = (float *)calloc(buf, sizeof(float));
    c->mag = (float *)calloc(H, sizeof(float)); c->phase = (float *)calloc(H, sizeof(float));
    c->prev_phase = (float *)calloc(H, sizeof(float)); c->prev_outphase = (float *)calloc(H, sizeof(float));
    c->locked = (float *)calloc(H, sizeof(float));
    c->packed = (cpx *)calloc(N + 2, sizeof(cpx));
    c->winacc[0] = 1.f; /* channelinfo.cc:108 */
    c->prev_increment = 0;
    rs_init(&c->res);
}

static void chan_free(chan_t *c) {
    free(c->inbuf.data); free(c->outbuf.data); free(c->iface); free(c->internal); free(c->outacc); free(c->winacc);
    free(c->mag); free(c->phase); free(c->prev_phase); free(c->prev_outphase); free(c->locked); free(c->packed);
    free(c->res.table); free(c->res.mem);
}

static int nextpow2(size_t value) { /* phasevocoderimpl.cc:159-167 */
    if (!(value & (value - 1))) return (int)value;
    int bits = 0;
    while (value) { ++bits; value >>= 1; }
    return 1 << bits;
}

static float hs_ratio(const pvo_t *p) { return p->time_ratio * p->pitch_scale; } /* impl.cc:144-147 */

pvo_t *pvo_create(int sr, int ch, float timeratio, float semitones, int mode, int coremode, int fftsize, int hopsize) {
    pvo_t *p = (pvo_t *)calloc(1, sizeof(pvo_t));
    int c;
    /* phasevocoder::phasevocoder, phasevocoder.cc:24-60 */
    p->sr = sr; p->ch = ch; p->mode = mode; p->coremode = coremode;
    p->time_ratio = timeratio;
    p->pitch_scale = semitones != 0 ? pow(2.0, semitones / 12) : 1.0;
    p->opt_gender = mode == MODE_GENDER; p->opt_formant = mode == MODE_FORMANT;
    p->opt_robotic = mode == MODE_ROBOTIC; p->opt_whisper = mode == MODE_WHISPER;
    /* Impl::calculateSizes, phasevocoderimpl.cc:169-263 */
    size_t windowSize = nextpow2((size_t)fftsize);
    if (p->pitch_scale <= 0.0) p->pitch_scale = 1.0;
    if (p->time_ratio <= 0.0) p->time_ratio = 1.0;
    float hsratio = hs_ratio(p);
    size_t inputHop, outputHop;
    if (hopsize > 0) {
        inputHop = hopsize;
        outputHop = (int)(floor(inputHop * hsratio));
    } else {
        float wir = 4.5;
        if (hsratio < 1) {
            if (hsratio == 1.0) wir = 4;
            else if (p->pitch_scale < 1.0) wir = 4.5;
            else wir = 6;
            inputHop = (int)(windowSize / wir);
            outputHop = (int)(inputHop * hsratio);
        } else {
            if (hsratio == 1.0) wir = 4;
            else wir = 8;
            outputHop = (int)(windowSize / wir);
            inputHop = (int)(outputHop / hsratio);
        }
    }
    (void)outputHop;
    p->N = (int)windowSize;
    p->hop = (int)inputHop;
    p->outbuf_size = hsratio > 1 ? (size_t)(windowSize * 16 * hsratio) : windowSize * 16;
    /* Impl::configure, phasevocoderimpl.cc:265-322 */
    p->win = (float *)malloc(sizeof(float) * p->N);
    p->area = make_hann(p->win, p->N);
    p->fft = fft_new(p->N);
    p->chan = (chan_t *)calloc(ch, sizeof(chan_t));
    p->carrier = (chan_t *)calloc(ch, sizeof(chan_t));
    for (c = 0; c < ch; ++c) { chan_init(&p->chan[c], p->N, p->outbuf_size); chan_init(&p->carrier[c], p->N, p->outbuf_size); }
    p->resamplebuf = (float *)calloc(p->N * 8 + 65536, sizeof(float));
    p->peak = (int *)malloc(sizeof(int) * (p->N / 2 + 2)); p->prev_peak = (int *)malloc(sizeof(int) * (p->N / 2 + 2));
    p->npeak = p->nprev = 0;
    p->first_locked = p->first_simple = 1;
    p->recovery = p->divergence = 0;
    grand_seed(&p->rng, 1);
    p->rosen = (rosen_t *)calloc(ch, sizeof(rosen_t));
    p->chord = (rosen_t *)calloc(3 * ch, sizeof(rosen_t));
    for (c = 0; c < ch; ++c) { /* impl.cc:312-320 */
        static const float chordmin[3] = {440, 523.251, 659.255};
        int k;
        rosen_init(&p->rosen[c], sr, 440, 0.01, 0.06);
        for (k = 0; k < 3; ++k) rosen_init(&p->chord[3 * c + k], sr, chordmin[k], 0.01, 0.06);
    }
    return p;
}

void pvo_destroy(pvo_t *p) {
    int c;
    if (!p) return;
    for (c = 0; c < p->ch; ++c) { chan_free(&p->chan[c]); chan_free(&p->carrier[c]); }
    free(p->chan); free(p->carrier); free(p->win); fft_free(p->fft); free(p->resamplebuf);
    free(p->peak); free(p->prev_peak); free(p->rosen); free(p->chord); free(p);
}

int pvo_fftsize(const pvo_t *p) { return p->N; }
int pvo_hop(const pvo_t *p) { return p->hop; }
float pvo_pitch_scale(const pvo_t *p) { return p->pitch_scale; }
long pvo_slices(const pvo_t *p) { return p->slices; }
long pvo_dropped(const pvo_t *p) { return p->dropped; }

/* fftshift + forwardPolar: analyzeSlice phasevocoderprocess.cc:492-503, impl.h:167-181 */
static void analyze(pvo_t *p, chan_t *c) {
    const int N = p->N, hs = N / 2;
    int i;
    for (i = 0; i < N; ++i) c->iface[i] *= p->win[i];
    for (i = 0; i < hs; ++i) c->internal[i] = c->iface[i + hs];
    for (i = 0; i < hs; ++i) c->internal[i + hs] = c->iface[i];
    fft_forward_polar(p->fft, c->packed, c->internal, c->mag, c->phase);
}

/* calculateThisIncrement, phasevocoderprocess.cc:379-410 */
static int this_increment(pvo_t *p, float ratio, size_t increment, size_t samplerate) {
    p->recovery = p->divergence / ((samplerate / 10.0) / increment);
    int incr = lrint(increment * ratio - p->recovery);
    if (incr < lrint((increment * ratio) / 2)) {
        incr = lrint((increment * ratio) / 2);
    } else if (incr > lrint(increment * ratio * 2)) {
        incr = lrint(increment * ratio * 2);
    }
    float divdiff = (increment * ratio) - incr;
    float prevDivergence = p->divergence;
    p->divergence -= divdiff;
    if ((prevDivergence < 0 && p->divergence > 0) || (prevDivergence > 0 && p->divergence < 0)) {
        p->recovery = p->divergence / ((samplerate / 10.0) / increment);
    }
    return incr;
}

/* modifySlicePhaseLocked, phasevocoderprocess.cc:574-706 */
static void modify_locked(pvo_t *p, chan_t *ad, size_t phaseIncrement) {
    const int halfsize = p->N / 2;
    const size_t m_hopsize = p->hop, m_fftSize = p->N;
    float *mag = ad->mag;
    int i, b = 2;
    p->npeak = 0;
    while (b + 2 < halfsize) {
        if (mag[b] > mag[b - 1] && mag[b] > mag[b - 2] && mag[b] > mag[b + 1] && mag[b] > mag[b + 2]) {
            p->peak[p->npeak++] = b;
            b += 3;
        } else {
            b += 1;
        }
    }
    if (p->first_locked) {
        for (i = 0; i < halfsize; i++) {
            float tp = ad->phase[i];
            ad->prev_phase[i] = tp;
            ad->phase[i] = tp;
            ad->prev_outphase[i] = tp;
        }
    } else if (p->npeak == 0 || p->nprev == 0) {
        for (i = 0; i < halfsize; i++) {
            float omega = (2 * M_PI * m_hopsize * i) / (m_fftSize);
            float delta_phi = omega + princarg(ad->phase[i] - ad->prev_phase[i] - omega);
            float advance = delta_phi * phaseIncrement / m_hopsize;
            float outphase = princarg(ad->prev_outphase[i] + advance);
            ad->prev_phase[i] = ad->phase[i];
            ad->phase[i] = outphase;
            ad->prev_outphase[i] = outphase;
        }
    } else {
        int prev_p = 0, pk;
        for (pk = 0; pk < p->npeak; pk++) {
            int p2 = p->peak[pk];
            while (prev_p < p->nprev - 1) {
                if (abs(p2 - p->prev_peak[prev_p + 1]) < abs(p2 - p->prev_peak[prev_p])) prev_p += 1;
                else break;
            }
            int p1 = p->prev_peak[prev_p];
            float avg_p = (p1 + p2) * 0.5;
            float pomega = (2 * M_PI * m_hopsize * (avg_p - 1)) / (m_fftSize);
            float peak_delta_phi = pomega + princarg(ad->phase[p2] - ad->prev_phase[p1] - pomega);
            float peak_target_phase = princarg(ad->prev_outphase[p1] + (peak_delta_phi * phaseIncrement) / m_hopsize);
            float peak_phase_rotation = princarg(peak_target_phase - ad->phase[p2]);
            int bin1 = 0, bin2 = 0;
            if (p->npeak == 1) {
                bin1 = 0; bin2 = halfsize;
            } else if (pk == 0) {
                bin1 = 0; bin2 = round((p->peak[pk + 1] + p2) * 0.5);
            } else if (pk == p->npeak - 1) {
                bin1 = round((p->peak[pk - 1] + p2) * 0.5); bin2 = halfsize;
            } else {
                bin1 = round((p->peak[pk - 1] + p2) * 0.5);
                bin2 = round((p->peak[pk + 1] + p2) * 0.5);
            }
            for (i = bin1; i < bin2; i++) ad->locked[i] = princarg(ad->phase[i] + peak_phase_rotation);
            if (p->rec_rot) { p->rec_rot[pk] = peak_phase_rotation; p->rec_bin1[pk] = bin1; p->rec_bin2[pk] = bin2; }
        }
        for (i = 0; i < halfsize; i++) {
            ad->prev_phase[i] = ad->phase[i];
            ad->prev_outphase[i] = ad->locked[i];
            ad->phase[i] = ad->locked[i];
        }
    }
    memcpy(p->prev_peak, p->peak, sizeof(int) * p->npeak);
    p->nprev = p->npeak;
    p->first_locked = 0;
}

/* modifySliceSimple, phasevocoderprocess.cc:708-753.  The shared peak vectors are only ever
   filled by the locked core, so with a single instance they are empty here and the
   "else if" is always taken after the first call. */
static void modify_simple(pvo_t *p, chan_t *ad, size_t phaseIncrement) {
    const int halfsize = p->N / 2;
    const size_t m_hopsize = p->hop, m_fftSize = p->N;
    int i;
    if (p->first_simple) {
        for (i = 0; i < halfsize; i++) {
            float tp = ad->phase[i];
            ad->prev_phase[i] = tp;
            ad->phase[i] = tp;
            ad->prev_outphase[i] = tp;
        }
    } else if (p->npeak == 0 || p->nprev == 0) {
        for (i = 0; i < halfsize; i++) {
            float omega = (2 * M_PI * m_hopsize * i) / (m_fftSize);
            float delta_phi = omega + princarg(ad->phase[i] - ad->prev_phase[i] - omega);
            float advance = delta_phi * phaseIncrement / m_hopsize;
            float outphase = princarg(ad->prev_outphase[i] + advance);
            ad->prev_phase[i] = ad->phase[i];
            ad->phase[i] = outphase;
            ad->prev_outphase[i] = outphase;
        }
    }
    p->first_simple = 0;
}

/* modifySliceIntRatio, phasevocoderprocess.cc:558-572 */
static void modify_intratio(pvo_t *p, chan_t *ad, size_t phaseIncrement) {
    const int halfsize = p->N / 2;
    const size_t m_hopsize = p->hop;
    int i;
    for (i = 0; i < halfsize; i++) ad->phase[i] = ad->phase[i] * phaseIncrement / m_hopsize;
}

/* freqCompSlice, phasevocoderprocess.cc:842-923 */
static void freq_comp(pvo_t *p, chan_t *ad, float freq_comp) {
    float *phi = ad->phase, *mag = ad->mag;
    const int halfsize = p->N / 2;
    const size_t m_hopsize = p->hop, m_fftSize = p->N;
    float absps = p->pitch_scale > 1 ? p->pitch_scale : 1 / p->pitch_scale;
    const float fixedgain = absps;
    int target, i;
    if (freq_comp > 1.0) {
        for (target = 0; target <= halfsize; ++target) {
            int source = lrint(target * freq_comp);
            float delta_omega = (2 * M_PI * m_hopsize * (target - source)) / (m_fftSize);
            if (source > halfsize) {
                mag[target] = 0.0;
                phi[target] = 0.0;
            } else {
                mag[target] = mag[source];
                phi[target] = phi[source] + delta_omega;
            }
        }
    } else {
        for (target = halfsize; target > 0;) {
            --target;
            int source = lrint(target * freq_comp);
            float delta_omega = (2 * M_PI * m_hopsize * (target - source)) / (m_fftSize);
            mag[target] = mag[source];
            phi[target] = phi[source] + delta_omega;
        }
    }
    for (i = 0; i < halfsize + 1; ++i) mag[i] *= fixedgain;
}

/* the synthesis half shared by synthesiseSlice (:1024-1073) and synthesiseSliceCarrier (:1077-1107) */
static void synth_ola(pvo_t *p, chan_t *ad) {
    const int N = p->N, halfsize = N / 2;
    int i;
    float factor = 1.f / N;
    for (i = 0; i < halfsize + 1; ++i) ad->mag[i] *= factor;
    fft_inverse_polar(p->fft, ad->packed, ad->mag, ad->phase, ad->internal);
    /* ifftshift, impl.h:183-198 */
    for (i = 0; i < halfsize; ++i) ad->iface[i] = ad->internal[i + halfsize];
    for (i = 0; i < halfsize; ++i) ad->iface[i + halfsize] = ad->internal[i];
    for (i = 0; i < N; ++i) ad->iface[i] *= p->win[i];
    for (i = 0; i < N; ++i) ad->outacc[i] += ad->iface[i];
    {
        float scale = p->area * 1.5; /* add2dst(windowAccumulator, GetArea()*1.5), :1073 */
        for (i = 0; i < N; ++i) ad->winacc[i] += p->win[i] * scale;
    }
}

/* synthesiseSlice, phasevocoderprocess.cc:1001-1075 */
static void synthesise(pvo_t *p, chan_t *ad) {
    if (p->opt_formant && (p->pitch_scale != 1.0)) freq_comp(p, ad, p->pitch_scale);
    if (p->opt_gender && (p->pitch_scale != 1.0)) {
        if (p->pitch_scale > 1) freq_comp(p, ad, 0.85 * p->pitch_scale);
        else freq_comp(p, ad, 1.17 * p->pitch_scale);
    } else if (p->opt_gender) {
        freq_comp(p, ad, 0.8);
    }
    synth_ola(p, ad);
}

static void shift_accumulators(pvo_t *p, chan_t *ad, size_t shiftIncrement) { /* :1185-1190 */
    const int N = p->N;
    memmove(ad->outacc, ad->outacc + shiftIncrement, sizeof(float) * (N - shiftIncrement));
    memset(ad->outacc + N - shiftIncrement, 0, sizeof(float) * shiftIncrement);
    memmove(ad->winacc, ad->winacc + shiftIncrement, sizeof(float) * (N - shiftIncrement));
    memset(ad->winacc + N - shiftIncrement, 0, sizeof(float) * shiftIncrement);
}

/* writeSlice, phasevocoderprocess.cc:1140-1194 */
static int write_slice(pvo_t *p, chan_t *ad, size_t shiftIncrement) {
    size_t i, outframes;
    for (i = 0; i < shiftIncrement; ++i) ad->outacc[i] /= ad->winacc[i];
    if (p->pitch_scale != 1.0) {
        outframes = rs_process(&ad->res, ad->outacc, (int)shiftIncrement, 1.0 / p->pitch_scale, p->resamplebuf);
        fifo_write(&ad->outbuf, p->resamplebuf, outframes);
    } else {
        outframes = shiftIncrement;
        fifo_write(&ad->outbuf, ad->outacc, shiftIncrement);
    }
    shift_accumulators(p, ad, shiftIncrement);
    return (int)outframes;
}

/* processSliceForChannel, phasevocoderprocess.cc:305-376 */
static void slice_for_channel(pvo_t *p, int c, size_t phaseIncrement, size_t shiftIncrement) {
    chan_t *ad = &p->chan[c];
    const int H = p->N / 2 + 1;
    int i;
    if (p->opt_robotic) { /* roboticSlice :805-812 */
        for (i = 0; i < H; i++) ad->phase[i] = 0;
    } else if (p->opt_whisper) { /* whisperSlice :814-822 */
        float two_pi = 2 * M_PI;
        for (i = 0; i < H; i++) ad->phase[i] = two_pi * (float)grand_next(&p->rng) / (float)RAND_MAX;
    } else {
        if (p->coremode == 1) modify_locked(p, ad, phaseIncrement);
        else if (p->coremode == 2) modify_intratio(p, ad, phaseIncrement);
        else modify_simple(p, ad, phaseIncrement);
    }
    synthesise(p, ad);
    int required = (int)(shiftIncrement / p->pitch_scale) + 1;
    int ws = (int)fifo_space(&ad->outbuf);
    if (ws < required) { p->dropped++; return; } /* slice dropped, :344-364 */
    write_slice(p, ad, shiftIncrement);
}

static int is_int_ratio(const pvo_t *p) { /* impl.cc:149-157; float abs overload (SURVEY.md s.8a S2) */
    float efr = hs_ratio(p);
    return fabsf(efr - floorf(efr)) <= 0.001;
}

/* processOneSlice, phasevocoderprocess.cc:236-287 */
static void one_slice(pvo_t *p) {
    int c;
    const int N = p->N;
    for (c = 0; c < p->ch; ++c) {
        chan_t *ad = &p->chan[c];
        if (ad->inbuf.fill < N) return;
        fifo_peek(&ad->inbuf, ad->iface, N);
        fifo_drop(&ad->inbuf, p->hop);
        analyze(p, ad);
    }
    size_t phaseIncrement, shiftIncrement;
    if (p->opt_robotic || p->opt_whisper) {
        phaseIncrement = p->hop; shiftIncrement = p->hop;
    } else if (is_int_ratio(p)) {
        phaseIncrement = p->hop * hs_ratio(p);
        shiftIncrement = p->hop * hs_ratio(p);
    } else { /* calculateIncrements :412-489 */
        chan_t *ad = &p->chan[0];
        int incr = this_increment(p, hs_ratio(p), p->hop, p->sr);
        shiftIncrement = incr;
        if (ad->prev_increment == 0) phaseIncrement = shiftIncrement;
        else phaseIncrement = ad->prev_increment;
        ad->prev_increment = shiftIncrement;
    }
    for (c = 0; c < p->ch; ++c) slice_for_channel(p, c, phaseIncrement, shiftIncrement);
    p->slices++;
}

/* processOneSliceConstant, phasevocoderprocess.cc:122-156 */
static void one_slice_constant(pvo_t *p) {
    int c;
    const int N = p->N;
    for (c = 0; c < p->ch; ++c) {
        chan_t *ad = &p->chan[c];
        if (ad->inbuf.fill < N) return;
        fifo_peek(&ad->inbuf, ad->iface, N);
        fifo_drop(&ad->inbuf, p->hop);
        analyze(p, ad);
    }
    for (c = 0; c < p->ch; ++c) {
        chan_t *ad = &p->chan[c];
        synthesise(p, ad);
        if (fifo_space(&ad->outbuf) < p->hop) { p->dropped++; return; }
        write_slice(p, ad, p->hop);
    }
    p->slices++;
}

/* processOneSliceVocoder :158-195, modifySliceVocoder :755-776, writeSliceCarrier :1196-1231 */
static void one_slice_vocoder(pvo_t *p) {
    int c, i;
    const int N = p->N, H = N / 2 + 1;
    for (c = 0; c < p->ch; ++c) {
        chan_t *ad = &p->chan[c];
        if (ad->inbuf.fill < N) return;
        fifo_peek(&ad->inbuf, ad->iface, N);
        fifo_drop(&ad->inbuf, p->hop);
        analyze(p, ad);
    }
    for (c = 0; c < p->ch; ++c) {
        chan_t *ca = &p->carrier[c];
        long ready = ca->inbuf.fill < N ? ca->inbuf.fill : N;
        memset(ca->iface, 0, sizeof(float) * N);
        fifo_peek(&ca->inbuf, ca->iface, ready);
        fifo_drop(&ca->inbuf, p->hop);
        analyze(p, ca);
    }
    for (c = 0; c < p->ch; ++c) {
        chan_t *ad = &p->chan[c], *ca = &p->carrier[c];
        int num_bands = 512;
        int band_len = (int)floor((float)(N) / (float)(num_bands * 2));
        int band_no, j;
        for (band_no = 0; band_no < num_bands; band_no++) {
            float mean_modul_mag = 0;
            for (i = 0, j = band_no * band_len; i < band_len; i++, j++) mean_modul_mag += ad->mag[j];
            mean_modul_mag /= (band_len * 2);
            for (i = 0, j = band_no * band_len; i < band_len; i++, j++) ca->mag[j] *= mean_modul_mag;
            ca->mag[0] = 0;
            ca->mag[H - 1] = 0;
        }
        synth_ola(p, ca);
        if (fifo_space(&ca->outbuf) < p->hop) { p->dropped++; continue; }
        for (i = 0; i < p->hop; ++i) ca->outacc[i] /= ca->winacc[i];
        fifo_write(&ca->outbuf, ca->outacc, p->hop);
        shift_accumulators(p, ca, p->hop);
    }
    p->slices++;
}

static int is_vocoder(const pvo_t *p) { return p->mode == MODE_VOC_ROSEN || p->mode == MODE_VOC_CHORD; }

static long min_avail(const pvo_t *p) { /* numsamples_available{,Carrier} :1240-1264 */
    long ret = 0;
    int c;
    for (c = 0; c < p->ch; ++c) {
        long a = is_vocoder(p) ? p->carrier[c].outbuf.fill : p->chan[c].outbuf.fill;
        if (c == 0 || a < ret) ret = a;
    }
    return ret;
}

/* phasevocoder::processInData (phasevocoder.cc:87-108) over Impl::processNormal /
   processConstant / processVocoder (phasevocoderimpl.cc:340-423) */
void pvo_process(pvo_t *p, const float *const *in, int n) {
    int c, allread = 0;
    long done[16] = {0};
    if (p->mode < -1 || p->mode > 7) { p->num_res = 0; return; }
    while (!allread) {
        for (c = 0; c < p->ch; ++c) {
            long w = n - done[c];
            if (is_vocoder(p)) { /* enbufferChannelVocoder :66-120 */
                chan_t *ad = &p->chan[c], *ca = &p->carrier[c];
                long i;
                if (fifo_space(&ad->inbuf) < w) w = fifo_space(&ad->inbuf);
                if (fifo_space(&ca->inbuf) < w) w = fifo_space(&ca->inbuf);
                fifo_write(&ad->inbuf, in[c] + done[c], w);
                float *tmp = (float *)malloc(sizeof(float) * (w + 1));
                if (p->mode == MODE_VOC_ROSEN) {
                    for (i = 0; i < w; i++) tmp[i] = rosen_next(&p->rosen[c]) * 0.3;
                } else {
                    for (i = 0; i < w; i++) {
                        float res = 0;
                        int k;
                        for (k = 0; k < 3; ++k) res += rosen_next(&p->chord[3 * c + k]) / 3; /* rosenbergchord.cc:38-43 */
                        tmp[i] = res * 0.3;
                    }
                }
                fifo_write(&ca->inbuf, tmp, w);
                free(tmp);
            } else { /* enbufferChannel :43-64 */
                w = fifo_write(&p->chan[c].inbuf, in[c] + done[c], w);
            }
            done[c] += w;
            allread = !(done[c] < n);
        }
        if (is_vocoder(p)) one_slice_vocoder(p);
        else if (p->mode == MODE_CONSTANT) one_slice_constant(p);
        else one_slice(p);
    }
    p->num_res = (int)min_avail(p);
}

int pvo_available(const pvo_t *p) { return p->num_res; }

/* phasevocoder::getOutData (phasevocoder.cc:110-124) over Impl::retrieve{,Carrier} (:1266-1304) */
int pvo_retrieve(pvo_t *p, float *const *out, int n) {
    int c;
    long ret = n;
    if (ret > p->num_res) ret = p->num_res;
    for (c = 0; c < p->ch; ++c) {
        fifo_t *f = is_vocoder(p) ? &p->carrier[c].outbuf : &p->chan[c].outbuf;
        long got = fifo_read(f, out[c], ret);
        if (got < ret) ret = got;
    }
    p->outready = 1;
    return (int)ret;
}

/* phasevocoder::processBlock (phasevocoder.cc:126-238): in place; 0 = block replaced,
   -1 = not enough output yet (outputReady() false, caller's buffer untouched).
   NORMAL_STRETCH is not routed by the reference's processBlock (does nothing, ready). */
int pvo_process_block(pvo_t *p, float *const *buf, int n) {
    int c;
    if (p->mode == MODE_STRETCH || p->mode < -1 || p->mode > 7) { p->outready = 1; return 0; }
    pvo_process(p, (const float *const *)buf, n);
    if (p->num_res >= n) {
        for (c = 0; c < p->ch; ++c) {
            fifo_t *f = is_vocoder(p) ? &p->carrier[c].outbuf : &p->chan[c].outbuf;
            fifo_read(f, buf[c], n);
        }
        p->outready = 1;
        return 0;
    }
    p->outready = 0;
    return -1;
}

/* The reference CLI protocol (main/main.cc:149,471-509) for one whole stream.
   in: planar [ch][n]; out: planar [ch][out_cap]; returns samples per channel written. */
long pvo_run_offline(int sr, int ch, float timeratio, float semitones, int mode, int coremode, int fftsize, int hopsize,
                     const float *in, long n, float *out, long out_cap, int block, long *slices_out) {
    pvo_t *p = pvo_create(sr, ch, timeratio, semitones, mode, coremode, fftsize, hopsize);
    float *bufs[16], *obufs[16];
    long produced = 0, i;
    int c;
    if (block <= 0) block = sr / 100 < 480 ? 480 : sr / 100;
    long ocap = p->outbuf_size + 4L * p->N + block;
    for (c = 0; c < ch; ++c) { bufs[c] = (float *)calloc(block, sizeof(float)); obufs[c] = (float *)malloc(sizeof(float) * ocap); }
    for (i = 0; i < n; i += block) {
        int m = (int)((n - i) < block ? (n - i) : block), k;
        for (c = 0; c < ch; ++c) memcpy(bufs[c], in + (long)c * n + i, sizeof(float) * m);
        pvo_process(p, (const float *const *)bufs, m);
        k = pvo_retrieve(p, obufs, pvo_available(p));
        if (produced + k > out_cap) k = (int)(out_cap - produced);
        for (c = 0; c < ch; ++c) memcpy(out + (long)c * out_cap + produced, obufs[c], sizeof(float) * k);
        produced += k;
    }
    if (mode != MODE_STRETCH) {
        for (c = 0; c < ch; ++c) memset(bufs[c], 0, sizeof(float) * block);
        while (produced < n) {
            int k;
            pvo_process(p, (const float *const *)bufs, block);
            k = pvo_retrieve(p, obufs, pvo_available(p));
            if (n - produced <= k) k = (int)(n - produced);
            if (produced + k > out_cap) k = (int)(out_cap - produced);
            for (c = 0; c < ch; ++c) memcpy(out + (long)c * out_cap + produced, obufs[c], sizeof(float) * k);
            produced += k;
            if (k == 0 && produced >= out_cap) break;
        }
    }
    if (slices_out) *slices_out = p->slices;
    for (c = 0; c < ch; ++c) { free(bufs[c]); free(obufs[c]); }
    pvo_destroy(p);
    return produced;
}

/* ---- component hooks for unit tests of the CUDA stages ---- */
void pvo_forward_polar(int N, const float *frame /* raw, un-windowed */, float *mag, float *phase, float *re_im /* 2*(N/2+1) or NULL */) {
    fftplan *f = fft_new(N);
    float *w = (float *)malloc(sizeof(float) * N), *x = (float *)malloc(sizeof(float) * N), *t = (float *)malloc(sizeof(float) * N);
    cpx *packed = (cpx *)calloc(N + 2, sizeof(cpx));
    int i, hs = N / 2;
    make_hann(w, N);
    for (i = 0; i < N; ++i) x[i] = frame[i] * w[i];
    for (i = 0; i < hs; ++i) { t[i] = x[i + hs]; t[i + hs] = x[i]; }
    fft_forward_polar(f, packed, t, mag, phase);
    if (re_im) memcpy(re_im, packed, sizeof(cpx) * (hs + 1));
    free(w); free(x); free(t); free(packed); fft_free(f);
}

void pvo_inverse_polar(int N, const float *mag, const float *phase, float *out /* N, after ifftshift+window */) {
    fftplan *f = fft_new(N);
    float *w = (float *)malloc(sizeof(float) * N), *t = (float *)malloc(sizeof(float) * N);
    cpx *packed = (cpx *)calloc(N + 2, sizeof(cpx));
    int i, hs = N / 2;
    make_hann(w, N);
    fft_inverse_polar(f, packed, mag, phase, t);
    for (i = 0; i < hs; ++i) { out[i] = t[i + hs]; out[i + hs] = t[i]; }
    for (i = 0; i < N; ++i) out[i] *= w[i];
    free(w); free(t); free(packed); fft_free(f);
}

float pvo_host_atan2f(float y, float x) { return atan2f(y, x); }
void pvo_host_atan2f_vec(const float *y, const float *x, float *out, long n) { long i; for (i = 0; i < n; ++i) out[i] = atan2f(y[i], x[i]); }
double pvo_princarg(double a) { return princarg(a); }
float pvo_hann(int N, float *w) { return make_hann(w, N); }
int pvo_rand_sequence(int *dst, int n) { grand_t g; int i; grand_seed(&g, 1); for (i = 0; i < n; ++i) dst[i] = grand_next(&g); return n; }
int pvo_host_rand(void) { return rand(); }

/* resampler table / parameters for a pitch scale (for checking the host-side table builder) */
int pvo_resampler_params(float pitch_scale, uint32_t *num, uint32_t *den, uint32_t *filt_len, uint32_t *oversample,
                         int *direct, float *table, int table_cap) {
    rs_t rs;
    int n;
    rs_init(&rs);
    rs_setratio(&rs, (float)(1.0 / pitch_scale));
    *num = rs.num; *den = rs.den; *filt_len = rs.filt_len; *oversample = rs.oversample; *direct = rs.direct;
    n = rs.table_len;
    if (table && table_cap >= n) memcpy(table, rs.table, sizeof(float) * n);
    free(rs.table); free(rs.mem);
    return n;
}

/* (re, im) -> (sqrtf(re*re + im*im), atan2f(im, re)), the polar step of forwardPolar (FFT.cc:2624-2629): polar spectra from given
   Cartesian ones, rounded as the reference rounds them.  re_im: [n][2]. */
void pvo_polar(long n, const float *re_im, float *mag, float *phase) {
    long i;
    for (i = 0; i < n; ++i) {
        const float r = re_im[2 * i], m = re_im[2 * i + 1];
        mag[i] = sqrtf(r * r + m * m);
        phase[i] = atan2f(m, r);
    }
}

/* The phase core of one stream (processSliceForChannel's modify call, :305-376) over given analysis frames, from the state of a fresh
   process: frames in order, the channels of a frame in order, sharing the peak lists.  N: FFT size, hop: input hop, ch channels,
   coremode 0 / 1 / 2, n frames with phase_inc[n].  mag, phase: [ch][n][N/2+1] analysis spectra.  Outputs per (channel, frame):
   branch [ch][n]  0 pass-through first frame, 1 classic propagation, 2 locked, 3 int ratio (coremode 2);
   npeak [ch][n], peaks [ch][n][maxpk]  the peaks picked (coremode 1; 0 otherwise);
   rot, bin1, bin2 [ch][n][maxpk]  locked frames: each peak's peak_phase_rotation and region [bin1, bin2);
   out_phase [ch][n][N/2+1]  the phases after the core (the Nyquist bin keeps its analysis phase).
   maxpk: room for N/6 + 2 peaks per frame. */
void pvo_phase_core_frames(int N, int hop, int ch, int coremode, int n, const int *phase_inc, const float *mag, const float *phase, int maxpk,
                           int *branch, int *npeak, int *peaks, float *rot, int *bin1, int *bin2, float *out_phase) {
    pvo_t *p = pvo_create(44100, ch, 1.0f, 0.0f, MODE_SHIFT, coremode, N, hop);
    const int H = p->N / 2 + 1;
    int f, c, i;
    for (f = 0; f < n; ++f)
        for (c = 0; c < ch; ++c) {
            chan_t *ad = &p->chan[c];
            const long o = (long)c * n + f;
            const int first = coremode == 1 ? p->first_locked : p->first_simple, nprev = p->nprev;
            memcpy(ad->mag, mag + o * H, sizeof(float) * H);
            memcpy(ad->phase, phase + o * H, sizeof(float) * H);
            p->rec_rot = rot + o * maxpk; p->rec_bin1 = bin1 + o * maxpk; p->rec_bin2 = bin2 + o * maxpk;
            if (coremode == 1) modify_locked(p, ad, (size_t)phase_inc[f]);
            else if (coremode == 2) modify_intratio(p, ad, (size_t)phase_inc[f]);
            else modify_simple(p, ad, (size_t)phase_inc[f]);
            p->rec_rot = NULL; p->rec_bin1 = p->rec_bin2 = NULL;
            if (coremode == 2) branch[o] = 3;
            else branch[o] = first ? 0 : (p->npeak == 0 || nprev == 0) ? 1 : 2;
            npeak[o] = coremode == 1 ? p->npeak : 0;
            for (i = 0; i < npeak[o] && i < maxpk; ++i) peaks[o * maxpk + i] = p->peak[i];
            memcpy(out_phase + o * H, ad->phase, sizeof(float) * H);
        }
    pvo_destroy(p);
}
