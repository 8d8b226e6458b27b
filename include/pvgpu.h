/*
 * pvgpu.h -- C ABI of the B200-native phase vocoder (libpvgpu.so).
 *
 * This is the drop-in boundary for the phase-vocoder path of tangkk/audiomod.  Nothing like it
 * exists in the reference (it is a single-threaded C++ library); each entry point below names the
 * reference interface it stands in for (file:line relative to the reference tree).  The C++ class
 * audiomod::phasevocoder in audiomod_b200/csrc/pv_dropin.hpp and the Python mirror in
 * audiomod_b200/phasevocoder.py are thin shims over these calls.
 *
 * Conventions: planar float32, one pointer per channel, caller-owned buffers valid only during the
 * call (include/dafx/modbase.h:43,89,97).  Every function returns PVGPU_OK (0) or a PVGPU_E* code and
 * never aborts (the reference aborts / throws, FFT.cc:3168,3220, memallocators.h:91);
 * pvgpu_last_error() gives the message for the calling thread.  All computation runs on the GPU;
 * there is no CPU fallback: without a usable CUDA device every create call fails with PVGPU_ECUDA.
 */
#ifndef PVGPU_H_
#define PVGPU_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum { PVGPU_OK = 0, PVGPU_EINVAL = 1, PVGPU_ECUDA = 2, PVGPU_ENOMEM = 3, PVGPU_ESTATE = 4 };

/* mode / coremode values: include/dafx/phasevocoder.h:22-36 */
enum { PVGPU_CONSTANT = -1, PVGPU_NORMAL_SHIFT = 0, PVGPU_GENDER_CHANGE = 1, PVGPU_FORMANT_PRESERVE = 2,
       PVGPU_VOCODER_ROSENBERG = 3, PVGPU_VOCODER_CHORD = 4, PVGPU_NORMAL_STRETCH = 5, PVGPU_ROBOTIC = 6, PVGPU_WHISPER = 7,
       /* Extensions, not reference modes: gender change / formant-preserving shift with the cepstral spectral-envelope routine
        * (formantShiftSlice, src/phasevocoder/phasevocoderprocess.cc:925-999 + FFT::inverseCepstral, FFT.cc:2723-2733) that the
        * reference keeps commented out in favour of freqCompSlice (:824-840).  They compute what the reference computes with
        * those comments swapped back; FFT sizes 512..8192. */
       PVGPU_GENDER_CEPSTRAL = 8, PVGPU_FORMANT_CEPSTRAL = 9 };
enum { PVGPU_NORMAL_PV = 0, PVGPU_PHASE_LOCKED = 1, PVGPU_INT_RATIO = 2 };

/* sample formats of the batch entry points */
enum { PVGPU_F32 = 0, PVGPU_S16 = 1 };

/* Constructor arguments of audiomod::phasevocoder (include/dafx/phasevocoder.h:54,
 * src/phasevocoder/phasevocoder.cc:24-60), plus the CUDA device ordinal. */
typedef struct pvgpu_config {
    int sample_rate;
    int channels;
    float time_ratio;        /* timeratio */
    float pitch_semitones;   /* pitchshift, in semitones */
    int mode;                /* PVGPU_NORMAL_SHIFT ... */
    int coremode;            /* PVGPU_PHASE_LOCKED ... */
    int fftsize;             /* rounded up to a power of two like the reference (phasevocoderimpl.cc:177-181) */
    int hopsize;             /* 0 = automatic (phasevocoderimpl.cc:209-226) */
    int device;              /* CUDA device ordinal */
} pvgpu_config;

/* Sizes the reference derives in Impl::calculateSizes (phasevocoderimpl.cc:169-263). */
typedef struct pvgpu_info {
    int fftsize, hop, bins;
    float pitch_scale, hs_ratio;
    int resampler_active, resampler_filt_len;
    uint32_t resampler_num, resampler_den;
    int64_t outbuf_capacity;
} pvgpu_info;

const char *pvgpu_last_error(void);
int pvgpu_version(void);
/* number of CUDA devices visible (0 when there is no driver/GPU) */
int pvgpu_device_count(void);
/* derived sizes only; needs no GPU */
int pvgpu_describe(const pvgpu_config *cfg, pvgpu_info *info);
/* Host-only dry run of one stream through the CLI block protocol (main/main.cc:149,471-509): how many samples come
 * out, how many slices run, how many would be dropped because the output ring is full (phasevocoderprocess.cc:337-364).
 * block = 0 uses max(480, sr/100).  Needs no GPU. */
int pvgpu_plan_counts(const pvgpu_config *cfg, int64_t n_in, int block, int64_t *n_out, int64_t *n_slices, int64_t *n_dropped);

/* ---------------------------------------------------------------------------------------------
 * Streaming instance == one audiomod::phasevocoder object with fresh-process semantics.
 * ------------------------------------------------------------------------------------------- */
typedef struct pvgpu_stream pvgpu_stream;

/* phasevocoder::phasevocoder + init (phasevocoder.cc:24-85) */
int pvgpu_create(const pvgpu_config *cfg, pvgpu_stream **out);
/* Live batch: n_streams phasevocoder objects of one configuration advancing in lock-step -- every pvgpu_process /
 * pvgpu_retrieve / pvgpu_process_block call passes n_streams * channels row pointers (stream-major: row = stream * channels
 * + channel) and the same n for all of them.  One set of kernel launches and one copy each way per call serve all streams
 * (the schedule does not depend on the data), so the per-call cost of a real-time block is paid once, not per stream.  Every
 * stream produces exactly the samples its own pvgpu_create instance would (tests/test_gpu_live_batch.py).
 * n_streams * channels <= 65535.  pvgpu_stream_count returns n_streams (1 for pvgpu_create). */
int pvgpu_create_multi(const pvgpu_config *cfg, int n_streams, pvgpu_stream **out);
int pvgpu_stream_count(const pvgpu_stream *s);
/* Device rows: the streaming calls for audio that already lives on the GPU (a decoder, a synthesis model, another effect).
 * d_in / d_out / d_buf point to float32 device memory of the instance's device, row r (= stream * channels + channel) at
 * ptr + r * pitch floats.  Everything is enqueued on `cuda_stream` (NULL = the legacy default stream) and NO call waits for
 * the device: the schedule does not depend on the data, so the counts (pvgpu_available, the return value of
 * pvgpu_retrieve_device, *ready) are known on the host at once.  Use one stream for all calls of an instance (or order them
 * yourself).  Same samples as the host-row calls, bit for bit (tests/test_gpu_live_batch.py).  An instance is fed either host
 * rows or device rows, not both (PVGPU_ESTATE). */
int pvgpu_process_device(pvgpu_stream *s, const float *d_in, int64_t in_pitch, int n, void *cuda_stream);
int pvgpu_retrieve_device(pvgpu_stream *s, float *d_out, int64_t out_pitch, int n, void *cuda_stream);   /* returns the count, < 0: -error */
int pvgpu_process_block_device(pvgpu_stream *s, float *d_buf, int64_t pitch, int n, void *cuda_stream, int *ready);
/* int16 twins of the streaming calls, for hosts that hold audio as 16-bit PCM: the same semantics, counts, *ready rule and
 * stream ordering as the float32 call of the same name without _s16.  Every stream of an instance fed int16 rows produces
 * exactly what a float32 instance produces with the same calls when its input is fed as (float)(s * (1.0/32768)) and every
 * output sample is quantised as (short)(int)clamp(x * 32768.f, -32768, 32767), truncating toward zero -- the batch's PVGPU_S16
 * rules (main/wavfile.cc:733-752, 1294-1306).  The samples stay int16 from the caller's rows to the device and back (half the
 * bytes of float32 to pack and copy); the kernels convert as they load and quantise as they store.  Device pitches are in int16
 * elements; device rows may start at any 2-byte boundary.  The first data call fixes an instance's rows: host or device,
 * float32 or int16 -- a call of another kind returns PVGPU_ESTATE and its message names the call to use. */
int pvgpu_process_s16(pvgpu_stream *s, const int16_t *const *in, int n);
int pvgpu_retrieve_s16(pvgpu_stream *s, int16_t *const *out, int n);                 /* returns the count, < 0: -error */
int pvgpu_process_block_s16(pvgpu_stream *s, int16_t *const *buf, int n, int *ready);
int pvgpu_process_device_s16(pvgpu_stream *s, const int16_t *d_in, int64_t in_pitch, int n, void *cuda_stream);
int pvgpu_retrieve_device_s16(pvgpu_stream *s, int16_t *d_out, int64_t out_pitch, int n, void *cuda_stream);   /* returns the count, < 0: -error */
int pvgpu_process_block_device_s16(pvgpu_stream *s, int16_t *d_buf, int64_t pitch, int n, void *cuda_stream, int *ready);
/* Post-chain of FFT-free effects (gain, compressor, limiter, biquad sections; the kinds, parameters and limits of
 * pvgpu_batch_set_postchain below, coefficients from cfg->sample_rate exactly as the batch computes them; at most 12 entries,
 * pvgpu_equalizer_chain output works unchanged) on a streaming instance or live batch -- the reference's effect objects chained
 * after the phase vocoder in SDK use (gain / compressor / limiter / equalizer after phasevocoder).
 *   What it runs on: the instance's output stream.  Every sample the instance produces goes through the chain once, in order,
 *   before it enters the output ring: the result is what the reference's effect objects compute when fed everything getOutData
 *   returns, in order.  Each effect's state is carried per row from call to call, so call sizes and partial retrieves do not
 *   change the result.  Sample counts, pvgpu_available and the *ready rule do not change; processBlock leaves the buffer
 *   untouched while output is not ready, and input that passes through unprocessed never meets the chain.
 *   Live batch: one chain serves all n_streams * channels rows; each stream gets what its own instance with the chain produces.
 *   Setting, changing, clearing: before the first data call or between calls.  A new chain takes effect at the next data call
 *   with fresh effect state, as if the effect objects had just been constructed; samples already in the output ring are not
 *   touched; n_fx = 0 clears the chain and later output is the plain output again, bit for bit.  The phase vocoder's own state
 *   is never touched.  Not a real-time call: it waits for the instance's outstanding device work.  Device-row calls enqueue the
 *   chain on their stream and still do not wait.
 *   int16 instances (*_s16): the chain runs on the float samples and its result is quantised by the int16 rule above, so each
 *   stream equals quantise(float32 instance with the same chain fed s / 32768).
 *   Errors: PVGPU_EINVAL for n_fx < 0 or > 12, a null chain with n_fx > 0, an unknown kind, a compressor ratio <= 0 (the
 *   batch's messages).  On an instance whose mode does nothing (an unknown mode) it succeeds and changes nothing. */
typedef struct pvgpu_fx pvgpu_fx;
int pvgpu_set_postchain(pvgpu_stream *s, const pvgpu_fx *chain, int n_fx);
/* Parameters of one stream's post-chain on a streaming instance or live batch (each user's level, EQ preset or limiter ceiling
 * on a voice server, changed while they talk).
 *   What it changes: the parameters of the chain pvgpu_set_postchain gave the instance, for one stream (all of its channel rows).
 *   n_fx and the kind in every position must equal the instance's chain; the parameters are the same constructor arguments,
 *   converted the same way at cfg->sample_rate.  Other streams are not touched, bit for bit.
 *   When it takes effect: every output sample produced by a data call after this one uses the new parameters, every sample
 *   produced earlier used the old ones; samples already in the output ring (host or device) keep their values.
 *   State is kept: the stream's effect state carries over (biquad x1, x2, y1, y2; the compressor's level; the limiter's peak,
 *   gain, delay line and position) and the new coefficients apply from the next sample on, as if the effect objects'
 *   coefficient members had been recomputed in place.  The limiter's delay length depends only on the sample rate.
 *   Real-time safe: no device work, never waits for the device, allocates nothing.  It converts one chain on the host and records
 *   the change; the next data call that runs the chain uploads the pending changes on that call's stream (host rows: the
 *   instance's stream; device rows: the caller's stream) before the chain runs.  Several updates between two calls coalesce;
 *   the last one for a stream wins.
 *   pvgpu_set_postchain is unchanged: it sets the kinds and gives every stream the same parameters with fresh state, discarding
 *   earlier per-stream parameters.  pvgpu_set_stream_postchain right after it, before the next data call, gives that stream its
 *   own parameters with fresh state -- per-user presets are one pvgpu_set_postchain, then one call per stream.
 *   A pvgpu_create instance is a live batch of one: stream 0.
 *   Errors (PVGPU_EINVAL, the instance unchanged): stream outside [0, n_streams); no chain on the instance; n_fx other than the
 *   instance's; a kind other than the instance's in some position (the message names the position and both kinds); a null
 *   chain; the argument errors of pvgpu_set_postchain (a compressor ratio <= 0, ...).  On an instance whose mode does nothing
 *   (an unknown mode) it succeeds and changes nothing. */
int pvgpu_set_stream_postchain(pvgpu_stream *s, int stream, const pvgpu_fx *chain, int n_fx);
/* Loudness meters on a streaming instance or live batch (ITU-R BS.1770-4 / EBU Tech 3341 momentary and short-term loudness,
 * sample peak).  Not the reference's loudnessmeter object: specified by the published standard, and nothing here restates
 * src/meter/loudnessmeter.cc.  Per stream: momentary and short-term loudness in LUFS; per row (stream * channels + channel): peak.
 *   What is measured: every sample the instance produces, once, in order, after the post-chain -- the chain's rule: input that
 *   passes through unprocessed is not measured.  float32 rows as the float value; int16 rows as delivered, s / 32768 in double.
 *   K-weighting: two direct-form-I biquad sections per row, shelf then high-pass, in double precision, each evaluated as
 *   b0*x + b1*x1 + b2*x2 - a1*y1 - a2*y2 from left to right with every product and sum rounded on its own (__dmul_rn /
 *   __dadd_rn / __dsub_rn, no contraction); the state carries from call to call.  Coefficients: pvgpu_kweighting_design.
 *   Windows: sub-blocks of L = (sample_rate + 5) / 10 samples (integer division) counted from the first measured sample; a row's
 *   sub-block energy is the sum of z^2 in double, in sample order; a stream's loudness over the last W sub-blocks is
 *   -0.691 + 10 log10(sum over channels of sum over sub-blocks of E / (W * L)), summed over the sub-blocks oldest to newest, then over
 *   the channels in order.  Momentary: W = 4 (400 ms); short-term: W = 30 (3 s).  No gating, every channel weighs 1.0; sub-blocks
 *   before the first measured sample count as silence; zero energy gives -inf.  Both values are updated at the end of every data
 *   call from the sub-blocks completed so far, and a call that completes no sub-block leaves them unchanged, so call sizes never
 *   change the values at equal `measured`.
 *   peak: the sample peak (not true peak), max |x| per row over the samples the most recent call that produced output produced.
 *   measured: samples per row measured since the meters were enabled.
 *   pvgpu_set_meters: before the first data call or between calls.  Not a real-time call: it allocates and waits for the
 *   instance's outstanding device work.  enable = 1 starts from fresh meter state (momentary and short-term -inf, peaks 0,
 *   measured 0), also when the meters were on already; enable = 0 stops every meter launch and copy, and the getters return
 *   PVGPU_ESTATE.  Meters never change output samples, counts, *ready or anything else.  On an instance whose mode does nothing
 *   (an unknown mode) it succeeds and nothing is ever measured.
 *   pvgpu_get_meters (host rows): reads a host mirror -- no device work, never waits, allocates nothing: real-time safe.  The
 *   values came back with the data call's own output copy, before its one synchronisation.  Any pointer may be NULL.
 *   pvgpu_get_meters_device (device rows): enqueues one device-to-device cudaMemcpyAsync of [2*S + S*C] floats (momentary S,
 *   short-term S, peak S*C) to d_dst on cuda_stream (NULL = the legacy default stream) and does not wait; it is ordered after the
 *   calls enqueued before it on that stream (use one stream for all calls of an instance).
 *   Before the first data call either getter works; afterwards the getter of the other kind of rows returns PVGPU_ESTATE and its
 *   message names the getter to use.  Errors: PVGPU_EINVAL for a null instance or d_dst, enable other than 0 or 1; PVGPU_ESTATE
 *   when the meters are off. */
int pvgpu_set_meters(pvgpu_stream *s, int enable);
int pvgpu_get_meters(const pvgpu_stream *s, float *momentary /*[S] or NULL*/, float *short_term /*[S] or NULL*/,
                     float *peak /*[S*C] or NULL*/, int64_t *measured /*or NULL*/);
int pvgpu_get_meters_device(pvgpu_stream *s, float *d_dst /*[2*S + S*C]: momentary, short-term, peak*/, void *cuda_stream,
                            int64_t *measured /*or NULL*/);
/* K-weighting at this sample rate, needs no GPU: {shelf b0, b1, b2, a1, a2, high-pass a1, a2} (high-pass b = {1, -2, 1}, a0 = 1).
 * libebur128's analog-prototype formulas restated in double: shelf f0 = 1681.974450955533, G = 3.999843853973347,
 * Q = 0.7071752369554196, K = tan(pi f0 / sr), Vh = 10^(G/20), Vb = Vh^0.4996667741545416, a0 = 1 + K/Q + K^2,
 * b = {(Vh + Vb K/Q + K^2)/a0, 2(K^2 - Vh)/a0, (Vh - Vb K/Q + K^2)/a0}, a1 = 2(K^2 - 1)/a0, a2 = (1 - K/Q + K^2)/a0; high-pass
 * f0 = 38.13547087602444, Q = 0.5003270373238773, the same a1 and a2.  At 48 kHz: BS.1770-4's tables.  sample_rate <= 0: PVGPU_EINVAL. */
int pvgpu_kweighting_design(int sample_rate, double *coeffs /*[7]*/);
/* phasevocoder::~phasevocoder (phasevocoder.cc:62-67) */
void pvgpu_destroy(pvgpu_stream *s);
/* modbase_offline::processInData (modbase.h:89, phasevocoder.cc:87-108): consume n samples per channel */
int pvgpu_process(pvgpu_stream *s, const float *const *in, int n);
/* modbase_offline::getOutSamples (modbase.h:114): samples available after the last pvgpu_process */
int pvgpu_available(const pvgpu_stream *s);
/* modbase_offline::getOutData (modbase.h:97, phasevocoder.cc:110-124): copies min(n, available); returns the count */
int pvgpu_retrieve(pvgpu_stream *s, float *const *out, int n);
/* modbase::processBlock (modbase.h:43, phasevocoder.cc:126-183): in place; returns 0 and sets *ready=1 when the
 * block was replaced, or returns 0 with *ready=0 (buffer untouched) when fewer than n samples were available --
 * i.e. *ready is modbase::outputReady() (modbase.h:61) */
int pvgpu_process_block(pvgpu_stream *s, float *const *buf, int n, int *ready);
int pvgpu_stream_info(const pvgpu_stream *s, pvgpu_info *info);

/* ---------------------------------------------------------------------------------------------
 * Batch: many independent streams with one configuration, each processed exactly as one fresh
 * `audiomod-exe <mode> in.wav out.wav ...` process would (main/main.cc:149,471-509: blocks of
 * max(480, sr/100); pitch modes are flushed with zero blocks and truncated to the input length,
 * time_stretch is not flushed).  Rows are channel-planar: row = stream * channels + channel.
 * ------------------------------------------------------------------------------------------- */
typedef struct pvgpu_batch pvgpu_batch;

int pvgpu_batch_create(const pvgpu_config *cfg, int n_streams, int64_t max_in_samples, pvgpu_batch **out);
void pvgpu_batch_destroy(pvgpu_batch *b);
/* Fix the per-stream input lengths (samples per channel) and get the per-stream output lengths.
 * block = 0 uses the CLI block size.  Must be called before a run; may be called again. */
int pvgpu_batch_plan(pvgpu_batch *b, const int64_t *n_in, int block, int64_t *n_out);
/* Inputs and outputs resident in device memory: d_in [rows][in_stride], d_out [rows][out_stride]
 * (elements of `fmt`), out_stride >= max n_out.  cuda_stream is the caller's cudaStream_t, with CUDA's own convention
 * that NULL is the legacy default stream: the run is ordered after everything queued on that stream before the call and
 * before everything queued on it afterwards.  The call only enqueues work and never blocks the host;
 * pvgpu_batch_synchronize waits for the last run. */
int pvgpu_batch_run_device(pvgpu_batch *b, const void *d_in, int64_t in_stride, void *d_out, int64_t out_stride, int fmt,
                           void *cuda_stream);
int pvgpu_batch_synchronize(pvgpu_batch *b);
/* Host buffers (pinned or pageable): one pointer per row; copies in, runs, copies out, synchronises.
 * Stream groups are pipelined so H2D, kernels and D2H overlap. */
int pvgpu_batch_run_host(pvgpu_batch *b, const void *const *in_rows, void *const *out_rows, int fmt);
/* FFT-free effects as a post-chain on the batch's float32 output rows (SURVEY.md 8(f) rank 4): applied, in order, to the columns
 * every frame chunk completes, with their state carried along the row -- exactly the reference objects' processBlock run over a
 * stream's whole output, whatever the block size.  kinds and parameters (the reference constructors' arguments):
 *   PVGPU_FX_GAIN        p = {gain}                                                          src/gain/gain.cc
 *   PVGPU_FX_COMPRESSOR  p = {dBThreshold, ratio, dBMakeUpGain, attackTimeMs, releaseTimeMs}  src/dynamics/compressor.cc
 *   PVGPU_FX_LIMITER     p = {dBThreshold, dBMakeUpGain, attackTimeMs, releaseTimeMs}          src/dynamics/limiter.cc (6 ms look-ahead)
 *   PVGPU_FX_BIQUAD      p = {type, cutoffFreq, q, dBGain}, type = biquadfilter::Type              src/common/filters/biquadfilter.cc
 *                        (0 highPass, 1 lowShelf, 2 peaking, 3 notch, 4 highShelf, 5 lowPass, 6 / 7 band-pass, 8 allpass)
 * n_fx = 0 clears the chain; at most 12 effects.  Takes effect at the next run. */
enum { PVGPU_FX_GAIN = 1, PVGPU_FX_COMPRESSOR = 2, PVGPU_FX_LIMITER = 3, PVGPU_FX_BIQUAD = 4 };
struct pvgpu_fx { int kind; float p[6]; };   /* typedef above, at pvgpu_set_postchain */
int pvgpu_batch_set_postchain(pvgpu_batch *b, const pvgpu_fx *chain, int n_fx);
/* the equalizer object (src/equalizer/equalizer.cc: eight biquad sections in a fixed order, paramlist = {use, cutoff, Q, gain} x 8,
 * NULL = its defaults) expanded into PVGPU_FX_BIQUAD entries for pvgpu_batch_set_postchain; chain must hold 8 entries */
int pvgpu_equalizer_chain(const float *paramlist /*[32] or NULL*/, pvgpu_fx *chain /*[8]*/, int *n_fx);
/* biquadfilter::computeCoeffs: {b0, b1, b2, a0, a1, a2} of one section (needs no GPU) */
int pvgpu_biquad_design(int type, int sample_rate, float cutoff, float q, float db_gain, float *coeffs /*[6]*/);
/* counters of the last run: kernels launched, slices per stream, H2D/D2H bytes */
int pvgpu_batch_stats(const pvgpu_batch *b, int64_t *kernel_launches, int64_t *slices, int64_t *h2d_bytes, int64_t *d2h_bytes);
int pvgpu_batch_info(const pvgpu_batch *b, pvgpu_info *info);
/* Per-kernel device timing with CUDA events recorded on the launching stream around every launch.  kinds:
 * 0 analyse, 1 phase core (polar), 2 synthesise, 3 overlap-add + resample, 4 fused synthesise + overlap-add + resample, 5 fixed phase (robotic/whisper on polar spectra) or the cepstral envelope kernel (modes 8 / 9),
 * 6 lock_peaks, 7 lock_chain (phase-locked core on Cartesian spectra).
 * pvgpu_batch_kernel_times synchronises the device and returns the totals since profiling was enabled. */
enum { PVGPU_KINDS = 8 };
int pvgpu_batch_profile(pvgpu_batch *b, int enable);
int pvgpu_batch_kernel_times(pvgpu_batch *b, double *ms /*[PVGPU_KINDS]*/, int64_t *count /*[PVGPU_KINDS]*/);
/* tuning (0 = keep): frames per chunk; rows per group (by default the whole batch is one group when its workspace fits,
 * and equal-length batches in evenly spaced host rows are pipelined along time; an explicit value selects pipelining
 * across row groups); how many row groups are in flight at once (1..4; each has its own stream, workspace and staging) */
int pvgpu_batch_tune(pvgpu_batch *b, int frames_per_chunk, int rows_per_group, int contexts);
/* Resynthesis back end: 0 = the split kernels (inverse FFT -> frame ring in HBM -> overlap-add + resampler); 1 = the fused
 * inverse-FFT + overlap-add + resampler kernel with the accumulator in shared memory wherever the FFT size has one
 * (512..8192); -1 (default) = automatic: the split kernels -- measured faster on B200, profiles/r02_summary.md -- unless the
 * stretch ratio overlaps more frames than their per-CTA tables hold, then the fused kernel, which has no such limit.  Both
 * produce bit-identical samples (tests/test_gpu_fused.py).  The environment variable PVGPU_FUSED=0/1 overrides the choice for
 * every instance, including streaming ones. */
int pvgpu_batch_set_fused(pvgpu_batch *b, int enable);

/* ---------------------------------------------------------------------------------------------
 * Multi-GPU batch: the same streams sharded across several devices of one box (BASELINE.json configs[3]: "4096 streams
 * ... sharded across 1/2/4/8 B200"; SURVEY.md 8(b)/(e)).  Nothing like it exists in the reference (one thread, no device).
 * A stream (all of its channels) shares nothing with any other stream, so there is no collective: the library partitions
 * the streams (equal lengths: contiguous balanced blocks; ragged: longest first, dealt boustrophedon), runs one
 * pvgpu_batch per device from one host thread per device, and every device's D2H copies land directly in the caller's
 * row pointers -- the "host-side gather".  Results are bit-identical to a single-device run.
 * ------------------------------------------------------------------------------------------- */
typedef struct pvgpu_mbatch pvgpu_mbatch;
/* devices == NULL (or n_dev <= 0): every visible device.  cfg->device is ignored. */
int pvgpu_mbatch_create(const pvgpu_config *cfg, int n_streams, int64_t max_in_samples, const int *devices, int n_dev, pvgpu_mbatch **out);
void pvgpu_mbatch_destroy(pvgpu_mbatch *m);
int pvgpu_mbatch_plan(pvgpu_mbatch *m, const int64_t *n_in, int block, int64_t *n_out);
/* rows in the caller's stream order: row = stream * channels + channel, exactly like pvgpu_batch_run_host */
int pvgpu_mbatch_run_host(pvgpu_mbatch *m, const void *const *in_rows, void *const *out_rows, int fmt);
int pvgpu_mbatch_stats(const pvgpu_mbatch *m, int64_t *kernel_launches, int64_t *h2d_bytes, int64_t *d2h_bytes, int *devices_used);
/* CUDA device ordinal that processes each stream (after pvgpu_mbatch_plan) */
int pvgpu_mbatch_owner(const pvgpu_mbatch *m, int *owner_device /*[n_streams]*/);
/* the partition rule on its own (needs no GPU): owner[s] in [0, n_dev) */
int pvgpu_shard_streams(const int64_t *n_in, int n_streams, int n_dev, int *owner);

/* Page-locked host buffers for batch I/O, placed on the NUMA node of `device` (a B200 box has two CPU sockets; pinned
 * pages on the far socket cross the inter-socket link and halve the copy rate once all eight GPUs move data).  flags: */
enum { PVGPU_HOST_NUMA_LOCAL = 1, PVGPU_HOST_HUGEPAGES = 2 /* explicit 2 MB pages (MAP_HUGETLB) when the box has a pool; else THP */ };
int pvgpu_host_alloc(void **ptr, size_t bytes, int device, int flags);
int pvgpu_host_free(void *ptr);
/* where a buffer ended up: node it was bound to (-1: not bound), whether explicit huge pages were granted, mapped bytes */
int pvgpu_host_info(const void *ptr, int *numa_node, int *hugepages, size_t *bytes);
/* NUMA node of a CUDA device from sysfs (-1 when unknown); pin the calling thread to that node's cores */
int pvgpu_device_numa_node(int device);
int pvgpu_bind_thread_to_device(int device);

/* ---------------------------------------------------------------------------------------------
 * File -> file: what `audiomod-exe <effect> in.wav out.wav <args>` does for one file (main/main.cc:95-161, 471-509 and the
 * RIFF reader / writer main/wavfile.cc:672-812, 848-1016, 1135-1182, 1294-1306, 1474-1526), for many files in one call.
 * Input: RIFF/WAVE integer PCM, 8/16/24/32 bit, mono or stereo; output: 16-bit PCM with the reference's 56-byte header
 * (main.cc:136).  cfg->sample_rate and cfg->channels are ignored (taken from each file; files are grouped into one batch per
 * (sample rate, channels, 16-bit or not)); devices as in pvgpu_mbatch_create.  Per-file results are reported in the jobs.
 * ------------------------------------------------------------------------------------------- */
typedef struct pvgpu_wav_job {
    const char *in_path, *out_path;
    int status;                         /* out: PVGPU_OK or this file's error code */
    int sample_rate, channels, bits;    /* out: from the input header */
    int64_t frames_in, frames_out;      /* out: samples per channel read / written */
    char message[160];                  /* out: error text */
} pvgpu_wav_job;
int pvgpu_run_wav_files(const pvgpu_config *cfg, pvgpu_wav_job *jobs, int n_jobs, const int *devices, int n_dev);

/* ---------------------------------------------------------------------------------------------
 * Stage hooks for the parity tests (tests/ compares each stage with the CPU oracle).  Device work,
 * host pointers.  frames: [n_frames][fftsize] raw (un-windowed) frames.
 * ------------------------------------------------------------------------------------------- */
/* analyzeSlice + FFT::forwardPolar (phasevocoderprocess.cc:492-503, FFT.cc:2617-2631) */
int pvgpu_test_forward_polar(int device, int fftsize, int n_frames, const float *frames, float *mag, float *phase);
/* 1/N scale + FFT::inversePolar + ifftshift + window (phasevocoderprocess.cc:1024-1056) */
int pvgpu_test_inverse_polar(int device, int fftsize, int n_frames, const float *mag, const float *phase, float *frames);
/* device atan2f restatement (FFT.cc:2629 -> glibc atan2f) */
int pvgpu_test_atan2f(int device, int64_t n, const float *y, const float *x, float *out);
/* princarg (src/common/system/sys.h:84-91) */
int pvgpu_test_princarg(int device, int64_t n, const double *a, double *out);
/* the post-chain once over [rows][n] float32 host samples, in place, from fresh effect state: the conversion and the kernel of
 * pvgpu_batch_set_postchain / pvgpu_set_postchain at this sample rate (a bit-exact anchor for the streaming post-chain's tests) */
int pvgpu_test_postchain(int device, int sample_rate, const pvgpu_fx *chain, int n_fx, int rows, int64_t n, float *samples);
/* the meter kernels of pvgpu_set_meters over [streams*channels][n] float32 host samples from fresh state, fed in pieces of `call`
 * samples; momentary / short_term [streams], peak [streams*channels] (over the last piece) */
int pvgpu_test_loudness(int device, int sample_rate, int channels, int streams, int64_t n, int call, const float *samples,
                        float *momentary, float *short_term, float *peak);
/* host-only self-test of the live batch's containers (ring FIFO, row-copy pool, non-temporal copies; float32 and int16 samples):
 * 0 = ok, else the number of the failed check (negative: an error code).  Needs no device. */
int pvgpu_test_host_structs(void);

#ifdef __cplusplus
}
#endif
#endif /* PVGPU_H_ */
