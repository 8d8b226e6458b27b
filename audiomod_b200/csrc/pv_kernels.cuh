// Device-side view of a batch and the kernel launchers (sm_100a).  See pv_kernels.cu.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "pv_plan.h"

namespace pvgpu {

constexpr int kMaxStages = 8;

// Constant tables + sizes, passed by value to every kernel.
struct DevPlan {
    int N, H, half, nc, hop, Hp;        // Hp: padded row length of a spectrum (floats)
    int nstages;
    int radix[kMaxStages], span[kMaxStages];
    const float *window;                // N
    const float2 *tw_fwd, *tw_inv;      // nc
    const float2 *tw2_fwd, *tw2_inv, *tw3_fwd, *tw3_inv;   // the same twiddles in the second / third pass's access order (pv_fft.cuh)
    const float2 *stw_fwd, *stw_inv;    // nc
    const uint16_t *perm;               // nc
    const float *omega;                 // half
    float inv_n;                        // 1.f / N
    double two_pi_hop;                  // 2*M_PI*hop  (double product, phasevocoderprocess.cc:625)
    // frequency-axis warp (formant / gender), 0 = off
    float freq_comp, fixed_gain;
    const float4 *warp_tab;             // Cartesian pipeline: per target bin (gain cos dw, gain sin dw, source bin as int bits, 0), or null
    // resampler
    int rs_active, rs_direct;
    uint32_t rs_num, rs_den, rs_filt_len, rs_oversample;
    int rs_int_adv, rs_frac_adv;
    const float *rs_table;
    const float4 *rs_quads;             // [rs_table_len] (tab[e-2], tab[e-1], tab[e], tab[e+1]) for the interpolated mode
    int rs_table_len;
};

// One group of channel rows being processed; all pointers are device pointers.
struct DevRows {
    int rows;                 // channel rows in this group (streams * channels)
    int channels;
    const void *in;           // [rows][in_stride] float32 or int16 PCM (fmt), element 0 is input sample in_base
    int fmt;                  // 0: float32 rows, 1: int16 rows (input, and output unless out_f32)
    int out_f32;              // 1: the resynthesis stores float32 rows whatever fmt is (an int16 streaming instance whose post-chain
                              //    quantises); 0: it stores fmt.  Read through out_fmt() (pv_synth.cuh)
    int64_t in_stride, in_base;
    const int64_t *n_in;      // per row: valid input samples (zeros beyond), global coordinates
    float *mag, *phase;       // [rows][F][Hp] spectra of the current frame chunk
    int F;                    // frame slots per row in mag/phase
    float *frames;            // [rows][Fr][N] synthesised frames, slot = frame % Fr
    int Fr;
    void *out;                // [rows][out_stride] (fmt), element 0 is output position out_base
    int64_t out_stride, out_base;
    const int64_t *n_out;     // per row: output positions >= n_out are not stored (truncation to the stream's length)
    float *prev_phase, *prev_out;   // [rows][half] phase-core state
    int *peaks;               // [streams][1 + maxpk]: count, then previous peak list (shared by a stream's channels)
    int maxpk;
    int *started;             // [streams] 0 until the first slice of the stream went through the core
    // phase-locked core on Cartesian spectra (pv_lock.cuh): k_lock_peaks -> k_lock_chain -> k_synthesise_t
    int2 *lock_hdr;           // [rows][F]: (peaks, frame kind: 0 pass-through first frame, 1 classic propagation, 2 locked)
    float4 *lock_rec;         // [rows][F][rec_stride]: per peak (phi[p2], prev_phase[p1], advance, p1 | region of p1 << 16);
    int rec_stride;           //   classic frames: float advance[half], prev_phase[half].  rec_stride = max(maxpk, half / 2)
    unsigned short *lock_map; // [rows][F][half]: region (= peak index) of every bin of the frame
    float2 *lock_csn;         // [rows][F][maxpk]: (cos, sin) of every region's rotation
    float *lock_tail;         // [rows][2][Hp]: (re, im) of the last frame of the previous launch
    int *lock_kind;           // [rows]: chain state of the channel (kind 0..3, see pv_lock.cuh)
    float *lock_rot;          // [rows][maxpk]: rotations of the channel's previous frame (kind 2); kind 1 keeps prev_out
    // fused inverse FFT + overlap-add + resampler (pv_fused.cu): what a row carries from one launch to the next
    float *ola_tail;          // [rows][N]: the unfinished part of the overlap-add accumulator (from the next slice's position on)
    float *res_hist;          // [rows][filt_len + 8]: the last normalised samples (resampler history), zeros before the stream
    int zero_mask;            // always 0; an operand the compiler cannot fold, used to tie load batches together (pv_synth.cuh)
    long aux_base;            // slice index of element 0 of the whisper table / carrier spectra
    int spec;                 // 0: spectra are (mag, phase); 1: Cartesian (re in mag[], im in phase[]) -- modes that never use the
                              //    analysis phase (robotic, whisper, vocoder, constant) and the phase-locked core of the plain
                              //    shift / stretch / formant / gender modes (k_lock_peaks + k_lock_chain) skip sqrtf/atan2f in the analysis kernel
    int synth_kind;           // 0: phases come from the spectra; 1: robotic (phase 0); 2: whisper (phase table); 3: constant;
                              // 4: Cartesian phase-locked core (rotate every bin by its region's (cos, sin))
    const float *whisper;     // [slices][channels][H] phases of the whisper mode (indexed by absolute slice - aux_base)
};

void launch_analyse(const DevPlan &p, const DevRows &g, long k0, int nframes, cudaStream_t st);
void launch_phase_core(const DevPlan &p, const DevRows &g, int coremode, const SliceRec *recs, long recs_base, long k0, int nframes, cudaStream_t st);
// the phase-locked core on Cartesian spectra (g.spec == 1): frame-parallel part, then the serial chain
void launch_lock_peaks(const DevPlan &p, const DevRows &g, const SliceRec *recs, long recs_base, long k0, int nframes, cudaStream_t st);
void launch_lock_chain(const DevPlan &p, const DevRows &g, int nframes, cudaStream_t st);
int lock_rec_stride(const DevPlan &p, int maxpk);
void launch_fixed_phase(const DevPlan &p, const DevRows &g, const float *table /*[slices][channels][H] indexed by absolute slice, or null = zeros*/,
                        long k0, int nframes, cudaStream_t st);
void launch_synthesise(const DevPlan &p, const DevRows &g, const float *car_mag, const float *car_phase /*[slices][Hp] indexed by absolute slice, or null*/,
                       long k0, int nframes, cudaStream_t st);
// Host-built work list of the resampler for one run of slices (see k_ola_resample): the run's outputs bucketed by
// sinc-table phase, output order inside a bucket, buckets padded to multiples of kResBlock.  Entry = (tap-0 position relative to
// u_lo + kResPad) << 16 | (output position relative to out_first); 0xffffffff = padding.  rs_frac holds the four cubic
// interpolation coefficients of each entry (interpolated mode, 16 bytes) or the table phase as raw bits (direct mode, 4 bytes).
constexpr int kMaxBuckets = 8;      // resampler table phases (oversample <= 8 at quality 4)
constexpr int kResPerThread = 4;    // outputs a thread of k_ola_resample accumulates at once
constexpr int kResBlock = 32 * kResPerThread;   // entries of a full warp step (the bank-aware ordering permutes a whole bucket of a run)
constexpr int kResPad = 1024;       // bias that keeps the packed tap-0 offset non-negative at the start of a stream
struct ResampleRun {
    int64_t u_lo;        // first normalised-stream position the run reads (clipped to 0)
    int64_t out_first;   // output position of the run's first slice
    int ent_off;         // offset of the run's entries in rs_ent / rs_frac
    int padded;          // entries including padding
    // what k_ola_resample would otherwise find by walking the slice records (four dependent loads before its tables can be filled):
    int64_t ola_base;    // ola_off of the first frame overlapping the run's slices and its resampler history
    int back_slices;     // ka - kmin: slices before the run that hold its resampler history
    int back_frames;     // ka - jmin: frames before the run's first slice that overlap those
    int rsv[5];
    int step_off;        // offset of the run's warp steps in rs_steps
    int n_steps;         // step = entry offset within the run | (rows - 1) << 20 | table phase << 24, rows <= kResPerThread
    int pad[1];
};
static_assert(sizeof(ResampleRun) == 72, "ResampleRun layout");

// largest run (slices per CTA) not above `run` that the packed entries and the CTA tables can hold
int ola_run_limit(const DevPlan &p, int run, int max_consumed, int max_out);
// size of k_ola_resample's per-CTA slice table (run + resampler history)
int ola_max_table_slices();
// dynamic shared memory of the phase-locked core's kernels on Cartesian spectra for C channels per stream
size_t lock_smem_bytes(const DevPlan &p, int channels, int maxpk);
// overlap-add + normalisation (+ resampler when p.rs_active); `run` consecutive slices per CTA starting at k0 (which must
// be run_origin + a multiple of run), max_consumed = the largest number of normalised samples any slice contributes
void launch_ola_resample(const DevPlan &p, const DevRows &g, const SliceRec *recs, const float *norm, int64_t norm_base, long recs_base,
                         long k0, int nframes, int run, int max_consumed, const ResampleRun *runs, const unsigned *rs_ent, const float *rs_frac,
                         const unsigned *rs_steps, long run_origin, cudaStream_t st);
// Fused inverse FFT + window + overlap-add + normalisation + resampler (k_synth_ola, pv_fused.cu): one CTA per row runs the
// frames [k0, k0 + nf) of a chunk in order, `run` frames per round (a multiple of the frames it has in flight).
struct FusedArgs {
    const SliceRec *recs; long recs_base;
    const float *norm; int64_t norm_base;
    long k0; int nf;
    int run;          // frames per round = slices per resampler work list
    int acc_len;      // floats of the shared-memory accumulator ring: power of two >= N + (run - 1) * largest shift increment
    int in_len;       // floats of the resampler input window: hist_len + run * largest per-slice contribution (+ pad)
    int hist_len;     // filt_len + 8 normalised samples carried between rounds / launches (0 without resampler)
    const ResampleRun *runs; const unsigned *rs_ent; const float *rs_frac; const unsigned *rs_steps; long run_origin;
    const float *car_mag, *car_phase;   // vocoder carrier spectra or null
};
int fused_frames_in_flight(int N);   // 0: this FFT size has no fused kernel
bool fused_plan(const DevPlan &p, int frames_per_chunk, int max_shift, int max_consumed, int max_out, size_t smem_limit, FusedArgs *out);
cudaError_t launch_synth_ola(const DevPlan &p, const DevRows &g, const FusedArgs &a, cudaStream_t st);

// cepstral spectral-envelope modification of the chunk's spectra in place (pv_cepstral.cu); false: no kernel for this FFT size
bool launch_cepstral(const DevPlan &p, const DevRows &g, float env_comp, int nframes, cudaStream_t st);
// ---- post-chain of FFT-free effects on the output rows (pv_post.cu) ----
constexpr int kMaxPostFx = 12;
enum { kFxGain = 1, kFxCompressor = 2, kFxLimiter = 3, kFxBiquad = 4 };
// coefficients as the reference's constructors compute them (host, glibc): gain p[0]; compressor p = {threshold dB, ratio,
// make-up dB, alphaAttack, alphaRelease}; limiter p = {makeUpGain, threshold (linear), alphaAttack, alphaRelease, initial xPeak},
// delay = (int)(sr * 0.001 * 6) + 1 samples of look-ahead; biquad p = {b0, b1, b2, a0, a1, a2} (biquadfilter::computeCoeffs)
struct PostFx { int kind; int delay; float p[6]; };
struct PostChain { int n; PostFx fx[kMaxPostFx]; };
int postchain_state_stride(const PostChain &pc);
void launch_postchain_reset(const PostChain &pc, float *state, int rows, cudaStream_t st);
void launch_postchain(const DevRows &g, const PostChain &pc, float *state, int64_t col0, int64_t col1, cudaStream_t st);
// the streaming instances' launch: g.out holds float32 rows, the chained samples go to dst (indexed like g.out) as dst_fmt
// (PVGPU_F32: dst == g.out, in place; PVGPU_S16: quantised like pcm_store); coef: null (pc's coefficients in every row) or
// per-stream coefficients [streams][pc.n][6] (the p[] of pc.fx; row r is stream r / g.channels)
void launch_postchain_stream(const DevRows &g, const PostChain &pc, float *state, int64_t col0, int64_t col1, void *dst, int dst_fmt, const float *coef,
                             cudaStream_t st);
// k records of 1 + n6 floats (stream index as int bits, then its n6 coefficients) into the rows of table ([streams][n6])
void launch_postchain_coef_scatter(const float *upd, int k, int n6, float *table, cudaStream_t st);

// ---- loudness meters on the output rows of streaming instances (pv_meter.cu) ----
constexpr int kMeterRing = 30;    // sub-blocks of the short-term window, the longest one kept
constexpr int kMeterState = 9;    // doubles per row: shelf x1 x2 y1 y2, high-pass x1 x2 y1 y2, energy of the open sub-block
struct KWeighting { double c[7]; };   // shelf b0, b1, b2, a1, a2; high-pass a1, a2 (b = 1, -2, 1); a0 = 1
void kweighting_design(int sample_rate, double *c /*[7]*/);
// Meters over columns [0, n) of rows = streams * channels rows of x (row r at x + r * pitch, float32 or int16 by fmt): the K-weighting
// state [kMeterState][rows] and the ring of sub-block energies [kMeterRing][rows] advance; out = [momentary S][short-term S][peak R]
// floats: the peaks are rewritten, the loudness values only when a sub-block completes.  *pos (samples in the open sub-block of L)
// and *ri (ring slot of the next completed sub-block) are the host's counters, advanced here.
void launch_meters(const void *x, int fmt, int64_t pitch, int n, int streams, int channels, const KWeighting &kw, int L, double *state,
                   double *ring, float *out, int *pos, int *ri, cudaStream_t st);

// row-wise copy with independent pitches (in elements) and any element alignment (live batch input placement); T = float or short
template <typename T>
void launch_place_rows(T *dst, int64_t dst_pitch, const T *src, int64_t src_pitch, int width, int rows, cudaStream_t st);
// the same with either side a ring of (mask + 1) elements per row starting at element `off` (mask = -1: a plain row)
template <typename T>
void launch_ring_rows(T *dst, int64_t dst_pitch, int64_t dst_off, int64_t dst_mask, const T *src, int64_t src_pitch, int64_t src_off, int64_t src_mask,
                      int width, int rows, cudaStream_t st);

void launch_test_atan2f(int64_t n, const float *y, const float *x, float *out, cudaStream_t st);
void launch_test_princarg(int64_t n, const double *a, double *out, cudaStream_t st);

// bytes of dynamic shared memory each kernel needs for this plan (for tests / occupancy notes)
size_t smem_analyse(const DevPlan &p);
size_t smem_phase_core(const DevPlan &p, int channels, int maxpk);
size_t smem_synthesise(const DevPlan &p);

// one-time opt-in for > 48 KB dynamic shared memory
cudaError_t configure_kernels();

}  // namespace pvgpu
