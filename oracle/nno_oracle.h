/*
 * nno_oracle.h -- CPU ORACLE for the nnnoiseless per-frame denoise path.
 *
 * TEST INFRASTRUCTURE ONLY.  This is a plain-C restatement of the reference
 * algorithm (jneem/nnnoiseless @ 7b47c9b, DenoiseState::process_frame) used as
 * the checker for the CUDA path and as the timed CPU baseline.  Nothing in the
 * product package (nnnoiseless_b200/) may include, link or call it; only
 * tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl
 * reference legs do.
 *
 * Pinning: the oracle reproduces the reference's only golden vector
 * (test_data/testing.raw -> test_data/reference_output.raw, metric of
 * src/lib.rs:184-194) -- see tests/test_oracle_golden.py.  Intermediates
 * (pitch index, VAD, features, gains) are NOT pinned by any reference test
 * (the reference has none); they are pinned transitively through that vector.
 * The Rust crate itself cannot be built here (no rustc/cargo), so the FFT
 * (easyfft 0.4.2 -> realfft 3.5.0 -> rustfft 6.4.1, not vendored) is restated
 * from its published semantics: unnormalised forward e^{-i}, unnormalised
 * inverse, bin 0 = DC, bin 480 = Nyquist.
 */
#ifndef NNO_ORACLE_H
#define NNO_ORACLE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NNO_FRAME_SIZE 480
#define NNO_NB_BANDS 22
#define NNO_NB_FEATURES 42

typedef struct nno_model nno_model;
typedef struct nno_state nno_state;

/* Per-frame intermediates of the most recent nno_process_frame call. */
typedef struct {
    int32_t pitch;     /* pitch period returned by PitchFinder::process, in [60, 768] */
    int32_t silence;   /* 1 if compute_frame_features returned true */
    float vad;         /* return value of process_frame */
    float pitch_gain;  /* PitchFinder last_gain */
    float features[NNO_NB_FEATURES];
    float gains[NNO_NB_BANDS]; /* g after the 0.6*lastg floor (== lastg); zeros on silent frames */
    float ex[NNO_NB_BANDS];
    float ep[NNO_NB_BANDS];
    float exp[NNO_NB_BANDS];
} nno_taps;

/* RnnModel::from_bytes (src/rnn.rs:75,116-232).  NULL on any format violation. */
nno_model *nno_model_from_bytes(const uint8_t *bytes, size_t len);
void nno_model_free(nno_model *m);
/* layer geometry, for tests: out[0..18) = {ni, nn, act} x 6 layers in file order */
void nno_model_describe(const nno_model *m, int32_t out[18]);

/* DenoiseState::with_model (src/denoise.rs:72-82): borrows the model. */
nno_state *nno_state_new(const nno_model *m);
void nno_state_free(nno_state *s);
/* DenoiseState::process_frame (src/denoise.rs:95-116).  out may alias in. */
float nno_process_frame(nno_state *s, float *out, const float *in);
void nno_get_taps(const nno_state *s, nno_taps *taps);

/* Exposed pieces for unit tests. */
void nno_rfft960(const float *in960, float *out_re481, float *out_im481);
void nno_irfft960(const float *re481, const float *im481, float *out960);
int32_t nno_pitch_only(nno_state *s, const float *buf1728);
/* FFT variant of every later transform (process-wide; test aid): 0 = f32 Stockham 4,4,5,3,2 (default, the pinned
 * oracle), 1 = f64 DFT sums rounded once, 2 = f32 Stockham 2,3,5,4,4. */
void nno_set_fft_mode(int mode);
float nno_tansig(float x);
float nno_sigmoid(float x);
/* the 201-entry table behind nno_tansig (src/util.rs:3-27) */
const float *nno_tansig_table(void);

/*
 * Batched driver used as the timed CPU baseline: n_streams independent states,
 * each advanced n_frames frames.  in/out: [n_streams][n_frames][480] floats
 * (out may be NULL to discard).  vad (may be NULL): [n_streams][n_frames].
 * pitch (may be NULL): [n_streams][n_frames].  Streams are distributed over
 * n_threads OpenMP threads (<=0: all).  Returns elapsed seconds of the
 * processing loop (state construction excluded) and the thread count used in
 * *threads_used.
 */
double nno_run_batch(const nno_model *m, const float *in, float *out, float *vad, int32_t *pitch,
                     int n_streams, int n_frames, int n_threads, int *threads_used);


/* ---- training-data rows: src/training.rs:113-161 (main loop) + :283-433 (NoiseSimulator) ---------------
 * One "lane" = one NoiseSimulator + its three DenoiseFeatures (clean / noise / combined).  The file readers and
 * the random draws of NoiseSimulator::randomize (src/training.rs:352-377, thread_rng: not reproducible) stay with
 * the caller, which hands their RESULT in as nno_sim_params; everything arithmetic per frame is restated here. */
#define NNO_TRAIN_ROW 87 /* 42 features + 22 gains + 22 noise levels + vad, src/training.rs:90,155-158 */
typedef struct {
    float signal_gain, noise_gain;         /* NoiseSimulator::{signal_gain, noise_gain}            */
    float sig_a[2], sig_b[2];              /* sig_filter   (Biquad a, b; Default = zeros)          */
    float noise_a[2], noise_b[2];          /* noise_filter                                         */
    int32_t band_lp;                       /* NoiseSimulator::band_lp (new(): NB_BANDS - 1)        */
} nno_sim_params;
typedef struct nno_trainer nno_trainer;
nno_trainer *nno_train_new(void);          /* NoiseSimulator::new + 3x DenoiseFeatures::new        */
void nno_train_free(nno_trainer *t);
void nno_train_set_params(nno_trainer *t, const nno_sim_params *p);
/* one iteration of the main loop: signal/noise are the raw frames SignalReader::frame yields (i16-valued f32) */
void nno_train_frame(nno_trainer *t, const float *signal480, const float *noise480, float *row87);
/* EBAND_5MS.position(|x| x << 2 > lowpass).unwrap_or(NB_BANDS - 1), src/training.rs:373-376 */
int32_t nno_train_band_lp(int32_t lowpass);


/* ---- file front-end: src/nnnoiseless.rs (the `nnnoiseless` binary) -------------------------------------
 * The resampler is dasp_interpolate 0.11.0's `Sinc<[f32; 16]>` over dasp_ring_buffer 0.11.0's `Fixed`
 * (Cargo.lock:292-300); both crates are NOT under /root/reference, so nno_resample restates their published
 * algorithm (depth-8 Hann-windowed sinc, taps accumulated in f32 in the order left(n), right(n), n = 0..depth;
 * ring indices wrap).  PARITY UNPINNED for the resampler: the reference holds no expected output for it
 * (tests/cli.rs only checks exit status and the "no RIFF tag found" message). */
/* Resample::next_sample (src/nnnoiseless.rs:104-131) until the source runs dry.  in: [n_in][channels] interleaved,
 * out: [cap][channels]; returns the number of output sample frames (they never exceed cap). */
long nno_resample(const float *in, long n_in, int channels, double ratio, float *out, long cap);
/* main's frame loop (src/nnnoiseless.rs:301-330): per channel one DenoiseState, 480-sample frames, the first
 * frame's output discarded, a trailing partial frame dropped, output clamped + rounded to i16 (:147-177).
 * in: [n_in][channels] at 48 kHz; out: [cap][channels]; returns output sample frames written. */
long nno_cli_frames(const nno_model *m, const float *in, long n_in, int channels, int16_t *out, long cap);

#ifdef __cplusplus
}
#endif
#endif
