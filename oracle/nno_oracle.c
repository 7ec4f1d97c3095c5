/*
 * nno_oracle.c -- CPU ORACLE (test infrastructure, see nno_oracle.h).
 *
 * Plain-C restatement of jneem/nnnoiseless @ 7b47c9b DenoiseState::process_frame.
 * Every function cites the reference file:line whose arithmetic (including the
 * ORDER of floating-point operations) it follows.  Build with
 *   gcc -O2 -ffp-contract=off -fno-fast-math   (see oracle/Makefile)
 * so no FMA contraction / reassociation changes the rounding.
 */
#include "nno_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#ifdef _OPENMP
#include <omp.h>
#endif

/* ---- constants: src/lib.rs:36-58 -------------------------------------------------------- */
#define FRAME_SIZE 480
#define WINDOW_SIZE 960
#define FREQ_SIZE 481
#define PITCH_MIN_PERIOD 60
#define PITCH_MAX_PERIOD 768
#define PITCH_FRAME_SIZE 960
#define PITCH_BUF_SIZE (PITCH_MAX_PERIOD + PITCH_FRAME_SIZE) /* 1728 */
#define NB_BANDS 22
#define CEPS_MEM 8
#define NB_DELTA_CEPS 6
#define NB_FEATURES 42
#define MAX_NEURONS 128

static const int EBAND_5MS[NB_BANDS] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 10, 12, 14, 16, 20, 24, 28, 34, 40, 48, 60, 78, 100};
/* src/pitch.rs:489 */
static const int SECOND_CHECK[16] = {0, 0, 3, 2, 3, 2, 5, 2, 3, 2, 3, 2, 5, 2, 3, 2};

/* ---- tables: src/lib.rs:99-136 (CommonState) + FFT twiddles ----------------------------- */
static float g_window[WINDOW_SIZE];
static float g_dct[NB_BANDS * NB_BANDS];
static float g_wnorm;
static float g_tw480_re[480], g_tw480_im[480]; /* exp(-2 pi i k / 480) */
static float g_tw960_re[481], g_tw960_im[481]; /* exp(-2 pi i k / 960), k = 0..480 */
static int g_tables_ready = 0;

static void build_tables(void) {
    const double pi = 3.14159265358979323846264338327950288;
    for (int i = 0; i < FRAME_SIZE; i++) {
        double s = sin(0.5 * pi * ((double)i + 0.5) / (double)FRAME_SIZE);
        float w = (float)sin(0.5 * pi * s * s);
        g_window[i] = w;
        g_window[WINDOW_SIZE - i - 1] = w;
    }
    float acc = 0.0f; /* f32 sequential sum, src/lib.rs:116 */
    for (int i = 0; i < WINDOW_SIZE; i++) acc += g_window[i] * g_window[i];
    g_wnorm = 1.0f / acc;
    for (int i = 0; i < NB_BANDS; i++) {
        for (int j = 0; j < NB_BANDS; j++) {
            float v = (float)cos(((double)i + 0.5) * (double)j * pi / (double)NB_BANDS);
            if (j == 0) v *= sqrtf(0.5f);
            g_dct[i * NB_BANDS + j] = v;
        }
    }
    for (int k = 0; k < 480; k++) {
        g_tw480_re[k] = (float)cos(-2.0 * pi * (double)k / 480.0);
        g_tw480_im[k] = (float)sin(-2.0 * pi * (double)k / 480.0);
    }
    for (int k = 0; k <= 480; k++) {
        g_tw960_re[k] = (float)cos(-2.0 * pi * (double)k / 960.0);
        g_tw960_im[k] = (float)sin(-2.0 * pi * (double)k / 960.0);
    }
    g_tables_ready = 1;
}

static void ensure_tables(void) {
    if (!g_tables_ready) {
#ifdef _OPENMP
#pragma omp critical(nno_tables)
#endif
        {
            if (!g_tables_ready) build_tables();
        }
    }
}

/* ---- FFT: restates easyfft::real_fft_using / real_ifft_using (call sites
 * src/features.rs:264,290).  960-point real transform = 480-point complex
 * Stockham (radix 4,4,5,3,2) + even/odd split, f32 throughout. ----------------------------- */
typedef struct {
    float re, im;
} cpx;

static inline cpx cmul(cpx a, cpx b) {
    cpx r = {a.re * b.re - a.im * b.im, a.re * b.im + a.im * b.re};
    return r;
}

/* One Stockham DIF pass of radix r: n = current sub-length, s = stride (product of previous radices). */
static void stockham_pass(int r, int n, int s, const cpx *x, cpx *y) {
    const int m = n / r;
    /* r-th roots of unity taken from the 480 table (480 divisible by 2,3,4,5) */
    for (int p = 0; p < m; p++) {
        for (int q = 0; q < s; q++) {
            cpx a[5], b[5] = {{0.0f, 0.0f}};
            for (int k = 0; k < r; k++) a[k] = x[q + s * (p + k * m)];
            if (r == 2) {
                b[0].re = a[0].re + a[1].re; b[0].im = a[0].im + a[1].im;
                b[1].re = a[0].re - a[1].re; b[1].im = a[0].im - a[1].im;
            } else if (r == 4) {
                cpx t0 = {a[0].re + a[2].re, a[0].im + a[2].im};
                cpx t1 = {a[0].re - a[2].re, a[0].im - a[2].im};
                cpx t2 = {a[1].re + a[3].re, a[1].im + a[3].im};
                cpx t3 = {a[1].re - a[3].re, a[1].im - a[3].im};
                /* -i * t3 = (t3.im, -t3.re) */
                b[0].re = t0.re + t2.re; b[0].im = t0.im + t2.im;
                b[1].re = t1.re + t3.im; b[1].im = t1.im - t3.re;
                b[2].re = t0.re - t2.re; b[2].im = t0.im - t2.im;
                b[3].re = t1.re - t3.im; b[3].im = t1.im + t3.re;
            } else {
                /* generic small DFT for r = 3, 5 */
                for (int j = 0; j < r; j++) {
                    cpx acc = a[0];
                    for (int k = 1; k < r; k++) {
                        int idx = ((j * k) % r) * (480 / r);
                        cpx w = {g_tw480_re[idx], g_tw480_im[idx]};
                        cpx t = cmul(a[k], w);
                        acc.re += t.re;
                        acc.im += t.im;
                    }
                    b[j] = acc;
                }
            }
            y[q + s * (r * p)] = b[0];
            for (int j = 1; j < r; j++) {
                int idx = (j * p * s) % 480;
                cpx w = {g_tw480_re[idx], g_tw480_im[idx]};
                y[q + s * (r * p + j)] = cmul(b[j], w);
            }
        }
    }
}

/* FFT variant (test aid, nno_set_fft_mode): 0 = the f32 Stockham above with radices 4,4,5,3,2 (default, the pinned
 * oracle); 1 = the transforms evaluated as plain DFT sums in f64 and rounded to f32 once; 2 = the same f32 Stockham
 * with the radix order 2,3,5,4,4 (a second, equally valid f32 FFT with a different rounding pattern).  Used by
 * tests/test_oracle_golden.py to show how much two correct FFTs may differ after signal -> digital silence -> signal. */
static int g_fft_mode = 0;
void nno_set_fft_mode(int mode) { g_fft_mode = mode; }

static double g_w960_re[960], g_w960_im[960];
static int g_w960_ready = 0;
static void ensure_w960(void) {
    if (g_w960_ready) return;
#ifdef _OPENMP
#pragma omp critical(nno_w960)
#endif
    {
        if (!g_w960_ready) {
            const double pi = 3.14159265358979323846264338327950288;
            for (int k = 0; k < 960; k++) {
                g_w960_re[k] = cos(-2.0 * pi * (double)k / 960.0);
                g_w960_im[k] = sin(-2.0 * pi * (double)k / 960.0);
            }
            g_w960_ready = 1;
        }
    }
}

/* forward (e^{-i}) unnormalised 480-point complex FFT, result in buf a */
static void cfft480(cpx *a, cpx *b) {
    static const int radices_a[5] = {4, 4, 5, 3, 2}, radices_b[5] = {2, 3, 5, 4, 4};
    const int *radices = g_fft_mode == 2 ? radices_b : radices_a;
    int n = 480, s = 1;
    cpx *x = a, *y = b;
    for (int i = 0; i < 5; i++) {
        stockham_pass(radices[i], n, s, x, y);
        n /= radices[i];
        s *= radices[i];
        cpx *t = x; x = y; y = t;
    }
    /* 5 passes: result is in b; copy back */
    if (x != a) memcpy(a, x, 480 * sizeof(cpx));
}

void nno_rfft960(const float *in, float *ore, float *oim) {
    ensure_tables();
    if (g_fft_mode == 1) {
        ensure_w960();
        for (int k = 0; k <= 480; k++) {
            double sr = 0.0, si = 0.0;
            for (int n = 0; n < 960; n++) {
                const int idx = (k * n) % 960;
                sr += (double)in[n] * g_w960_re[idx];
                si += (double)in[n] * g_w960_im[idx];
            }
            ore[k] = (float)sr;
            oim[k] = (float)si;
        }
        oim[0] = 0.0f;
        oim[480] = 0.0f;
        return;
    }
    cpx z[480], w[480];
    for (int n = 0; n < 480; n++) {
        z[n].re = in[2 * n];
        z[n].im = in[2 * n + 1];
    }
    cfft480(z, w);
    for (int k = 0; k <= 480; k++) {
        cpx zk = z[k % 480];
        cpx zc = z[(480 - k) % 480];
        /* E = (Z[k] + conj Z[N-k]) / 2 ; O = (Z[k] - conj Z[N-k]) / (2i) */
        float er = 0.5f * (zk.re + zc.re), ei = 0.5f * (zk.im - zc.im);
        float dr = 0.5f * (zk.re - zc.re), di = 0.5f * (zk.im + zc.im);
        /* O = d / i = (di, -dr) */
        cpx o = {di, -dr};
        cpx tw = {g_tw960_re[k], g_tw960_im[k]};
        cpx t = cmul(o, tw);
        ore[k] = er + t.re;
        oim[k] = ei + t.im;
    }
    oim[0] = 0.0f;
    oim[480] = 0.0f;
}

void nno_irfft960(const float *re, const float *im, float *out) {
    ensure_tables();
    if (g_fft_mode == 1) {
        /* unnormalised inverse of a real signal's half spectrum; imaginary parts of DC / Nyquist ignored (realfft) */
        ensure_w960();
        for (int n = 0; n < 960; n++) {
            double acc = (double)re[0] + ((n & 1) ? -(double)re[480] : (double)re[480]);
            for (int k = 1; k < 480; k++) {
                const int idx = (k * n) % 960; /* e^{+i} = conj of the table entry */
                acc += 2.0 * ((double)re[k] * g_w960_re[idx] + (double)im[k] * g_w960_im[idx]);
            }
            out[n] = (float)acc;
        }
        return;
    }
    cpx z[480], w[480];
    for (int k = 0; k < 480; k++) {
        /* imag parts of DC / Nyquist are ignored, as realfft does */
        float xr = re[k], xi = (k == 0) ? 0.0f : im[k];
        float yr = re[480 - k], yi = (k == 0) ? 0.0f : -im[480 - k]; /* conj X[480-k] */
        float sr = xr + yr, si = xi + yi; /* X[k] + conj X[N-k]  = 2E */
        float dr = xr - yr, di = xi - yi; /* X[k] - conj X[N-k]  = 2 w^k O */
        /* i * conj(w^k) * d */
        cpx cw = {g_tw960_re[k], -g_tw960_im[k]};
        cpx d = {dr, di};
        cpx t = cmul(d, cw);
        /* Z = 2E + i*(2O) ; we feed conj(Z) to the forward FFT and conjugate the result */
        float zr = sr - t.im, zi = si + t.re;
        z[k].re = zr;
        z[k].im = -zi;
    }
    cfft480(z, w);
    for (int n = 0; n < 480; n++) {
        out[2 * n] = z[n].re;
        out[2 * n + 1] = -z[n].im;
    }
}

/* ---- activations: src/util.rs:3-53 ------------------------------------------------------- */
static const float TANSIG_TABLE[201] = {
    0.000000f, 0.039979f, 0.079830f, 0.119427f, 0.158649f, 0.197375f, 0.235496f, 0.272905f, 0.309507f,
    0.345214f, 0.379949f, 0.413644f, 0.446244f, 0.477700f, 0.507977f, 0.537050f, 0.564900f, 0.591519f,
    0.616909f, 0.641077f, 0.664037f, 0.685809f, 0.706419f, 0.725897f, 0.744277f, 0.761594f, 0.777888f,
    0.793199f, 0.807569f, 0.821040f, 0.833655f, 0.845456f, 0.856485f, 0.866784f, 0.876393f, 0.885352f,
    0.893698f, 0.901468f, 0.908698f, 0.915420f, 0.921669f, 0.927473f, 0.932862f, 0.937863f, 0.942503f,
    0.946806f, 0.950795f, 0.954492f, 0.957917f, 0.961090f, 0.964028f, 0.966747f, 0.969265f, 0.971594f,
    0.973749f, 0.975743f, 0.977587f, 0.979293f, 0.980869f, 0.982327f, 0.983675f, 0.984921f, 0.986072f,
    0.987136f, 0.988119f, 0.989027f, 0.989867f, 0.990642f, 0.991359f, 0.992020f, 0.992631f, 0.993196f,
    0.993718f, 0.994199f, 0.994644f, 0.995055f, 0.995434f, 0.995784f, 0.996108f, 0.996407f, 0.996682f,
    0.996937f, 0.997172f, 0.997389f, 0.997590f, 0.997775f, 0.997946f, 0.998104f, 0.998249f, 0.998384f,
    0.998508f, 0.998623f, 0.998728f, 0.998826f, 0.998916f, 0.999000f, 0.999076f, 0.999147f, 0.999213f,
    0.999273f, 0.999329f, 0.999381f, 0.999428f, 0.999472f, 0.999513f, 0.999550f, 0.999585f, 0.999617f,
    0.999646f, 0.999673f, 0.999699f, 0.999722f, 0.999743f, 0.999763f, 0.999781f, 0.999798f, 0.999813f,
    0.999828f, 0.999841f, 0.999853f, 0.999865f, 0.999875f, 0.999885f, 0.999893f, 0.999902f, 0.999909f,
    0.999916f, 0.999923f, 0.999929f, 0.999934f, 0.999939f, 0.999944f, 0.999948f, 0.999952f, 0.999956f,
    0.999959f, 0.999962f, 0.999965f, 0.999968f, 0.999970f, 0.999973f, 0.999975f, 0.999977f, 0.999978f,
    0.999980f, 0.999982f, 0.999983f, 0.999984f, 0.999986f, 0.999987f, 0.999988f, 0.999989f, 0.999990f,
    0.999990f, 0.999991f, 0.999992f, 0.999992f, 0.999993f, 0.999994f, 0.999994f, 0.999994f, 0.999995f,
    0.999995f, 0.999996f, 0.999996f, 0.999996f, 0.999997f, 0.999997f, 0.999997f, 0.999997f, 0.999997f,
    0.999998f, 0.999998f, 0.999998f, 0.999998f, 0.999998f, 0.999998f, 0.999999f, 0.999999f, 0.999999f,
    0.999999f, 0.999999f, 0.999999f, 0.999999f, 0.999999f, 0.999999f, 0.999999f, 0.999999f, 0.999999f,
    0.999999f, 1.000000f, 1.000000f, 1.000000f, 1.000000f, 1.000000f, 1.000000f, 1.000000f, 1.000000f,
    1.000000f, 1.000000f, 1.000000f,
};

/* src/util.rs:29-45 */
float nno_tansig(float x) {
    if (!(x < 8.0f)) return 1.0f;
    if (!(x > -8.0f)) return -1.0f;
    float sign = 1.0f;
    if (x < 0.0f) {
        x = -x;
        sign = -1.0f;
    }
    float fi = floorf(0.5f + 25.0f * x);
    x -= 0.04f * fi;
    float y = TANSIG_TABLE[(int)fi];
    float dy = 1.0f - y * y;
    y = y + x * dy * (1.0f - y * x);
    return sign * y;
}
const float *nno_tansig_table(void) { return TANSIG_TABLE; }
/* src/util.rs:47-49 */
float nno_sigmoid(float x) { return 0.5f + 0.5f * nno_tansig(0.5f * x); }
/* src/util.rs:51-53 */
static inline float relu(float x) { return fmaxf(x, 0.0f); }

static inline float activate(int act, float x) {
    switch (act) {
    case 0: return nno_tansig(x);
    case 1: return nno_sigmoid(x);
    default: return relu(x);
    }
}

/* ---- model: src/rnn.rs:24-62,116-232 ----------------------------------------------------- */
typedef struct {
    int ni, nn, act;
    const int8_t *w;    /* [ni][nn] */
    const int8_t *bias; /* [nn] */
} dense_layer;

typedef struct {
    int ni, nn, act;
    const int8_t *w;    /* [ni][3nn] */
    const int8_t *r;    /* [nn][3nn] */
    const int8_t *bias; /* [3nn] */
} gru_layer;

struct nno_model {
    int8_t *blob;
    size_t len;
    dense_layer input_dense;
    gru_layer vad_gru, noise_gru, denoise_gru;
    dense_layer denoise_output, vad_output;
};

static int read_dense(const int8_t **p, size_t *left, dense_layer *l) {
    if (*left < 3) return 0;
    const int8_t *b = *p;
    if (b[0] < 0 || b[1] < 0) return 0;
    l->ni = b[0]; /* header order is [nb_inputs, nb_neurons, activation]: src/rnn.rs:150-152 */
    l->nn = b[1];
    if (b[2] < 0 || b[2] > 2) return 0;
    l->act = b[2];
    size_t need = (size_t)l->ni * l->nn + l->nn;
    if (*left - 3 < need) return 0;
    l->w = b + 3;
    l->bias = l->w + (size_t)l->ni * l->nn;
    *p = b + 3 + need;
    *left -= 3 + need;
    return 1;
}

static int read_gru(const int8_t **p, size_t *left, gru_layer *l) {
    if (*left < 3) return 0;
    const int8_t *b = *p;
    if (b[0] < 0 || b[1] < 0) return 0;
    l->ni = b[0];
    l->nn = b[1];
    if (b[2] < 0 || b[2] > 2) return 0;
    l->act = b[2];
    size_t nw = (size_t)3 * l->nn * l->ni, nr = (size_t)3 * l->nn * l->nn, nb = (size_t)3 * l->nn;
    if (*left - 3 < nw + nr + nb) return 0;
    l->w = b + 3;
    l->r = l->w + nw;
    l->bias = l->r + nr;
    *p = b + 3 + nw + nr + nb;
    *left -= 3 + nw + nr + nb;
    return 1;
}

nno_model *nno_model_from_bytes(const uint8_t *bytes, size_t len) {
    nno_model *m = (nno_model *)calloc(1, sizeof(*m));
    if (!m) return NULL;
    m->blob = (int8_t *)malloc(len ? len : 1);
    m->len = len;
    memcpy(m->blob, bytes, len);
    const int8_t *p = m->blob;
    size_t left = len;
    int ok = read_dense(&p, &left, &m->input_dense) && read_gru(&p, &left, &m->vad_gru) &&
             read_gru(&p, &left, &m->noise_gru) && read_gru(&p, &left, &m->denoise_gru) &&
             read_dense(&p, &left, &m->denoise_output) && read_dense(&p, &left, &m->vad_output);
    ok = ok && left == 0;
    /* src/rnn.rs:204-222 */
    ok = ok && m->input_dense.ni == 42 && m->denoise_output.nn == 22 && m->vad_output.nn == 1;
    ok = ok && m->input_dense.nn == m->vad_gru.ni && m->vad_gru.nn == m->vad_output.ni;
    ok = ok && 42 + m->input_dense.nn + m->vad_gru.nn == m->noise_gru.ni;
    ok = ok && 42 + m->vad_gru.nn + m->noise_gru.nn == m->denoise_gru.ni;
    ok = ok && m->denoise_gru.nn == m->denoise_output.ni;
    if (!ok) {
        nno_model_free(m);
        return NULL;
    }
    return m;
}

void nno_model_free(nno_model *m) {
    if (!m) return;
    free(m->blob);
    free(m);
}

void nno_model_describe(const nno_model *m, int32_t out[18]) {
    const int v[18] = {m->input_dense.ni,    m->input_dense.nn,    m->input_dense.act,   m->vad_gru.ni,    m->vad_gru.nn,
                       m->vad_gru.act,       m->noise_gru.ni,      m->noise_gru.nn,      m->noise_gru.act, m->denoise_gru.ni,
                       m->denoise_gru.nn,    m->denoise_gru.act,   m->denoise_output.ni, m->denoise_output.nn,
                       m->denoise_output.act, m->vad_output.ni,    m->vad_output.nn,     m->vad_output.act};
    for (int i = 0; i < 18; i++) out[i] = v[i];
}

/* ---- state: src/features.rs:18-46, src/pitch.rs:4-17, src/rnn.rs:65-70, src/denoise.rs:37-42 */
struct nno_state {
    const nno_model *model;
    float lastg[NB_BANDS];
    float vad_gru_state[MAX_NEURONS], noise_gru_state[MAX_NEURONS], denoise_gru_state[MAX_NEURONS];
    float input_mem[PITCH_BUF_SIZE];
    float cepstral_mem[CEPS_MEM][NB_BANDS];
    int mem_id;
    float mem_hp_x[2];
    float synthesis_mem[FRAME_SIZE];
    float window_buf[WINDOW_SIZE];
    float x_re[FREQ_SIZE], x_im[FREQ_SIZE];
    float p_re[FREQ_SIZE], p_im[FREQ_SIZE];
    float ex[NB_BANDS], ep[NB_BANDS], exp[NB_BANDS];
    float features[NB_FEATURES];
    /* PitchFinder */
    int last_period;
    float last_gain;
    float pitch_buf[PITCH_BUF_SIZE / 2];
    float scratch[PITCH_MAX_PERIOD + 1];
    float scratch2[PITCH_FRAME_SIZE / 4];
    float scratch3[(PITCH_MAX_PERIOD - 3 * PITCH_MIN_PERIOD) / 2];
    nno_taps taps;
};

nno_state *nno_state_new(const nno_model *m) {
    ensure_tables();
    nno_state *s = (nno_state *)calloc(1, sizeof(*s));
    if (s) s->model = m;
    return s;
}
void nno_state_free(nno_state *s) { free(s); }
void nno_get_taps(const nno_state *s, nno_taps *t) { *t = s->taps; }

/* ---- band ops: src/lib.rs:65-97 ---------------------------------------------------------- */
static void compute_band_corr(float *out, const float *xr, const float *xi, const float *pr, const float *pi_) {
    for (int i = 0; i < NB_BANDS; i++) out[i] = 0.0f;
    for (int i = 0; i < NB_BANDS - 1; i++) {
        int band_size = (EBAND_5MS[i + 1] - EBAND_5MS[i]) << 2;
        for (int j = 0; j < band_size; j++) {
            float frac = (float)j / (float)band_size;
            int idx = (EBAND_5MS[i] << 2) + j;
            float corr = xr[idx] * pr[idx] + xi[idx] * pi_[idx];
            out[i] += (1.0f - frac) * corr;
            out[i + 1] += frac * corr;
        }
    }
    out[0] *= 2.0f;
    out[NB_BANDS - 1] *= 2.0f;
}

static void interp_band_gain(float *out /*[481]*/, const float *band_e) {
    for (int i = 0; i < FREQ_SIZE; i++) out[i] = 0.0f;
    for (int i = 0; i < NB_BANDS - 1; i++) {
        int band_size = (EBAND_5MS[i + 1] - EBAND_5MS[i]) << 2;
        for (int j = 0; j < band_size; j++) {
            float frac = (float)j / (float)band_size;
            int idx = (EBAND_5MS[i] << 2) + j;
            out[idx] = (1.0f - frac) * band_e[i] + frac * band_e[i + 1];
        }
    }
}

/* src/lib.rs:139-148 */
static void dct22(float *out, const float *x) {
    for (int i = 0; i < NB_BANDS; i++) {
        float sum = 0.0f;
        for (int j = 0; j < NB_BANDS; j++) sum += x[j] * g_dct[j * NB_BANDS + i];
        out[i] = (float)((double)sum * sqrt(2.0 / (double)NB_BANDS));
    }
}

/* ---- biquad: src/util.rs:68-71,95-107 ---------------------------------------------------- */
static void biquad_hp(float *out, float mem[2], const float *in, int n) {
    const double a0 = (double)-1.99599f, a1 = (double)0.99600f, b0 = (double)-2.0f, b1 = (double)1.0f;
    for (int i = 0; i < n; i++) {
        double x64 = (double)in[i];
        double y64 = x64 + (double)mem[0];
        mem[0] = (float)((double)mem[1] + (b0 * x64 - a0 * y64));
        mem[1] = (float)(b1 * x64 - a1 * y64);
        out[i] = (float)y64;
    }
}

/* ---- pitch: src/pitch.rs ----------------------------------------------------------------- */
/* src/pitch.rs:225-244 */
static float inner_prod(const float *xs, const float *ys, int n) {
    float s0 = 0.0f, s1 = 0.0f, s2 = 0.0f, s3 = 0.0f;
    int n4 = n - n % 4;
    for (int i = 0; i < n4; i += 4) {
        s0 += xs[i] * ys[i];
        s1 += xs[i + 1] * ys[i + 1];
        s2 += xs[i + 2] * ys[i + 2];
        s3 += xs[i + 3] * ys[i + 3];
    }
    float sum = s0 + s1 + s2 + s3;
    for (int i = n4; i < n; i++) sum += xs[i] * ys[i];
    return sum;
}

/* src/pitch.rs:296-363.  Every xcorr[i] is the in-order sum over j of xs[j]*ys[i+j]
 * (the 4x4 unrolling of the reference keeps each accumulator sequential in j). */
static void pitch_xcorr(const float *xs, int xlen, const float *ys, float *xcorr, int nlag) {
    for (int i = 0; i < nlag; i++) {
        float c = 0.0f;
        for (int j = 0; j < xlen; j++) c += xs[j] * ys[i + j];
        xcorr[i] = c;
    }
}

/* src/pitch.rs:372-405 */
static void find_best_pitch(const float *xcorr, int nlag, const float *ys, int len, int *best, int *second) {
    float best_num = -1.0f, second_best_num = -1.0f;
    float best_den = 0.0f, second_best_den = 0.0f;
    int best_pitch = 0, second_best_pitch = 1;
    float y_sq_norm = 1.0f;
    for (int j = 0; j < len; j++) y_sq_norm += ys[j] * ys[j];
    for (int i = 0; i < nlag; i++) {
        float corr = xcorr[i];
        if (corr > 0.0f) {
            float num = corr * corr;
            if (num * second_best_den > second_best_num * y_sq_norm) {
                if (num * best_den > best_num * y_sq_norm) {
                    second_best_num = best_num;
                    second_best_den = best_den;
                    second_best_pitch = best_pitch;
                    best_num = num;
                    best_den = y_sq_norm;
                    best_pitch = i;
                } else {
                    second_best_num = num;
                    second_best_den = y_sq_norm;
                    second_best_pitch = i;
                }
            }
        }
        y_sq_norm += ys[i + len] * ys[i + len] - ys[i] * ys[i];
        y_sq_norm = fmaxf(y_sq_norm, 1.0f);
    }
    *best = best_pitch;
    *second = second_best_pitch;
}

/* src/pitch.rs:257-292 */
static void lpc4(float *lpc, const float *ac) {
    const int p = 4;
    float error = ac[0];
    for (int i = 0; i < p; i++) lpc[i] = 0.0f;
    if (ac[0] == 0.0f) return;
    for (int i = 0; i < p; i++) {
        float rr = 0.0f;
        for (int j = 0; j < i; j++) rr += lpc[j] * ac[i - j];
        rr += ac[i + 1];
        float r = -rr / error;
        lpc[i] = r;
        for (int j = 0; j < (i + 1) / 2; j++) {
            float tmp1 = lpc[j];
            float tmp2 = lpc[i - 1 - j];
            lpc[j] = tmp1 + r * tmp2;
            lpc[i - 1 - j] = tmp2 + r * tmp1;
        }
        error = error - r * r * error;
        if (error < 0.001f * ac[0]) return;
    }
}

/* src/pitch.rs:448-483 incl. celt_autocorr (433-446) and fir5_in_place (407-429) */
static void pitch_downsample(const float *x /*1728*/, float *x_lp /*864*/) {
    const int half = PITCH_BUF_SIZE / 2;
    float ac[5], lpc[4], lpc2[5];
    for (int i = 1; i < half; i++) x_lp[i] = ((x[2 * i - 1] + x[2 * i + 1]) / 2.0f + x[2 * i]) / 2.0f;
    x_lp[0] = (x[1] / 2.0f + x[0]) / 2.0f;

    /* celt_autocorr: n = 864, lag = 4, fast_n = 860 */
    const int n = half, lag = 4, fast_n = n - lag;
    pitch_xcorr(x_lp, fast_n, x_lp, ac, lag + 1);
    for (int k = 0; k <= lag; k++) {
        float d = 0.0f;
        for (int i = k + fast_n; i < n; i++) d += x_lp[i] * x_lp[i - k];
        ac[k] += d;
    }
    ac[0] *= 1.0001f;
    for (int i = 1; i < 5; i++) ac[i] -= ac[i] * (0.008f * (float)i) * (0.008f * (float)i);

    lpc4(lpc, ac);
    float tmp = 1.0f;
    for (int i = 0; i < 4; i++) {
        tmp *= 0.9f;
        lpc[i] *= tmp;
    }
    lpc2[0] = lpc[0] + 0.8f;
    lpc2[1] = lpc[1] + 0.8f * lpc[0];
    lpc2[2] = lpc[2] + 0.8f * lpc[1];
    lpc2[3] = lpc[3] + 0.8f * lpc[2];
    lpc2[4] = 0.8f * lpc[3];

    float m0 = 0, m1 = 0, m2 = 0, m3 = 0, m4 = 0;
    for (int i = 0; i < n; i++) {
        float xi = x_lp[i];
        float out = xi + lpc2[0] * m0 + lpc2[1] * m1 + lpc2[2] * m2 + lpc2[3] * m3 + lpc2[4] * m4;
        m4 = m3; m3 = m2; m2 = m1; m1 = m0; m0 = xi;
        x_lp[i] = out;
    }
}

/* src/pitch.rs:63-115 */
static int pitch_search(nno_state *s) {
    const float *x_lp = s->pitch_buf + PITCH_MAX_PERIOD / 2;
    const float *y = s->pitch_buf;
    const int len = PITCH_FRAME_SIZE;                             /* 960 */
    const int max_pitch = PITCH_MAX_PERIOD - 3 * PITCH_MIN_PERIOD; /* 588 */
    float *x_lp4 = s->scratch2;                                    /* 240 */
    float *y_lp4 = s->scratch;                                     /* 387 */
    float *xcorr = s->scratch3;                                    /* 294 */
    const int n4 = len / 4, ny4 = len / 4 + max_pitch / 4;
    for (int j = 0; j < n4; j++) x_lp4[j] = x_lp[2 * j];
    for (int j = 0; j < ny4; j++) y_lp4[j] = y[2 * j];

    pitch_xcorr(x_lp4, n4, y_lp4, xcorr, max_pitch / 4);
    int best, second;
    find_best_pitch(xcorr, max_pitch / 4, y_lp4, n4, &best, &second);

    for (int i = 0; i < max_pitch / 2; i++) {
        xcorr[i] = 0.0f;
        if (abs(i - 2 * best) > 2 && abs(i - 2 * second) > 2) continue;
        xcorr[i] = fmaxf(inner_prod(x_lp, y + i, len / 2), -1.0f);
    }
    int dummy;
    find_best_pitch(xcorr, max_pitch / 2, y, len / 2, &best, &dummy);

    int offset = 0;
    if (best > 0 && best < max_pitch / 2 - 1) {
        float a = xcorr[best - 1], b = xcorr[best], c = xcorr[best + 1];
        if (c - a > 0.7f * (b - a)) offset = 1;
        else if (a - c > 0.7f * (b - c)) offset = -1;
    }
    return 2 * best - offset;
}

/* src/pitch.rs:485-487 */
static inline float pitch_gain(float xy, float xx, float yy) { return xy / sqrtf(1.0f + xx * yy); }

/* src/pitch.rs:118-221 */
static int remove_doubling(nno_state *s, int pitch_idx, float *gain_out) {
    const float *x = s->pitch_buf;
    const int min_period = PITCH_MIN_PERIOD / 2, max_period = PITCH_MAX_PERIOD / 2, n = PITCH_FRAME_SIZE / 2;
    int t0 = pitch_idx / 2;
    if (t0 > max_period - 1) t0 = max_period - 1;
    const int prev_period = s->last_period / 2;
    float *yy_lookup = s->scratch;
    int t = t0;

    float xx = inner_prod(x + max_period, x + max_period, n);
    float xy = inner_prod(x + max_period, x + max_period - t0, n);
    yy_lookup[0] = xx;
    float yy = xx;
    for (int i = 1; i <= max_period; i++) {
        yy += x[max_period - i] * x[max_period - i] - x[max_period + n - i] * x[max_period + n - i];
        yy_lookup[i] = fmaxf(yy, 0.0f);
    }
    yy = yy_lookup[t0];
    float best_xy = xy, best_yy = yy;
    const float g0 = pitch_gain(xy, xx, yy);
    float g = g0;

    for (int k = 2; k <= 15; k++) {
        int t1 = (2 * t0 + k) / (2 * k);
        if (t1 < min_period) break;
        int t1b;
        if (k == 2) t1b = (t1 + t0 > max_period) ? t0 : t0 + t1;
        else t1b = (2 * SECOND_CHECK[k] * t0 + k) / (2 * k);
        xy = inner_prod(x + max_period, x + max_period - t1, n);
        float xy2 = inner_prod(x + max_period, x + max_period - t1b, n);
        xy = (xy + xy2) / 2.0f;
        yy = (yy_lookup[t1] + yy_lookup[t1b]) / 2.0f;
        float g1 = pitch_gain(xy, xx, yy);
        float cont;
        int d = abs(t1 - prev_period);
        if (d <= 1) cont = s->last_gain;
        else if (d <= 2 && 5 * k * k < t0) cont = s->last_gain / 2.0f;
        else cont = 0.0f;
        float thresh;
        if (t1 < 3 * min_period) thresh = fmaxf(0.85f * g0 - cont, 0.4f);
        else if (t1 < 2 * min_period) thresh = fmaxf(0.9f * g0 - cont, 0.5f); /* unreachable, kept as in the reference */
        else thresh = fmaxf(0.7f * g0 - cont, 0.3f);
        if (g1 > thresh) {
            best_xy = xy;
            best_yy = yy;
            t = t1;
            g = g1;
        }
    }
    best_xy = fmaxf(best_xy, 0.0f);
    float pg = (best_yy <= best_xy) ? 1.0f : best_xy / (best_yy + 1.0f);

    float xc[3];
    for (int k = 0; k < 3; k++) xc[k] = inner_prod(x + max_period, x + max_period - (t + k - 1), n);
    int offset = 0;
    if (xc[2] - xc[0] > 0.7f * (xc[1] - xc[0])) offset = 1;
    else if (xc[0] - xc[2] > 0.7f * (xc[1] - xc[2])) offset = -1;

    pg = fminf(pg, g);
    int tf = 2 * t + offset;
    if (tf < PITCH_MIN_PERIOD) tf = PITCH_MIN_PERIOD;
    *gain_out = pg;
    return tf;
}

/* src/pitch.rs:45-54 */
static int pitch_process(nno_state *s, const float *input /*1728*/) {
    pitch_downsample(input, s->pitch_buf);
    int idx = pitch_search(s);
    idx = PITCH_MAX_PERIOD - idx;
    float gain;
    int period = remove_doubling(s, idx, &gain);
    s->last_period = period;
    s->last_gain = gain;
    return period;
}

int32_t nno_pitch_only(nno_state *s, const float *buf1728) { return pitch_process(s, buf1728); }

/* ---- features: src/features.rs ----------------------------------------------------------- */
/* src/features.rs:281-298 */
static void transform_input(nno_state *s, int lag, float *re, float *im, float *e) {
    const float *in = s->input_mem + (PITCH_BUF_SIZE - WINDOW_SIZE - lag);
    for (int i = 0; i < WINDOW_SIZE; i++) s->window_buf[i] = in[i] * g_window[i];
    nno_rfft960(s->window_buf, re, im);
    for (int i = 0; i < FREQ_SIZE; i++) {
        re[i] *= g_wnorm;
        im[i] *= g_wnorm;
    }
    compute_band_corr(e, re, im, re, im);
}

/* src/features.rs:115-219 */
static int compute_frame_features(nno_state *s) {
    float ly[NB_BANDS], tmp[NB_BANDS];
    transform_input(s, 0, s->x_re, s->x_im, s->ex);
    int pitch_idx = pitch_process(s, s->input_mem);
    s->taps.pitch = pitch_idx;
    s->taps.pitch_gain = s->last_gain;
    transform_input(s, pitch_idx, s->p_re, s->p_im, s->ep);
    compute_band_corr(s->exp, s->x_re, s->x_im, s->p_re, s->p_im);
    for (int i = 0; i < NB_BANDS; i++) s->exp[i] /= sqrtf(0.001f + s->ex[i] * s->ep[i]);
    dct22(tmp, s->exp);
    for (int i = 0; i < NB_DELTA_CEPS; i++) s->features[NB_BANDS + 2 * NB_DELTA_CEPS + i] = tmp[i];
    s->features[NB_BANDS + 2 * NB_DELTA_CEPS] -= 1.3f;
    s->features[NB_BANDS + 2 * NB_DELTA_CEPS + 1] -= 0.9f;
    s->features[NB_BANDS + 3 * NB_DELTA_CEPS] = 0.01f * ((float)pitch_idx - 300.0f);
    float log_max = -2.0f, follow = -2.0f, e = 0.0f;
    for (int i = 0; i < NB_BANDS; i++) {
        ly[i] = fmaxf(fmaxf(log10f(1e-2f + s->ex[i]), log_max - 7.0f), follow - 1.5f);
        log_max = fmaxf(log_max, ly[i]);
        follow = fmaxf(follow - 1.5f, ly[i]);
        e += s->ex[i];
    }
    if (e < 0.04f) {
        for (int i = 0; i < NB_FEATURES; i++) s->features[i] = 0.0f;
        return 1;
    }
    dct22(s->features, ly);
    s->features[0] -= 12.0f;
    s->features[1] -= 4.0f;
    int c0 = s->mem_id;
    int c1 = (s->mem_id < 1) ? CEPS_MEM + s->mem_id - 1 : s->mem_id - 1;
    int c2 = (s->mem_id < 2) ? CEPS_MEM + s->mem_id - 2 : s->mem_id - 2;
    for (int i = 0; i < NB_BANDS; i++) s->cepstral_mem[c0][i] = s->features[i];
    s->mem_id += 1;
    for (int i = 0; i < NB_DELTA_CEPS; i++) {
        float a = s->cepstral_mem[c0][i], b = s->cepstral_mem[c1][i], c = s->cepstral_mem[c2][i];
        s->features[i] = a + b + c;
        s->features[NB_BANDS + i] = a - c;
        s->features[NB_BANDS + NB_DELTA_CEPS + i] = a - 2.0f * b + c;
    }
    float spec_variability = 0.0f;
    if (s->mem_id == CEPS_MEM) s->mem_id = 0;
    for (int i = 0; i < CEPS_MEM; i++) {
        float min_dist = 1e15f;
        for (int j = 0; j < CEPS_MEM; j++) {
            float dist = 0.0f;
            for (int k = 0; k < NB_BANDS; k++) {
                float t = s->cepstral_mem[i][k] - s->cepstral_mem[j][k];
                dist += t * t;
            }
            if (j != i) min_dist = fminf(min_dist, dist);
        }
        spec_variability += min_dist;
    }
    s->features[NB_BANDS + 3 * NB_DELTA_CEPS + 1] = spec_variability / (float)CEPS_MEM - 2.1f;
    return 0;
}

/* src/features.rs:223-257 */
static void pitch_filter(nno_state *s, const float *gain) {
    float r[NB_BANDS], rf[FREQ_SIZE], new_e[NB_BANDS];
    for (int i = 0; i < NB_BANDS; i++) {
        if (s->exp[i] > gain[i]) {
            r[i] = 1.0f;
        } else {
            float exp_sq = s->exp[i] * s->exp[i];
            float g_sq = gain[i] * gain[i];
            r[i] = exp_sq * (1.0f - g_sq) / (0.001f + g_sq * (1.0f - exp_sq));
        }
        /* f32::clamp(0,1): NaN propagates */
        if (r[i] < 0.0f) r[i] = 0.0f;
        if (r[i] > 1.0f) r[i] = 1.0f;
        r[i] = sqrtf(r[i]);
        r[i] *= sqrtf(s->ex[i] / (1e-8f + s->ep[i]));
    }
    interp_band_gain(rf, r);
    s->x_re[0] += s->p_re[0] * rf[0]; /* offset (DC) is a real scalar */
    for (int i = 1; i < FREQ_SIZE; i++) {
        s->x_re[i] += s->p_re[i] * rf[i];
        s->x_im[i] += s->p_im[i] * rf[i];
    }
    compute_band_corr(new_e, s->x_re, s->x_im, s->x_re, s->x_im);
    for (int i = 0; i < NB_BANDS; i++) r[i] = sqrtf(s->ex[i] / (1e-8f + new_e[i]));
    interp_band_gain(rf, r);
    for (int i = 0; i < FREQ_SIZE; i++) {
        s->x_re[i] *= rf[i];
        s->x_im[i] *= rf[i];
    }
}

/* src/features.rs:263-275 */
static void frame_synthesis(nno_state *s, float *out) {
    nno_irfft960(s->x_re, s->x_im, s->window_buf);
    for (int i = 0; i < WINDOW_SIZE; i++) s->window_buf[i] /= 2.0f;
    for (int i = 0; i < WINDOW_SIZE; i++) s->window_buf[i] *= g_window[i];
    for (int i = 0; i < FRAME_SIZE; i++) {
        out[i] = s->window_buf[i] + s->synthesis_mem[i];
        s->synthesis_mem[i] = s->window_buf[FRAME_SIZE + i];
    }
}

/* ---- RNN: src/rnn.rs:251-409 -------------------------------------------------------------- */
#define WEIGHTS_SCALE (1.0f / 256.0f)

/* SubMatrix::mul_add, src/rnn.rs:402-409 */
static void mul_add(const int8_t *data, int stride, int offset, int rows, float *out, int nout, const float *in) {
    for (int j = 0; j < rows; j++) {
        const int8_t *col = data + (size_t)j * stride + offset;
        float xj = in[j];
        for (int i = 0; i < nout; i++) out[i] += (float)col[i] * xj;
    }
}

/* src/rnn.rs:251-272 */
static void dense_compute(const dense_layer *l, float *out, const float *in) {
    for (int i = 0; i < l->nn; i++) out[i] = (float)l->bias[i];
    mul_add(l->w, l->nn, 0, l->ni, out, l->nn, in);
    for (int i = 0; i < l->nn; i++) out[i] = activate(l->act, out[i] * WEIGHTS_SCALE);
}

/* src/rnn.rs:292-327 */
static void gru_compute(const gru_layer *l, float *state, const float *in) {
    float z[MAX_NEURONS], r[MAX_NEURONS], h[MAX_NEURONS];
    const int n = l->nn, st = 3 * n;
    for (int i = 0; i < n; i++) z[i] = (float)l->bias[i];
    mul_add(l->w, st, 0, l->ni, z, n, in);
    mul_add(l->r, st, 0, n, z, n, state);
    for (int i = 0; i < n; i++) z[i] = nno_sigmoid(WEIGHTS_SCALE * z[i]);

    for (int i = 0; i < n; i++) r[i] = (float)l->bias[n + i];
    mul_add(l->w, st, n, l->ni, r, n, in);
    mul_add(l->r, st, n, n, r, n, state);
    for (int i = 0; i < n; i++) r[i] = state[i] * nno_sigmoid(WEIGHTS_SCALE * r[i]);

    for (int i = 0; i < n; i++) h[i] = (float)l->bias[2 * n + i];
    mul_add(l->w, st, 2 * n, l->ni, h, n, in);
    mul_add(l->r, st, 2 * n, n, h, n, r);
    for (int i = 0; i < n; i++) {
        float hh = activate(l->act, WEIGHTS_SCALE * h[i]);
        state[i] = z[i] * state[i] + (1.0f - z[i]) * hh;
    }
}

/* src/rnn.rs:343-379 */
static void rnn_compute(nno_state *s, float *gains, float *vad, const float *input) {
    const nno_model *m = s->model;
    float buf[MAX_NEURONS * 3], dbuf[MAX_NEURONS * 3];
    memset(buf, 0, sizeof buf);
    memset(dbuf, 0, sizeof dbuf);
    const int nd = m->input_dense.nn, nv = m->vad_gru.nn, nn = m->noise_gru.nn;
    dense_compute(&m->input_dense, buf, input);
    gru_compute(&m->vad_gru, s->vad_gru_state, buf);
    dense_compute(&m->vad_output, vad, s->vad_gru_state);
    memcpy(buf + nd, s->vad_gru_state, nv * sizeof(float));
    memcpy(buf + nd + nv, input, 42 * sizeof(float));
    gru_compute(&m->noise_gru, s->noise_gru_state, buf);
    memcpy(dbuf, s->vad_gru_state, nv * sizeof(float));
    memcpy(dbuf + nv, s->noise_gru_state, nn * sizeof(float));
    memcpy(dbuf + nv + nn, input, 42 * sizeof(float));
    gru_compute(&m->denoise_gru, s->denoise_gru_state, dbuf);
    dense_compute(&m->denoise_output, gains, s->denoise_gru_state);
}

/* ---- frame driver: src/denoise.rs:95-116 -------------------------------------------------- */
float nno_process_frame(nno_state *s, float *out, const float *in) {
    float g[NB_BANDS], gf[FREQ_SIZE];
    float vad_prob = 0.0f;
    for (int i = 0; i < NB_BANDS; i++) g[i] = 0.0f;

    /* shift_and_filter_input, src/features.rs:97-104 */
    memmove(s->input_mem, s->input_mem + FRAME_SIZE, (PITCH_BUF_SIZE - FRAME_SIZE) * sizeof(float));
    biquad_hp(s->input_mem + (PITCH_BUF_SIZE - FRAME_SIZE), s->mem_hp_x, in, FRAME_SIZE);

    int silence = compute_frame_features(s);
    if (!silence) {
        rnn_compute(s, g, &vad_prob, s->features);
        pitch_filter(s, g);
        for (int i = 0; i < NB_BANDS; i++) {
            g[i] = fmaxf(g[i], 0.6f * s->lastg[i]);
            s->lastg[i] = g[i];
        }
        interp_band_gain(gf, g);
        for (int i = 0; i < FREQ_SIZE; i++) {
            s->x_re[i] *= gf[i];
            s->x_im[i] *= gf[i];
        }
    }
    frame_synthesis(s, out);

    s->taps.silence = silence;
    s->taps.vad = vad_prob;
    memcpy(s->taps.features, s->features, sizeof s->features);
    memcpy(s->taps.gains, g, sizeof g);
    memcpy(s->taps.ex, s->ex, sizeof s->ex);
    memcpy(s->taps.ep, s->ep, sizeof s->ep);
    memcpy(s->taps.exp, s->exp, sizeof s->exp);
    return vad_prob;
}

/* ---- batched CPU driver (timed baseline) --------------------------------------------------- */
static double now_s(void) {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}

double nno_run_batch(const nno_model *m, const float *in, float *out, float *vad, int32_t *pitch, int n_streams,
                     int n_frames, int n_threads, int *threads_used) {
    ensure_tables();
    nno_state **st = (nno_state **)malloc(sizeof(nno_state *) * (size_t)n_streams);
    for (int i = 0; i < n_streams; i++) st[i] = nno_state_new(m);
    int used = 1;
#ifdef _OPENMP
    if (n_threads <= 0) n_threads = omp_get_max_threads();
    used = n_threads;
#else
    (void)n_threads;
#endif
    double t0 = now_s();
#ifdef _OPENMP
#pragma omp parallel for schedule(dynamic, 1) num_threads(n_threads)
#endif
    for (int i = 0; i < n_streams; i++) {
        float tmp[FRAME_SIZE];
        for (int f = 0; f < n_frames; f++) {
            size_t off = ((size_t)i * n_frames + f) * FRAME_SIZE;
            float v = nno_process_frame(st[i], out ? out + off : tmp, in + off);
            if (vad) vad[(size_t)i * n_frames + f] = v;
            if (pitch) pitch[(size_t)i * n_frames + f] = st[i]->taps.pitch;
        }
    }
    double t1 = now_s();
    for (int i = 0; i < n_streams; i++) nno_state_free(st[i]);
    free(st);
    if (threads_used) *threads_used = used;
    return t1 - t0;
}

/* ---- training-data rows: src/training.rs ---------------------------------------------------- */
/* Biquad::filter_in_place, src/util.rs:113-124 (f64 arithmetic, f32 state) */
static void biquad_in_place(const float a[2], const float b[2], float *data, float mem[2], int n) {
    const double a0 = (double)a[0], a1 = (double)a[1], b0 = (double)b[0], b1 = (double)b[1];
    for (int i = 0; i < n; i++) {
        double x64 = (double)data[i];
        double y64 = x64 + (double)mem[0];
        mem[0] = (float)((double)mem[1] + (b0 * x64 - a0 * y64));
        mem[1] = (float)(b1 * x64 - a1 * y64);
        data[i] = (float)y64;
    }
}

struct nno_trainer {
    nno_sim_params p;
    int vad_count;                              /* NoiseSimulator::vad_count, src/training.rs:288 */
    float signal_resp_mem[2], noise_resp_mem[2]; /* :299-300 */
    nno_state *clean, *noise, *comb;            /* src/training.rs:113-115 */
};

nno_trainer *nno_train_new(void) {
    nno_trainer *t = (nno_trainer *)calloc(1, sizeof(*t));
    if (!t) return NULL;
    /* NoiseSimulator::new, src/training.rs:319-340 */
    t->p.signal_gain = 1.0f;
    t->p.noise_gain = 1.0f;
    t->p.band_lp = NB_BANDS - 1;
    t->clean = nno_state_new(NULL);
    t->noise = nno_state_new(NULL);
    t->comb = nno_state_new(NULL);
    return t;
}

void nno_train_free(nno_trainer *t) {
    if (!t) return;
    nno_state_free(t->clean);
    nno_state_free(t->noise);
    nno_state_free(t->comb);
    free(t);
}

void nno_train_set_params(nno_trainer *t, const nno_sim_params *p) { t->p = *p; }

int32_t nno_train_band_lp(int32_t lowpass) {
    for (int i = 0; i < NB_BANDS; i++)
        if ((EBAND_5MS[i] << 2) > lowpass) return i;
    return NB_BANDS - 1;
}

/* DenoiseFeatures::shift_and_filter_input, src/features.rs:97-104 */
static void shift_and_filter(nno_state *s, const float *in) {
    memmove(s->input_mem, s->input_mem + FRAME_SIZE, (PITCH_BUF_SIZE - FRAME_SIZE) * sizeof(float));
    biquad_hp(s->input_mem + (PITCH_BUF_SIZE - FRAME_SIZE), s->mem_hp_x, in, FRAME_SIZE);
}

void nno_train_frame(nno_trainer *t, const float *signal, const float *noise, float *row) {
    float sig_buf[FRAME_SIZE], noise_buf[FRAME_SIZE], out_buf[FRAME_SIZE];
    /* NoiseSimulator::next_frame, src/training.rs:399-432 (the randomize() trigger is the caller's) */
    for (int i = 0; i < FRAME_SIZE; i++) noise_buf[i] = noise[i] * t->p.noise_gain; /* read_noise :342-348 */
    float sig_e = 0.0f;                                                            /* read_signal :351-359 */
    for (int i = 0; i < FRAME_SIZE; i++) {
        sig_e += signal[i] * signal[i];
        sig_buf[i] = signal[i] * t->p.signal_gain;
    }
    biquad_in_place(t->p.sig_a, t->p.sig_b, sig_buf, t->signal_resp_mem, FRAME_SIZE);
    biquad_in_place(t->p.noise_a, t->p.noise_b, noise_buf, t->noise_resp_mem, FRAME_SIZE);
    for (int i = 0; i < FRAME_SIZE; i++) out_buf[i] = sig_buf[i] + noise_buf[i];
    /* NoiseSimulator::vad, :380-397 */
    if (sig_e > 1e9f) t->vad_count = 0;
    else if (sig_e > 1e8f) t->vad_count -= 5;
    else if (sig_e > 1e7f) t->vad_count += 1;
    else t->vad_count += 2;
    if (t->vad_count < 0) t->vad_count = 0;
    if (t->vad_count > 15) t->vad_count = 15;
    const float vad = t->vad_count >= 10 ? 0.0f : (t->vad_count > 0 ? 0.5f : 1.0f);
    int cutoff = (vad == 0.0f && t->p.noise_gain == 0.0f) ? 0 : t->p.band_lp + 1;

    /* main loop body, src/training.rs:126-159 */
    shift_and_filter(t->clean, sig_buf);
    shift_and_filter(t->noise, noise_buf);
    shift_and_filter(t->comb, out_buf);
    compute_frame_features(t->clean);
    compute_frame_features(t->noise);
    const int silence = compute_frame_features(t->comb);
    if (silence) cutoff = 0;
    float *gains = row + NB_FEATURES, *noise_level = row + NB_FEATURES + NB_BANDS;
    for (int i = 0; i < NB_BANDS; i++) {
        if (i < cutoff) {
            const float ce = t->clean->ex[i], me = t->comb->ex[i];
            gains[i] = (ce < 5e-2f && me < 5e-2f) ? -1.0f : fminf(sqrtf((ce + 1e-3f) / (me + 1e-3f)), 1.0f);
        } else {
            gains[i] = -1.0f;
        }
        noise_level[i] = log10f(t->noise->ex[i] + 1e-2f);
    }
    memcpy(row, t->comb->features, NB_FEATURES * sizeof(float));
    row[NB_FEATURES + 2 * NB_BANDS] = vad;
}

/* ---- file front-end: src/nnnoiseless.rs --------------------------------------------------- */
/* dasp_interpolate::sinc::Sinc<[f32; 16]> (0.11.0, restated): ring of 16 frames, idx saturating at depth. */
typedef struct {
    float ring[16]; /* logical order: ring[(first + i) % 16] = frames[i] */
    int first;
    int idx;
} sinc16;

static inline float sinc_at(const sinc16 *s, int i) { return s->ring[(s->first + i) % 16]; } /* Fixed::get wraps */

/* Sinc::next_source_frame: Fixed::push overwrites the oldest frame, which becomes the newest */
static void sinc_push(sinc16 *s, float x) {
    s->ring[s->first] = x;
    s->first = (s->first + 1) % 16;
    if (s->idx < 8) s->idx += 1;
}

/* Sinc::interpolate */
static float sinc_interpolate(const sinc16 *s, double x) {
    const double pi = 3.14159265358979323846264338327950288;
    const int depth = 8, len = 16;
    const double phil = x, phir = 1.0 - x;
    const int nl = s->idx, nr = s->idx + 1;
    const int rightmost = nl + depth, leftmost = nr - depth;
    int max_depth;
    if (rightmost >= len) max_depth = len - depth;
    else if (leftmost < 0) max_depth = depth + leftmost;
    else max_depth = depth;
    float v = 0.0f;
    for (int n = 0; n < max_depth; n++) {
        double a = pi * (phil + (double)n);
        double first = (a == 0.0) ? 1.0 : sin(a) / a;
        double second = 0.5 + 0.5 * cos(a / (double)depth);
        v += (float)(first * second * (double)sinc_at(s, nl - n));
        a = pi * (phir + (double)n);
        first = (a == 0.0) ? 1.0 : sin(a) / a;
        second = 0.5 + 0.5 * cos(a / (double)depth);
        v += (float)(first * second * (double)sinc_at(s, nr + n));
    }
    return v;
}

long nno_resample(const float *in, long n_in, int channels, double ratio, float *out, long cap) {
    sinc16 *st = (sinc16 *)calloc((size_t)channels, sizeof(sinc16));
    double pos = 0.0;
    long src = 0, k = 0;
    for (;; k++) {
        pos += ratio;
        int dry = 0;
        while (pos >= 1.0) {
            pos -= 1.0;
            if (src >= n_in) {
                dry = 1;
                break;
            }
            for (int c = 0; c < channels; c++) sinc_push(&st[c], in[src * channels + c]);
            src++;
        }
        if (dry || k >= cap) break;
        for (int c = 0; c < channels; c++) out[k * channels + c] = sinc_interpolate(&st[c], pos);
    }
    free(st);
    return k;
}

long nno_cli_frames(const nno_model *m, const float *in, long n_in, int channels, int16_t *out, long cap) {
    nno_state **st = (nno_state **)malloc(sizeof(nno_state *) * (size_t)channels);
    for (int c = 0; c < channels; c++) st[c] = nno_state_new(m);
    float ib[FRAME_SIZE], ob[FRAME_SIZE];
    long written = 0;
    for (long f = 0; (f + 1) * FRAME_SIZE <= n_in; f++) {
        if (f > 0 && written + FRAME_SIZE > cap) break;
        for (int c = 0; c < channels; c++) {
            for (int i = 0; i < FRAME_SIZE; i++) ib[i] = in[(f * FRAME_SIZE + i) * channels + c];
            nno_process_frame(st[c], ob, ib);
            if (f == 0) continue; /* `first` frame is not written, src/nnnoiseless.rs:319-327 */
            for (int i = 0; i < FRAME_SIZE; i++) {
                float v = fminf(fmaxf(ob[i], -32768.0f), 32767.0f); /* :152-153, :167 */
                out[(written + i) * channels + c] = (int16_t)roundf(v);
            }
        }
        if (f > 0) written += FRAME_SIZE;
    }
    for (int c = 0; c < channels; c++) nno_state_free(st[c]);
    free(st);
    return written;
}
