/*
 * wavenet_oracle.c -- CPU oracle (TEST INFRASTRUCTURE ONLY, see wavenet_oracle.h).
 *
 * Plain-C restatement of NVIDIA/nv-wavenet's CPU model.  "ref:" comments give the
 * reference file:line each block follows.  All matrices are column-major exactly
 * as the reference API passes them (README.md:38): W[row + k*M].
 *
 * Operation order is the reference CPU order, NOT the reference GPU order:
 *   dot products   sum = 0; sum += a*b  left to right, separate mul and add
 *                  (matrix.cpp:85-102)
 *   pre-activation (a_prev + a_cur) + Bh, then + Lh           (reference.cpp:67-72)
 *   residual       (Wres.h + Bres) + Xin                      (reference.cpp:82-84)
 *   skip           (Wskip.h + skipIn) + Bskip, relu on last   (reference.cpp:86-90)
 *   softmax        max starts at 0.f, sequential sum, p = e/sum   (matrix.cpp:167-183)
 *   select         first row with sel < running sum of p      (reference.cpp:106-121)
 *
 * Build WITHOUT -ffast-math / -mfma / -march=native so that float mul+add are
 * never contracted (the pin test against oracle/_ref is bit-exact).
 */
#include "wavenet_oracle.h"

#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

/* ------------------------------------------------------------------------- */
/* portable transcendental functions (DESIGN.md §4): only IEEE-754 double       */
/* +,*,/,fma,rint and one double->float rounding, so a CUDA transcription is    */
/* bit-identical.                                                               */
/* ------------------------------------------------------------------------- */

static double wno_exp_core(double x)
{
    /* caller guarantees -150 <= x <= 100 */
    const double LOG2E = 0x1.71547652b82fep+0;
    const double LN2_HI = 0x1.62e42fee00000p-1;
    const double LN2_LO = 0x1.a39ef35793c76p-33;
    double kd = rint(x * LOG2E);
    double r = fma(-kd, LN2_HI, x);
    r = fma(-kd, LN2_LO, r);
    /* degree-13 Taylor polynomial of exp(r), |r| <= ln2/2, Estrin association (fixed: the CUDA
     * kernel evaluates exactly this tree) */
    double a0 = fma(1.0, r, 1.0);                                           /* c0 + c1 r   */
    double a1 = fma(0x1.5555555555555p-3, r, 0.5);                           /* c2 + c3 r   */
    double a2 = fma(0x1.1111111111111p-7, r, 0x1.5555555555555p-5);          /* c4 + c5 r   */
    double a3 = fma(0x1.a01a01a01a01ap-13, r, 0x1.6c16c16c16c17p-10);        /* c6 + c7 r   */
    double a4 = fma(0x1.71de3a556c734p-19, r, 0x1.a01a01a01a01ap-16);        /* c8 + c9 r   */
    double a5 = fma(0x1.ae64567f544e4p-26, r, 0x1.27e4fb7789f5cp-22);        /* c10 + c11 r */
    double a6 = fma(0x1.6124613a86d09p-33, r, 0x1.1eed8eff8d898p-29);        /* c12 + c13 r */
    double r2 = r * r;
    double b0 = fma(a1, r2, a0);
    double b1 = fma(a3, r2, a2);
    double b2 = fma(a5, r2, a4);
    double r4 = r2 * r2;
    double d0 = fma(b1, r4, b0);
    double d1 = fma(a6, r4, b2);
    double r8 = r4 * r4;
    double p = fma(d1, r8, d0);
    int64_t k = (int64_t)kd;                 /* -217 .. 145: 2^k is a normal double */
    uint64_t bits = (uint64_t)(k + 1023) << 52;
    double scale;
    memcpy(&scale, &bits, sizeof scale);
    return p * scale;
}

float wno_expf_portable(float x)
{
    if (x != x) return x;
    if (x < -150.0f) return 0.0f;
    if (x > 100.0f) return INFINITY;
    return (float)wno_exp_core((double)x);
}

float wno_tanhf_portable(float x)
{
    if (x != x) return x;
    double xd = (double)x;
    double ax = fabs(xd);
    double t;
    if (ax < 0x1p-12) {
        double x2 = ax * ax;
        t = fma(-(x2 * ax), 0x1.5555555555555p-2, ax);   /* x - x^3/3 */
    } else if (ax >= 20.0) {
        t = 1.0;
    } else {
        double e = wno_exp_core(2.0 * ax);
        t = (e - 1.0) / (e + 1.0);
    }
    return (float)(xd < 0.0 ? -t : t);
}

/* ref: nv_wavenet_reference.cpp:36  sigmoid(f) = 1.f / (1.f + exp(-f)) in float */
float wno_sigmoidf_portable(float x)
{
    float e = wno_expf_portable(-x);
    float den = 1.0f + e;
    return 1.0f / den;
}

/* (float)(_Float16)x, round to nearest even, in integer arithmetic: the compiler's conversion is a library call on x86-64
 * without F16C, and the fp16-contract model rounds every weight of every dot product (equal for all 2^32 inputs). */
static inline float round_fp16(float x)
{
    uint32_t u, a, s;
    float r;
    memcpy(&u, &x, 4);
    a = u & 0x7FFFFFFFu; s = u & 0x80000000u;
    if (a >= 0x7F800000u) return x;                                   /* inf, nan */
    if (a >= 0x477FF000u) u = s | 0x7F800000u;                        /* rounds past 65504 */
    else if (a >= 0x38800000u) u = s | ((a + 0x0FFFu + ((a >> 13) & 1u)) & ~0x1FFFu);    /* normal: 11 significant bits */
    else {                                                            /* subnormal: a multiple of 2^-24, the ulp of [0.5, 1) */
        float m;
        memcpy(&m, &a, 4);
        m = (m + 0.5f) - 0.5f;
        memcpy(&u, &m, 4);
        u |= s;
    }
    memcpy(&r, &u, 4);
    return r;
}

float wno_round_fp16(float x) { return round_fp16(x); }

/* ------------------------------------------------------------------------- */

struct wno_model {
    int L, B, N, R, S, A, maxDil;
    int math_mode, prec_mode, tanh_embed;
    const int* forced;
    float* logit_trace;

    float *embPrev, *embCur;            /* [A][R] : emb[y*R + r]  (reference.cpp:52, Matrix(R,A) col-major) */
    float *Wprev, *Wcur, *Bh;           /* per layer: 2R x R col-major, 2R */
    float *Wres, *Bres;                 /* R x R, R */
    float *Wskip, *Bskip;               /* S x R, S */
    float *Wzs, *Bzs, *Wza, *Bza;       /* A x S, A, A x A, A */

    float* Lh;                          /* [N][L][B][2R] */
    float* sel;                         /* [N][B] */
    int *yPrev, *yCur;                  /* [B] */

    /* ring of layer inputs: [(maxDil+1)][L+1][B][R]  (fp32 residual stream) */
    float* ring;
    float* skipOut;                     /* [L][B][S]  last computed sample */
    float* xtOut;                       /* [L][B][R]  last computed sample (layer outputs) */
    float *Zs, *Za, *P;                 /* [B][A] */
};

static float* fzalloc(size_t n) { return (float*)calloc(n ? n : 1, sizeof(float)); }

wno_model* wno_create(int num_layers, int max_batch, int max_samples, int R, int S, int A, int max_dilation)
{
    wno_model* m = (wno_model*)calloc(1, sizeof *m);
    m->L = num_layers; m->B = max_batch; m->N = max_samples;
    m->R = R; m->S = S; m->A = A; m->maxDil = max_dilation;
    m->math_mode = WNO_MATH_LIBM; m->prec_mode = WNO_PREC_FP32; m->tanh_embed = 1;
    size_t L = (size_t)num_layers;
    m->embPrev = fzalloc((size_t)A * R); m->embCur = fzalloc((size_t)A * R);
    m->Wprev = fzalloc(L * 2 * R * R); m->Wcur = fzalloc(L * 2 * R * R); m->Bh = fzalloc(L * 2 * R);
    m->Wres = fzalloc(L * R * R); m->Bres = fzalloc(L * R);
    m->Wskip = fzalloc(L * S * R); m->Bskip = fzalloc(L * S);
    m->Wzs = fzalloc((size_t)A * S); m->Bzs = fzalloc(A); m->Wza = fzalloc((size_t)A * A); m->Bza = fzalloc(A);
    m->Lh = fzalloc((size_t)max_samples * L * max_batch * 2 * R);
    m->sel = fzalloc((size_t)max_samples * max_batch);
    m->yPrev = (int*)calloc(max_batch, sizeof(int)); m->yCur = (int*)calloc(max_batch, sizeof(int));
    m->ring = fzalloc((size_t)(max_dilation + 1) * (L + 1) * max_batch * R);
    m->skipOut = fzalloc(L * max_batch * S);
    m->xtOut = fzalloc(L * max_batch * R);
    m->Zs = fzalloc((size_t)max_batch * A); m->Za = fzalloc((size_t)max_batch * A); m->P = fzalloc((size_t)max_batch * A);
    for (int b = 0; b < max_batch; b++) { m->yPrev[b] = 128; m->yCur[b] = 128; }
    return m;
}

void wno_destroy(wno_model* m)
{
    if (!m) return;
    free(m->embPrev); free(m->embCur); free(m->Wprev); free(m->Wcur); free(m->Bh);
    free(m->Wres); free(m->Bres); free(m->Wskip); free(m->Bskip);
    free(m->Wzs); free(m->Bzs); free(m->Wza); free(m->Bza);
    free(m->Lh); free(m->sel); free(m->yPrev); free(m->yCur);
    free(m->ring); free(m->skipOut); free(m->xtOut); free(m->Zs); free(m->Za); free(m->P);
    free(m);
}

void wno_set_math(wno_model* m, int mode) { m->math_mode = mode; }
void wno_set_precision(wno_model* m, int mode) { m->prec_mode = mode; }
void wno_set_tanh_embed(wno_model* m, int t) { m->tanh_embed = t; }
void wno_set_forced(wno_model* m, const int* forced) { m->forced = forced; }
void wno_set_logit_trace(wno_model* m, float* trace) { m->logit_trace = trace; }

/* ref: nv_wavenet_reference.cpp:205-208 */
void wno_set_embeddings(wno_model* m, const float* embedPrev, const float* embedCur)
{
    memcpy(m->embPrev, embedPrev, sizeof(float) * m->A * m->R);
    memcpy(m->embCur, embedCur, sizeof(float) * m->A * m->R);
}

/* ref: nv_wavenet_reference.cpp:210-219 */
void wno_set_layer_weights(wno_model* m, int l, const float* Wprev, const float* Wcur, const float* Bh,
                           const float* Wres, const float* Bres, const float* Wskip, const float* Bskip)
{
    int R = m->R, S = m->S;
    memcpy(m->Wprev + (size_t)l * 2 * R * R, Wprev, sizeof(float) * 2 * R * R);
    memcpy(m->Wcur + (size_t)l * 2 * R * R, Wcur, sizeof(float) * 2 * R * R);
    memcpy(m->Bh + (size_t)l * 2 * R, Bh, sizeof(float) * 2 * R);
    memcpy(m->Wres + (size_t)l * R * R, Wres, sizeof(float) * R * R);
    memcpy(m->Bres + (size_t)l * R, Bres, sizeof(float) * R);
    memcpy(m->Wskip + (size_t)l * S * R, Wskip, sizeof(float) * S * R);
    memcpy(m->Bskip + (size_t)l * S, Bskip, sizeof(float) * S);
}

/* ref: nv_wavenet_reference.cpp:221-226 */
void wno_set_out_weights(wno_model* m, const float* Wzs, const float* Bzs, const float* Wza, const float* Bza)
{
    memcpy(m->Wzs, Wzs, sizeof(float) * m->A * m->S);
    memcpy(m->Bzs, Bzs, sizeof(float) * m->A);
    memcpy(m->Wza, Wza, sizeof(float) * m->A * m->A);
    memcpy(m->Bza, Bza, sizeof(float) * m->A);
}

/* ref: nv_wavenet_reference.cpp:228-247 (history reset to 128, Lh [N][L][B][2R], selectors [N][B]) */
void wno_set_inputs(wno_model* m, const float* Lh, const float* outputSelectors)
{
    for (int b = 0; b < m->B; b++) { m->yPrev[b] = 128; m->yCur[b] = 128; }
    memcpy(m->Lh, Lh, sizeof(float) * (size_t)m->N * m->L * m->B * 2 * m->R);
    memcpy(m->sel, outputSelectors, sizeof(float) * (size_t)m->N * m->B);
}

void wno_get_xt_out(wno_model* m, int layer, float* out) { memcpy(out, m->xtOut + (size_t)layer * m->B * m->R, sizeof(float) * m->B * m->R); }
void wno_get_skip_out(wno_model* m, int layer, float* out) { memcpy(out, m->skipOut + (size_t)layer * m->B * m->S, sizeof(float) * m->B * m->S); }
void wno_get_zs(wno_model* m, float* out) { memcpy(out, m->Zs, sizeof(float) * m->B * m->A); }
void wno_get_za(wno_model* m, float* out) { memcpy(out, m->Za, sizeof(float) * m->B * m->A); }
void wno_get_p(wno_model* m, float* out) { memcpy(out, m->P, sizeof(float) * m->B * m->A); }

/* ------------------------------------------------------------------------- */

static inline float m_exp(const wno_model* m, float x) { return m->math_mode == WNO_MATH_LIBM ? expf(x) : wno_expf_portable(x); }
static inline float m_tanh(const wno_model* m, float x) { return m->math_mode == WNO_MATH_LIBM ? tanhf(x) : wno_tanhf_portable(x); }
/* ref: nv_wavenet_reference.cpp:36 */
static inline float m_sigmoid(const wno_model* m, float x) { return 1.f / (1.f + m_exp(m, -x)); }
static inline float q16(const wno_model* m, float x) { return m->prec_mode == WNO_PREC_FP16 ? round_fp16(x) : x; }

/* ref: matrix.cpp:85-102 matrix_multiply, one output element.
 * W is M x K col-major; x has K contiguous elements.  In PREC_FP16 both operands arrive rounded to fp16 (see wno_run). */
static inline float dot_row(const float* W, int M, int K, int row, const float* x)
{
    float sum = 0;
    for (int k = 0; k < K; k++) sum += W[row + (size_t)k * M] * x[k];
    return sum;
}

/* PREC_FP16 operands: the weights rounded once per run, an activation vector once per use (into buf) */
static float* rounded_copy(const float* W, size_t n)
{
    float* q = fzalloc(n);
    for (size_t i = 0; i < n; i++) q[i] = round_fp16(W[i]);
    return q;
}
static inline const float* q16v(const wno_model* m, const float* x, int n, float* buf)
{
    if (m->prec_mode != WNO_PREC_FP16) return x;
    for (int i = 0; i < n; i++) buf[i] = round_fp16(x[i]);
    return buf;
}

int wno_run(wno_model* m, int num_samples, int batch_size, int* yOut)
{
    const int L = m->L, R = m->R, S = m->S, A = m->A, B = m->B;
    const int slots = m->maxDil + 1;
    int status = 0;
    float* a_prev = fzalloc(2 * R); float* a_cur = fzalloc(2 * R); float* hp = fzalloc(2 * R);
    float* h = fzalloc(R); float* zeroR = fzalloc(R); float* skipv = fzalloc(S); float* zs = fzalloc(A);
    float* qa = fzalloc(R); float* qb = fzalloc(R); float* qh = fzalloc(R); float* qs = fzalloc(S); float* qz = fzalloc(A);
    const float *Wprev = m->Wprev, *Wcur = m->Wcur, *Wres = m->Wres, *Wskip = m->Wskip, *Wzs = m->Wzs, *Wza = m->Wza;
    float* wq[6] = {NULL, NULL, NULL, NULL, NULL, NULL};
    if (m->prec_mode == WNO_PREC_FP16) {
        Wprev = wq[0] = rounded_copy(m->Wprev, (size_t)L * 2 * R * R); Wcur = wq[1] = rounded_copy(m->Wcur, (size_t)L * 2 * R * R);
        Wres = wq[2] = rounded_copy(m->Wres, (size_t)L * R * R); Wskip = wq[3] = rounded_copy(m->Wskip, (size_t)L * S * R);
        Wzs = wq[4] = rounded_copy(m->Wzs, (size_t)A * S); Wza = wq[5] = rounded_copy(m->Wza, (size_t)A * A);
    }

    for (int t = 0; t < num_samples; t++) {
        float* ring_t = m->ring + (size_t)(t % slots) * (L + 1) * B * R;
        for (int b = 0; b < batch_size; b++) {
            /* ref: nv_wavenet_reference.cpp:42-57 nvWavenetEmbed */
            float* x0 = ring_t + (size_t)b * R;
            for (int r = 0; r < R; r++) {
                float e = q16(m, m->embPrev[m->yPrev[b] * R + r]) + q16(m, m->embCur[m->yCur[b] * R + r]);
                x0[r] = m->tanh_embed ? m_tanh(m, e) : e;
            }
            /* ref: nv_wavenet_reference.cpp:283-293 layer loop and dilation schedule */
            int dilation = 1;
            for (int l = 0; l < L; l++) {
                const float* xin = ring_t + ((size_t)l * B + b) * R;
                const float* xtmd = (t < dilation) ? zeroR
                    : m->ring + (size_t)((t - dilation) % slots) * (L + 1) * B * R + ((size_t)l * B + b) * R;
                dilation *= 2;
                if (dilation > m->maxDil) dilation = 1;
                /* ref: nv_wavenet_reference.cpp:59-72 nvWavenetLayer, pre-activation */
                const float* Wp = Wprev + (size_t)l * 2 * R * R;
                const float* Wc = Wcur + (size_t)l * 2 * R * R;
                const float* lh = m->Lh + (((size_t)t * L + l) * B + b) * 2 * R;
                const float* xtmd_q = q16v(m, xtmd, R, qa);
                const float* xin_q = q16v(m, xin, R, qb);
                for (int row = 0; row < 2 * R; row++) {
                    a_prev[row] = dot_row(Wp, 2 * R, R, row, xtmd_q);
                    a_cur[row] = dot_row(Wc, 2 * R, R, row, xin_q);
                    float v = a_prev[row] + a_cur[row];
                    v = v + q16(m, m->Bh[(size_t)l * 2 * R + row]);
                    v = v + q16(m, lh[row]);
                    hp[row] = v;
                }
                /* ref: nv_wavenet_reference.cpp:74-80 gate */
                for (int r = 0; r < R; r++) h[r] = m_tanh(m, hp[r]) * m_sigmoid(m, hp[r + R]);
                const float* h_q = q16v(m, h, R, qh);
                /* ref: nv_wavenet_reference.cpp:82-84 residual */
                const float* Wr = Wres + (size_t)l * R * R;
                float* xout = ring_t + ((size_t)(l + 1) * B + b) * R;
                for (int r = 0; r < R; r++) {
                    float v = dot_row(Wr, R, R, r, h_q);
                    v = v + q16(m, m->Bres[(size_t)l * R + r]);
                    v = v + xin[r];
                    xout[r] = v;
                    m->xtOut[((size_t)l * B + b) * R + r] = v;
                }
                /* ref: nv_wavenet_reference.cpp:86-90 skip accumulate (+relu on the last layer) */
                const float* Ws = Wskip + (size_t)l * S * R;
                float* so = m->skipOut + ((size_t)l * B + b) * S;
                const float* si = l ? m->skipOut + ((size_t)(l - 1) * B + b) * S : NULL;
                for (int s = 0; s < S; s++) {
                    float v = dot_row(Ws, S, R, s, h_q);
                    v = v + (si ? si[s] : 0.f);
                    v = v + q16(m, m->Bskip[(size_t)l * S + s]);
                    if (l == L - 1) v = (v < 0) ? 0.f : v;
                    so[s] = v;
                }
            }
            /* ref: nv_wavenet_reference.cpp:93-104 nvWavenetFinal */
            const float* skipL = m->skipOut + ((size_t)(L - 1) * B + b) * S;
            for (int s = 0; s < S; s++) skipv[s] = skipL[s];
            float* Zs = m->Zs + (size_t)b * A; float* Za = m->Za + (size_t)b * A; float* P = m->P + (size_t)b * A;
            const float* skip_q = q16v(m, skipv, S, qs);
            for (int a = 0; a < A; a++) {
                float v = dot_row(Wzs, A, S, a, skip_q);
                v = v + q16(m, m->Bzs[a]);
                v = (v < 0) ? 0.f : v;
                Zs[a] = v; zs[a] = v;
            }
            const float* zs_q = q16v(m, zs, A, qz);
            for (int a = 0; a < A; a++) {
                float v = dot_row(Wza, A, A, a, zs_q);
                v = v + q16(m, m->Bza[a]);
                Za[a] = v;
            }
            if (m->logit_trace) memcpy(m->logit_trace + ((size_t)t * batch_size + b) * A, Za, sizeof(float) * A);
            /* ref: matrix.cpp:167-183 matrix_softmax (max is initialised to 0.f, not to the first element) */
            float mx = 0.f;
            for (int a = 0; a < A; a++) if (Za[a] > mx) mx = Za[a];
            float sum = 0.f;
            for (int a = 0; a < A; a++) sum += m_exp(m, Za[a] - mx);
            for (int a = 0; a < A; a++) P[a] = m_exp(m, Za[a] - mx) / sum;
            /* ref: nv_wavenet_reference.cpp:106-121 nvWavenetSelect; selectors are Matrix(batch,samples)
             * col-major, i.e. sel[t*B + b] */
            float sel = m->sel[(size_t)t * B + b];
            float cs = 0.f;
            int y = -1;
            for (int a = 0; a < A; a++) {
                cs += P[a];
                if (sel < cs) { y = a; break; }
            }
            if (y < 0) { status = -1; y = A - 1; }   /* reference asserts here (reference.cpp:119) */
            /* ref: nv_wavenet_reference.cpp:296-300 feedback */
            yOut[(size_t)b * num_samples + t] = y;
            int fb = m->forced ? m->forced[(size_t)b * num_samples + t] : y;
            m->yPrev[b] = m->yCur[b];
            m->yCur[b] = fb;
        }
    }
    free(a_prev); free(a_cur); free(hp); free(h); free(zeroR); free(skipv); free(zs);
    free(qa); free(qb); free(qh); free(qs); free(qz);
    for (int i = 0; i < 6; i++) free(wq[i]);
    return status;
}

/* ------------------------------------------------------------------------- */
/* Test support: glibc rand() (random_r TYPE_3: r[i] = r[i-3] + r[i-31], output >> 1)
 * stepped on caller-held state, so that tests/refgen.py can replay the reference
 * test's srand(seed)/rand() input construction without depending on the host libc.
 * state[0..30] = ring, state[31] = front index, state[32] = rear index.          */
void wno_glibc_rand_fill(uint32_t* state, long n, int32_t* out)
{
    uint32_t f = state[31], r = state[32];
    for (long i = 0; i < n; i++) {
        uint32_t v = state[f] + state[r];
        state[f] = v;
        out[i] = (int32_t)(v >> 1);
        if (++f == 31) f = 0;
        if (++r == 31) r = 0;
    }
    state[31] = f; state[32] = r;
}
