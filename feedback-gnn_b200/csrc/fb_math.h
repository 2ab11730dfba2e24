/* fb_math.h -- the arithmetic specification of the fbgnn hot path.
 *
 * Every floating-point step of the decoder (quaternary BP, binary BP, feedback GNN) is
 * written in terms of the functions below.  They use only IEEE-754 binary32 operations
 * with a fixed evaluation order (add, mul, fma, div, integer bit manipulation), so the
 * same source gives bit-identical results on the host (gcc, -ffp-contract=off) and on
 * the device (nvcc, explicit __f*_rn intrinsics which are never contracted).  That is
 * what lets the CUDA kernels be compared BIT-EXACTLY with the CPU oracle instead of
 * within a tolerance that BP's chaotic dynamics would blow through (SURVEY.md F6/H1).
 *
 * The formulas restate the TensorFlow ops the reference calls:
 *   tf.math.softplus        decoding_q.py:265,270,373,458,462   (Eigen softplus functor:
 *                           x > 13.942385 -> x ; x < -13.942385 -> exp(x) ; else log1p(exp(x)))
 *   tf.reduce_logsumexp     decoding_q.py:266,271,459,463       (max-shifted, log not log1p)
 *   _phi (quaternary)       decoding_q.py:365-373
 *   _phi (binary)           decoding.py:625-633
 *   tanh activation         gnn.py:55-58 (Keras Dense(..., "tanh"))
 * exp/log/tanh themselves are polynomial / rational approximations accurate to about
 * 1-2 ulp (measured in tests/test_math.py against float64).
 *
 * This header is plain C99 / CUDA C++ and has no dependencies.
 */
#ifndef FBGNN_FB_MATH_H
#define FBGNN_FB_MATH_H

#include <stdint.h>

#if defined(__CUDA_ARCH__)
#  define FB_HD __host__ __device__ __forceinline__
#  define FB_FMA(a, b, c) __fmaf_rn((a), (b), (c))
#  define FB_ADD(a, b)    __fadd_rn((a), (b))
#  define FB_SUB(a, b)    __fsub_rn((a), (b))
#  define FB_MUL(a, b)    __fmul_rn((a), (b))
#  define FB_DIV(a, b)    __fdiv_rn((a), (b))
#  define FB_F2I(f)       __float_as_int(f)
#  define FB_I2F(i)       __int_as_float(i)
#  define FB_FMAX(a, b)   fmaxf((a), (b))
#  define FB_FMIN(a, b)   fminf((a), (b))
#else
#  include <math.h>
#  include <string.h>
#  if defined(__CUDACC__)
#    define FB_HD __host__ __device__ inline
#  else
#    define FB_HD static inline
#  endif
#  define FB_FMA(a, b, c) fmaf((a), (b), (c))
#  define FB_ADD(a, b)    ((float)((float)(a) + (float)(b)))
#  define FB_SUB(a, b)    ((float)((float)(a) - (float)(b)))
#  define FB_MUL(a, b)    ((float)((float)(a) * (float)(b)))
#  define FB_DIV(a, b)    ((float)((float)(a) / (float)(b)))
static inline int32_t fb_f2i_(float f) { int32_t i; memcpy(&i, &f, 4); return i; }
static inline float fb_i2f_(int32_t i) { float f; memcpy(&f, &i, 4); return f; }
#  define FB_F2I(f)       fb_f2i_(f)
#  define FB_I2F(i)       fb_i2f_(i)
/* operands are never NaN on the decoder path; ties (+0/-0) do not occur with a<b tests */
#  define FB_FMAX(a, b)   (((a) < (b)) ? (b) : (a))
#  define FB_FMIN(a, b)   (((b) < (a)) ? (b) : (a))
#endif

/* ---- constants of the reference ------------------------------------------------- */
#define FB_PHI_CLIP_LO   8.5e-8f          /* decoding_q.py:372, decoding.py:632 */
#define FB_PHI_CLIP_HI   16.635532f
#define FB_SOFTPLUS_THR  13.942385f       /* -(log(FLT_EPSILON) + 2), Eigen softplus */
#define FB_LLR_MAX       20.0f            /* decoding_q.py:51, decoding.py:320 */
#define FB_ATANH_CLIP    0.9999999f       /* 1 - 1e-7 in float32, decoding_q.py:49 */

/* ---- exp ------------------------------------------------------------------------- */
/* exp(x) for x >= -87.0 (no underflow handling), x <= 88.  Cephes-style: n = rint(x/ln2),
 * r = x - n*ln2 (two-step), degree-5 polynomial on r^2 plus 1 + r, scaled by 2^n through
 * the exponent field. */
FB_HD float fb_expf_core(float x) {
    const float magic = 12582912.0f;                 /* 1.5 * 2^23 : round-to-nearest-even */
    float t = FB_FMA(x, 1.44269504088896341f, magic);
    int32_t n = FB_F2I(t) - 0x4B400000;
    float fn = FB_SUB(t, magic);
    float r = FB_FMA(fn, -0.693359375f, x);
    r = FB_FMA(fn, 2.12194440e-4f, r);
    float p = 1.9875691500e-4f;
    p = FB_FMA(p, r, 1.3981999507e-3f);
    p = FB_FMA(p, r, 8.3334519073e-3f);
    p = FB_FMA(p, r, 4.1665795894e-2f);
    p = FB_FMA(p, r, 1.6666665459e-1f);
    p = FB_FMA(p, r, 5.0000001201e-1f);
    float r2 = FB_MUL(r, r);
    p = FB_FMA(p, r2, r);
    p = FB_ADD(p, 1.0f);
    return FB_I2F(FB_F2I(p) + (int32_t)((uint32_t)n << 23));
}

/* exp(x) for any finite x <= 88; arguments below -87 are clamped (exp(-87) = 1.6e-38 is the
 * smallest value returned, still a normal float32). */
FB_HD float fb_expf(float x) {
    return fb_expf_core(FB_FMAX(x, -87.0f));
}

/* ---- log ------------------------------------------------------------------------- */
/* log(x) for positive normal x.  Cephes-style: x = m * 2^e with m in [sqrt(1/2), sqrt(2)),
 * f = m - 1, log(1+f) = f - f^2/2 + f^3 P(f), plus e*ln2 split in two parts. */
FB_HD float fb_logf(float x) {
    int32_t ix = FB_F2I(x);
    int32_t eb = (ix - 0x3f3504f3) & (int32_t)0xff800000;   /* e * 2^23 */
    float m = FB_I2F(ix - eb);
    float fe = (float)eb;                                   /* exact: |e| <= 128 */
    float f = FB_SUB(m, 1.0f);
    float z = FB_MUL(f, f);
    float p = 7.0376836292e-2f;
    p = FB_FMA(p, f, -1.1514610310e-1f);
    p = FB_FMA(p, f, 1.1676998740e-1f);
    p = FB_FMA(p, f, -1.2420140846e-1f);
    p = FB_FMA(p, f, 1.4249322787e-1f);
    p = FB_FMA(p, f, -1.6668057665e-1f);
    p = FB_FMA(p, f, 2.0000714765e-1f);
    p = FB_FMA(p, f, -2.4999993993e-1f);
    p = FB_FMA(p, f, 3.3333331174e-1f);
    float y = FB_MUL(FB_MUL(p, f), z);                      /* f^3 P(f) */
    y = FB_FMA(fe, -2.12194440e-4f * 1.1920928955078125e-7f, y);      /* e * ln2_lo (constants carry 2^-23) */
    y = FB_FMA(z, -0.5f, y);
    float r = FB_ADD(f, y);
    return FB_FMA(fe, 0.693359375f * 1.1920928955078125e-7f, r);      /* + e * ln2_hi */
}

/* crude reciprocal (relative error < 1e-3) used only to scale a half-ulp correction */
FB_HD float fb_rcp_crude(float u) {
    float y = FB_I2F(0x7EF311C7 - FB_F2I(u));
    float t = FB_FMA(-u, y, 2.0f);
    y = FB_MUL(y, t);
    t = FB_FMA(-u, y, 2.0f);
    return FB_MUL(y, t);
}

/* log1p(e) for e > 0 : log(u) + c/u with u = fl(1+e), c = the rounding error of that sum */
FB_HD float fb_log1pf_pos(float e) {
    float u = FB_ADD(1.0f, e);
    float hi = FB_FMAX(e, 1.0f);
    float lo = FB_FMIN(e, 1.0f);
    float c = FB_SUB(lo, FB_SUB(u, hi));              /* Fast2Sum error term (exact) */
    float l = fb_logf(u);
    return FB_FMA(c, fb_rcp_crude(u), l);
}

/* ---- TensorFlow composites ------------------------------------------------------- */
/* log1p(e) for e >= 1: log(fl(1 + e)); the rounding of the sum costs at most half an ulp */
FB_HD float fb_log1pf_ge1(float e) {
    return fb_logf(FB_ADD(1.0f, e));
}

/* tf.math.softplus */
FB_HD float fb_softplusf(float x) {
    float xc = FB_FMIN(x, FB_SOFTPLUS_THR);                 /* keeps exp finite; unused when x is large */
    float e = fb_expf(xc);
    float l = fb_log1pf_pos(e);
    float r = (x < -FB_SOFTPLUS_THR) ? e : l;
    return (x > FB_SOFTPLUS_THR) ? x : r;
}

/* tf.reduce_logsumexp over the two values (a, b); both finite. */
FB_HD float fb_logaddexpf(float a, float b) {
    float mx = FB_FMAX(a, b);
    float mn = FB_FMIN(a, b);
    float t = fb_expf(FB_SUB(mn, mx));                /* the larger term is exp(0) = 1 */
    float s = FB_ADD(1.0f, t);
    return FB_ADD(fb_logf(s), mx);
}

/* quaternary decoder phi, decoding_q.py:365-373: softplus(x) - log(exp(x) - 1) after clipping */
FB_HD float fb_phi4f(float x) {
    x = FB_FMIN(FB_FMAX(x, FB_PHI_CLIP_LO), FB_PHI_CLIP_HI);
    float e = fb_expf_core(x);                              /* e >= 1 */
    float sp = (x > FB_SOFTPLUS_THR) ? x : fb_log1pf_ge1(e);
    return FB_SUB(sp, fb_logf(FB_SUB(e, 1.0f)));
}

/* binary decoder phi, decoding.py:625-633: log(exp(x) + 1) - log(exp(x) - 1) after clipping */
FB_HD float fb_phi2f(float x) {
    x = FB_FMIN(FB_FMAX(x, FB_PHI_CLIP_LO), FB_PHI_CLIP_HI);
    float e = fb_expf_core(x);
    return FB_SUB(fb_logf(FB_ADD(e, 1.0f)), fb_logf(FB_SUB(e, 1.0f)));
}

/* tanh: rational approximation x*P(x^2)/Q(x^2) on the clamped argument (the scheme Eigen's
 * float tanh, i.e. the TF CPU kernel, uses).  Q stays in [4.8e-3, 0.91], so the quotient is
 * formed branch-free with a fixed sequence: bit-trick seed, one Newton step (1.4e-2), then the
 * series 1/(1-e) = 1 + e + e^2 + e^3. */
FB_HD float fb_tanhf(float x) {
    float xc = FB_FMIN(FB_FMAX(x, -7.90531110763549805f), 7.90531110763549805f);
    float x2 = FB_MUL(xc, xc);
    float p = -2.76076847742355e-16f;
    p = FB_FMA(p, x2, 2.00018790482477e-13f);
    p = FB_FMA(p, x2, -8.60467152213735e-11f);
    p = FB_FMA(p, x2, 5.12229709037114e-08f);
    p = FB_FMA(p, x2, 1.48572235717979e-05f);
    p = FB_FMA(p, x2, 6.37261928875436e-04f);
    p = FB_FMA(p, x2, 4.89352455891786e-03f);
    p = FB_MUL(p, xc);
    float q = 1.19825839466702e-06f;
    q = FB_FMA(q, x2, 1.18534705686654e-04f);
    q = FB_FMA(q, x2, 2.26843463243900e-03f);
    q = FB_FMA(q, x2, 4.89352518554385e-03f);
    float y = FB_I2F(0x7EF311C7 - FB_F2I(q));
    y = FB_MUL(y, FB_FMA(-q, y, 2.0f));
    float e = FB_FMA(-q, y, 1.0f);
    float r0 = FB_MUL(p, y);
    float t = FB_FMA(e, e, e);
    t = FB_FMA(t, e, e);
    return FB_FMA(r0, t, r0);
}

/* atanh for |x| <= 1 - 1e-7 (tanh check-node variant, decoding_q.py:356-361):
 * 0.5 * (log(1 + x) - log(1 - x)) */
FB_HD float fb_atanhf(float x) {
    float a = fb_logf(FB_ADD(1.0f, x));
    float b = fb_logf(FB_SUB(1.0f, x));
    return FB_MUL(0.5f, FB_SUB(a, b));
}

/* ================================================================================================
 * SFU arithmetic (FBGNN_MATH_SFU): exp, log and reciprocal on the GPU's special-function unit -- MUFU.EX2
 * (ex2.approx), MUFU.LG2 (lg2.approx), MUFU.RCP (rcp.approx) -- with every formula arranged so that the
 * MUFU inputs fall in finite sets.  The hardware functions are then TABLES: the repository carries them as
 * measured on a B200 (tests/golden/sfu_b200_*.xz, written by tools/dump_sfu_tables.py), the CPU oracle
 * looks the values up, and the CUDA kernels stay bit-identical to the oracle in this arithmetic too.
 *
 *   2^(x c): n = round(x c) from one FMA against the 1.5 * 2^23 constant, then u = FMA(x, c, 1 - n) is the
 *            fraction plus one, rounded once: u in [0.5, 1.5], 12 582 913 float32 values.  MUFU.EX2(u) =
 *            2 * 2^frac, and n - 1 goes into the exponent field.  Five instructions; exp(x) is c = log2(e),
 *            exp(-x) and exp(-2x) only change the constant.
 *   log    : of 1 + t, t in [0, 1]: lg2 on [1, 2] directly.  Of 1 - t: every such float32 is a multiple of 2^-24
 *            in [0, 1], so lg2 sees k 2^-24, k = 1 .. 2^24, directly as well -- no exponent split in either case.
 *            (General positive arguments -- atanh only -- split off the exponent; mantissa in [sqrt(1/2), sqrt(2)).)
 *   phi(x) = softplus(x) - log(expm1(x)) with softplus(x) = x + log(1 + t), log(expm1(x)) = x + log(1 - t),
 *            t = exp(-x); the two terms are rounded separately, as the reference's are.  1 - t is kept >= 2^-23,
 *            which bounds phi by 24 ln 2 = 16.635532, the reference's phi(8.5e-8).
 *   softplus(x) = max(x, 0) + log(1 + exp(-|x|));  logaddexp(a, b) = max + log(1 + exp(min - max)).
 *   tanh(x) = sign(x) (1 - t) / (1 + t), t = exp(-2|x|), MUFU.RCP on [1, 2] (2^23 + 1 values).
 *
 * Accuracy: 2-3 ulp per exp / log instead of 1.  The saturation constants of phi (phi(<= 8.5e-8) = 16.635532,
 * phi(>= 16.635532) = 0: the reference's known answers), softplus(x < -thr) = exp(x), softplus(x > thr) = x and
 * the rule that a second term below e^-17.5 leaves logaddexp at its larger argument are part of this
 * specification, not consequences of rounding.
 * ================================================================================================ */
#define FB_SFU_EX2_BASE   0x3F000000          /* bits of u for table entry 0: 0.5                          */
#define FB_SFU_EX2_COUNT  (0x00C00000 + 1)    /* consecutive float32 values up to and including 1.5        */
#define FB_SFU_LG2_BASE   0x3f3504f3          /* bits of the smallest mantissa, sqrt(1/2)                  */
#define FB_SFU_LG2_COUNT  (0x40000000 - 0x3f3504f3 + 1)   /* up to and including 2.0                       */
#define FB_SFU_LG2B_COUNT 11863284            /* k 2^-24 for k = 0 .. ceil(sqrt(1/2) 2^24) (entry 0 unused) */
#define FB_SFU_RCP_BASE   0x3F800000          /* q = 1.0                                                   */
#define FB_SFU_RCP_COUNT  ((1 << 23) + 1)     /* up to and including 2.0                                   */
#define FB_LOG2E          1.44269504088896341f
#define FB_LN2            0.693147180559945f

#if defined(__CUDA_ARCH__)
__device__ __forceinline__ float fb_mufu_ex2(float u) {
    float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(u)); return y;
}
__device__ __forceinline__ float fb_mufu_lg2(float m) {
    float y; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(m)); return y;
}
__device__ __forceinline__ float fb_mufu_rcp(float q) {
    float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(q)); return y;
}
#elif !defined(__CUDACC__)
/* host: the MUFU as measured on the hardware (tables installed through fb_sfu_set_tables) */
static const float *fb_sfu_ex2_tab = 0, *fb_sfu_lg2_tab = 0, *fb_sfu_lg2b_tab = 0, *fb_sfu_rcp_tab = 0;
static inline void fb_sfu_set_tables(const float *ex2_tab, const float *lg2_tab, const float *lg2b_tab,
                                     const float *rcp_tab) {
    fb_sfu_ex2_tab = ex2_tab; fb_sfu_lg2_tab = lg2_tab; fb_sfu_lg2b_tab = lg2b_tab; fb_sfu_rcp_tab = rcp_tab;
}
static inline float fb_mufu_ex2(float u) {
    int64_t i = (int64_t)FB_F2I(u) - FB_SFU_EX2_BASE;
    if (i < 0) i = 0;
    if (i >= FB_SFU_EX2_COUNT) i = FB_SFU_EX2_COUNT - 1;
    return fb_sfu_ex2_tab[i];
}
static inline float fb_mufu_lg2(float m) {
    int64_t i = (int64_t)FB_F2I(m) - FB_SFU_LG2_BASE;
    if (i < 0) {                                  /* below sqrt(1/2): the multiples of 2^-24 (1 - t) */
        int64_t k = (int64_t)(m * 16777216.0f);
        if (k < 1) k = 1;
        if (k >= FB_SFU_LG2B_COUNT) k = FB_SFU_LG2B_COUNT - 1;
        return fb_sfu_lg2b_tab[k];
    }
    if (i >= FB_SFU_LG2_COUNT) i = FB_SFU_LG2_COUNT - 1;
    return fb_sfu_lg2_tab[i];
}
static inline float fb_mufu_rcp(float q) {
    int64_t i = (int64_t)FB_F2I(q) - FB_SFU_RCP_BASE;
    if (i < 0) i = 0;
    if (i >= FB_SFU_RCP_COUNT) i = FB_SFU_RCP_COUNT - 1;
    return fb_sfu_rcp_tab[i];
}
#else
/* host side of a .cu file: never evaluated (the library has no CPU compute path) */
static inline float fb_mufu_ex2(float u) { (void)u; return 0.0f; }
static inline float fb_mufu_lg2(float m) { (void)m; return 0.0f; }
static inline float fb_mufu_rcp(float q) { (void)q; return 0.0f; }
#endif

/* 2^(x c) for -125 <= x c <= 126 */
FB_HD float fb_sfu_exp2s(float x, float c) {
    const float magic = 12582912.0f;                          /* 1.5 * 2^23: ulp 1 */
    float t = FB_FMA(x, c, 12582911.0f);                      /* magic + (n - 1), n = round(x c) */
    float fn = FB_SUB(t, magic);                              /* n - 1 */
    float u = FB_FMA(x, c, -fn);                              /* x c - n + 1, one rounding */
    float y = fb_mufu_ex2(u);
    return FB_I2F(FB_F2I(y) + (int32_t)((uint32_t)FB_F2I(t) << 23));
}
FB_HD float fb_sfu_expf_core(float x) { return fb_sfu_exp2s(x, FB_LOG2E); }
FB_HD float fb_sfu_expf(float x) { return fb_sfu_expf_core(FB_FMAX(x, -86.0f)); }

/* log(x) for positive normal x (general argument: exponent split) */
FB_HD float fb_sfu_logf(float x) {
    int32_t ix = FB_F2I(x);
    int32_t eb = (ix - 0x3f3504f3) & (int32_t)0xff800000;
    float m = FB_I2F(ix - eb);
    float fe = (float)eb;
    float l2 = fb_mufu_lg2(m);
    return FB_FMA(fe, FB_LN2 * 1.1920928955078125e-7f, FB_MUL(l2, FB_LN2));
}

FB_HD float fb_sfu_softplusf(float x) {
    float ax = FB_FMIN(FB_I2F(FB_F2I(x) & 0x7fffffff), 86.0f);
    float e = fb_sfu_exp2s(ax, -FB_LOG2E);                    /* exp(-|x|), 0 < e <= 1 */
    float r = FB_FMA(fb_mufu_lg2(FB_ADD(1.0f, e)), FB_LN2, FB_FMAX(x, 0.0f));
    r = (x < -FB_SOFTPLUS_THR) ? e : r;
    return (x > FB_SOFTPLUS_THR) ? x : r;
}

/* log(exp(a) + exp(b)) for mn - mx >= -17.5 (the caller's side of the specification handles the rest) */
FB_HD float fb_sfu_logaddexp_open(float mx, float d) {
    float t = fb_sfu_expf_core(d);                            /* 0 < t <= 1 */
    return FB_FMA(fb_mufu_lg2(FB_ADD(1.0f, t)), FB_LN2, mx);
}
FB_HD float fb_sfu_logaddexpf(float a, float b) {
    float mx = FB_FMAX(a, b);
    float mn = FB_FMIN(a, b);
    float d = FB_SUB(mn, mx);
    float f = fb_sfu_logaddexp_open(mx, FB_FMAX(d, -17.5f));
    return (d < -17.5f) ? FB_ADD(0.0f, mx) : f;
}

/* Variable-node update of the quaternary decoder in SFU arithmetic.  The outgoing messages of one side are
 *     num - logaddexp(-(l1 - a_k), -(ly - a_k))  =  num - ((a_k - min(l1, ly)) + log(1 + exp(-|ly - l1|)))
 * (l1 = lz for the x edges, lx for the z edges; a_k the incoming message of edge k): the correction term does not depend
 * on the edge, so it is evaluated ONCE per side and variable instead of once per edge -- two exp / log pairs per variable
 * node instead of 2 DV.  A correction below e^-17.5 is zero (as in logaddexp). */
FB_HD float fb_sfu_vn_corr(float l1, float ly) {
    float d = FB_SUB(ly, l1);
    d = FB_I2F(FB_F2I(d) | (int32_t)0x80000000);              /* -|ly - l1| */
    float f = fb_sfu_logaddexp_open(0.0f, FB_FMAX(d, -17.5f));
    return (d < -17.5f) ? 0.0f : f;
}
FB_HD float fb_sfu_vn_msg(float num, float a, float u, float corr) {      /* u = min(l1, ly) */
    return FB_SUB(num, FB_ADD(FB_SUB(a, u), corr));
}

/* phi on the open interval (8.5e-8, 16.635532), t = exp(-x):  softplus(x) = x + log(1 + t) and log(expm1(x)) =
 * x + log(1 - t), each rounded to float32 where the reference rounds them (at the magnitude of x), then subtracted --
 * the reference's phi with its float32 cancellation for large x reproduced, which the decoder's error rates depend
 * on (profiles/r02_ler_phi_forms.txt).  Never negative: lg2 >= 0 on [1, 2], <= 0 on (0, 1], and the two FMAs round
 * monotonically. */
FB_HD float fb_sfu_phi_open(float x) {
    float t = fb_sfu_exp2s(x, -FB_LOG2E);
    float la = fb_mufu_lg2(FB_ADD(1.0f, t));
    float lb = fb_mufu_lg2(FB_FMAX(FB_SUB(1.0f, t), 1.1920928955078125e-7f));
    return FB_SUB(FB_FMA(la, FB_LN2, x), FB_FMA(lb, FB_LN2, x));
}
FB_HD float fb_sfu_phi4_open(float x) { return fb_sfu_phi_open(x); }
FB_HD float fb_sfu_phi2_open(float x) { return fb_sfu_phi_open(x); }
FB_HD float fb_sfu_phi4f(float x) {
    float f = fb_sfu_phi_open(FB_FMIN(FB_FMAX(x, FB_PHI_CLIP_LO), FB_PHI_CLIP_HI));
    f = (x <= FB_PHI_CLIP_LO) ? FB_PHI_CLIP_HI : f;
    return (x >= FB_PHI_CLIP_HI) ? 0.0f : f;
}
FB_HD float fb_sfu_phi2f(float x) { return fb_sfu_phi4f(x); }

/* tanh(x) = sign(x) (1 - t) / (1 + t), t = exp(-2 |x|); |x| >= 10 gives exactly 1 */
FB_HD float fb_sfu_tanhf(float x) {
    float ax = FB_FMIN(FB_I2F(FB_F2I(x) & 0x7fffffff), 10.0f);
    float t = fb_sfu_exp2s(ax, -2.0f * FB_LOG2E);
    float r = FB_MUL(FB_SUB(1.0f, t), fb_mufu_rcp(FB_ADD(1.0f, t)));
    return FB_I2F(FB_F2I(r) | (FB_F2I(x) & (int32_t)0x80000000));
}
/* atanh for |x| <= 1 - 1e-7 */
FB_HD float fb_sfu_atanhf(float x) {
    return FB_MUL(0.5f, FB_SUB(fb_sfu_logf(FB_ADD(1.0f, x)), fb_sfu_logf(FB_SUB(1.0f, x))));
}

#if defined(__CUDACC__) && (!defined(__CUDA_ARCH__) || __CUDA_ARCH__ >= 1000)
/* ---- paired SFU arithmetic (device only, sm_100 and later) -----------------------------------------------------------------------
 * float2 forms of the SFU functions above for sm_100's packed FP32 instructions fma.rn.f32x2 / add.rn.f32x2 /
 * mul.rn.f32x2 (SASS FFMA2 / FADD2 / FMUL2): two float32 operations in one issue slot, each lane rounded to nearest
 * exactly as the scalar __fmaf_rn / __fadd_rn / __fmul_rn round it, without flushing subnormals.  Each lane performs
 * the scalar function's IEEE operations in the same order with the same constants; the MUFU, the exponent splices,
 * min / max and the compares stay scalar per lane.  The scalar functions remain the specification (the CPU oracle
 * evaluates those), and tests/test_gpu_sfu_pairs.py holds every paired form to its scalar form bit for bit.
 * a - b is formed as a + (-b), which IEEE-754 defines it to be (signed zeros included). */
__device__ __forceinline__ float2 fb2(float a, float b) { return make_float2(a, b); }
__device__ __forceinline__ float2 fb2s(float a) { return make_float2(a, a); }
__device__ __forceinline__ float2 fb2_neg(float2 a) { return make_float2(-a.x, -a.y); }
#define FB_FMA2(a, b, c) __ffma2_rn((a), (b), (c))
#define FB_ADD2(a, b)    __fadd2_rn((a), (b))
#define FB_SUB2(a, b)    __fadd2_rn((a), fb2_neg(b))
#define FB_MUL2(a, b)    __fmul2_rn((a), (b))

__device__ __forceinline__ float2 fb_sfu_exp2s2(float2 x, float c) {
    const float2 t = FB_FMA2(x, fb2s(c), fb2s(12582911.0f));
    const float2 fn = FB_SUB2(t, fb2s(12582912.0f));
    const float2 u = FB_FMA2(x, fb2s(c), fb2_neg(fn));
    const float yx = fb_mufu_ex2(u.x), yy = fb_mufu_ex2(u.y);
    return fb2(FB_I2F(FB_F2I(yx) + (int32_t)((uint32_t)FB_F2I(t.x) << 23)),
               FB_I2F(FB_F2I(yy) + (int32_t)((uint32_t)FB_F2I(t.y) << 23)));
}
__device__ __forceinline__ float2 fb_sfu_logaddexp_open2(float2 mx, float2 d) {
    const float2 s = FB_ADD2(fb2s(1.0f), fb_sfu_exp2s2(d, FB_LOG2E));
    return FB_FMA2(fb2(fb_mufu_lg2(s.x), fb_mufu_lg2(s.y)), fb2s(FB_LN2), mx);
}
__device__ __forceinline__ float2 fb_sfu_softplusf2(float2 x) {
    const float2 ax = fb2(FB_FMIN(FB_I2F(FB_F2I(x.x) & 0x7fffffff), 86.0f), FB_FMIN(FB_I2F(FB_F2I(x.y) & 0x7fffffff), 86.0f));
    const float2 e = fb_sfu_exp2s2(ax, -FB_LOG2E);
    const float2 s = FB_ADD2(fb2s(1.0f), e);
    float2 r = FB_FMA2(fb2(fb_mufu_lg2(s.x), fb_mufu_lg2(s.y)), fb2s(FB_LN2), fb2(FB_FMAX(x.x, 0.0f), FB_FMAX(x.y, 0.0f)));
    r.x = (x.x < -FB_SOFTPLUS_THR) ? e.x : r.x;
    r.y = (x.y < -FB_SOFTPLUS_THR) ? e.y : r.y;
    return fb2((x.x > FB_SOFTPLUS_THR) ? x.x : r.x, (x.y > FB_SOFTPLUS_THR) ? x.y : r.y);
}
__device__ __forceinline__ float2 fb_sfu_vn_corr2(float2 l1, float2 ly) {
    float2 d = FB_SUB2(ly, l1);
    d = fb2(FB_I2F(FB_F2I(d.x) | (int32_t)0x80000000), FB_I2F(FB_F2I(d.y) | (int32_t)0x80000000));
    const float2 f = fb_sfu_logaddexp_open2(fb2s(0.0f), fb2(FB_FMAX(d.x, -17.5f), FB_FMAX(d.y, -17.5f)));
    return fb2((d.x < -17.5f) ? 0.0f : f.x, (d.y < -17.5f) ? 0.0f : f.y);
}
__device__ __forceinline__ float2 fb_sfu_vn_msg2(float2 num, float2 a, float2 u, float2 corr) {
    return FB_SUB2(num, FB_ADD2(FB_SUB2(a, u), corr));
}
__device__ __forceinline__ float2 fb_sfu_phi_open2(float2 x) {
    const float2 t = fb_sfu_exp2s2(x, -FB_LOG2E);
    const float2 sa = FB_ADD2(fb2s(1.0f), t), sb = FB_SUB2(fb2s(1.0f), t);
    const float2 la = fb2(fb_mufu_lg2(sa.x), fb_mufu_lg2(sa.y));
    const float2 lb = fb2(fb_mufu_lg2(FB_FMAX(sb.x, 1.1920928955078125e-7f)), fb_mufu_lg2(FB_FMAX(sb.y, 1.1920928955078125e-7f)));
    return FB_SUB2(FB_FMA2(la, fb2s(FB_LN2), x), FB_FMA2(lb, fb2s(FB_LN2), x));
}
__device__ __forceinline__ float2 fb_sfu_tanhf2(float2 x) {
    const float2 ax = fb2(FB_FMIN(FB_I2F(FB_F2I(x.x) & 0x7fffffff), 10.0f), FB_FMIN(FB_I2F(FB_F2I(x.y) & 0x7fffffff), 10.0f));
    const float2 t = fb_sfu_exp2s2(ax, -2.0f * FB_LOG2E);
    const float2 q = FB_ADD2(fb2s(1.0f), t);
    const float2 r = FB_MUL2(FB_SUB2(fb2s(1.0f), t), fb2(fb_mufu_rcp(q.x), fb_mufu_rcp(q.y)));
    return fb2(FB_I2F(FB_F2I(r.x) | (FB_F2I(x.x) & (int32_t)0x80000000)),
               FB_I2F(FB_F2I(r.y) | (FB_F2I(x.y) & (int32_t)0x80000000)));
}
#endif

#if !defined(__CUDACC__)
/* ---- host-side arithmetic selection (the CPU oracle): 0 = exact (default), 1 = SFU ------------ */
static int fb_math_mode = 0;
static inline float fb_m_softplusf(float x) { return fb_math_mode ? fb_sfu_softplusf(x) : fb_softplusf(x); }
static inline float fb_m_logaddexpf(float a, float b) { return fb_math_mode ? fb_sfu_logaddexpf(a, b) : fb_logaddexpf(a, b); }
static inline float fb_m_phi4f(float x) { return fb_math_mode ? fb_sfu_phi4f(x) : fb_phi4f(x); }
static inline float fb_m_phi2f(float x) { return fb_math_mode ? fb_sfu_phi2f(x) : fb_phi2f(x); }
static inline float fb_m_tanhf(float x) { return fb_math_mode ? fb_sfu_tanhf(x) : fb_tanhf(x); }
static inline float fb_m_atanhf(float x) { return fb_math_mode ? fb_sfu_atanhf(x) : fb_atanhf(x); }
#endif

#endif /* FBGNN_FB_MATH_H */
