/*
 * nmch_oracle.c -- CPU oracle for the Heston Monte-Carlo hot path.
 *
 * TEST INFRASTRUCTURE ONLY (see nmch_oracle.h).  Plain C99 + OpenMP; single
 * precision where the reference is single precision, explicit fmaf() where
 * nvcc contracts the reference's expressions (SURVEY.md Appendix B, read off
 * the SASS of FE_k2<XORWOW> at sm_100).
 *
 * Parity status: pinned -- see tests/test_oracle_*.py (Philox KATs, cuRAND
 * host build, reference CUDA build fixtures).  Host libm (logf/sinf/cosf)
 * differs from the device in the last bits (cuRAND's device Box-Muller uses
 * __sincosf, curand_normal.h:76-83), so float outputs are compared with the
 * tolerances written in the tests; integer streams are bit exact.
 */
#include "nmch_oracle.h"

#include <complex.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

/* ======================================================================== */
/* Philox4x32-10  (curand_philox4x32_x.h:88-91, 160-192; Random123)          */
/* ======================================================================== */
#define PHILOX_M0 0xD2511F53u
#define PHILOX_M1 0xCD9E8D57u
#define PHILOX_W0 0x9E3779B9u
#define PHILOX_W1 0xBB67AE85u

void orc_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4])
{
    uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3];
    uint32_t k0 = key[0], k1 = key[1];
    for (int round = 0; round < 10; ++round) {
        uint64_t p0 = (uint64_t)PHILOX_M0 * c0;
        uint64_t p1 = (uint64_t)PHILOX_M1 * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        uint32_t n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += PHILOX_W0; k1 += PHILOX_W1;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

/* ======================================================================== */
/* XORWOW  (curand_kernel.h:863-874 step, :800-825 init, :721-736 skip)      */
/* ======================================================================== */
static inline void xorwow_advance_v(uint32_t v[5])
{
    uint32_t t = v[0] ^ (v[0] >> 2);
    v[0] = v[1]; v[1] = v[2]; v[2] = v[3]; v[3] = v[4];
    v[4] = (v[4] ^ (v[4] << 4)) ^ (t ^ (t << 1));
}

/* 160x160 GF(2) matrices as 160 rows of 5 words; row b is the image of the
 * unit vector e_b, so   v*M = XOR of the rows selected by the set bits of v
 * (the convention of __curand_matvec_inplace, curand_kernel.h:315-334).
 * cuRAND ships these as tables (curand_precalc.h); the oracle derives them:
 * seq[m] advances by 2^67 * 4^m draws, off[m] by 4^m draws. */
typedef struct { uint32_t row[160][5]; } gf2mat_t;

static void gf2_matvec(const uint32_t v[5], const gf2mat_t *M, uint32_t out[5])
{
    uint32_t r[5] = {0, 0, 0, 0, 0};
    for (int i = 0; i < 5; ++i)
        for (int j = 0; j < 32; ++j)
            if (v[i] & (1u << j))
                for (int k = 0; k < 5; ++k) r[k] ^= M->row[i * 32 + j][k];
    memcpy(out, r, sizeof r);
}

static void gf2_square(const gf2mat_t *M, gf2mat_t *out)
{
    gf2mat_t tmp;
    for (int b = 0; b < 160; ++b) gf2_matvec(M->row[b], M, tmp.row[b]);
    *out = tmp;
}

static gf2mat_t g_seq[32], g_off[32];
static int g_mats_ready = 0;

static void xorwow_build_matrices(void)
{
    if (g_mats_ready) return;
#ifdef _OPENMP
#pragma omp critical(orc_mats)
#endif
    {
        if (!g_mats_ready) {
            gf2mat_t cur;
            for (int b = 0; b < 160; ++b) {
                uint32_t e[5] = {0, 0, 0, 0, 0};
                e[b / 32] = 1u << (b % 32);
                xorwow_advance_v(e);
                memcpy(cur.row[b], e, sizeof e);
            }
            /* off[m] = T^(4^m), m = 0..31 ; after 64 squarings cur = T^(2^64) */
            for (int m = 0; m < 32; ++m) {
                g_off[m] = cur;
                gf2_square(&cur, &cur);
                gf2_square(&cur, &cur);
            }
            /* three more squarings: T^(2^67) */
            gf2_square(&cur, &cur);
            gf2_square(&cur, &cur);
            gf2_square(&cur, &cur);
            for (int m = 0; m < 32; ++m) {
                g_seq[m] = cur;
                gf2_square(&cur, &cur);
                gf2_square(&cur, &cur);
            }
            g_mats_ready = 1;
        }
    }
}

static void xorwow_init(orc_rng_t *s, uint64_t seed, uint64_t subsequence, uint64_t offset)
{
    xorwow_build_matrices();
    /* seed scramble, curand_kernel.h:807-818 */
    uint32_t s0 = (uint32_t)seed ^ 0xaad26b49u;
    uint32_t s1 = (uint32_t)(seed >> 32) ^ 0xf7dcefddu;
    uint32_t t0 = 1099087573u * s0;
    uint32_t t1 = 2591861531u * s1;
    s->d = 6615241u + t1 + t0;
    s->v[0] = 123456789u + t0;
    s->v[1] = 362436069u ^ t0;
    s->v[2] = 521288629u + t1;
    s->v[3] = 88675123u ^ t1;
    s->v[4] = 5783321u + t0;
    /* subsequence skip: 2-bit digits, LSB first (curand_kernel.h:721-736) */
    uint64_t x = subsequence;
    for (int m = 0; x; ++m, x >>= 2)
        for (unsigned t = 0; t < (x & 3u); ++t) gf2_matvec(s->v, &g_seq[m], s->v);
    /* offset skip (curand_kernel.h:703-719) */
    x = offset;
    for (int m = 0; x; ++m, x >>= 2)
        for (unsigned t = 0; t < (x & 3u); ++t) gf2_matvec(s->v, &g_off[m], s->v);
    s->d += 362437u * (uint32_t)offset;
}

static inline uint32_t xorwow_next(orc_rng_t *s)
{
    xorwow_advance_v(s->v);
    s->d += 362437u;
    return s->v[4] + s->d;
}

/* ======================================================================== */
/* MRG32k3a  (L'Ecuyer 1999; cuRAND curand_kernel.h:1061-1150 generator,       */
/* :1274-1300 init, :1181-1225 skip-ahead by 3x3 matrix powers mod m)          */
/* ======================================================================== */
#define MRG_M1 4294967087ull
#define MRG_M2 4294944443ull
typedef struct { uint64_t a[3][3]; } mat3_t;

static void mat3_mul(const mat3_t *A, const mat3_t *B, uint64_t m, mat3_t *out)
{
    mat3_t t;
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            unsigned __int128 acc = 0;
            for (int k = 0; k < 3; ++k) acc += (unsigned __int128)A->a[i][k] * B->a[k][j];
            t.a[i][j] = (uint64_t)(acc % m);
        }
    *out = t;
}

static void mat3_pow(const mat3_t *A, uint64_t e, uint64_t m, mat3_t *out)
{
    mat3_t r = {{{1, 0, 0}, {0, 1, 0}, {0, 0, 1}}}, b = *A;
    while (e) {
        if (e & 1ull) mat3_mul(&b, &r, m, &r);
        mat3_mul(&b, &b, m, &b);
        e >>= 1;
    }
    *out = r;
}

static void mat3_apply(const mat3_t *A, uint32_t v[3], uint64_t m)
{
    uint64_t t[3];
    for (int k = 0; k < 3; ++k) {
        unsigned __int128 acc = 0;
        for (int j = 0; j < 3; ++j) acc += (unsigned __int128)A->a[k][j] * v[j];
        t[k] = (uint64_t)(acc % m);
    }
    for (int k = 0; k < 3; ++k) v[k] = (uint32_t)t[k];
}

static const mat3_t MRG_A1 = {{{0, 1, 0}, {0, 0, 1}, {MRG_M1 - 810728ull, 1403580ull, 0}}};
static const mat3_t MRG_A2 = {{{0, 1, 0}, {0, 0, 1}, {MRG_M2 - 1370589ull, 0, 527612ull}}};

static void mrg_skip(orc_rng_t *s, int log2_stride, uint64_t n)
{   /* advance by n * 2^log2_stride draws: (A^(2^log2_stride))^n */
    mat3_t b1 = MRG_A1, b2 = MRG_A2, p;
    for (int i = 0; i < log2_stride; ++i) { mat3_mul(&b1, &b1, MRG_M1, &b1); mat3_mul(&b2, &b2, MRG_M2, &b2); }
    mat3_pow(&b1, n, MRG_M1, &p); mat3_apply(&p, s->s1, MRG_M1);
    mat3_pow(&b2, n, MRG_M2, &p); mat3_apply(&p, s->s2, MRG_M2);
}

static void mrg_init(orc_rng_t *s, uint64_t seed, uint64_t subsequence, uint64_t offset)
{
    for (int i = 0; i < 3; ++i) { s->s1[i] = 12345u; s->s2[i] = 12345u; }
    if (seed != 0ull) {                                       /* curand_kernel.h:1284-1293 */
        const uint64_t x1 = (uint32_t)seed ^ 0x55555555u;
        const uint64_t x2 = (uint32_t)((seed >> 32) ^ 0xAAAAAAAAu);
        s->s1[0] = (uint32_t)((x1 * s->s1[0]) % MRG_M1);
        s->s1[1] = (uint32_t)((x2 * s->s1[1]) % MRG_M1);
        s->s1[2] = (uint32_t)((x1 * s->s1[2]) % MRG_M1);
        s->s2[0] = (uint32_t)((x2 * s->s2[0]) % MRG_M2);
        s->s2[1] = (uint32_t)((x1 * s->s2[1]) % MRG_M2);
        s->s2[2] = (uint32_t)((x2 * s->s2[2]) % MRG_M2);
    }
    if (subsequence) mrg_skip(s, 76, subsequence);            /* subsequences are 2^76 draws apart */
    if (offset) mrg_skip(s, 0, offset);
}

static inline double mrg_next(orc_rng_t *s)
{   /* one draw in [1, m1]: p1 - p2 (+ m1 if <= 0) */
    const int64_t p1 = (int64_t)((1403580ull * s->s1[1] + 810728ull * (MRG_M1 - s->s1[0])) % MRG_M1);
    s->s1[0] = s->s1[1]; s->s1[1] = s->s1[2]; s->s1[2] = (uint32_t)p1;
    const int64_t p2 = (int64_t)((527612ull * s->s2[2] + 1370589ull * (MRG_M2 - s->s2[0])) % MRG_M2);
    s->s2[0] = s->s2[1]; s->s2[1] = s->s2[2]; s->s2[2] = (uint32_t)p2;
    return (p1 <= p2) ? (double)(p1 - p2 + (int64_t)MRG_M1) : (double)(p1 - p2);
}
#define MRG_NORM 2.3283065498378288e-10
#define MRG_BITS_NORM 1.000000048662

/* ======================================================================== */
/* generic stream front-end                                                  */
/* ======================================================================== */
static void philox_incr(uint32_t c[4], uint64_t n)
{   /* Philox_State_Incr(s, n), curand_philox4x32_x.h:107-122 */
    uint32_t nlo = (uint32_t)n, nhi = (uint32_t)(n >> 32);
    c[0] += nlo;
    if (c[0] < nlo) nhi++;
    c[1] += nhi;
    if (nhi <= c[1]) return;
    if (++c[2]) return;
    ++c[3];
}

void orc_rng_init(orc_rng_t *s, int kind, uint64_t seed, uint64_t subsequence, uint64_t offset)
{
    memset(s, 0, sizeof *s);
    s->kind = kind;
    if (kind == ORC_RNG_XORWOW) {
        xorwow_init(s, seed, subsequence, offset);
    } else if (kind == ORC_RNG_MRG32K3A) {
        mrg_init(s, seed, subsequence, offset);
    } else if (kind == ORC_RNG_PHILOX_DENSE) {
        s->key[0] = (uint32_t)seed;
        s->key[1] = (uint32_t)(seed >> 32);
        s->ctr[2] = (uint32_t)subsequence;
        s->ctr[3] = (uint32_t)(subsequence >> 32);
        s->dense_step = offset / 2;                          /* two logical draws per step */
    } else {
        /* curand_init for Philox, curand_kernel.h:1022-1037, skipahead :971-981 */
        s->key[0] = (uint32_t)seed;
        s->key[1] = (uint32_t)(seed >> 32);
        s->ctr[2] = (uint32_t)subsequence;
        s->ctr[3] = (uint32_t)(subsequence >> 32);
        s->pos = (int)(offset & 3u);
        philox_incr(s->ctr, offset / 4);
        orc_philox4x32_10(s->ctr, s->key, s->out);
    }
}

uint32_t orc_rng_next(orc_rng_t *s)
{
    if (s->kind == ORC_RNG_XORWOW) return xorwow_next(s);
    if (s->kind == ORC_RNG_MRG32K3A) return (uint32_t)(mrg_next(s) * MRG_BITS_NORM);    /* curand_kernel.h:1161-1167 */
    /* curand(), curand_kernel.h:888-912 */
    uint32_t r = s->out[s->pos++];
    if (s->pos == 4) {
        philox_incr(s->ctr, 1);
        orc_philox4x32_10(s->ctr, s->key, s->out);
        s->pos = 0;
    }
    return r;
}

/* ======================================================================== */
/* float transforms                                                          */
/* ======================================================================== */
#define TWO_POW32_INV      2.3283064e-10f
#define TWO_POW32_INV_2PI  (2.3283064e-10f * 6.2831855f)
#define TWO_POW53_INV_D    1.1102230246251565e-16

static inline float uniform_from_u32(uint32_t x)
{   /* _curand_uniform, curand_uniform.h:69-72 ; nvcc contracts to one FFMA */
    return fmaf((float)x, TWO_POW32_INV, TWO_POW32_INV / 2.0f);
}

float orc_uniform(orc_rng_t *s)
{
    if (s->kind == ORC_RNG_MRG32K3A) return (float)(mrg_next(s) * MRG_NORM);             /* curand_uniform.h:177-180 */
    return uniform_from_u32(orc_rng_next(s));
}

static inline void box_muller(uint32_t x, uint32_t y, float *gx, float *gy)
{   /* _curand_box_muller, curand_normal.h:70-87 : .x pairs with sin */
    float u = fmaf((float)x, TWO_POW32_INV, TWO_POW32_INV / 2);
    float v = fmaf((float)y, TWO_POW32_INV_2PI, TWO_POW32_INV_2PI / 2);
    float s = sqrtf(-2.0f * logf(u));
    *gx = sinf(v) * s;
    *gy = cosf(v) * s;
}

void orc_normal2(orc_rng_t *s, float *gx, float *gy)
{   /* curand_normal2, curand_normal.h:405-408, 424-427 */
    if (s->kind == ORC_RNG_PHILOX_DENSE) {                   /* restates dense_fields + fe_step_dense of fe_kernels.cu */
        const uint64_t blk = s->dense_step / 3;
        const int phase = (int)(s->dense_step % 3);
        const uint32_t ctr[4] = {(uint32_t)blk, (uint32_t)(blk >> 32), s->ctr[2], s->ctr[3]};
        uint32_t w[4];
        orc_philox4x32_10(ctr, s->key, w);
        uint32_t k23, k19;
        if (phase == 0) { k23 = w[0] >> 9; k19 = ((w[0] & 0x1ffu) << 10) | (w[1] >> 22); }
        else if (phase == 1) { k23 = ((w[1] & 0x3fffffu) << 1) | (w[2] >> 31); k19 = (w[2] >> 12) & 0x7ffffu; }
        else { k23 = ((w[2] & 0xfffu) << 11) | (w[3] >> 21); k19 = (w[3] >> 2) & 0x7ffffu; }
        const float u = ((float)k23 + 0.5f) * 1.1920929e-07f;            /* 2^-23 */
        const float ang = (1.0f + (float)k19 * 1.9073486e-06f) * 6.2831855f;  /* 2^-19 */
        const float r = sqrtf(-2.0f * logf(u));
        *gx = sinf(ang) * r;
        *gy = cosf(ang) * r;
        s->dense_step++;
        return;
    }
    if (s->kind == ORC_RNG_MRG32K3A) {                       /* curand_box_muller_mrg, curand_normal.h:89-108 */
        const float x = orc_uniform(s);
        const float y = orc_uniform(s) * 6.2831855f;
        const float r = sqrtf(-2.0f * logf(x));
        *gx = sinf(y) * r;
        *gy = cosf(y) * r;
        return;
    }
    uint32_t x = orc_rng_next(s);
    uint32_t y = orc_rng_next(s);
    box_muller(x, y, gx, gy);
}

float orc_normal(orc_rng_t *s)
{   /* curand_normal (cached pair), curand_normal.h:313-326 / 345-358 */
    if (s->bm_flag != 1) {
        float gx, gy;
        orc_normal2(s, &gx, &gy);
        s->bm_extra = gy;
        s->bm_flag = 1;
        return gx;
    }
    s->bm_flag = 0;
    return s->bm_extra;
}

double orc_normal_double(orc_rng_t *s)
{   /* curand_normal_double, curand_normal.h:581-596 / 615-627 ;
       _curand_box_muller_double :110-133 (host branch: sin/cos(v*pi)) */
    if (s->bm_flag_d != 1 && s->kind == ORC_RNG_MRG32K3A) {  /* curand_box_muller_mrg_double, curand_normal.h:135-155 */
        const double x = mrg_next(s) * MRG_NORM;
        const double y = mrg_next(s) * MRG_NORM * 2.0;
        const double r = sqrt(-2.0 * log(x));
        s->bm_extra_d = cos(y * 3.1415926535897932) * r;
        s->bm_flag_d = 1;
        return sin(y * 3.1415926535897932) * r;
    }
    if (s->bm_flag_d != 1) {
        uint32_t x0 = orc_rng_next(s), x1 = orc_rng_next(s);
        uint32_t y0 = orc_rng_next(s), y1 = orc_rng_next(s);
        uint64_t zx = (uint64_t)x0 ^ ((uint64_t)x1 << (53 - 32));
        double u = zx * TWO_POW53_INV_D + (TWO_POW53_INV_D / 2.0);
        uint64_t zy = (uint64_t)y0 ^ ((uint64_t)y1 << (53 - 32));
        double v = zy * (TWO_POW53_INV_D * 2.0) + TWO_POW53_INV_D;
        double r = sqrt(-2.0 * log(u));
        double gx = sin(v * 3.1415926535897932) * r;
        double gy = cos(v * 3.1415926535897932) * r;
        s->bm_extra_d = gy;
        s->bm_flag_d = 1;
        return gx;
    }
    s->bm_flag_d = 0;
    return s->bm_extra_d;
}

/* ---- curand_poisson, curand_poisson.h:594-601 ---------------------------- */
/* host branches of __cr_* (curand_poisson.h:74-113) use exact libm; the
 * device uses rsqrt/ex2/lg2/rcp.approx -- accept/reject may differ in rare
 * edge cases, so EM parity host-vs-device is statistical (tests say so). */
static inline float cr_rsqrt(float a) { return 1.0f / sqrtf(a); }
static inline float cr_exp(float a) { return expf(a); }
static inline float cr_log(float a) { return logf(a); }
static inline float cr_rcp(float a) { return 1.0f / a; }

static float cr_pgammainc(float a, float x)
{   /* curand_poisson.h:116-147 */
    const float ma1 = 1.43248035075540910f, ma2 = 0.12400979329415655f, ma3 = 0.00025361074907033f,
                mb1 = 0.21096734870196546f, mb2 = 1.97381164089999420f, mb3 = 0.94201734077887530f;
    float alpha = cr_rsqrt(a - ma2);
    alpha = ma1 * alpha + ma3;
    float beta = cr_rsqrt(a - mb2);
    beta = mb1 * beta + mb3;
    float t = a - x;
    t = alpha * t - beta;
    t = 1.0f + cr_exp(t);
    t = t * t;
    t = cr_rcp(t);
    return t;
}

static float cr_pgammaincinv(float a, float y)
{   /* curand_poisson.h:150-180 */
    const float ma1 = 1.43248035075540910f, ma2 = 0.12400979329415655f, ma3 = 0.00025361074907033f,
                mb1 = 0.21096734870196546f, mb2 = 1.97381164089999420f, mb3 = 0.94201734077887530f;
    float alpha = cr_rsqrt(a - ma2);
    alpha = ma1 * alpha + ma3;
    float beta = cr_rsqrt(a - mb2);
    beta = mb1 * beta + mb3;
    float t = cr_rsqrt(y) - 1.0f;
    t = cr_log(t);
    t = beta + t;
    t = -t * cr_rcp(alpha) + a;
    return t;
}

/* device float->int conversion saturates (cvt.rzi.s32.f32: NaN -> 0, +-inf -> INT_MAX/INT_MIN);
 * x86 would give INT_MIN.  Reached when curand_uniform returns exactly 1.0f (x = +inf, rejected). */
static inline int sat_f2i(float f)
{
    if (f != f) return 0;
    if (f >= 2147483648.0f) return 2147483647;
    if (f <= -2147483648.0f) return (-2147483647 - 1);
    return (int)f;
}

static double cr_lgamma_integer(int a)
{   /* curand_poisson.h:199-243 (Stirling, Hart et al. 5404) */
    static const double table[] = {0.0, 0.0, 6.931471805599453094e-1, 1.791759469228055001e0,
        3.178053830347945620e0, 4.787491742782045994e0, 6.579251212010100995e0,
        8.525161361065414300e0, 1.060460290274525023e1};
    double s, t, sum;
    double fa = fabs((float)a);
    if (a > 8) {
        s = 1.0 / fa;
        t = s * s;
        sum = -0.1633436431e-2;
        sum = sum * t + 0.83645878922e-3;
        sum = sum * t - 0.5951896861197e-3;
        sum = sum * t + 0.793650576493454e-3;
        sum = sum * t - 0.277777777735865004e-2;
        sum = sum * t + 0.833333333333331018375e-1;
        sum = sum * s + 0.918938533204672;
        s = 0.5 * log(fa);
        t = fa - 0.5;
        s = s * t;
        t = s - fa;
        s = s + sum;
        t = t + s;
        return t;
    }
    int idx = (int)fa - 1;
    if (idx < 0 || idx > 8) return 0.0;     /* device reads out of the table here; the draw is rejected anyway */
    return table[idx];
}

static unsigned poisson_knuth(orc_rng_t *s, float lambda)
{   /* curand_poisson.h:246-257 */
    unsigned k = 0;
    float p = expf(lambda);
    do {
        k++;
        p *= orc_uniform(s);
    } while (p > 1.0);
    return k - 1;
}

static unsigned poisson_gammainc(orc_rng_t *s, float lambda)
{   /* curand_poisson.h:464-481 */
    float y, x, t, z, v;
    float logl = cr_log(lambda);
    for (;;) {
        y = orc_uniform(s);
        x = cr_pgammaincinv(lambda, y);
        x = floorf(x);
        z = orc_uniform(s);
        v = (cr_pgammainc(lambda, x + 1.0f) - cr_pgammainc(lambda, x)) * 1.3f;
        z = z * v;
        t = (float)cr_exp(-lambda + x * logl - (float)cr_lgamma_integer(sat_f2i(1.0f + x)));
        if ((z < t) && (v >= 1e-20)) break;
    }
    return (unsigned)x;
}

unsigned orc_poisson(orc_rng_t *s, double lambda)
{
    if (lambda < 64) return poisson_knuth(s, (float)lambda);
    if (lambda > 4000) return (unsigned)((sqrt(lambda) * orc_normal_double(s)) + lambda + 0.5);
    return poisson_gammainc(s, (float)lambda);
}

/* ---- gamma_distribution, src/NMCH/methods/NMCH_EM.cu:11-55 --------------- */
float orc_gamma(orc_rng_t *s, float alpha)
{
    float d, c, x, v, u, x2;
    float C = 1.0f;
    if (alpha < 1.0f) {                       /* NMCH_EM.cu:35-38 */
        C = powf(orc_uniform(s), 1.0f / alpha);
        alpha += 1.0f;
    }
    d = alpha - 1.0f / 3.0f;                  /* :41 */
    c = 1.0f / sqrtf(9.0f * d);               /* :42 */
    for (;;) {                                /* :44-54 */
        do { x = orc_normal(s); v = fmaf(c, x, 1.0f); } while (v <= 0.0f);
        v = v * v * v;
        u = orc_uniform(s);
        x2 = x * x;
        if (u < 1.0f - 0.0331f * x2 * x2 ||
            logf(u) < 0.5f * x2 + d * (1.0f - v + logf(v))) return d * v * C;
    }
}

/* ======================================================================== */
/* FE  (NMCH_FE.cu:145-175; contraction as SURVEY.md Appendix B)             */
/* ======================================================================== */
static inline void fe_step(float *S, float *V, float gx, float gy, float r, float k, float rho,
                           float theta, float sigma, float dt, float sqrt_dt, float sqrt_rho,
                           int floor_kind)
{
    float St = *S, Vt = *V;
    float sv = sqrtf(Vt);
    float a = r * St;          a = fmaf(a, dt, St);
    float z = gy * sqrt_rho;   z = fmaf(gx, rho, z);
    float b = sv * St;         b = b * sqrt_dt;
    float Sn = fmaf(b, z, a);
    float c = theta - Vt;      c = c * k;   c = fmaf(c, dt, Vt);
    float e = sv * sigma;      e = e * sqrt_dt;
    float Vn = fmaf(gx, e, c);
    Vn = (floor_kind == ORC_FLOOR_ABS) ? fabsf(Vn) : fmaxf(Vn, 0.0f);
    *S = Sn; *V = Vn;
}

static void fe_run_impl(const orc_params_t *p, int rng_kind, int floor_kind, uint64_t seed, uint64_t offset,
                        uint64_t first_path, uint64_t n_paths, int calls,
                        float *S_out, float *V_out, double *sum, double *sumsq, int threads);

void orc_fe_run(const orc_params_t *p, int rng_kind, int floor_kind, uint64_t seed,
                uint64_t first_path, uint64_t n_paths, int calls,
                float *S_out, float *V_out, double *sum, double *sumsq, int threads)
{
    fe_run_impl(p, rng_kind, floor_kind, seed, 0, first_path, n_paths, calls, S_out, V_out, sum, sumsq, threads);
}

/* same, with the streams started at curand_init's `offset` (the reference always passes 0) */
void orc_fe_run_at(const orc_params_t *p, int rng_kind, int floor_kind, uint64_t seed, uint64_t offset,
                   uint64_t first_path, uint64_t n_paths, int calls,
                   float *S_out, float *V_out, double *sum, double *sumsq, int threads)
{
    fe_run_impl(p, rng_kind, floor_kind, seed, offset, first_path, n_paths, calls, S_out, V_out, sum, sumsq, threads);
}

static void fe_run_impl(const orc_params_t *p, int rng_kind, int floor_kind, uint64_t seed, uint64_t offset,
                        uint64_t first_path, uint64_t n_paths, int calls,
                        float *S_out, float *V_out, double *sum, double *sumsq, int threads)
{
    const float dt = p->T / p->N;                       /* NMCH.cu:9 */
    const float K = p->S_0;                             /* NMCH.cu:7 */
    const float sqrt_dt = sqrtf(dt);                    /* NMCH_FE.cu:152 */
    const float sqrt_rho = sqrtf(1 - p->rho * p->rho);  /* NMCH_FE.cu:153 */
    double acc = 0.0, acc2 = 0.0;
    xorwow_build_matrices();
    if (threads <= 0) threads = orc_max_threads();
#ifdef _OPENMP
#pragma omp parallel for reduction(+ : acc, acc2) num_threads(threads) schedule(static)
#endif
    for (int64_t i = 0; i < (int64_t)n_paths; ++i) {
        orc_rng_t st;
        orc_rng_init(&st, rng_kind, seed, first_path + (uint64_t)i, offset);   /* random.cu:8-9 (offset 0 there) */
        float St = 0, Vt = 0;
        for (int call = 0; call < calls; ++call) {
            St = p->S_0; Vt = p->v_0;
            for (int n = 0; n < p->N; ++n) {
                float gx, gy;
                orc_normal2(&st, &gx, &gy);
                fe_step(&St, &Vt, gx, gy, p->r, p->k, p->rho, p->theta, p->sigma, dt, sqrt_dt,
                        sqrt_rho, floor_kind);
            }
        }
        float pay = fmaxf(0.0f, St - K);                /* NMCH_FE.cu:171 */
        acc += (double)pay;
        acc2 += (double)pay * (double)pay;
        if (S_out) S_out[i] = St;
        if (V_out) V_out[i] = Vt;
    }
    if (sum) *sum = acc;
    if (sumsq) *sumsq = acc2;
}

/* FE with the pathwise tangent in v_0 (checker of the product's compute_greeks; the reference has no
 * sensitivities).  (S, V) advance by the reference's step (NMCH_FE.cu:156-163, fe_step above); the tangent
 * A = dV/dv_0, B = dS/dv_0 is that step differentiated by hand and carried in DOUBLE, so that the checker does not
 * share the rounding of the float tangent it checks:
 *   sv = sqrt(V), z = rho gx + sqrt(1-rho^2) gy, h = A / (2 sv)
 *   B' = B (1 + r dt + sv sqrt(dt) z) + S sqrt(dt) z h
 *   A'' = A (1 - k dt) + sigma sqrt(dt) gx h,   A' = sign(V'') A'' for |.|,  1{V'' > 0} A'' for (.)+
 * V = 0 (only the (.)+ floor parks paths there, with A = 0 from the parking step on) takes h = 0. */
void orc_fe_tangent_run(const orc_params_t *p, int rng_kind, int floor_kind, uint64_t seed,
                        uint64_t first_path, uint64_t n_paths, float *S_out, float *V_out, double *B_out, int threads)
{
    const float dt = p->T / p->N;
    const float sqrt_dt = sqrtf(dt);
    const float sqrt_rho = sqrtf(1 - p->rho * p->rho);
    xorwow_build_matrices();
    if (threads <= 0) threads = orc_max_threads();
#ifdef _OPENMP
#pragma omp parallel for num_threads(threads) schedule(static)
#endif
    for (int64_t i = 0; i < (int64_t)n_paths; ++i) {
        orc_rng_t st;
        orc_rng_init(&st, rng_kind, seed, first_path + (uint64_t)i, 0);
        float St = p->S_0, Vt = p->v_0;
        double A = 1.0, B = 0.0;
        for (int n = 0; n < p->N; ++n) {
            float gx, gy;
            orc_normal2(&st, &gx, &gy);
            const double sv = sqrt((double)Vt);
            const double z = (double)p->rho * gx + (double)sqrt_rho * gy;
            const double h = Vt > 0.0f ? A / (2.0 * sv) : 0.0;
            const double Bn = B * (1.0 + (double)p->r * dt + sv * sqrt_dt * z) + (double)St * sqrt_dt * z * h;
            const double An = A * (1.0 - (double)p->k * dt) + (double)p->sigma * sqrt_dt * gx * h;
            /* the sign of the pre-floor variance, from the same float expression the step evaluates */
            float c = p->theta - Vt;   c = c * p->k;   c = fmaf(c, dt, Vt);
            float e = sqrtf(Vt) * p->sigma;   e = e * sqrt_dt;
            const float Vpre = fmaf(gx, e, c);
            fe_step(&St, &Vt, gx, gy, p->r, p->k, p->rho, p->theta, p->sigma, dt, sqrt_dt, sqrt_rho, floor_kind);
            B = Bn;
            if (floor_kind == ORC_FLOOR_ABS) A = Vpre < 0.0f ? -An : An;
            else A = Vpre > 0.0f ? An : 0.0;
        }
        if (S_out) S_out[i] = St;
        if (V_out) V_out[i] = Vt;
        if (B_out) B_out[i] = B;
    }
}

/* The exploration sweep (exploration.cu:71-88): one set_* + compute() per point on CONTINUED
 * per-path streams; sums[2*i], sums[2*i+1] = raw payoff moments of point i. */
void orc_fe_sweep(const orc_params_t *p, int rng_kind, int floor_kind, uint64_t seed,
                  uint64_t first_path, uint64_t n_paths, int n_points, const float *k, const float *theta,
                  const float *sigma, double *sums, int threads)
{
    const float dt = p->T / p->N;
    const float K = p->S_0;
    const float sqrt_dt = sqrtf(dt);
    const float sqrt_rho = sqrtf(1 - p->rho * p->rho);
    xorwow_build_matrices();
    if (threads <= 0) threads = orc_max_threads();
    for (int i = 0; i < 2 * n_points; ++i) sums[i] = 0.0;
#ifdef _OPENMP
#pragma omp parallel num_threads(threads)
#endif
    {
        double *loc = (double *)calloc((size_t)2 * n_points, sizeof(double));
#ifdef _OPENMP
#pragma omp for schedule(static)
#endif
        for (int64_t i = 0; i < (int64_t)n_paths; ++i) {
            orc_rng_t st;
            orc_rng_init(&st, rng_kind, seed, first_path + (uint64_t)i, 0);
            for (int pt = 0; pt < n_points; ++pt) {
                float St = p->S_0, Vt = p->v_0;
                for (int n = 0; n < p->N; ++n) {
                    float gx, gy;
                    orc_normal2(&st, &gx, &gy);
                    fe_step(&St, &Vt, gx, gy, p->r, k[pt], p->rho, theta[pt], sigma[pt], dt, sqrt_dt, sqrt_rho,
                            floor_kind);
                }
                float pay = fmaxf(0.0f, St - K);
                loc[2 * pt] += (double)pay;
                loc[2 * pt + 1] += (double)pay * (double)pay;
            }
        }
#ifdef _OPENMP
#pragma omp critical(orc_sweep)
#endif
        for (int i = 0; i < 2 * n_points; ++i) sums[i] += loc[i];
        free(loc);
    }
}

/* ======================================================================== */
/* EM  (NMCH_EM.cu:213-260)                                                  */
/* ======================================================================== */
void orc_em_run(const orc_params_t *p, int rng_kind, uint64_t seed,
                uint64_t first_path, uint64_t n_paths, int calls,
                float *S_out, float *V_out, double *sum, double *sumsq, int threads)
{
    const float dt = p->T / p->N;
    const float K = p->S_0;
    const float k = p->k, theta = p->theta, sigma = p->sigma, rho = p->rho, v_0 = p->v_0;
    const float exp_kdt = expf(-k * dt);                                           /* :226 */
    const float d = 2.0f * k * theta / (sigma * sigma);                            /* :227 */
    const float lambda_const = (2 * k * exp_kdt) / (sigma * sigma * (1 - exp_kdt)); /* :229 */
    const float scale = sigma * sigma * (1.0f - exp_kdt) / (2.0f * k);             /* :240 */
    double acc = 0.0, acc2 = 0.0;
    xorwow_build_matrices();
    if (threads <= 0) threads = orc_max_threads();
#ifdef _OPENMP
#pragma omp parallel for reduction(+ : acc, acc2) num_threads(threads) schedule(dynamic, 64)
#endif
    for (int64_t i = 0; i < (int64_t)n_paths; ++i) {
        orc_rng_t st;
        orc_rng_init(&st, rng_kind, seed, first_path + (uint64_t)i, 0);
        float St = 0, Vt = 0;
        for (int call = 0; call < calls; ++call) {
            Vt = v_0;
            float vI = 0.0f;
            for (int n = 0; n < p->N; ++n) {
                float lambda = lambda_const * Vt;
                int N_p = (int)orc_poisson(&st, lambda);
                float gamma = orc_gamma(&st, d + N_p);
                float Vt_next = scale * gamma;
                vI += (Vt + Vt_next);
                Vt = Vt_next;
            }
            vI = (float)(vI * (dt * 0.5));                    /* :247, double multiply */
            float m = (1.0f / sigma) * (Vt - v_0 - k * theta + k * vI);   /* :249, T=1 assumed */
            m = -0.5f * vI + rho * m;                          /* :251 */
            float sigma2 = (1.0f - rho * rho) * vI;            /* :253 */
            St = expf(m + sqrtf(sigma2) * orc_normal(&st));    /* :260, S_0=1, r=0 assumed */
        }
        float pay = fmaxf(0.0f, St - K);
        acc += (double)pay;
        acc2 += (double)pay * (double)pay;
        if (S_out) S_out[i] = St;
        if (V_out) V_out[i] = Vt;
    }
    if (sum) *sum = acc;
    if (sumsq) *sumsq = acc2;
}

/* ---- scheme-level EM with exact samplers (statistical oracle) ------------ */
static inline uint64_t splitmix64(uint64_t *x)
{
    uint64_t z = (*x += 0x9E3779B97F4A7C15ull);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
static inline double sm_uniform(uint64_t *x) { return ((splitmix64(x) >> 11) + 0.5) * (1.0 / 9007199254740992.0); }
static inline double sm_normal(uint64_t *x)
{
    double u = sm_uniform(x), v = sm_uniform(x);
    return sqrt(-2.0 * log(u)) * cos(6.283185307179586 * v);
}
static double sm_gamma(uint64_t *x, double alpha)
{
    double boost = 1.0;
    if (alpha < 1.0) { boost = pow(sm_uniform(x), 1.0 / alpha); alpha += 1.0; }
    double d = alpha - 1.0 / 3.0, c = 1.0 / sqrt(9.0 * d);
    for (;;) {
        double z, v;
        do { z = sm_normal(x); v = 1.0 + c * z; } while (v <= 0.0);
        v = v * v * v;
        double u = sm_uniform(x);
        if (log(u) < 0.5 * z * z + d * (1.0 - v + log(v))) return d * v * boost;
    }
}
static unsigned sm_poisson(uint64_t *x, double lambda)
{
    if (lambda < 30.0) {
        double L = exp(-lambda), p = 1.0; unsigned k = 0;
        do { k++; p *= sm_uniform(x); } while (p > L);
        return k - 1;
    }
    /* Hoermann PTRS (transformed rejection with squeeze), exact */
    double slam = sqrt(lambda), loglam = log(lambda);
    double b = 0.931 + 2.53 * slam, a = -0.059 + 0.02483 * b;
    double invalpha = 1.1239 + 1.1328 / (b - 3.4), vr = 0.9277 - 3.6224 / (b - 2.0);
    for (;;) {
        double U = sm_uniform(x) - 0.5, V = sm_uniform(x);
        double us = 0.5 - fabs(U);
        double kf = floor((2.0 * a / us + b) * U + lambda + 0.43);
        if (us >= 0.07 && V <= vr) return (unsigned)kf;
        if (kf < 0 || (us < 0.013 && V > us)) continue;
        if (log(V) + log(invalpha) - log(a / (us * us) + b) <= -lambda + kf * loglam - lgamma(kf + 1.0))
            return (unsigned)kf;
    }
}

void orc_em_exact_run(const orc_params_t *p, uint64_t seed, uint64_t n_paths,
                      double *sum, double *sumsq, double *sum_ST, int threads)
{
    const double dt = (double)p->T / p->N, k = p->k, theta = p->theta, sigma = p->sigma, rho = p->rho;
    const double e = exp(-k * dt), om = -expm1(-k * dt);
    const double d = 2.0 * k * theta / (sigma * sigma);
    const double lc = 2.0 * k * e / (sigma * sigma * om), scale = sigma * sigma * om / (2.0 * k);
    const double K = p->S_0;
    double acc = 0, acc2 = 0, accS = 0;
    if (threads <= 0) threads = orc_max_threads();
#ifdef _OPENMP
#pragma omp parallel for reduction(+ : acc, acc2, accS) num_threads(threads) schedule(dynamic, 64)
#endif
    for (int64_t i = 0; i < (int64_t)n_paths; ++i) {
        uint64_t x = seed * 0x9E3779B97F4A7C15ull + (uint64_t)i * 0xD1B54A32D192ED03ull;
        double V = p->v_0, vI = 0.0;
        for (int n = 0; n < p->N; ++n) {
            unsigned Np = sm_poisson(&x, lc * V);
            double Vn = scale * sm_gamma(&x, d + Np);
            vI += V + Vn;
            V = Vn;
        }
        vI *= 0.5 * dt;
        double m = (V - p->v_0 - k * theta * p->T + k * vI) / sigma;
        double lnS = log((double)p->S_0) + p->r * p->T - 0.5 * vI + rho * m
                   + sqrt((1.0 - rho * rho) * vI) * sm_normal(&x);
        double S = exp(lnS);
        double pay = fmax(0.0, S - K);
        acc += pay; acc2 += pay * pay; accS += S;
    }
    if (sum) *sum = acc;
    if (sumsq) *sumsq = acc2;
    if (sum_ST) *sum_ST = accS;
}

/* ======================================================================== */
/* QE-M (Andersen 2008), the product's third method: no reference counterpart */
/* ======================================================================== */
/* Restates nmch_b200/csrc/qe_kernels.cu on the SAME draws (one Philox block per (path, step), counter =
 * (step, call, path_lo, path_hi), 23-bit uniforms) with libm in place of the MUFU approximations, so the kernel can
 * be checked path by path; the scheme itself is checked against the semi-analytic price in the tests. */
void orc_qe_run(const orc_params_t *p, uint64_t seed, uint64_t first_path, uint64_t n_paths, uint32_t call,
                float *S_out, float *V_out, double *sum, double *sumsq, int threads)
{
    const double k = p->k, theta = p->theta, sigma = p->sigma, rho = p->rho, dt = (double)p->T / p->N;
    const double e = exp(-k * dt), om = -expm1(-k * dt);
    const float fe = (float)e, m0 = (float)(theta * om), c1 = (float)(sigma * sigma * e * om / k),
                c2 = (float)(theta * sigma * sigma * om * om / (2.0 * k));
    const double dK2 = 0.5 * dt * (k * rho / sigma - 0.5) + rho / sigma, dK3 = 0.5 * dt * (1.0 - rho * rho);
    const float K2 = (float)dK2, K3 = (float)dK3, K4 = (float)dK3, A = (float)(dK2 + 0.5 * dK3);
    const float hV = (float)(-0.5 * (dK3 + dK3 * e)), h0 = (float)((double)(p->r * (p->T / (float)p->N)) - 0.5 * dK3 * theta * om);
    const float K = p->S_0;
    const uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
    double acc = 0.0, acc2 = 0.0;
    if (threads <= 0) threads = orc_max_threads();
#ifdef _OPENMP
#pragma omp parallel for reduction(+ : acc, acc2) num_threads(threads) schedule(static)
#endif
    for (int64_t i = 0; i < (int64_t)n_paths; ++i) {
        const uint64_t g = first_path + (uint64_t)i;
        float V = p->v_0, lnS = 0.0f;     /* ln(S / S_0), as the kernel accumulates it */
        for (int n = 0; n < p->N; ++n) {
            const uint32_t ctr[4] = {(uint32_t)n, call, (uint32_t)g, (uint32_t)(g >> 32)};
            uint32_t w[4];
            orc_philox4x32_10(ctr, key, w);
            const float u1 = ((float)(w[0] >> 9) + 0.5f) * 1.1920929e-07f;
            const float rad = sqrtf(-2.0f * logf(u1));
            const float ang = (1.0f + (float)(w[1] >> 9) * 1.1920929e-07f) * 6.2831855f;
            const float zv = rad * sinf(ang), zs = rad * cosf(ang);
            const float u = ((float)(w[2] >> 9) + 0.5f) * 1.1920929e-07f;
            const float m = fmaf(V, fe, m0), s2 = fmaf(V, c1, c2), mm = m * m, psi = s2 / mm;
            /* dlog = K2 (V' - m) - (ln M - A m): the kernel's form of K2 V' - ln M without the cancellation */
            float Vn, dlog;
            if (psi <= 1.5f) {
                const float t = 2.0f / psi, b2 = t - 1.0f + sqrtf(t * (t - 1.0f)), a = m / (1.0f + b2);
                const float b = sqrtf(b2), q = b + zv, dV = a * fmaf(zv, fmaf(2.0f, b, zv), -1.0f);
                const float x = 2.0f * A * a, den = fmaxf(1.0f - x, 1e-6f);
                Vn = a * q * q;
                const float tail = fabsf(x) < 0.0625f ? x * x * fmaf(x, fmaf(x, fmaf(x, 0.2f, 0.25f), 0.33333334f), 0.5f)
                                                      : -(logf(den) + x);
                dlog = fmaf(K2, dV, 0.5f * fmaf(b2 * x, -x / den, -tail));
            } else {
                const float pp = (psi - 1.0f) / (psi + 1.0f), beta = (1.0f - pp) / m;
                Vn = (u <= pp) ? 0.0f : logf((1.0f - pp) / (1.0f - u)) / beta;
                const float lnM = logf(pp + beta * (1.0f - pp) / fmaxf(beta - A, 1e-6f));
                dlog = fmaf(K2, Vn - m, fmaf(A, m, -lnM));
            }
            if (!(mm >= 1.17549435e-38f)) {     /* absorbed at zero: theta = 0 and V = 0, or m^2 below FLT_MIN */
                Vn = 0.0f;
                dlog = 0.0f;
            }
            lnS += fmaf(hV, V, h0) + dlog + sqrtf(fmaf(K3, V, K4 * Vn)) * zs;
            V = Vn;
        }
        const float S = p->S_0 * expf(lnS), pay = fmaxf(0.0f, S - K);
        acc += (double)pay;
        acc2 += (double)pay * (double)pay;
        if (S_out) S_out[i] = S;
        if (V_out) V_out[i] = V;
    }
    if (sum) *sum = acc;
    if (sumsq) *sumsq = acc2;
}

/* ======================================================================== */
/* native EM sampler of the product (no reference counterpart: its scheme, own draws) */
/* ======================================================================== */
/* Restates nmch_b200/csrc/em_kernels.cu (em_native_kernel) on the SAME Philox words with libm in place of the MUFU
 * approximations, so the kernel's bit fields, trial order, boost recycling and commit logic can be checked path by
 * path (a flipped accept/reject re-routes a path: the tests ask for the overwhelming majority, and for the aggregate).
 * The SCHEME is the reference's (NMCH_EM.cu:226-260: exact CIR transition per step, trapezoid integral, one
 * conditional log-normal draw); the SAMPLER is the product's: chi-square split for d > 1/2, Poisson mixture below.
 * counter = (trial block, call, path_lo, path_hi), key = seed.  In the split samplers the block counter is shared by
 * the 32 paths of an aligned group (the kernel's loop is warp-uniform), so the terminal draw of a path sits behind the
 * SLOWEST path of its group: paths are processed in aligned groups of 32 here too. */
typedef struct {
    float scale, lc, d, mt_d, inv_a, f_c, f_dl, f_g2s, f_t1, f_ev, f_hs, f_lg2s, k, ktheta_T, inv_sigma;
    int kind;                                    /* 0 split + boost, 1 mixture, 2 split without boost */
} em_native_point_t;

static em_native_point_t em_native_fold(const orc_params_t *p)
{
    const double k = p->k, theta = p->theta, sigma = p->sigma, dt = (double)p->T / p->N;
    const double e = exp(-k * dt), om = -expm1(-k * dt);
    const double c0 = 1.1774100225154747, log2e = 1.4426950408889634;
    em_native_point_t pt;
    memset(&pt, 0, sizeof pt);
    const double cc = sigma * sigma * om / (2.0 * k);
    pt.scale = (float)cc;
    pt.lc = (float)(2.0 * k * e / (sigma * sigma * om));
    pt.d = (float)(2.0 * k * theta / (sigma * sigma));
    double a = 2.0 * k * theta / (sigma * sigma) - 0.5;
    const float af = (float)a;
    float mt_c = 0.0f;
    if (a > 0.0) {
        if (a < 1.0) { pt.inv_a = (float)(1.0 / a); a += 1.0; }
        const double md = a - 1.0 / 3.0;
        pt.mt_d = (float)md;
        mt_c = (float)(1.0 / sqrt(9.0 * md));
    }
    pt.f_c = (float)(mt_c * c0);
    pt.f_dl = (float)(pt.mt_d * log2e);
    pt.f_g2s = (float)(pt.mt_d * cc);
    pt.f_t1 = (float)(c0 * sqrt(0.5 * cc));
    pt.f_ev = (float)e;
    pt.f_hs = (mt_c > 0.0f) ? (float)(0.5 * log2e / ((double)mt_c * (double)mt_c)) : 0.0f;
    pt.f_lg2s = (pt.mt_d > 0.0f) ? (float)log2((double)pt.mt_d * cc) : 0.0f;
    pt.k = p->k;
    pt.ktheta_T = (float)(k * theta * (double)p->T);
    pt.inv_sigma = (float)(1.0 / sigma);
    pt.kind = !(af > 1e-3f) ? 1 : (pt.inv_a != 0.0f ? 0 : 2);
    return pt;
}

static inline float em_u01(uint32_t w) { return ((float)(w >> 9) + 0.5f) * 1.1920929e-07f; }
static inline float em_bits(uint32_t m) { union { uint32_t u; float f; } x; x.u = m | 0x3f800000u; return x.f; }

/* one 64-bit split trial (em_split_trial): returns accept */
static int em_native_split_trial(uint32_t wa, uint32_t wc, const em_native_point_t *pc, int boost, float *zp, float *g2)
{
    const float rad = sqrtf(-log2f(em_u01(wa)));
    const float ang = em_bits(((wa << 14) | (wc >> 18)) & 0x7fffe0u) * 6.2831855f;
    *zp = rad * sinf(ang);
    const float xs = (rad * pc->f_c) * cosf(ang);
    const float v1 = xs + 1.0f, v = v1 * v1 * v1;
    const float lv = log2f(v);                                   /* v <= 0: NaN or -inf, the test fails */
    float rhs = (xs * xs) * pc->f_hs;
    rhs = fmaf(1.0f - v, pc->f_dl, rhs);
    rhs = fmaf(lv, pc->mt_d, rhs);
    const float lu = log2f(em_bits(wc & 0x7fffffu) - 0.99999994f);
    *g2 = boost ? exp2f(fmaf(lu - rhs, pc->inv_a, lv + pc->f_lg2s)) : pc->f_g2s * v;
    return lu < rhs;
}

static const float em_lg2fact[10] = {0.0f, 0.0f, 1.0f, 2.5849625f, 4.5849625f, 6.9068906f, 9.4918531f, 12.2992080f,
                                     15.2992080f, 18.4691330f};

static int em_native_ptrs(float mu, float u_raw, float v, float *k_out)
{
    const float kLn2 = 0.69314718f, kLog2e = 1.44269504f;
    const float smu = sqrtf(mu), b = fmaf(2.53f, smu, 0.931f), a = fmaf(0.02483f, b, -0.059f);
    const float inv_alpha = fmaf(1.1328f, 1.0f / (b - 3.4f), 1.1239f);
    const float u = u_raw - 0.5f, us = 0.5f - fabsf(u), inv_us = 1.0f / us;
    const float k = floorf(fmaf(fmaf(2.0f * a, inv_us, b), u, mu + 0.43f));
    *k_out = k;
    const int big = k >= 10.0f;
    const float t = v * inv_alpha * (1.0f / fmaf(a * inv_us, inv_us, b));
    const float lhs = 0.5f * log2f(big ? (t * t) * (6.28318531f * k) : t * t);
    const float ik = 1.0f / (big ? k : 1.0f);
    const float delta = (k - mu) * ik, sv = delta * (1.0f / (2.0f - delta)), s2 = sv * sv;
    float poly = fmaf(s2, 1.0f / 11.0f, 1.0f / 9.0f);
    poly = fmaf(poly, s2, 1.0f / 7.0f);
    poly = fmaf(poly, s2, 1.0f / 5.0f);
    poly = fmaf(poly, s2, 1.0f / 3.0f);
    const float f_series = -fmaf(2.0f * sv * s2, poly, delta * sv);
    const float lgx = log2f(big ? mu * ik : mu);
    const float f_log = fmaf(lgx, kLn2, delta);
    const float stirling = ik * fmaf(ik * ik, 1.0f / 360.0f, -1.0f / 12.0f);
    const float rhs_big = fmaf(k, (fabsf(sv) < 0.3f) ? f_series : f_log, stirling) * kLog2e;
    int ki = big ? 0 : (int)k;
    if (ki < 0) ki = 0;
    const float rhs_small = fmaf(k, lgx, -fmaf(mu, kLog2e, em_lg2fact[ki]));
    const float rhs = big ? rhs_big : rhs_small;
    return (k >= 0.0f) && !(us < 0.013f && v > us) && (lhs <= rhs);
}

static float em_native_terminal(const orc_params_t *p, const em_native_point_t *pc, const uint32_t w[4], float V, float acc)
{
    const float half_dt = 0.5f * (p->T / (float)p->N), one_m_rho2 = 1.0f - p->rho * p->rho;
    const float lnS0_rT = (float)(log((double)p->S_0) + (double)p->r * (double)p->T);
    const float r = sqrtf(-1.38629436f * log2f(em_u01(w[0])));
    const float z = r * sinf(em_bits(w[1] >> 9) * 6.2831855f);
    const float vI = fmaf(2.0f, acc, p->v_0 - V) * half_dt;
    float m = pc->inv_sigma * fmaf(pc->k, vI, V - p->v_0 - pc->ktheta_T);
    m = fmaf(p->rho, m, fmaf(-0.5f, vI, lnS0_rT));
    return expf(fmaf(sqrtf(one_m_rho2 * vI), z, m));
}

void orc_em_native_run(const orc_params_t *p, uint64_t seed, uint64_t first_path, uint64_t n_paths, uint32_t call,
                       float *S_out, float *V_out, double *sum, double *sumsq, int threads)
{
    const em_native_point_t pc = em_native_fold(p);
    const uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
    const float K = p->S_0;
    const int N = p->N;
    double acc_sum = 0.0, acc_sq = 0.0;
    if (threads <= 0) threads = orc_max_threads();
    const uint64_t g_begin = first_path, g_end = first_path + n_paths;
    const int64_t grp0 = (int64_t)(g_begin / 32u), grp1 = (int64_t)((g_end + 31u) / 32u);
#ifdef _OPENMP
#pragma omp parallel for reduction(+ : acc_sum, acc_sq) num_threads(threads) schedule(dynamic, 8)
#endif
    for (int64_t grp = grp0; grp < grp1; ++grp) {
        float Vt[32], At[32];
        uint32_t blk_end[32];
        uint32_t blk_group = 0;
        for (int lane = 0; lane < 32; ++lane) {
            const uint64_t g = (uint64_t)grp * 32u + (uint64_t)lane;
            blk_end[lane] = 0;
            if (g < g_begin || g >= g_end) continue;
            uint32_t ctr[4] = {0, call, (uint32_t)g, (uint32_t)(g >> 32)}, w[8];
            float V = p->v_0, acc = 0.0f;
            int step = 0;
            uint32_t blk = 0;
            if (pc.kind != 1) {
                while (step < N) {                                /* two blocks = four trials per iteration */
                    ctr[0] = blk; orc_philox4x32_10(ctr, key, w);
                    ctr[0] = blk + 1u; orc_philox4x32_10(ctr, key, w + 4);
                    blk += 2u;
                    for (int j = 0; j < 4; ++j) {
                        float zp, g2;
                        const int ok = em_native_split_trial(w[2 * j], w[2 * j + 1], &pc, pc.kind == 0, &zp, &g2);
                        const float t = fmaf(pc.f_t1, zp, sqrtf(pc.f_ev * V));
                        const float Vn = fmaf(t, t, g2);
                        if (ok && step < N) { acc += Vn; V = Vn; ++step; }
                    }
                }
                if (blk > blk_group) blk_group = blk;             /* the group ends with its slowest path */
            } else {
                int have_np = 0;
                float np = 0.0f;
                const float inv_d = 1.0f / pc.d;
                while (step < N) {
                    ctr[0] = blk++; orc_philox4x32_10(ctr, key, w);
                    if (!have_np) {
                        const float mu = pc.lc * V;
                        if (mu < 10.0f) {
                            float pp = exp2f(-1.44269504f * mu), cdf = pp, kk = 0.0f;
                            const float u = em_u01(w[0]);
                            while (u > cdf && kk < 80.0f) { kk += 1.0f; pp *= mu * (1.0f / kk); cdf += pp; }
                            np = kk;
                            have_np = 1;
                        } else {
                            have_np = em_native_ptrs(mu, em_u01(w[0]), em_u01(w[1]), &np);
                        }
                    }
                    const float shape0 = pc.d + np;
                    const int small = shape0 < 1.0f;
                    const float md = (small ? shape0 + 1.0f : shape0) - (1.0f / 3.0f);
                    const float rad = sqrtf(-log2f(em_u01(w[2])));
                    const float ang = em_bits(((w[2] << 14) | (w[3] >> 18)) & 0x7fffe0u) * 6.2831855f;
                    const float xs = (rad * (1.1774100f * (1.0f / sqrtf(9.0f * md)))) * cosf(ang);
                    const float v1 = xs + 1.0f, v = v1 * v1 * v1, lv = log2f(v);
                    const float rhs = md * fmaf(fmaf(4.5f * xs, xs, 1.0f - v), 1.44269504f, lv);
                    const float lu = log2f(em_bits(w[3] & 0x7fffffu) - 0.99999994f);
                    const float boost = exp2f((lu - rhs) * inv_d);
                    const float gam = md * v * (small ? boost : 1.0f);
                    if (have_np && lu < rhs) {
                        const float Vn = pc.scale * gam;
                        acc += Vn; V = Vn; ++step; have_np = 0;
                    }
                }
                blk_end[lane] = blk;                              /* per-lane counter in the mixture loop */
            }
            Vt[lane] = V;
            At[lane] = acc;
        }
        for (int lane = 0; lane < 32; ++lane) {
            const uint64_t g = (uint64_t)grp * 32u + (uint64_t)lane;
            if (g < g_begin || g >= g_end) continue;
            const uint32_t ctr[4] = {pc.kind != 1 ? blk_group : blk_end[lane], call, (uint32_t)g, (uint32_t)(g >> 32)};
            uint32_t w[4];
            orc_philox4x32_10(ctr, key, w);
            const float S = em_native_terminal(p, &pc, w, Vt[lane], At[lane]);
            const float pay = fmaxf(0.0f, S - K);
            acc_sum += (double)pay;
            acc_sq += (double)pay * (double)pay;
            if (S_out) S_out[g - g_begin] = S;
            if (V_out) V_out[g - g_begin] = Vt[lane];
        }
    }
    if (sum) *sum = acc_sum;
    if (sumsq) *sumsq = acc_sq;
}

/* ======================================================================== */
/* host statistics                                                           */
/* ======================================================================== */
float orc_get_err(int state_numbers, float strike_price, float price_squared)
{   /* NMCH_FE.hpp:50-55 verbatim in meaning: 1.0f/(n-1) in float, n*E[X^2] in float */
    float err = 1.96 * sqrt((double)(1.0f / (state_numbers - 1)) *
                            (state_numbers * price_squared - (strike_price * strike_price))) /
                sqrt((double)state_numbers);
    return err;
}

double orc_NP(double x)
{   /* utils.cu:5-25, Abramowitz-Stegun 26.2.17 */
    const double p = 0.2316419, b1 = 0.319381530, b2 = -0.356563782, b3 = 1.781477937,
                 b4 = -1.821255978, b5 = 1.330274429, one_over_twopi = 0.39894228;
    double t;
    if (x >= 0.0) {
        t = 1.0 / (1.0 + p * x);
        return 1.0 - one_over_twopi * exp(-x * x / 2.0) * t * (t * (t * (t * (t * b5 + b4) + b3) + b2) + b1);
    }
    t = 1.0 / (1.0 - p * x);
    return one_over_twopi * exp(-x * x / 2.0) * t * (t * (t * (t * (t * b5 + b4) + b3) + b2) + b1);
}

float orc_print_true_price(float S_0, float K, float r, float sigma)
{   /* NMCH_FE.cu:336-338 : Black-Scholes with vol:=sigma, T:=1 */
    float real_price = S_0 * orc_NP((r + 0.5 * sigma * sigma) / sigma) -
                       K * expf(-r) * orc_NP((r - 0.5 * sigma * sigma) / sigma);
    return real_price;
}

/* Semi-analytic Heston call: Heston (1993) P1/P2 with the Albrecher et al.
 * "little trap" branch choice; composite 16-point Gauss-Legendre on [0, 400]. */
static double complex heston_cf(double phi, int j, double lnS0, double v0, double r, double kappa,
                                double theta, double sigma, double rho, double T)
{
    const double u = (j == 1) ? 0.5 : -0.5;
    const double b = (j == 1) ? kappa - rho * sigma : kappa;
    const double a = kappa * theta;
    double complex iphi = I * phi;
    double complex rsi = rho * sigma * iphi;
    double complex d = csqrt((rsi - b) * (rsi - b) - sigma * sigma * (2.0 * u * iphi - phi * phi));
    double complex g = (b - rsi - d) / (b - rsi + d);
    double complex edT = cexp(-d * T);
    double complex C = r * iphi * T + a / (sigma * sigma) * ((b - rsi - d) * T - 2.0 * clog((1.0 - g * edT) / (1.0 - g)));
    double complex D = (b - rsi - d) / (sigma * sigma) * (1.0 - edT) / (1.0 - g * edT);
    return cexp(C + D * v0 + iphi * lnS0);
}

double orc_heston_call(double S0, double K, double v0, double r, double kappa,
                       double theta, double sigma, double rho, double T)
{
    static const double gx[8] = {0.0950125098376374, 0.2816035507792589, 0.4580167776572274,
        0.6178762444026438, 0.7554044083550030, 0.8656312023878318, 0.9445750230732326, 0.9894009349916499};
    static const double gw[8] = {0.1894506104550685, 0.1826034150449236, 0.1691565193950025,
        0.1495959888165767, 0.1246289712555339, 0.0951585116824928, 0.0622535239386479, 0.0271524594117541};
    const double lnS0 = log(S0), lnK = log(K);
    const double upper = 400.0;
    const int panels = 4000;
    const double h = upper / panels;
    double I1 = 0.0, I2 = 0.0;
    for (int pnl = 0; pnl < panels; ++pnl) {
        double mid = (pnl + 0.5) * h, half = 0.5 * h;
        for (int q = 0; q < 8; ++q)
            for (int sgn = -1; sgn <= 1; sgn += 2) {
                double phi = mid + sgn * half * gx[q];
                double complex e = cexp(-I * phi * lnK) / (I * phi);
                I1 += gw[q] * half * creal(e * heston_cf(phi, 1, lnS0, v0, r, kappa, theta, sigma, rho, T));
                I2 += gw[q] * half * creal(e * heston_cf(phi, 2, lnS0, v0, r, kappa, theta, sigma, rho, T));
            }
    }
    double P1 = 0.5 + I1 / M_PI, P2 = 0.5 + I2 / M_PI;
    return S0 * P1 - K * exp(-r * T) * P2;
}

/* ======================================================================== */
/* exploration grid (exploration.cu:46-52, 71-88)                            */
/* ======================================================================== */
int orc_exploration_grid(int steps, int apply_filter, float *k_out, float *theta_out, float *sigma_out, int cap)
{
    float k_min = 0.1f, k_max = 10.0f;
    float theta_min = 0.01f, theta_max = 0.5f;
    float sigma_min = 0.1f, sigma_max = 1.0f;
    float sigma_step = (sigma_max - sigma_min) / steps;
    float theta_step = (theta_max - theta_min) / steps;
    float k_step = (k_max - k_min) / steps;
    int n = 0;
    for (float sigma = sigma_min; sigma <= sigma_max; sigma += sigma_step)
        for (float theta = theta_min; theta <= theta_max; theta += theta_step)
            for (float k = k_min; k <= k_max; k += k_step) {
                if (apply_filter && (20 * k * theta < sigma * sigma)) continue;
                if (n < cap) { k_out[n] = k; theta_out[n] = theta; sigma_out[n] = sigma; }
                ++n;
            }
    return n;
}

/* Generator initialisation alone for paths [first_path, first_path + n_paths): what the reference's init_curand_state_k
 * does (random.cu:6-10) and reports as Tim_init, outside Tim_exec.  bench.py times this next to orc_fe_run / orc_em_run
 * (which initialise inside their path loop) so that the CPU baseline can be quoted on the same span as the GPU arm.
 * Returns a checksum of the states so that the work cannot be optimised away. */
uint64_t orc_rng_init_only(int rng_kind, uint64_t seed, uint64_t first_path, uint64_t n_paths, int threads)
{
    uint64_t acc = 0;
    xorwow_build_matrices();
    if (threads <= 0) threads = orc_max_threads();
#ifdef _OPENMP
#pragma omp parallel for reduction(+ : acc) num_threads(threads) schedule(static)
#endif
    for (int64_t i = 0; i < (int64_t)n_paths; ++i) {
        orc_rng_t st;
        orc_rng_init(&st, rng_kind, seed, first_path + (uint64_t)i, 0);
        acc += (uint64_t)orc_rng_next(&st);
    }
    return acc;
}

int orc_max_threads(void)
{
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}
