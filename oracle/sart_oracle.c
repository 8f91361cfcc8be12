/*
 * TEST INFRASTRUCTURE ONLY -- fp64 restatement of the adjoint projector and of ordered-subset SART
 * (ipdm_fbp_project_adjoint, ipdm_fbp_sart_tv with ntv = 0, csrc/sart.cu).
 *
 * The rays and Joseph weights are those of oracle/project_oracle.c (ray_sum): along the dominant axis one
 * sample per column / row m at u(m) = u0 + (m - 255.5) g, weight 1 - w on pixel floor(u) and w on floor(u) + 1
 * of the other axis, times dx / |cos| (or |sin|); every m of the grid is visited, taps outside the grid are dropped.
 *
 * adjoint_oracle scatters each ray's weights times its value.  Under OpenMP the views are split statically over
 * per-thread image buffers that are summed in thread order, so the result is fixed for a given thread count.
 * sart_oracle runs the plain SART loop of ipdm_fbp_sart_tv in fp64 with R = A 1 and C_s = A_s^T 1 from the same weights.
 * Both work in the native frame; flip = 1 reverses the detector axis of the sinogram and the columns of the image.
 * Nothing under ipdm-pytorch_b200/ links or loads this file.
 */
#include <math.h>
#include <stddef.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define ND 912
#define NP 512
#define NV 2000

typedef struct {
    int xmajor;
    double u0, g, scale;
} ray_t;

static ray_t ray_setup(double ct, double st, double ca, double sa, double D, double dx)
{
    const double c = ct * ca + st * sa, s = st * ca - ct * sa;   /* cos, sin of phi = theta - alpha */
    const double p = D * sa / dx;
    ray_t r;
    r.xmajor = fabs(c) >= fabs(s);
    const double a = r.xmajor ? c : s, o = r.xmajor ? s : c;
    r.u0 = r.xmajor ? 255.5 - p / a : 255.5 + p / a;
    r.g = o / a;
    r.scale = dx / fabs(a);
    return r;
}

/* native pixel index of tap k of sample m, -1 outside the grid */
static long tap(const ray_t *r, int m, int k)
{
    if (k < 0 || k >= NP) return -1;
    return r->xmajor ? (long)k * NP + m : (long)m * NP + k;
}

/* A row of the ray applied to a native fp64 image */
static double ray_project(const double *img, const ray_t *r)
{
    double acc = 0.0;
    for (int m = 0; m < NP; ++m) {
        const double u = r->u0 + (m - 255.5) * r->g;
        const double kf = floor(u);
        const int k = (int)kf;
        const double w = u - kf;
        const long a = tap(r, m, k), b = tap(r, m, k + 1);
        const double v0 = a >= 0 ? img[a] : 0.0, v1 = b >= 0 ? img[b] : 0.0;
        acc += v0 + w * (v1 - v0);
    }
    return acc * r->scale;
}

/* img += y * (A row of the ray)^T, native */
static void ray_scatter(double *img, const ray_t *r, double y)
{
    const double ys = y * r->scale;
    for (int m = 0; m < NP; ++m) {
        const double u = r->u0 + (m - 255.5) * r->g;
        const double kf = floor(u);
        const int k = (int)kf;
        const double w = u - kf;
        const long a = tap(r, m, k), b = tap(r, m, k + 1);
        if (a >= 0) img[a] += ys * (1.0 - w);
        if (b >= 0) img[b] += ys * w;
    }
}

static int n_threads(void)
{
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}

static int thread_id(void)
{
#ifdef _OPENMP
    return omp_get_thread_num();
#else
    return 0;
#endif
}

/* out = sum of the per-thread buffers in thread order */
static void reduce(const double *buf, int nt, double *out)
{
    memcpy(out, buf, sizeof(double) * NP * NP);
    for (int t = 1; t < nt; ++t)
        for (long q = 0; q < (long)NP * NP; ++q) out[q] += buf[(size_t)t * NP * NP + q];
}

/* native sino [nv][912] (rows = the views theta[vlist[n]], vlist NULL: n) -> native img = A^T sino */
static void adjoint_native(const double *sino, double *img, int nv, const int *vlist, const double *theta, const double *ca,
                           const double *sa, double D, double dx)
{
    const int nt = n_threads();
    double *buf = calloc((size_t)nt * NP * NP, sizeof(double));
#pragma omp parallel num_threads(nt)
    {
        double *mine = buf + (size_t)thread_id() * NP * NP;
#pragma omp for schedule(static)
        for (int n = 0; n < nv; ++n) {
            const double th = theta[vlist ? vlist[n] : n];
            const double ct = cos(th), st = sin(th);
            for (int k = 0; k < ND; ++k) {
                const double y = sino[(size_t)n * ND + k];
                if (y == 0.0) continue;
                const ray_t r = ray_setup(ct, st, ca[k], sa[k], D, dx);
                ray_scatter(mine, &r, y);
            }
        }
    }
    reduce(buf, nt, img);
    free(buf);
}

/* sino [batch][nv][912] f64 (frame flip) -> img [batch][512][512] f64 (frame flip); theta [nv], alpha [912] */
void adjoint_oracle(const double *sino, double *img, int batch, int nv, int flip, const double *theta, const double *alpha, double D,
                    double dx)
{
    double ca[ND], sa[ND];
    for (int k = 0; k < ND; ++k) { ca[k] = cos(alpha[k]); sa[k] = sin(alpha[k]); }
    double *sn = malloc(sizeof(double) * (size_t)nv * ND), *im = malloc(sizeof(double) * NP * NP);
    for (int b = 0; b < batch; ++b) {
        const double *s = sino + (size_t)b * nv * ND;
        for (int n = 0; n < nv; ++n)
            for (int k = 0; k < ND; ++k) sn[(size_t)n * ND + k] = s[(size_t)n * ND + (flip ? ND - 1 - k : k)];
        adjoint_native(sn, im, nv, NULL, theta, ca, sa, D, dx);
        double *o = img + (size_t)b * NP * NP;
        for (int i = 0; i < NP; ++i)
            for (int j = 0; j < NP; ++j) o[(size_t)i * NP + j] = im[(size_t)i * NP + (flip ? NP - 1 - j : j)];
    }
    free(sn);
    free(im);
}

static int gcd(int a, int b) { while (b) { const int t = a % b; a = b; b = t; } return a; }

/* the visit step of ipdm_fbp_sart_tv: the integer in [1, S) coprime to S closest to 0.382 S, smaller on a tie; 1 when S <= 2 */
int sart_visit_step(int S)
{
    if (S <= 2) return 1;
    const double t = 0.382 * S;
    int best = 1;
    double bd = 1e300;
    for (int q = 1; q < S; ++q)
        if (gcd(q, S) == 1 && fabs(q - t) < bd) { bd = fabs(q - t); best = q; }
    return best;
}

/* sino [batch][2000][912] f32 (frame flip) -> img [batch][512][512] f64 (frame flip) after `iterations` sweeps; history
 * (NULL or [batch][iterations][512][512]) receives the iterate after every sweep.  theta [2000], alpha [912]. */
void sart_oracle(const float *sino, double *img, double *history, int batch, int flip, int iterations, int S, double lambda,
                 const double *theta, const double *alpha, double D, double dx)
{
    const int nv = NV / S, nt = n_threads();
    double ca[ND], sa[ND];
    for (int k = 0; k < ND; ++k) { ca[k] = cos(alpha[k]); sa[k] = sin(alpha[k]); }
    /* R = A 1 (native [2000][912]) and C_s = A_s^T 1 (native [S][512][512]) */
    double *ones = malloc(sizeof(double) * NP * NP), *R = malloc(sizeof(double) * NV * ND);
    for (long q = 0; q < (long)NP * NP; ++q) ones[q] = 1.0;
#pragma omp parallel for schedule(static)
    for (int v = 0; v < NV; ++v) {
        const double ct = cos(theta[v]), st = sin(theta[v]);
        for (int k = 0; k < ND; ++k) {
            const ray_t r = ray_setup(ct, st, ca[k], sa[k], D, dx);
            R[(size_t)v * ND + k] = ray_project(ones, &r);
        }
    }
    double *C = malloc(sizeof(double) * (size_t)S * NP * NP), *sub1 = malloc(sizeof(double) * (size_t)nv * ND);
    int *vlist = malloc(sizeof(int) * nv);
    for (long q = 0; q < (long)nv * ND; ++q) sub1[q] = 1.0;
    for (int s = 0; s < S; ++s) {
        for (int n = 0; n < nv; ++n) vlist[n] = s + n * S;
        adjoint_native(sub1, C + (size_t)s * NP * NP, nv, vlist, theta, ca, sa, D, dx);
    }
    const int step = sart_visit_step(S);
    double *x = malloc(sizeof(double) * NP * NP), *bp = malloc(sizeof(double) * NP * NP);
    double *buf = malloc(sizeof(double) * (size_t)nt * NP * NP);
    for (int b = 0; b < batch; ++b) {
        const float *bs = sino + (size_t)b * NV * ND;
        memset(x, 0, sizeof(double) * NP * NP);
        for (int it = 0; it < iterations; ++it) {
            for (int n = 0; n < S; ++n) {
                const int s = (int)((long long)n * step % S);
                memset(buf, 0, sizeof(double) * (size_t)nt * NP * NP);
#pragma omp parallel num_threads(nt)
                {
                    double *mine = buf + (size_t)thread_id() * NP * NP;
#pragma omp for schedule(static)
                    for (int q = 0; q < nv; ++q) {
                        const int v = s + q * S;
                        const double ct = cos(theta[v]), st = sin(theta[v]);
                        for (int k = 0; k < ND; ++k) {
                            const double rs = R[(size_t)v * ND + k];
                            if (!(rs > 0.0)) continue;
                            const ray_t r = ray_setup(ct, st, ca[k], sa[k], D, dx);
                            const double y = ((double)bs[(size_t)v * ND + (flip ? ND - 1 - k : k)] - ray_project(x, &r)) / rs;
                            ray_scatter(mine, &r, y);
                        }
                    }
                }
                reduce(buf, nt, bp);
                const double *c = C + (size_t)s * NP * NP;
                for (long q = 0; q < (long)NP * NP; ++q)
                    if (c[q] > 0.0) x[q] = fmax(0.0, x[q] + lambda * bp[q] / c[q]);
            }
            if (history) {
                double *h = history + ((size_t)b * iterations + it) * NP * NP;
                for (int i = 0; i < NP; ++i)
                    for (int j = 0; j < NP; ++j) h[(size_t)i * NP + j] = x[(size_t)i * NP + (flip ? NP - 1 - j : j)];
            }
        }
        double *o = img + (size_t)b * NP * NP;
        for (int i = 0; i < NP; ++i)
            for (int j = 0; j < NP; ++j) o[(size_t)i * NP + j] = x[(size_t)i * NP + (flip ? NP - 1 - j : j)];
    }
    free(ones); free(R); free(C); free(sub1); free(vlist); free(x); free(bp); free(buf);
}
