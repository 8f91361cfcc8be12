/*
 * TEST INFRASTRUCTURE ONLY -- fp64 restatement of the total-variation steps and of SART-TV
 * (ipdm_fbp_tv_descent, ipdm_fbp_sart_tv, csrc/tv.cu and csrc/sart.cu).
 *
 * TV_eps(x) = sum_{i,j} sqrt(dx^2 + dy^2 + eps^2), forward differences dx = x[i][j+1] - x[i][j], dy = x[i+1][j] - x[i][j]
 * (0 where they would leave the image), in the native frame.  Its gradient is
 *   g[i][j] = -(dx[i][j] + dy[i][j]) / n[i][j] + dx[i][j-1] / n[i][j-1] + dy[i-1][j] / n[i-1][j],  n = sqrt(dx^2 + dy^2 + eps^2),
 * out-of-range terms dropped.  A TV step of length t is x <- max(0, x - t g / |g|_2) (no change where |g| = 0).
 *
 * sart_tv_oracle is the loop of sart_oracle.c (included below, so the rays, weights, R and C_s are its own) with a start x0
 * (NULL: 0) and, after every sweep, ntv TV steps of length t = tv_alpha |x - x_prev|_2, x_prev the iterate before the sweep
 * (ASD-POCS, Sidky & Pan 2008, with a fixed step fraction).  The SART loop is restated here rather than changed in place, so
 * that sart_oracle.c stays the reference of plain SART.
 * Nothing under ipdm-pytorch_b200/ links or loads this file.
 */
#include "sart_oracle.c"

/* native x [512][512] -> native g = grad TV_eps(x) */
static void tv_grad_native(const double *x, double *g, double eps)
{
    const double e2 = eps * eps;
#define X(i, j) x[(size_t)(i) * NP + (j)]
#define DX(i, j) ((j) < NP - 1 ? X(i, (j) + 1) - X(i, j) : 0.0)
#define DY(i, j) ((i) < NP - 1 ? X((i) + 1, j) - X(i, j) : 0.0)
#define NRM(i, j) sqrt(DX(i, j) * DX(i, j) + DY(i, j) * DY(i, j) + e2)
#pragma omp parallel for schedule(static)
    for (int i = 0; i < NP; ++i)
        for (int j = 0; j < NP; ++j) {
            double v = -(DX(i, j) + DY(i, j)) / NRM(i, j);
            if (j > 0) v += DX(i, j - 1) / NRM(i, j - 1);
            if (i > 0) v += DY(i - 1, j) / NRM(i - 1, j);
            g[(size_t)i * NP + j] = v;
        }
#undef X
#undef DX
#undef DY
#undef NRM
}

static double norm2(const double *a, const double *b)
{
    double s = 0.0;
    for (long q = 0; q < (long)NP * NP; ++q) {
        const double d = b ? a[q] - b[q] : a[q];
        s += d * d;
    }
    return sqrt(s);
}

/* steps TV steps of length t on a native image; g is scratch [512][512] */
static void tv_steps_native(double *x, double *g, int steps, double t, double eps)
{
    for (int s = 0; s < steps; ++s) {
        tv_grad_native(x, g, eps);
        const double gn = norm2(g, NULL);
        if (!(gn > 0.0)) continue;
        for (long q = 0; q < (long)NP * NP; ++q) x[q] = fmax(0.0, x[q] - t * g[q] / gn);
    }
}

static void to_native(const double *in, double *out, int flip)
{
    for (int i = 0; i < NP; ++i)
        for (int j = 0; j < NP; ++j) out[(size_t)i * NP + j] = in[(size_t)i * NP + (flip ? NP - 1 - j : j)];
}

/* img [batch][512][512] (frame flip) -> g [batch][512][512] (frame flip) */
void tv_grad_oracle(const double *img, double *g, int batch, int flip, double eps)
{
    double *xn = malloc(sizeof(double) * NP * NP), *gn = malloc(sizeof(double) * NP * NP);
    for (int b = 0; b < batch; ++b) {
        to_native(img + (size_t)b * NP * NP, xn, flip);
        tv_grad_native(xn, gn, eps);
        to_native(gn, g + (size_t)b * NP * NP, flip);          /* the column mirror is its own inverse */
    }
    free(xn);
    free(gn);
}

/* img [batch][512][512] (frame flip), in place: steps TV steps of length step */
void tv_descent_oracle(double *img, int batch, int flip, int steps, double step, double eps)
{
    double *xn = malloc(sizeof(double) * NP * NP), *g = malloc(sizeof(double) * NP * NP);
    for (int b = 0; b < batch; ++b) {
        double *o = img + (size_t)b * NP * NP;
        to_native(o, xn, flip);
        tv_steps_native(xn, g, steps, step, eps);
        to_native(xn, o, flip);
    }
    free(xn);
    free(g);
}

/* sart_oracle with a start x0 ([batch][512][512] f64, frame flip, clamped at 0; NULL: 0) and ntv TV steps after every sweep */
void sart_tv_oracle(const float *sino, const double *x0, double *img, double *history, int batch, int flip, int iterations, int S,
                    double lambda, int ntv, double tv_alpha, double tv_eps, const double *theta, const double *alpha, double D,
                    double dx)
{
    const int nv = NV / S, nt = n_threads();
    double ca[ND], sa[ND];
    for (int k = 0; k < ND; ++k) { ca[k] = cos(alpha[k]); sa[k] = sin(alpha[k]); }
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
    double *xp = malloc(sizeof(double) * NP * NP), *g = malloc(sizeof(double) * NP * NP);
    double *buf = malloc(sizeof(double) * (size_t)nt * NP * NP);
    for (int b = 0; b < batch; ++b) {
        const float *bs = sino + (size_t)b * NV * ND;
        if (x0) {
            to_native(x0 + (size_t)b * NP * NP, x, flip);
            for (long q = 0; q < (long)NP * NP; ++q) x[q] = fmax(0.0, x[q]);
        } else {
            memset(x, 0, sizeof(double) * NP * NP);
        }
        for (int it = 0; it < iterations; ++it) {
            memcpy(xp, x, sizeof(double) * NP * NP);
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
            if (ntv > 0) tv_steps_native(x, g, ntv, tv_alpha * norm2(x, xp), tv_eps);
            if (history) to_native(x, history + ((size_t)b * iterations + it) * NP * NP, flip);
        }
        to_native(x, img + (size_t)b * NP * NP, flip);
    }
    free(ones); free(R); free(C); free(sub1); free(vlist); free(x); free(bp); free(xp); free(g); free(buf);
}
