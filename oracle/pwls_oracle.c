/*
 * TEST INFRASTRUCTURE ONLY -- fp64 restatement of penalised weighted least squares solved by ordered-subset SQS
 * (ipdm_fbp_pwls, ipdm_fbp_pwls_penalty, csrc/pwls.cu and csrc/sart.cu).
 *
 * Phi(x) = 1/2 sum_i w_i ([A x]_i - b_i)^2 + beta R(x), x >= 0, with A the Joseph matrix of sart_oracle.c (included below, so the
 * rays and weights are its own) and w_i = 1 / sigma^2(max(b_i, 0)), sigma^2(p) = e^p / (f N0) (1 + Ne e^p / (f N0)), the
 * variance of a measurement at dose f (N0 = 1.4e5, Ne = 5.8, the constants of the dose-reduction noise).
 * R(x) = sum_j sum_{k in N+(j)} kappa_jk psi(x_j - x_k): N+ = right, down, down-left, down-right (native frame, each pair once),
 * kappa = 1 (edge) or 1/sqrt(2) (diagonal), psi(t) = delta^2 (sqrt(1 + (t / delta)^2) - 1), no terms outside the image.
 * grad R_j = sum over the 8 neighbours of kappa psi'(x_j - x_k), psi'(t) = t omega(t), omega(t) = 1 / sqrt(1 + (t / delta)^2);
 * the SQS curvature is d^R_j = 2 sum over the 8 neighbours of kappa omega(x_j - x_k) (De Pierro's bound for a pairwise term).
 * D^L = A^T (w o A 1).  One OS-SQS subset s (views v = s mod S, visited in sart_visit_step order):
 *   x <- max(0, x + (S A_s^T (w_s o (b_s - A_s x)) - beta grad R(x)) / (D^L + beta d^R(x)))   (x kept where the denominator is 0)
 * Everything is computed in the native frame; flip = 1 reverses the detector axis of the sinogram and the columns of the image.
 * Nothing under ipdm-pytorch_b200/ links or loads this file.
 */
#include "sart_oracle.c"

#define PWLS_N0 1.4e5
#define PWLS_NE 5.8

static double weight(double b, double dose)
{
    const double q = exp(fmax(b, 0.0)) / (dose * PWLS_N0);
    return 1.0 / (q * (1.0 + PWLS_NE * q));
}

/* n sinogram values -> weights */
void pwls_weights_oracle(const float *b, double *w, long n, double dose)
{
    for (long q = 0; q < n; ++q) w[q] = weight((double)b[q], dose);
}

/* native x: R(x) and, when g / c are given, grad R and d^R (native) */
static double penalty_native(const double *x, double *g, double *c, double delta)
{
    static const int di[8] = {-1, -1, -1, 0, 0, 1, 1, 1}, dj[8] = {-1, 0, 1, -1, 1, -1, 0, 1};
    const double kd = 1.0 / sqrt(2.0), id = 1.0 / delta;
    double val = 0.0;
#pragma omp parallel for schedule(static) reduction(+ : val)
    for (int i = 0; i < NP; ++i)
        for (int j = 0; j < NP; ++j) {
            const double xv = x[(size_t)i * NP + j];
            double gs = 0.0, cs = 0.0;
            for (int n = 0; n < 8; ++n) {
                const int ii = i + di[n], jj = j + dj[n];
                if (ii < 0 || ii >= NP || jj < 0 || jj >= NP) continue;
                const double kap = (di[n] != 0 && dj[n] != 0) ? kd : 1.0;
                const double t = xv - x[(size_t)ii * NP + jj], u = t * id;
                const double om = 1.0 / sqrt(1.0 + u * u);
                gs += kap * t * om;
                cs += kap * om;
                /* forward neighbours (right, down-left, down, down-right) carry the pair's value */
                if (di[n] > 0 || (di[n] == 0 && dj[n] > 0)) val += kap * delta * delta * (sqrt(1.0 + u * u) - 1.0);
            }
            if (g) g[(size_t)i * NP + j] = gs;
            if (c) c[(size_t)i * NP + j] = 2.0 * cs;
        }
    return val;
}

static void to_native(const double *in, double *out, int flip)
{
    for (int i = 0; i < NP; ++i)
        for (int j = 0; j < NP; ++j) out[(size_t)i * NP + j] = in[(size_t)i * NP + (flip ? NP - 1 - j : j)];
}

/* img [batch][512][512] (frame flip) -> val [batch], grad / curv [batch][512][512] (frame flip; either may be NULL) */
void pwls_penalty_oracle(const double *img, double *val, double *grad, double *curv, int batch, int flip, double delta)
{
    double *xn = malloc(sizeof(double) * NP * NP), *g = malloc(sizeof(double) * NP * NP), *c = malloc(sizeof(double) * NP * NP);
    for (int b = 0; b < batch; ++b) {
        to_native(img + (size_t)b * NP * NP, xn, flip);
        val[b] = penalty_native(xn, g, c, delta);
        if (grad) to_native(g, grad + (size_t)b * NP * NP, flip);   /* the column mirror is its own inverse */
        if (curv) to_native(c, curv + (size_t)b * NP * NP, flip);
    }
    free(xn); free(g); free(c);
}

typedef struct {
    double ca[ND], sa[ND];
    const double *theta;
    double D, dx;
} geom_t;

static void geom_init(geom_t *G, const double *theta, const double *alpha, double D, double dx)
{
    for (int k = 0; k < ND; ++k) { G->ca[k] = cos(alpha[k]); G->sa[k] = sin(alpha[k]); }
    G->theta = theta; G->D = D; G->dx = dx;
}

/* native out = A^T y over the views s + n S (n < NV / S), y(v, k) = w(b) * (b - [A x]) (x non-NULL) or w(b) * [A 1] (x NULL),
 * b[v][k] read in the sinogram's frame; buf: per-thread scratch [nt][512][512].  Returns sum of 1/2 w (A x - b)^2 over the
 * views when x is given (the data term restricted to them). */
static double weighted_backproject(const float *bs, const double *x, double *out, double *buf, int s, int S, int flip, double dose,
                                   const geom_t *G)
{
    const int nv = NV / S, nt = n_threads();
    double *ones = NULL;
    if (!x) {
        ones = malloc(sizeof(double) * NP * NP);
        for (long q = 0; q < (long)NP * NP; ++q) ones[q] = 1.0;
    }
    double val = 0.0;
    memset(buf, 0, sizeof(double) * (size_t)nt * NP * NP);
#pragma omp parallel num_threads(nt) reduction(+ : val)
    {
        double *mine = buf + (size_t)thread_id() * NP * NP;
#pragma omp for schedule(static)
        for (int q = 0; q < nv; ++q) {
            const int v = s + q * S;
            const double ct = cos(G->theta[v]), st = sin(G->theta[v]);
            for (int k = 0; k < ND; ++k) {
                const ray_t r = ray_setup(ct, st, G->ca[k], G->sa[k], G->D, G->dx);
                const double b = (double)bs[(size_t)v * ND + (flip ? ND - 1 - k : k)], w = weight(b, dose);
                double y;
                if (x) {
                    const double res = b - ray_project(x, &r);
                    val += 0.5 * w * res * res;
                    y = w * res;
                } else {
                    y = w * ray_project(ones, &r);
                }
                ray_scatter(mine, &r, y);
            }
        }
    }
    reduce(buf, nt, out);
    free(ones);
    return val;
}

/* sino [batch][2000][912] f32 (frame flip) -> D^L [batch][512][512] (frame flip) */
void pwls_denom_oracle(const float *sino, double *dl, int batch, int flip, double dose, const double *theta, const double *alpha,
                       double D, double dx)
{
    geom_t G;
    geom_init(&G, theta, alpha, D, dx);
    double *n = malloc(sizeof(double) * NP * NP), *buf = malloc(sizeof(double) * (size_t)n_threads() * NP * NP);
    for (int b = 0; b < batch; ++b) {
        weighted_backproject(sino + (size_t)b * NV * ND, NULL, n, buf, 0, 1, flip, dose, &G);
        to_native(n, dl + (size_t)b * NP * NP, flip);
    }
    free(n); free(buf);
}

/* the data term L(x) = 1/2 sum w (A x - b)^2 of every slice -> val [batch], and grad L = A^T (w o (A x - b)) (frame flip) when
 * grad is non-NULL */
void pwls_data_oracle(const float *sino, const double *img, double *val, double *grad, int batch, int flip, double dose,
                      const double *theta, const double *alpha, double D, double dx)
{
    geom_t G;
    geom_init(&G, theta, alpha, D, dx);
    double *xn = malloc(sizeof(double) * NP * NP), *n = malloc(sizeof(double) * NP * NP);
    double *buf = malloc(sizeof(double) * (size_t)n_threads() * NP * NP);
    for (int b = 0; b < batch; ++b) {
        to_native(img + (size_t)b * NP * NP, xn, flip);
        val[b] = weighted_backproject(sino + (size_t)b * NV * ND, xn, n, buf, 0, 1, flip, dose, &G);
        if (grad) {
            double *o = grad + (size_t)b * NP * NP;
            to_native(n, o, flip);
            for (long q = 0; q < (long)NP * NP; ++q) o[q] = -o[q];
        }
    }
    free(xn); free(n); free(buf);
}

/* OS-SQS from x0 ([batch][512][512] f64, frame flip, clamped at 0; NULL: 0): img [batch][512][512] (frame flip) after `iterations`
 * sweeps, history (NULL or [batch][iterations][512][512]) after every sweep */
void pwls_oracle(const float *sino, const double *x0, double *img, double *history, int batch, int flip, int iterations, int S,
                 double dose, double beta, double delta, const double *theta, const double *alpha, double D, double dx)
{
    geom_t G;
    geom_init(&G, theta, alpha, D, dx);
    const int step = sart_visit_step(S);
    double *x = malloc(sizeof(double) * NP * NP), *bp = malloc(sizeof(double) * NP * NP), *dl = malloc(sizeof(double) * NP * NP);
    double *g = malloc(sizeof(double) * NP * NP), *c = malloc(sizeof(double) * NP * NP);
    double *buf = malloc(sizeof(double) * (size_t)n_threads() * NP * NP);
    for (int b = 0; b < batch; ++b) {
        const float *bs = sino + (size_t)b * NV * ND;
        weighted_backproject(bs, NULL, dl, buf, 0, 1, flip, dose, &G);
        if (x0) {
            to_native(x0 + (size_t)b * NP * NP, x, flip);
            for (long q = 0; q < (long)NP * NP; ++q) x[q] = fmax(0.0, x[q]);
        } else {
            memset(x, 0, sizeof(double) * NP * NP);
        }
        for (int it = 0; it < iterations; ++it) {
            for (int n = 0; n < S; ++n) {
                const int s = (int)((long long)n * step % S);
                penalty_native(x, g, c, delta);
                weighted_backproject(bs, x, bp, buf, s, S, flip, dose, &G);
#pragma omp parallel for schedule(static)
                for (long q = 0; q < (long)NP * NP; ++q) {
                    const double den = dl[q] + beta * c[q];
                    if (den > 0.0) x[q] = fmax(0.0, x[q] + (S * bp[q] - beta * g[q]) / den);
                }
            }
            if (history) to_native(x, history + ((size_t)b * iterations + it) * NP * NP, flip);
        }
        to_native(x, img + (size_t)b * NP * NP, flip);
    }
    free(x); free(bp); free(dl); free(g); free(c); free(buf);
}
