/*
 * TEST INFRASTRUCTURE ONLY -- fp64 restatement of the forward projector (ipdm_fbp_project, csrc/project.cu).
 *
 * Equiangular fan beam in the geometry of the reference FBP (Recon/FBP_kernel.py:32-44) and of
 * synthetic.fan_sinogram: source at D, view angle theta[v], ray k at fan angle alpha[k] (= nda[k] + da/2),
 * pixel (i, j) centred at x = (j - 255.5) dx, y = (255.5 - i) dx, zero outside the grid.  In the native
 * frame ray (v, k) is the line x sin(phi) + y cos(phi) = D sin(alpha), phi = theta - alpha.
 *
 * Joseph's method: along the dominant axis (columns j when |cos phi| >= |sin phi|, rows i otherwise) one
 * sample per column / row m at the fractional index u(m) = u0 + (m - 255.5) g of the other axis, linear
 * between the two pixel centres that straddle it, sum times dx / |cos| (or |sin|).  Every m of the grid is
 * visited (taps outside the grid read 0), in ascending order, in fp64.
 *
 * flip = 1: img is column-flipped (the convertor's output frame), sino is written with the detector axis
 * reversed (its input frame); flip = 0: both native.  Threads split the views.
 * Nothing under ipdm-pytorch_b200/ links or loads this file.
 */
#include <math.h>
#include <stddef.h>

#define ND 912
#define NP 512

static double pix(const float *img, int i, int j, int flip)
{
    if (i < 0 || i >= NP || j < 0 || j >= NP) return 0.0;
    return (double)img[(size_t)i * NP + (flip ? NP - 1 - j : j)];
}

/* one ray: theta / alpha given by their cos and sin */
static double ray_sum(const float *img, double ct, double st, double ca, double sa, double D, double dx, int flip)
{
    const double c = ct * ca + st * sa, s = st * ca - ct * sa;   /* cos, sin of phi = theta - alpha */
    const double p = D * sa / dx;
    const int xmajor = fabs(c) >= fabs(s);
    const double a = xmajor ? c : s, o = xmajor ? s : c;
    const double u0 = xmajor ? 255.5 - p / a : 255.5 + p / a, g = o / a;
    double acc = 0.0;
    for (int m = 0; m < NP; ++m) {
        const double u = u0 + (m - 255.5) * g;
        const double kf = floor(u);
        const int k = (int)kf;
        const double w = u - kf;
        double v0, v1;
        if (xmajor) { v0 = pix(img, k, m, flip); v1 = pix(img, k + 1, m, flip); }   /* column m, rows k, k+1 */
        else        { v0 = pix(img, m, k, flip); v1 = pix(img, m, k + 1, flip); }   /* row m, columns k, k+1 */
        acc += v0 + w * (v1 - v0);
    }
    return acc * dx / fabs(a);
}

/* img [batch][512][512] -> sino [batch][nv][912]; theta [nv] (all 2000 views, or a subset), alpha [912] in radians */
void project_oracle(const float *img, double *sino, int batch, int nv, int flip, const double *theta, const double *alpha, double D,
                    double dx)
{
    for (int b = 0; b < batch; ++b) {
        const float *im = img + (size_t)b * NP * NP;
        double *out = sino + (size_t)b * nv * ND;
#pragma omp parallel for schedule(static)
        for (int v = 0; v < nv; ++v) {
            const double ct = cos(theta[v]), st = sin(theta[v]);
            for (int k = 0; k < ND; ++k)
                out[(size_t)v * ND + (flip ? ND - 1 - k : k)] = ray_sum(im, ct, st, cos(alpha[k]), sin(alpha[k]), D, dx, flip);
        }
    }
}
