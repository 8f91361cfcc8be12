// The FBP plan (geometry tables + workspace), shared by the convertor (fbp.cu), the forward projector (project.cu) and its
// adjoint / SART (sart.cu), and the device helpers more than one of them evaluates.
#pragma once
#include "common.cuh"

#include <map>
#include <vector>

namespace ipdm {

struct FbpTables {
    std::vector<double> theta;   // [2000]
    std::vector<float> nda;      // [912]
    std::vector<float> h;        // [1823]
    std::vector<float> wcos;     // [912]
    double dtheta, D, da;
};

}  // namespace ipdm

struct ipdm_fbp_plan {
    ipdm::FbpTables host;
    float* d_wcos = nullptr;     // [912]
    float* d_htap = nullptr;     // [2][911]  H_c[d + 455] = h[2d + 2c - 1 + 911]
    float2* d_cs = nullptr;      // [2000] (cos theta, sin theta) from fp64
    float2* d_ray = nullptr;     // [912] (cos alpha, sin alpha) from fp64, alpha = nda[k] + da/2: the fan angle filtered sample k is read at
    float* d_work = nullptr;     // filtered sinograms [cap][2000][912]; the projector's transposed images [cap][512][512]
    int cap = 0;
    float h0 = 0.f, inv_da = 0.f, u_off = 0.f, dtheta_f = 0.f;
    double dtheta = 0.0;
    // SART (sart.cu): row sums R = A 1 [2000][912] (native detector order), column sums C_s = A_s^T 1 [S][512][512] (native
    // columns) per subset count S, and the subset projections [sart_bytes / 4]; all built by the first call that needs them
    float* d_rowsum = nullptr;
    std::map<int, float*> colsum;
    float* d_sart = nullptr;
    size_t sart_bytes = 0;
};

namespace ipdm {
// grows plan->d_work to `batch` filtered sinograms (it is never shrunk)
int ensure_workspace(ipdm_fbp_plan* plan, int batch);
// frees the SART tables and workspace (sart.cu)
void release_sart(ipdm_fbp_plan* plan);
// transpose + Joseph projection of the views v0 + n * vstep, n < nv: img [B][512][512] -> sino [B][nv][912] (project.cu)
int launch_project(ipdm_fbp_plan* p, const float* img, float* sino, int batch, int flip, int v0, int vstep, int nv, cudaStream_t st);

// atan(t) = t * P(t^2), |t| <= 0.62, |err| < 1.3e-10 in exact arithmetic (fit: see DESIGN.md)
__device__ __forceinline__ float atan_small(float t) {
    const float z = t * t;
    float p = -2.018183097e-02f;
    p = fmaf(p, z, 5.469628051e-02f);
    p = fmaf(p, z, -8.460120857e-02f);
    p = fmaf(p, z, 1.100626141e-01f);
    p = fmaf(p, z, -1.427598149e-01f);
    p = fmaf(p, z, 1.999954879e-01f);
    p = fmaf(p, z, -3.333332539e-01f);
    p = fmaf(p, z, 1.0f);
    return t * p;
}

// One Joseph ray in the native frame (see project.cu): the line x sin(phi) + y cos(phi) = D sin(alpha), phi = theta - alpha, from
// th = (cos theta, sin theta) and al = (cos alpha, sin alpha).  Along the dominant axis (columns j when xmajor, rows i otherwise)
// the sample of column / row m sits at the fractional index joseph_u(r, m) of the other axis; the sum of the samples is scaled by
// `scale` = dx / |cos| (or |sin|).  The projector and its adjoint both take their weights from here, so the adjoint is the exact
// transpose of the fp32 matrix the projector applies.
struct JosephRay {
    float u0, g, scale;
    bool xmajor;
};

__device__ __forceinline__ JosephRay joseph_ray(float2 th, float2 al) {
    constexpr float dx = 42.0f / 512.0f;
    const float cphi = fmaf(th.x, al.x, th.y * al.y);                // cos(theta - alpha)
    const float sphi = fmaf(th.y, al.x, -th.x * al.y);               // sin(theta - alpha)
    const float p = (59.5f / dx) * al.y;                              // D sin(alpha) in pixel units
    JosephRay r;
    r.xmajor = fabsf(cphi) >= fabsf(sphi);
    // x-major: row index r(j) = 255.5 - p / cos + (j - 255.5) tan;  y-major: column index c(i) = 255.5 + p / sin + (i - 255.5) cot
    const float a = r.xmajor ? cphi : sphi, o = r.xmajor ? sphi : cphi;
    const float ra = 1.0f / a;
    r.u0 = r.xmajor ? fmaf(-p, ra, 255.5f) : fmaf(p, ra, 255.5f);
    r.g = o * ra;
    r.scale = dx * fabsf(ra);
    return r;
}

__device__ __forceinline__ float joseph_u(const JosephRay& r, int m) { return fmaf((float)m - 255.5f, r.g, r.u0); }

}  // namespace ipdm
