// The FBP plan (geometry tables + workspace), shared by the convertor (fbp.cu), the forward projector (project.cu), its
// adjoint / SART / PWLS (sart.cu), the TV steps (tv.cu) and the PWLS penalty (pwls.cu), and the device helpers more than one of
// them evaluates.
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

// a device buffer that grows to the largest size a call has asked of it and is never shrunk, so that after the first call of a
// shape a call allocates nothing; it holds nothing from one call to the next
struct GrowBuffer {
    void* ptr = nullptr;
    size_t bytes = 0;
    int reserve(size_t need) {
        if (need <= bytes) return IPDM_OK;
        IPDM_CHECK_CUDA(cudaFree(ptr));
        ptr = nullptr;
        bytes = 0;
        IPDM_CHECK_CUDA(cudaMalloc(&ptr, need));
        bytes = need;
        return IPDM_OK;
    }
    void release() {
        cudaFree(ptr);
        ptr = nullptr;
        bytes = 0;
    }
    float* f32() const { return static_cast<float*>(ptr); }
};

}  // namespace ipdm

struct ipdm_fbp_plan {
    ipdm::FbpTables host;
    float* d_wcos = nullptr;     // [912]
    float* d_htap = nullptr;     // [2][911]  H_c[d + 455] = h[2d + 2c - 1 + 911]
    float2* d_cs = nullptr;      // [2000] (cos theta, sin theta) from fp64
    float2* d_ray = nullptr;     // [912] (cos alpha, sin alpha) from fp64, alpha = nda[k] + da/2: the fan angle filtered sample k is read at
    float h0 = 0.f, inv_da = 0.f, u_off = 0.f, dtheta_f = 0.f;
    double dtheta = 0.0;
    // SART (sart.cu): row sums R = A 1 [2000][912] (native detector order) and column sums C_s = A_s^T 1 [S][512][512] (native
    // columns) per subset count S, built by the first call that needs them and kept
    float* d_rowsum = nullptr;
    std::map<int, float*> colsum;
    // per-call scratch, laid out for the call's batch B.  work: the filtered sinograms [B][2000][912], or the projector's transposed
    // images [B][512][512], always reserved at the sinograms' size (work_bytes) so that only a larger batch grows it
    ipdm::GrowBuffer work;
    ipdm::GrowBuffer subset;     // the subset projections A_s x [B][2000 / S][912] (SART, PWLS)
    ipdm::GrowBuffer tv;         // the TV steps (tv.cu): see tv_scratch_bytes
    ipdm::GrowBuffer pwls;       // PWLS: D^L, grad R and d^R [B][512][512] f32 each
};

namespace ipdm {
inline size_t work_bytes(int batch) { return (size_t)batch * IPDM_N_VIEWS * IPDM_N_DET * sizeof(float); }
// the TV scratch of `batch` slices in plan->tv: x_prev (the iterate before a SART sweep, first, so at plan->tv.ptr) and g
// [B][512][512] f32, per-tile partial sums [B][2][256] and step lengths [B] f64 (tv.cu)
size_t tv_scratch_bytes(int batch);
// `steps` TV steps on img [B][512][512] (column-flipped iff flip), in place, in plan->tv (reserved by the caller for `batch`).
// sweep: the step length is alpha_or_step times |img - x_prev| of each slice, taken at the first step; otherwise alpha_or_step
// itself (tv.cu)
int launch_tv(ipdm_fbp_plan* p, float* img, int batch, int flip, int steps, bool sweep, double alpha_or_step, float eps, cudaStream_t st);
// grad R and d^R of the hyperbola penalty of img [B][512][512] (column-flipped iff flip), in the same frame (pwls.cu)
int launch_pwls_penalty(const float* img, float* grad, float* curv, int batch, int flip, float delta, cudaStream_t st);
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
