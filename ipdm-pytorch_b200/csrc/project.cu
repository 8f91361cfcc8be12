// Low-dose input simulation for sm_100a: fan-beam forward projector (an operation of the FBP plan) and the dose-reduction
// noise of the reference's Utils/Low_dose_CT_simulate.py add_noise (:38-44).
//
// Geometry: exactly the rays synthetic.fan_sinogram traces and the backprojector reads (fbp.cu): source at D = 59.5 cm, view
// theta_v = v * 0.18 deg, filtered sample k read at fan angle alpha_k = nda[k] + da/2, pixel (i, j) centred at
// x = (j - 255.5) dx, y = (255.5 - i) dx, dx = 42/512 cm, zero outside the grid.  In the native frame the ray (v, k) is the line
//   x sin(phi) + y cos(phi) = D sin(alpha_k),   phi = theta_v - alpha_k,   direction (cos phi, -sin phi).
//
// Discrete model: Joseph's method.  Along the dominant axis of the ray (columns j when |cos phi| >= |sin phi|, rows i otherwise)
// one sample per column / row m, at the fractional index u(m) = u0 + (m - 255.5) g of the other axis, linear between the two pixel
// centres that straddle it (weights in fp32, no texture filtering), times the step dx / |cos| (or |sin|); fp32 accumulation in
// ascending m.  The test suite's C checker restates the same sums in fp64.  The per-ray setup (u0, g, dominant axis, step) is
// joseph_ray in fbp_plan.cuh, which the adjoint (sart.cu) evaluates too.
//
// Kernel 1  project_transpose_kernel  one 32 x 32 tile per CTA: T[b][j][i] = native[b][i][j].  Column-major rays then read T
//           along a row, so a warp of adjacent detectors reads adjacent words of one row in either case (1 MB per slice).
// Kernel 2  fbp_project_kernel        one thread per ray (of all views, or of one SART subset), a warp on 32 adjacent detectors
//           of one view; each ray only loops over
//           the columns / rows where it is inside the grid.  Bound: gather through L1 (about 0.75 G samples, 2 loads each, per
//           slice; compulsory HBM bytes 1 MB image + 7.3 MB sinogram per slice).
// Kernel 3  low_dose_noise_kernel     one thread per 4 bins: out = p + sqrt((1-f) e^p (1 + (1+f) Ne e^p / (f N0)) / (f N0)) n,
//           n from the caller's tape or Philox keyed by (seed, slice id, bin / 4).  HBM bound (8 or 12 bytes per bin).
#include "fbp_plan.cuh"

#include <cmath>

namespace ipdm {

constexpr int NV = IPDM_N_VIEWS, ND = IPDM_N_DET, NP = IPDM_N_PIX;
constexpr int PROJ_THREADS = 256;

__global__ void __launch_bounds__(256) project_transpose_kernel(const float* __restrict__ img, float* __restrict__ t, int flip) {
    __shared__ float tile[32][33];
    const size_t off = (size_t)blockIdx.z * NP * NP;
    const int i0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
#pragma unroll
    for (int r = threadIdx.y; r < 32; r += 8) tile[r][threadIdx.x] = img[off + (size_t)(i0 + r) * NP + c0 + threadIdx.x];
    __syncthreads();
#pragma unroll
    for (int c = threadIdx.y; c < 32; c += 8) {
        const int j = flip ? NP - 1 - (c0 + c) : c0 + c;               // native column
        t[off + (size_t)j * NP + i0 + threadIdx.x] = tile[threadIdx.x][c];
    }
}

// sum over m in [m_lo, m_hi] of the linear interpolation of row m of `plane` at u(m) = u0 + (m - 255.5) g; MIRROR reads column
// NP-1-k for k (a column-flipped image read in the native frame)
template <bool MIRROR>
__device__ __forceinline__ float joseph_sum(const float* __restrict__ plane, int m_lo, int m_hi, float u0, float g) {
    float acc = 0.f;
#pragma unroll 4
    for (int m = m_lo; m <= m_hi; ++m) {
        const float u = fmaf((float)m - 255.5f, g, u0);
        const float kf = floorf(u);
        const int k = (int)kf;
        const float w = u - kf;
        const float* row = plane + (size_t)m * NP;
        const float v0 = (unsigned)k < (unsigned)NP ? __ldg(row + (MIRROR ? NP - 1 - k : k)) : 0.f;
        const float v1 = (unsigned)(k + 1) < (unsigned)NP ? __ldg(row + (MIRROR ? NP - 2 - k : k + 1)) : 0.f;
        acc += fmaf(w, v1 - v0, v0);
    }
    return acc;
}

// rays of the views v0 + n * vstep, n < nv (all 2000 views: 0, 1, 2000); sino is [B][nv][912]
__global__ void __launch_bounds__(PROJ_THREADS)
fbp_project_kernel(const float* __restrict__ img, const float* __restrict__ imgT, float* __restrict__ sino,
                   const float2* __restrict__ cs_view, const float2* __restrict__ cs_ray, int flip, int v0, int vstep, int nv) {
    const int ray = blockIdx.x * PROJ_THREADS + threadIdx.x;          // n * ND + k
    if (ray >= nv * ND) return;
    const int n = ray / ND, k = ray - n * ND;
    const size_t b = blockIdx.y;
    const JosephRay r = joseph_ray(__ldg(cs_view + v0 + n * vstep), __ldg(cs_ray + k));
    const float u0 = r.u0, g = r.g;
    // columns / rows where -1 <= u < 512 (the only ones with a non-zero tap), one of slack on either side
    int m_lo = 0, m_hi = NP - 1;
    if (fabsf(g) > 1e-6f) {
        const float ma = 255.5f + (-1.0f - u0) / g, mb = 255.5f + (512.0f - u0) / g;
        m_lo = max(0, (int)floorf(fmaxf(fminf(ma, mb), -2.0f)) - 1);
        m_hi = min(NP - 1, (int)ceilf(fminf(fmaxf(ma, mb), (float)NP + 1.0f)) + 1);
    }
    float acc;
    if (r.xmajor) acc = joseph_sum<false>(imgT + b * NP * NP, m_lo, m_hi, u0, g);
    else if (flip) acc = joseph_sum<true>(img + b * NP * NP, m_lo, m_hi, u0, g);
    else acc = joseph_sum<false>(img + b * NP * NP, m_lo, m_hi, u0, g);
    sino[b * nv * ND + (size_t)n * ND + (flip ? ND - 1 - k : k)] = acc * r.scale;
}

__global__ void __launch_bounds__(256)
low_dose_noise_kernel(const float* sino, const float* __restrict__ noise, float* out, size_t n, float ka, float kc, int clip,
                      uint64_t seed, const uint64_t* __restrict__ slice_ids) {
    const size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t e0 = 4 * q;
    if (e0 >= n) return;
    const size_t base = (size_t)blockIdx.y * n;
    float nz[4];
    if (!noise) {
        const uint64_t sid = slice_ids ? slice_ids[blockIdx.y] : (uint64_t)blockIdx.y;
        const float4 r = philox_normal4_keyed((uint32_t)q, (uint32_t)sid, (uint32_t)(sid >> 32), 0u, (uint32_t)seed, (uint32_t)(seed >> 32));
        nz[0] = r.x; nz[1] = r.y; nz[2] = r.z; nz[3] = r.w;
    }
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const size_t i = e0 + e;
        if (i >= n) break;
        const float pv = sino[base + i];
        const float ex = expf(pv);
        const float nv = noise ? noise[base + i] : nz[e];
        float r = fmaf(sqrtf(ka * ex * fmaf(kc, ex, 1.0f)), nv, pv);
        if (clip) r = fmaxf(r, 0.0f);
        out[base + i] = r;
    }
}

int launch_project(ipdm_fbp_plan* p, const float* img, float* sino, int batch, int flip, int v0, int vstep, int nv, cudaStream_t st) {
    IPDM_CHECK(p->work.reserve(work_bytes(batch)));
    float* imgT = p->work.f32();
    project_transpose_kernel<<<dim3(NP / 32, NP / 32, batch), dim3(32, 8), 0, st>>>(img, imgT, flip);
    count_launch();
    IPDM_CHECK_LAUNCH();
    fbp_project_kernel<<<dim3(ceil_div((long long)nv * ND, PROJ_THREADS), batch), PROJ_THREADS, 0, st>>>(img, imgT, sino, p->d_cs,
                                                                                                          p->d_ray, flip, v0, vstep, nv);
    count_launch();
    IPDM_CHECK_LAUNCH();
    return IPDM_OK;
}

}  // namespace ipdm

using namespace ipdm;

extern "C" int ipdm_fbp_project(ipdm_fbp_plan* p, const float* img, float* sino, int batch, int flip, void* stream) {
    IPDM_REQUIRE(p && img && sino && batch > 0 && batch <= 65535, "ipdm_fbp_project: bad arguments");
    return launch_project(p, img, sino, batch, flip, 0, 1, NV, (cudaStream_t)stream);
}

extern "C" int ipdm_low_dose_noise(const float* sino, const float* noise, float* out, int batch, size_t n_per_slice, float dose,
                                   int clip, uint64_t seed, const uint64_t* slice_ids, void* stream) {
    IPDM_REQUIRE(sino && out && batch > 0 && batch <= 65535 && n_per_slice > 0 && n_per_slice / 4 < (1ull << 32),
                 "ipdm_low_dose_noise: bad arguments");
    IPDM_REQUIRE(dose > 0.f && dose <= 1.f, "ipdm_low_dose_noise: dose must be in (0, 1], got %g", (double)dose);
    const double f = dose, ne = kDoseNe, n0 = kDoseN0;
    const float ka = (float)((1.0 - f) / (f * n0)), kc = (float)((1.0 + f) * ne / (f * n0));
    const size_t quads = (n_per_slice + 3) / 4;
    low_dose_noise_kernel<<<dim3(ceil_div((long long)quads, 256), batch), 256, 0, (cudaStream_t)stream>>>(
        sino, noise, out, n_per_slice, ka, kc, clip, seed, slice_ids);
    count_launch();
    IPDM_CHECK_LAUNCH();
    return IPDM_OK;
}
