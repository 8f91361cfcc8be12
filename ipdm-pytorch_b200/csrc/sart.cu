// Iterative convertor for sm_100a: the exact adjoint of the forward projector (project.cu) and ordered-subset SART around the
// projector / adjoint pair, in the FBP plan's geometry and flip frames, optionally started from the FBP image and regularised by
// TV steps between the sweeps (SART-TV, tv.cu).  A new convertor, not a port of the reference's Windows-only TASART2DNSL0.pyd:
// its area-integral projector and its NSL0 formula are not ported (the TV steps here are ASD-POCS on a smoothed isotropic TV).
//
// A is the fp32 matrix ipdm_fbp_project applies: ray (v, k) samples column / row m of its dominant axis at u = joseph_u(m) and
// puts the weights 1 - w on pixel floor(u) and w on floor(u) + 1 of the other axis (w = u - floor(u)), times the ray's step.
//
// Kernel 1  fbp_adjoint_kernel<SART>  pixel-driven gather, one CTA per 32 x 32 pixel tile and slice, ascending views.  Per
//           16-view chunk the CTA stages, for the detector segment its tile can touch, each ray's (u0, g, step * value, axis)
//           in shared memory; the ray setup is joseph_ray, so every weight is the projector's own fp32 weight.  A pixel then
//           tries the rays within dx / (L da) + 1 pitches of its own fan angle (L its distance from the source): a ray passes
//           within one pixel pitch of every pixel it touches.  About 5-7 candidates per (view, pixel), each one FMA for u, a
//           floor and a compare.  No atomics: each output pixel is one thread's sum in a fixed order.
//           SART: the staged value is the ray's residual (b - A_s x) / R (0 where R = 0), and the epilogue applies
//           x <- max(0, x + lambda * A_s^T r / C_s) (pixels with C_s = 0 keep x).  Bound: FP32 issue on the candidate loop.
// Kernel 2  fill_kernel                the all-ones image / sinogram the tables R = A 1 and C_s = A_s^T 1 are computed from.
// Kernel 3  clamp_nonneg_kernel        x0 = max(0, FBP) of the FBP start.
// SART-TV: before every sweep the iterate is copied to the TV workspace's x_prev, after it ntv TV steps run (launch_tv).
#include "fbp_plan.cuh"

#include <cmath>
#include <cstdint>
#include <numeric>

namespace ipdm {

constexpr int NV = IPDM_N_VIEWS, ND = IPDM_N_DET, NP = IPDM_N_PIX;
constexpr int ADJ_VC = 16;                 // views per staged chunk
constexpr int ADJ_SEG = 160;               // staged rays per view (a 32 x 32 tile touches at most about 135)
constexpr int ADJ_RPT = 4;                 // pixel rows per thread
constexpr int ADJ_TH = 8 * ADJ_RPT;        // tile rows
constexpr float DXP = 42.0f / 512.0f;

// continuous ray index kc of the pixel centre (x, y) in view cs = (cos theta, sin theta), and the half width hw of its candidate
// window: dx / (L da) pitches plus one of slack (the rounding of kc is about 1e-4 pitch)
__device__ __forceinline__ void pixel_window(float x, float y, float2 cs, float inv_da, float k_off, float& kc, float& hw) {
    const float s = fmaf(x, cs.y, y * cs.x);
    const float c = fmaf(x, cs.x, fmaf(-y, cs.y, 59.5f));
    kc = fmaf(atan_small(s * __frcp_rn(c)), inv_da, k_off);
    hw = fmaf(DXP * inv_da, rsqrtf(fmaf(s, s, c * c)), 1.0f);
}

// staged entry of ray (v, k): (u0, g, step * value, xmajor); value = y[v][k'] (plain adjoint) or the SART residual of the ray,
// k' = k in the sinogram's frame.  yb / pb / R are per-slice; pb (the subset projection, row n) is null when x = 0.
template <bool SART>
__device__ __forceinline__ float4 adj_entry(const float* __restrict__ yb, const float* __restrict__ pb, const float* __restrict__ R,
                                            const float2* __restrict__ cs_view, const float2* __restrict__ cs_ray, int v, int n, int k,
                                            int flip) {
    const JosephRay r = joseph_ray(__ldg(cs_view + v), __ldg(cs_ray + k));
    const int kk = flip ? ND - 1 - k : k;
    float val = __ldg(yb + (size_t)v * ND + kk);
    if (SART) {
        const float rs = __ldg(R + (size_t)v * ND + k);
        if (pb) val -= __ldg(pb + (size_t)n * ND + kk);
        val = rs > 0.f ? val / rs : 0.f;
    }
    return make_float4(r.u0, r.g, r.scale * val, r.xmajor ? 1.f : 0.f);
}

// the same, out of line: a ray outside the staged segment (kept off the candidate loop's registers)
template <bool SART>
__device__ __noinline__ float4 adj_entry_far(const float* yb, const float* pb, const float* R, const float2* cs_view, const float2* cs_ray,
                                             int v, int n, int k, int flip) {
    return adj_entry<SART>(yb, pb, R, cs_view, cs_ray, v, n, k, flip);
}

// views v0 + n * vstep, n < nv.  y: [B][2000][912] (the sinogram, or b for SART); psub: [B][nv][912] A_s x (SART, may be null);
// R: [2000][912]; colsum: C_s [512][512] native; img: written (plain) or updated in place (SART), column-flipped iff flip
template <bool SART>
__global__ void __launch_bounds__(256)
fbp_adjoint_kernel(const float* __restrict__ y, const float* __restrict__ psub, const float* __restrict__ R,
                   const float* __restrict__ colsum, float* __restrict__ img, const float2* __restrict__ cs_view,
                   const float2* __restrict__ cs_ray, int v0, int vstep, int nv, float inv_da, float k_off, float lambda, int flip) {
    __shared__ float4 seg[ADJ_VC][ADJ_SEG];
    __shared__ int seg0[ADJ_VC];
    __shared__ float2 scs[ADJ_VC];
    const int tid = threadIdx.x, lane = tid & 31, wrp = tid >> 5;
    const int j = blockIdx.x * 32 + lane;                    // native column
    const int i_base = blockIdx.y * ADJ_TH + wrp;            // first row of this thread
    const float* yb = y + (size_t)blockIdx.z * NV * ND;
    const float* pb = psub ? psub + (size_t)blockIdx.z * nv * ND : nullptr;
    const float x = ((float)j - 255.5f) * DXP;
    float yp[ADJ_RPT], acc[ADJ_RPT];
#pragma unroll
    for (int p = 0; p < ADJ_RPT; ++p) { yp[p] = (255.5f - (float)(i_base + 8 * p)) * DXP; acc[p] = 0.f; }
    const float xc0 = ((float)(blockIdx.x * 32) - 255.5f) * DXP, xc1 = xc0 + 31 * DXP;
    const float yc0 = (255.5f - (float)(blockIdx.y * ADJ_TH)) * DXP, yc1 = yc0 - (ADJ_TH - 1) * DXP;

    for (int c0 = 0; c0 < nv; c0 += ADJ_VC) {
        const int nvc = min(ADJ_VC, nv - c0);
        __syncthreads();                                     // previous chunk consumed
        if (tid < nvc) {                                     // segment: the tile's fan-angle range (extremes at its corners) +- 5
            const float2 c = __ldg(cs_view + v0 + (c0 + tid) * vstep);
            float kc, hw, kmin;
            pixel_window(xc0, yc0, c, inv_da, k_off, kc, hw); kmin = kc;
            pixel_window(xc1, yc0, c, inv_da, k_off, kc, hw); kmin = fminf(kmin, kc);
            pixel_window(xc0, yc1, c, inv_da, k_off, kc, hw); kmin = fminf(kmin, kc);
            pixel_window(xc1, yc1, c, inv_da, k_off, kc, hw); kmin = fminf(kmin, kc);
            seg0[tid] = max(0, min((int)floorf(kmin) - 5, ND - ADJ_SEG));
            scs[tid] = c;
        }
        __syncthreads();
        for (int e = tid; e < nvc * ADJ_SEG; e += 256) {
            const int vv = e / ADJ_SEG, o = e - vv * ADJ_SEG;
            seg[vv][o] = adj_entry<SART>(yb, pb, R, cs_view, cs_ray, v0 + (c0 + vv) * vstep, c0 + vv, seg0[vv] + o, flip);
        }
        __syncthreads();
        for (int vv = 0; vv < nvc; ++vv) {
            const float2 c = scs[vv];
            const int k0 = seg0[vv];
#pragma unroll
            for (int p = 0; p < ADJ_RPT; ++p) {
                const int i = i_base + 8 * p;
                float kc, hw;
                pixel_window(x, yp[p], c, inv_da, k_off, kc, hw);
                const int klo = max(0, (int)ceilf(kc - hw)), khi = min(ND - 1, (int)floorf(kc + hw));
                for (int k = klo; k <= khi; ++k) {
                    const int o = k - k0;
                    const float4 e = (unsigned)o < (unsigned)ADJ_SEG
                                         ? seg[vv][o]
                                         : adj_entry_far<SART>(yb, pb, R, cs_view, cs_ray, v0 + (c0 + vv) * vstep, c0 + vv, k, flip);
                    const bool xm = e.w != 0.f;
                    const float u = fmaf((float)(xm ? j : i) - 255.5f, e.y, e.x);     // joseph_u at this pixel's column / row
                    const float kf = floorf(u);
                    const int d = (xm ? i : j) - (int)kf;    // 0: tap floor(u), weight 1 - w; 1: tap floor(u) + 1, weight w
                    const float w = u - kf;
                    if (d == 0) acc[p] = fmaf(e.z, 1.0f - w, acc[p]);
                    else if (d == 1) acc[p] = fmaf(e.z, w, acc[p]);
                }
            }
        }
    }
    float* ob = img + (size_t)blockIdx.z * NP * NP;
    const int jo = flip ? NP - 1 - j : j;
#pragma unroll
    for (int p = 0; p < ADJ_RPT; ++p) {
        const int i = i_base + 8 * p;
        if (!SART) {
            ob[(size_t)i * NP + jo] = acc[p];
        } else {
            const float cs = __ldg(colsum + (size_t)i * NP + j);
            if (cs > 0.f) ob[(size_t)i * NP + jo] = fmaxf(0.f, fmaf(lambda, acc[p] / cs, ob[(size_t)i * NP + jo]));
        }
    }
}

__global__ void fill_kernel(float* p, float v, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

__global__ void clamp_nonneg_kernel(float4* p, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        float4 v = p[i];
        v.x = fmaxf(0.f, v.x); v.y = fmaxf(0.f, v.y); v.z = fmaxf(0.f, v.z); v.w = fmaxf(0.f, v.w);
        p[i] = v;
    }
}

template <bool SART>
static int launch_adjoint(ipdm_fbp_plan* p, const float* y, const float* psub, const float* colsum, float* img, int batch, int flip, int v0,
                          int vstep, int nv, float lambda, cudaStream_t st) {
    const float k_off = (float)(-0.5 - (double)p->host.nda[0] / p->host.da);     // ray k is at fan angle nda[0] + (k + 1/2) da
    fbp_adjoint_kernel<SART><<<dim3(NP / 32, NP / ADJ_TH, batch), 256, 0, st>>>(y, psub, p->d_rowsum, colsum, img, p->d_cs, p->d_ray, v0,
                                                                                vstep, nv, p->inv_da, k_off, lambda, flip);
    count_launch();
    IPDM_CHECK_LAUNCH();
    return IPDM_OK;
}

// visit order of the subsets: s_n = n * step mod S, step the integer in [1, S) coprime to S closest to 0.382 S (smaller on a tie)
static int sart_visit_step(int S) {
    if (S <= 2) return 1;
    const double t = 0.382 * S;
    int best = 1;
    double bd = 1e300;
    for (int q = 1; q < S; ++q)
        if (std::gcd(q, S) == 1 && std::fabs(q - t) < bd) { bd = std::fabs(q - t); best = q; }
    return best;
}

// R = A 1 (once per plan) and C_s = A_s^T 1 for every subset of S (once per plan and S), in fp32 with the same kernels
static int ensure_sart_tables(ipdm_fbp_plan* p, int S, cudaStream_t st) {
    const bool need_r = p->d_rowsum == nullptr, need_c = p->colsum.count(S) == 0;
    if (!need_r && !need_c) return IPDM_OK;
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    IPDM_CHECK_CUDA(cudaStreamIsCapturing(st, &cap));
    IPDM_REQUIRE(cap == cudaStreamCaptureStatusNone,
                 "ipdm_fbp_sart: the first call with %d subsets builds the plan's tables and cannot be captured; run it once eagerly", S);
    float* ones = nullptr;
    IPDM_CHECK_CUDA(cudaMalloc(&ones, (size_t)NV * ND * sizeof(float)));       // all-ones sinogram, and image (its first 512 x 512)
    int rc = IPDM_OK;
    fill_kernel<<<ceil_div(NV * ND, 256), 256, 0, st>>>(ones, 1.0f, NV * ND);
    count_launch();
    if (cudaGetLastError() != cudaSuccess) rc = IPDM_ERR_CUDA;
    if (rc == IPDM_OK && need_r) {
        if (cudaMalloc(&p->d_rowsum, (size_t)NV * ND * sizeof(float)) != cudaSuccess) rc = IPDM_ERR_CUDA;
        if (rc == IPDM_OK) rc = launch_project(p, ones, p->d_rowsum, 1, 0, 0, 1, NV, st);
    }
    if (rc == IPDM_OK && need_c) {
        float* c = nullptr;
        if (cudaMalloc(&c, (size_t)S * NP * NP * sizeof(float)) != cudaSuccess) rc = IPDM_ERR_CUDA;
        for (int s = 0; rc == IPDM_OK && s < S; ++s)
            rc = launch_adjoint<false>(p, ones, nullptr, nullptr, c + (size_t)s * NP * NP, 1, 0, s, S, NV / S, 0.f, st);
        if (rc == IPDM_OK) p->colsum[S] = c;
        else cudaFree(c);
    }
    if (cudaStreamSynchronize(st) != cudaSuccess && rc == IPDM_OK) rc = IPDM_ERR_CUDA;
    cudaFree(ones);
    if (rc == IPDM_ERR_CUDA) set_error("ipdm_fbp_sart: building the tables failed: %s", cudaGetErrorString(cudaGetLastError()));
    return rc;
}

void release_sart(ipdm_fbp_plan* p) {
    cudaFree(p->d_rowsum);
    cudaFree(p->d_sart);
    for (auto& kv : p->colsum) cudaFree(kv.second);
    p->d_rowsum = p->d_sart = nullptr;
    p->colsum.clear();
    p->sart_bytes = 0;
    release_tv(p);
}

// SART (ntv = 0) or SART-TV, from x0 = 0 (init_fbp = 0) or x0 = max(0, FBP(sino)) (init_fbp = 1); arguments checked by the callers
static int run_sart(ipdm_fbp_plan* p, const float* sino, float* img, int batch, int flip, int iterations, int subsets, float relaxation,
                    int ntv, float tv_alpha, float tv_eps, int init_fbp, cudaStream_t st) {
    IPDM_CHECK(ensure_sart_tables(p, subsets, st));
    IPDM_CHECK(ensure_workspace(p, batch));                                    // the projector's transposed iterates
    if (ntv > 0) IPDM_CHECK(ensure_tv_workspace(p, batch));                    // g, x_prev and the partial sums of the TV steps
    const int nv = NV / subsets;
    const size_t need = (size_t)batch * nv * ND * sizeof(float);               // A_s x of one subset
    if (need > p->sart_bytes) {
        IPDM_CHECK_CUDA(cudaFree(p->d_sart));
        p->d_sart = nullptr;
        p->sart_bytes = 0;
        IPDM_CHECK_CUDA(cudaMalloc(&p->d_sart, need));
        p->sart_bytes = need;
    }
    const float* colsum = p->colsum[subsets];
    const int step = sart_visit_step(subsets);
    const size_t img_bytes = (size_t)batch * NP * NP * sizeof(float);
    if (init_fbp) {                                                            // x0 = max(0, FBP(sino)), unsharpened
        IPDM_CHECK(ipdm_fbp_forward(p, sino, img, batch, flip, st));
        const size_t n4 = (size_t)batch * NP * NP / 4;
        clamp_nonneg_kernel<<<ceil_div((long long)n4, 256), 256, 0, st>>>(reinterpret_cast<float4*>(img), n4);
        count_launch();
        IPDM_CHECK_LAUNCH();
    } else {
        IPDM_CHECK_CUDA(cudaMemsetAsync(img, 0, img_bytes, st));              // x0 = 0
    }
    for (int it = 0; it < iterations; ++it) {
        if (ntv > 0) IPDM_CHECK_CUDA(cudaMemcpyAsync(tv_prev(p), img, img_bytes, cudaMemcpyDeviceToDevice, st));
        for (int n = 0; n < subsets; ++n) {
            const int s = (int)((long long)n * step % subsets);
            const float* proj = nullptr;                                       // A_s x0 = 0: the first subset from 0 needs no projection
            if (init_fbp || it > 0 || n > 0) {
                IPDM_CHECK(launch_project(p, img, p->d_sart, batch, flip, s, subsets, nv, st));
                proj = p->d_sart;
            }
            IPDM_CHECK(launch_adjoint<true>(p, sino, proj, colsum + (size_t)s * NP * NP, img, batch, flip, s, subsets, nv, relaxation, st));
        }
        if (ntv > 0) IPDM_CHECK(launch_tv(p, img, batch, flip, ntv, true, (double)tv_alpha, tv_eps, st));
    }
    return IPDM_OK;
}

}  // namespace ipdm

using namespace ipdm;

extern "C" int ipdm_fbp_project_adjoint(ipdm_fbp_plan* p, const float* sino, float* img, int batch, int flip, void* stream) {
    IPDM_REQUIRE(p && sino && img && batch > 0 && batch <= 65535, "ipdm_fbp_project_adjoint: bad arguments");
    return launch_adjoint<false>(p, sino, nullptr, nullptr, img, batch, flip, 0, 1, NV, 0.f, (cudaStream_t)stream);
}

// the argument checks both SART entries share
#define SART_CHECK_ARGS(fn)                                                                                                       \
    IPDM_REQUIRE(p && sino && img && sino != img && batch > 0 && batch <= 65535, fn ": bad arguments");                          \
    IPDM_REQUIRE(iterations >= 1, fn ": iterations must be >= 1, got %d", iterations);                                          \
    IPDM_REQUIRE(subsets >= 1 && subsets <= NV && NV % subsets == 0, fn ": subsets must divide %d, got %d", NV, subsets);       \
    IPDM_REQUIRE(relaxation > 0.f && relaxation < 2.f, fn ": relaxation must be in (0, 2), got %g", (double)relaxation)

extern "C" int ipdm_fbp_sart(ipdm_fbp_plan* p, const float* sino, float* img, int batch, int flip, int iterations, int subsets,
                             float relaxation, void* stream) {
    SART_CHECK_ARGS("ipdm_fbp_sart");
    return run_sart(p, sino, img, batch, flip, iterations, subsets, relaxation, 0, 0.f, 0.f, 0, (cudaStream_t)stream);
}

extern "C" int ipdm_fbp_sart_tv(ipdm_fbp_plan* p, const float* sino, float* img, int batch, int flip, int iterations, int subsets,
                                float relaxation, int ntv, float tv_alpha, float tv_eps, int init_fbp, void* stream) {
    SART_CHECK_ARGS("ipdm_fbp_sart_tv");
    IPDM_REQUIRE(ntv >= 0, "ipdm_fbp_sart_tv: ntv must be >= 0, got %d", ntv);
    IPDM_REQUIRE(std::isfinite(tv_alpha) && tv_alpha > 0.f, "ipdm_fbp_sart_tv: tv_alpha must be finite and > 0, got %g", (double)tv_alpha);
    IPDM_REQUIRE(std::isfinite(tv_eps) && tv_eps > 0.f, "ipdm_fbp_sart_tv: tv_eps must be finite and > 0, got %g", (double)tv_eps);
    IPDM_REQUIRE(init_fbp == 0 || init_fbp == 1, "ipdm_fbp_sart_tv: init_fbp must be 0 or 1, got %d", init_fbp);
    IPDM_REQUIRE(((uintptr_t)img & 15) == 0, "ipdm_fbp_sart_tv: img must be 16-byte aligned");
    return run_sart(p, sino, img, batch, flip, iterations, subsets, relaxation, ntv, tv_alpha, tv_eps, init_fbp, (cudaStream_t)stream);
}
