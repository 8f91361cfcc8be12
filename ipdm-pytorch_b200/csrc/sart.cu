// Iterative convertors for sm_100a: the exact adjoint of the forward projector (project.cu), ordered-subset SART around the
// projector / adjoint pair, in the FBP plan's geometry and flip frames, optionally started from the FBP image and regularised by
// TV steps between the sweeps (SART-TV, tv.cu), and penalised weighted least squares solved by ordered-subset SQS (PWLS, with the
// penalty of pwls.cu).  A new convertor, not a port of the reference's Windows-only TASART2DNSL0.pyd:
// its area-integral projector and its NSL0 formula are not ported (the TV steps here are ASD-POCS on a smoothed isotropic TV).
//
// A is the fp32 matrix ipdm_fbp_project applies: ray (v, k) samples column / row m of its dominant axis at u = joseph_u(m) and
// puts the weights 1 - w on pixel floor(u) and w on floor(u) + 1 of the other axis (w = u - floor(u)), times the ray's step.
//
// Kernel 1  fbp_adjoint_kernel<MODE>  pixel-driven gather, one CTA per 32 x 32 pixel tile and slice, ascending views.  Per
//           16-view chunk the CTA stages, for the detector segment its tile can touch, each ray's (u0, g, step * value, axis)
//           in shared memory; the ray setup is joseph_ray, so every weight is the projector's own fp32 weight.  A pixel then
//           tries the rays within dx / (L da) + 1 pitches of its own fan angle (L its distance from the source): a ray passes
//           within one pixel pitch of every pixel it touches.  About 5-7 candidates per (view, pixel), each one FMA for u, a
//           floor and a compare.  No atomics: each output pixel is one thread's sum in a fixed order.
//           SART: the staged value is the ray's residual (b - A_s x) / R (0 where R = 0), and the epilogue applies
//           x <- max(0, x + lambda * A_s^T r / C_s) (pixels with C_s = 0 keep x).  Bound: FP32 issue on the candidate loop.
//           PWLS: DENOM stages w(b) R and writes D^L = A^T (w o R); SQS stages w(b) (b - A_s x) and the epilogue applies
//           x <- max(0, x + (S A_s^T(...) - beta grad R) / (D^L + beta d^R)) (pixels with a zero denominator keep x), with
//           w(b) = 1 / sigma^2(max(b, 0)) computed from b in fp32 (no weight sinogram is stored).
// Kernel 2  fill_kernel                the all-ones image / sinogram the tables R = A 1 and C_s = A_s^T 1 are computed from.
// Kernel 3  clamp_nonneg_kernel        x0 = max(0, FBP) of the FBP start.
// SART-TV: before every sweep the iterate is copied to x_prev in the TV scratch, after it ntv TV steps run (launch_tv).
// PWLS: D^L once per call, then per subset transpose, projection, penalty (launch_pwls_penalty) and the SQS adjoint.
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

// what fbp_adjoint_kernel stages per ray and does with the sums
enum AdjMode { ADJ_PLAIN, ADJ_SART, ADJ_DENOM, ADJ_SQS };

// the PWLS operands of the DENOM and SQS modes: wk = 1 / (dose N0); dl, grad, curv [B][512][512] in the image's frame (SQS)
struct PwlsArgs {
    const float* dl = nullptr;
    const float* grad = nullptr;
    const float* curv = nullptr;
    float wk = 0.f, beta = 0.f;
};

// w = 1 / sigma^2(max(b, 0)), sigma^2(p) = q (1 + Ne q), q = e^p / (dose N0): the inverse variance of a measurement at the dose
__device__ __forceinline__ float pwls_weight(float b, float wk) {
    const float q = expf(fmaxf(b, 0.f)) * wk;
    return 1.0f / (q * fmaf((float)kDoseNe, q, 1.0f));
}

// continuous ray index kc of the pixel centre (x, y) in view cs = (cos theta, sin theta), and the half width hw of its candidate
// window: dx / (L da) pitches plus one of slack (the rounding of kc is about 1e-4 pitch)
__device__ __forceinline__ void pixel_window(float x, float y, float2 cs, float inv_da, float k_off, float& kc, float& hw) {
    const float s = fmaf(x, cs.y, y * cs.x);
    const float c = fmaf(x, cs.x, fmaf(-y, cs.y, 59.5f));
    kc = fmaf(atan_small(s * __frcp_rn(c)), inv_da, k_off);
    hw = fmaf(DXP * inv_da, rsqrtf(fmaf(s, s, c * c)), 1.0f);
}

// staged entry of ray (v, k): (u0, g, step * value, xmajor); value = y[v][k'] (plain adjoint), the SART residual of the ray,
// w(b) R (DENOM) or w(b) (b - A_s x) (SQS), k' = k in the sinogram's frame.  yb / pb / R are per-slice; pb (the subset
// projection, row n) is null when x = 0.
template <int MODE>
__device__ __forceinline__ float4 adj_entry(const float* __restrict__ yb, const float* __restrict__ pb, const float* __restrict__ R,
                                            const float2* __restrict__ cs_view, const float2* __restrict__ cs_ray, int v, int n, int k,
                                            int flip, float wk) {
    const JosephRay r = joseph_ray(__ldg(cs_view + v), __ldg(cs_ray + k));
    const int kk = flip ? ND - 1 - k : k;
    float val = __ldg(yb + (size_t)v * ND + kk);
    if (MODE == ADJ_SART) {
        const float rs = __ldg(R + (size_t)v * ND + k);
        if (pb) val -= __ldg(pb + (size_t)n * ND + kk);
        val = rs > 0.f ? val / rs : 0.f;
    } else if (MODE == ADJ_DENOM) {
        val = pwls_weight(val, wk) * __ldg(R + (size_t)v * ND + k);
    } else if (MODE == ADJ_SQS) {
        const float w = pwls_weight(val, wk);
        if (pb) val -= __ldg(pb + (size_t)n * ND + kk);
        val *= w;
    }
    return make_float4(r.u0, r.g, r.scale * val, r.xmajor ? 1.f : 0.f);
}

// the same, out of line: a ray outside the staged segment (kept off the candidate loop's registers)
template <int MODE>
__device__ __noinline__ float4 adj_entry_far(const float* yb, const float* pb, const float* R, const float2* cs_view, const float2* cs_ray,
                                             int v, int n, int k, int flip, float wk) {
    return adj_entry<MODE>(yb, pb, R, cs_view, cs_ray, v, n, k, flip, wk);
}

// views v0 + n * vstep, n < nv.  y: [B][2000][912] (the sinogram, or b for SART / PWLS); psub: [B][nv][912] A_s x (SART / SQS,
// may be null); R: [2000][912]; colsum: C_s [512][512] native (SART); img: written (plain, DENOM) or updated in place (SART,
// SQS), column-flipped iff flip; lambda: the relaxation (SART) or S (SQS)
template <int MODE>
__global__ void __launch_bounds__(256)
fbp_adjoint_kernel(const float* __restrict__ y, const float* __restrict__ psub, const float* __restrict__ R,
                   const float* __restrict__ colsum, float* __restrict__ img, const float2* __restrict__ cs_view,
                   const float2* __restrict__ cs_ray, int v0, int vstep, int nv, float inv_da, float k_off, float lambda, int flip,
                   PwlsArgs pw) {
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
            seg[vv][o] = adj_entry<MODE>(yb, pb, R, cs_view, cs_ray, v0 + (c0 + vv) * vstep, c0 + vv, seg0[vv] + o, flip, pw.wk);
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
                                         : adj_entry_far<MODE>(yb, pb, R, cs_view, cs_ray, v0 + (c0 + vv) * vstep, c0 + vv, k, flip,
                                                               pw.wk);
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
    const size_t slice = (size_t)blockIdx.z * NP * NP;
    float* ob = img + slice;
    const int jo = flip ? NP - 1 - j : j;
#pragma unroll
    for (int p = 0; p < ADJ_RPT; ++p) {
        const int i = i_base + 8 * p;
        if (MODE == ADJ_PLAIN || MODE == ADJ_DENOM) {
            ob[(size_t)i * NP + jo] = acc[p];
        } else if (MODE == ADJ_SART) {
            const float cs = __ldg(colsum + (size_t)i * NP + j);
            if (cs > 0.f) ob[(size_t)i * NP + jo] = fmaxf(0.f, fmaf(lambda, acc[p] / cs, ob[(size_t)i * NP + jo]));
        } else {
            const size_t m = slice + (size_t)i * NP + jo;
            const float den = fmaf(pw.beta, __ldg(pw.curv + m), __ldg(pw.dl + m));
            if (den > 0.f) {
                const float num = fmaf(lambda, acc[p], -pw.beta * __ldg(pw.grad + m));
                ob[(size_t)i * NP + jo] = fmaxf(0.f, ob[(size_t)i * NP + jo] + num / den);
            }
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

template <int MODE>
static int launch_adjoint(ipdm_fbp_plan* p, const float* y, const float* psub, const float* colsum, float* img, int batch, int flip, int v0,
                          int vstep, int nv, float lambda, cudaStream_t st, const PwlsArgs& pw = PwlsArgs()) {
    const float k_off = (float)(-0.5 - (double)p->host.nda[0] / p->host.da);     // ray k is at fan angle nda[0] + (k + 1/2) da
    fbp_adjoint_kernel<MODE><<<dim3(NP / 32, NP / ADJ_TH, batch), 256, 0, st>>>(y, psub, p->d_rowsum, colsum, img, p->d_cs, p->d_ray, v0,
                                                                                vstep, nv, p->inv_da, k_off, lambda, flip, pw);
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

// a table build allocates and synchronises, so it cannot run inside a stream capture
static int require_eager(cudaStream_t st, const char* what) {
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    IPDM_CHECK_CUDA(cudaStreamIsCapturing(st, &cap));
    IPDM_REQUIRE(cap == cudaStreamCaptureStatusNone, "%s cannot be captured; run it once eagerly", what);
    return IPDM_OK;
}

// an all-ones sinogram [2000][912]; its first 512 x 512 values serve as the all-ones image
static int make_ones(float** ones, cudaStream_t st) {
    IPDM_CHECK_CUDA(cudaMalloc(ones, (size_t)NV * ND * sizeof(float)));
    fill_kernel<<<ceil_div(NV * ND, 256), 256, 0, st>>>(*ones, 1.0f, NV * ND);
    count_launch();
    return IPDM_OK;
}

// ends a table build: waits for it, frees the ones buffer and reports a CUDA failure under fn's name
static int finish_build(int rc, float* ones, const char* fn, cudaStream_t st) {
    if (rc == IPDM_OK && cudaGetLastError() != cudaSuccess) rc = IPDM_ERR_CUDA;
    if (cudaStreamSynchronize(st) != cudaSuccess && rc == IPDM_OK) rc = IPDM_ERR_CUDA;
    cudaFree(ones);
    if (rc == IPDM_ERR_CUDA) set_error("%s: building the tables failed: %s", fn, cudaGetErrorString(cudaGetLastError()));
    return rc;
}

// R = A 1, once per plan, in fp32 with the projector; fn names the calling entry in messages
static int ensure_rowsum(ipdm_fbp_plan* p, const char* fn, cudaStream_t st) {
    if (p->d_rowsum) return IPDM_OK;
    char what[96];
    snprintf(what, sizeof what, "%s: the first call of a plan builds its row sums and", fn);
    IPDM_CHECK(require_eager(st, what));
    float* ones = nullptr;
    IPDM_CHECK(make_ones(&ones, st));
    int rc = cudaMalloc(&p->d_rowsum, (size_t)NV * ND * sizeof(float)) == cudaSuccess ? IPDM_OK : IPDM_ERR_CUDA;
    if (rc == IPDM_OK) rc = launch_project(p, ones, p->d_rowsum, 1, 0, 0, 1, NV, st);
    return finish_build(rc, ones, fn, st);
}

// R (ensure_rowsum) and C_s = A_s^T 1 for every subset of S (once per plan and S), in fp32 with the same kernels
static int ensure_sart_tables(ipdm_fbp_plan* p, int S, cudaStream_t st) {
    IPDM_CHECK(ensure_rowsum(p, "ipdm_fbp_sart_tv", st));
    if (p->colsum.count(S)) return IPDM_OK;
    char what[96];
    snprintf(what, sizeof what, "ipdm_fbp_sart_tv: the first call with %d subsets builds the plan's tables and", S);
    IPDM_CHECK(require_eager(st, what));
    float* ones = nullptr;
    IPDM_CHECK(make_ones(&ones, st));
    float* c = nullptr;
    int rc = cudaMalloc(&c, (size_t)S * NP * NP * sizeof(float)) == cudaSuccess ? IPDM_OK : IPDM_ERR_CUDA;
    for (int s = 0; rc == IPDM_OK && s < S; ++s)
        rc = launch_adjoint<ADJ_PLAIN>(p, ones, nullptr, nullptr, c + (size_t)s * NP * NP, 1, 0, s, S, NV / S, 0.f, st);
    if (rc == IPDM_OK) p->colsum[S] = c;
    else cudaFree(c);
    return finish_build(rc, ones, "ipdm_fbp_sart_tv", st);
}

// the start of an iterative convertor: x0 = max(0, FBP(sino)), unsharpened (init_fbp = 1), or x0 = 0
static int set_start(ipdm_fbp_plan* p, const float* sino, float* img, int batch, int flip, int init_fbp, cudaStream_t st) {
    if (init_fbp) {
        IPDM_CHECK(ipdm_fbp_forward(p, sino, img, batch, flip, st));
        const size_t n4 = (size_t)batch * NP * NP / 4;
        clamp_nonneg_kernel<<<ceil_div((long long)n4, 256), 256, 0, st>>>(reinterpret_cast<float4*>(img), n4);
        count_launch();
        IPDM_CHECK_LAUNCH();
    } else {
        IPDM_CHECK_CUDA(cudaMemsetAsync(img, 0, (size_t)batch * NP * NP * sizeof(float), st));
    }
    return IPDM_OK;
}

// proj = A_s x of the iterate, in the plan's subset buffer (reserved by the caller), or null when x is known to be 0: A_s 0 = 0,
// so the first subset from the zero start needs no projection
static int project_subset(ipdm_fbp_plan* p, const float* img, bool zero, int batch, int flip, int s, int subsets, const float** proj,
                          cudaStream_t st) {
    *proj = nullptr;
    if (zero) return IPDM_OK;
    *proj = p->subset.f32();
    return launch_project(p, img, p->subset.f32(), batch, flip, s, subsets, NV / subsets, st);
}

// SART (ntv = 0) or SART-TV, from x0 = 0 (init_fbp = 0) or x0 = max(0, FBP(sino)) (init_fbp = 1); arguments checked by the caller
static int run_sart(ipdm_fbp_plan* p, const float* sino, float* img, int batch, int flip, int iterations, int subsets, float relaxation,
                    int ntv, float tv_alpha, float tv_eps, int init_fbp, cudaStream_t st) {
    IPDM_CHECK(ensure_sart_tables(p, subsets, st));
    const int nv = NV / subsets;
    IPDM_CHECK(p->work.reserve(work_bytes(batch)));                           // the projector's transposed iterates
    IPDM_CHECK(p->subset.reserve((size_t)batch * nv * ND * sizeof(float)));   // A_s x of one subset
    if (ntv > 0) IPDM_CHECK(p->tv.reserve(tv_scratch_bytes(batch)));           // x_prev, g and the partial sums of the TV steps
    const float* colsum = p->colsum[subsets];
    const int step = sart_visit_step(subsets);
    const size_t img_bytes = (size_t)batch * NP * NP * sizeof(float);
    IPDM_CHECK(set_start(p, sino, img, batch, flip, init_fbp, st));
    for (int it = 0; it < iterations; ++it) {
        if (ntv > 0) IPDM_CHECK_CUDA(cudaMemcpyAsync(p->tv.ptr, img, img_bytes, cudaMemcpyDeviceToDevice, st));     // x_prev
        for (int n = 0; n < subsets; ++n) {
            const int s = (int)((long long)n * step % subsets);
            const float* proj;
            IPDM_CHECK(project_subset(p, img, !init_fbp && it == 0 && n == 0, batch, flip, s, subsets, &proj, st));
            IPDM_CHECK(launch_adjoint<ADJ_SART>(p, sino, proj, colsum + (size_t)s * NP * NP, img, batch, flip, s, subsets, nv, relaxation,
                                                st));
        }
        if (ntv > 0) IPDM_CHECK(launch_tv(p, img, batch, flip, ntv, true, (double)tv_alpha, tv_eps, st));
    }
    return IPDM_OK;
}

// PWLS by OS-SQS (subsets and visit order of SART), from x0 = 0 or max(0, FBP(sino)); arguments checked by the caller
static int run_pwls(ipdm_fbp_plan* p, const float* sino, float* img, int batch, int flip, int iterations, int subsets, float dose,
                    float beta, float delta, int init_fbp, cudaStream_t st) {
    IPDM_CHECK(ensure_rowsum(p, "ipdm_fbp_pwls", st));                         // R, no C_s tables
    const int nv = NV / subsets;
    const size_t plane = (size_t)batch * NP * NP;
    IPDM_CHECK(p->work.reserve(work_bytes(batch)));
    IPDM_CHECK(p->subset.reserve((size_t)batch * nv * ND * sizeof(float)));
    IPDM_CHECK(p->pwls.reserve(3 * plane * sizeof(float)));
    float* dl = p->pwls.f32();
    float* grad = dl + plane;
    float* curv = grad + plane;
    PwlsArgs pw;
    pw.dl = dl;
    pw.grad = grad;
    pw.curv = curv;
    pw.wk = (float)(1.0 / ((double)dose * kDoseN0));
    pw.beta = beta;
    IPDM_CHECK(launch_adjoint<ADJ_DENOM>(p, sino, nullptr, nullptr, dl, batch, flip, 0, 1, NV, 0.f, st, pw));
    IPDM_CHECK(set_start(p, sino, img, batch, flip, init_fbp, st));
    const int step = sart_visit_step(subsets);
    for (int it = 0; it < iterations; ++it) {
        for (int n = 0; n < subsets; ++n) {
            const int s = (int)((long long)n * step % subsets);
            const float* proj;
            IPDM_CHECK(project_subset(p, img, !init_fbp && it == 0 && n == 0, batch, flip, s, subsets, &proj, st));
            IPDM_CHECK(launch_pwls_penalty(img, grad, curv, batch, flip, delta, st));
            IPDM_CHECK(launch_adjoint<ADJ_SQS>(p, sino, proj, nullptr, img, batch, flip, s, subsets, nv, (float)subsets, st, pw));
        }
    }
    return IPDM_OK;
}

}  // namespace ipdm

using namespace ipdm;

extern "C" int ipdm_fbp_project_adjoint(ipdm_fbp_plan* p, const float* sino, float* img, int batch, int flip, void* stream) {
    IPDM_REQUIRE(p && sino && img && batch > 0 && batch <= 65535, "ipdm_fbp_project_adjoint: bad arguments");
    return launch_adjoint<ADJ_PLAIN>(p, sino, nullptr, nullptr, img, batch, flip, 0, 1, NV, 0.f, (cudaStream_t)stream);
}

// the argument checks both iterative entries share
#define ITER_CHECK_ARGS(fn)                                                                                                       \
    IPDM_REQUIRE(p && sino && img && sino != img && batch > 0 && batch <= 65535, fn ": bad arguments");                          \
    IPDM_REQUIRE(iterations >= 1, fn ": iterations must be >= 1, got %d", iterations);                                          \
    IPDM_REQUIRE(subsets >= 1 && subsets <= NV && NV % subsets == 0, fn ": subsets must divide %d, got %d", NV, subsets)

extern "C" int ipdm_fbp_sart_tv(ipdm_fbp_plan* p, const float* sino, float* img, int batch, int flip, int iterations, int subsets,
                                float relaxation, int ntv, float tv_alpha, float tv_eps, int init_fbp, void* stream) {
    ITER_CHECK_ARGS("ipdm_fbp_sart_tv");
    IPDM_REQUIRE(relaxation > 0.f && relaxation < 2.f, "ipdm_fbp_sart_tv: relaxation must be in (0, 2), got %g", (double)relaxation);
    IPDM_REQUIRE(ntv >= 0, "ipdm_fbp_sart_tv: ntv must be >= 0, got %d", ntv);
    IPDM_REQUIRE(std::isfinite(tv_alpha) && tv_alpha > 0.f, "ipdm_fbp_sart_tv: tv_alpha must be finite and > 0, got %g", (double)tv_alpha);
    IPDM_REQUIRE(std::isfinite(tv_eps) && tv_eps > 0.f, "ipdm_fbp_sart_tv: tv_eps must be finite and > 0, got %g", (double)tv_eps);
    IPDM_REQUIRE(init_fbp == 0 || init_fbp == 1, "ipdm_fbp_sart_tv: init_fbp must be 0 or 1, got %d", init_fbp);
    // the TV steps and the FBP start's clamp work on float4
    IPDM_REQUIRE((ntv == 0 && init_fbp == 0) || ((uintptr_t)img & 15) == 0,
                 "ipdm_fbp_sart_tv: img must be 16-byte aligned when ntv > 0 or init_fbp = 1");
    return run_sart(p, sino, img, batch, flip, iterations, subsets, relaxation, ntv, tv_alpha, tv_eps, init_fbp, (cudaStream_t)stream);
}

extern "C" int ipdm_fbp_pwls(ipdm_fbp_plan* p, const float* sino, float* img, int batch, int flip, int iterations, int subsets, float dose,
                             float beta, float delta, int init_fbp, void* stream) {
    ITER_CHECK_ARGS("ipdm_fbp_pwls");
    IPDM_REQUIRE(dose > 0.f && dose <= 1.f, "ipdm_fbp_pwls: dose must be in (0, 1], got %g", (double)dose);
    IPDM_REQUIRE(std::isfinite(beta) && beta >= 0.f, "ipdm_fbp_pwls: beta must be finite and >= 0, got %g", (double)beta);
    IPDM_REQUIRE(std::isfinite(delta) && delta > 0.f, "ipdm_fbp_pwls: delta must be finite and > 0, got %g", (double)delta);
    IPDM_REQUIRE(init_fbp == 0 || init_fbp == 1, "ipdm_fbp_pwls: init_fbp must be 0 or 1, got %d", init_fbp);
    IPDM_REQUIRE(((uintptr_t)img & 15) == 0, "ipdm_fbp_pwls: img must be 16-byte aligned");
    return run_pwls(p, sino, img, batch, flip, iterations, subsets, dose, beta, delta, init_fbp, (cudaStream_t)stream);
}
