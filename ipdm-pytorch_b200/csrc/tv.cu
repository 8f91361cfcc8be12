// Total-variation steps for sm_100a, the regulariser of SART-TV (sart.cu): normalised steepest descent on the isotropic,
// eps-smoothed TV of every slice (ASD-POCS, Sidky & Pan, Phys. Med. Biol. 53 (2008) 4777, with a fixed step fraction).
//
// TV_eps(x) = sum sqrt(dx^2 + dy^2 + eps^2), forward differences dx = x[i][j+1] - x[i][j], dy = x[i+1][j] - x[i][j] in the native
// frame (0 where they would leave the image), so p = dx / n and q = dy / n (n the square root) give the gradient
//   g[i][j] = p[i][j-1] + q[i-1][j] - (p[i][j] + q[i][j])      (out-of-range terms dropped).
// A step of length t is x <- max(0, x - t g / |g|_2), per slice; |g| = 0 leaves the slice as it is.
//
// Kernel 1  tv_grad_kernel    one CTA per 32 x 32 native tile and slice: stages x with a one-pixel halo (34 x 34), then p and q of
//                             the 33 x 33 pixels the tile's gradient reads, then g.  Writes g in the image's own memory frame and the
//                             tile's sum of g^2 (fp64) to a per-tile partial; at the first step of a SART-TV sweep also the tile's
//                             sum of (x - x_prev)^2.  Column j of the native frame is memory column 511 - j when flip = 1, and all
//                             arithmetic is indexed natively, so a flip = 1 result is the column mirror of the flip = 0 one, bit
//                             for bit.  Bound: HBM / L2 traffic (x read, g written; x_prev read at a sweep's first step).
// Kernel 2  tv_update_kernel  one CTA per 4096 pixels of a slice: folds the slice's 256 partials in a fixed tree order (fp64), takes
//                             t (given, or alpha |x - x_prev| at a sweep's first step, kept per slice for the later steps) and
//                             applies the step elementwise.  Bound: HBM / L2 traffic (x, g read, x written).
// No atomics: every sum has a fixed order, so results are bit-identical from run to run and slice k of a batch equals slice k alone.
#include "fbp_plan.cuh"

#include <cmath>
#include <cstdint>

namespace ipdm {

constexpr int TV_NP = IPDM_N_PIX;
constexpr int TV_T = 32;                           // tile edge
constexpr int TV_TILES = (TV_NP / TV_T) * (TV_NP / TV_T);   // 256 partials per slice
constexpr int TV_UPD_PIX = 4096;                   // pixels per update CTA (256 threads x 4 float4)
static_assert(TV_TILES == 256, "the update kernel folds one partial per thread");

// fixed-order sum of one double per thread of a 256-thread CTA; the result is valid in every thread
__device__ __forceinline__ double block_sum_256(double v, double* red) {
    const int tid = threadIdx.x;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    __syncthreads();                               // red may still be read by a previous call
    if ((tid & 31) == 0) red[tid >> 5] = v;
    __syncthreads();
    double s = red[0];
#pragma unroll
    for (int w = 1; w < 8; ++w) s += red[w];
    return s;
}

// x, xprev, g: [B][512][512] in the memory frame (column-flipped iff flip); part: [B][2][256] (sum g^2, sum (x - xprev)^2)
template <bool WITH_D>
__global__ void __launch_bounds__(256)
tv_grad_kernel(const float* __restrict__ x, const float* __restrict__ xprev, float* __restrict__ g, double* __restrict__ part,
               float eps2, int flip) {
    __shared__ float sx[TV_T + 2][TV_T + 3];       // native rows i0 - 1 .. i0 + 32, columns j0 - 1 .. j0 + 32
    __shared__ float sp[TV_T + 1][TV_T + 2];       // p, q of rows i0 - 1 .. i0 + 31, columns j0 - 1 .. j0 + 31
    __shared__ float sq[TV_T + 1][TV_T + 2];
    __shared__ double red[8];
    const int tid = threadIdx.x, lane = tid & 31, wrp = tid >> 5;
    const int i0 = blockIdx.y * TV_T, j0 = blockIdx.x * TV_T;
    const size_t base = (size_t)blockIdx.z * TV_NP * TV_NP;
    const float* xb = x + base;
    auto mcol = [flip](int j) { return flip ? TV_NP - 1 - j : j; };
    for (int e = tid; e < (TV_T + 2) * (TV_T + 2); e += 256) {
        const int r = e / (TV_T + 2), c = e - r * (TV_T + 2);
        const int i = i0 - 1 + r, j = j0 - 1 + c;
        sx[r][c] = (i >= 0 && i < TV_NP && j >= 0 && j < TV_NP) ? __ldg(xb + (size_t)i * TV_NP + mcol(j)) : 0.f;
    }
    __syncthreads();
    for (int e = tid; e < (TV_T + 1) * (TV_T + 1); e += 256) {
        const int r = e / (TV_T + 1), c = e - r * (TV_T + 1);
        const int i = i0 - 1 + r, j = j0 - 1 + c;
        float p = 0.f, q = 0.f;
        if (i >= 0 && j >= 0) {                    // i, j <= 511 always
            const float v = sx[r][c];
            const float dx = j < TV_NP - 1 ? sx[r][c + 1] - v : 0.f;
            const float dy = i < TV_NP - 1 ? sx[r + 1][c] - v : 0.f;
            const float n = sqrtf(fmaf(dx, dx, fmaf(dy, dy, eps2)));
            p = dx / n;
            q = dy / n;
        }
        sp[r][c] = p;                              // 0 outside the image: the dropped terms
        sq[r][c] = q;
    }
    __syncthreads();
    double g2 = 0.0, d2 = 0.0;
    float* gb = g + base;
    const int j = j0 + lane;
#pragma unroll
    for (int k = 0; k < TV_T / 8; ++k) {
        const int r = wrp + 8 * k, i = i0 + r;
        const float gv = (sp[r + 1][lane] + sq[r][lane + 1]) - (sp[r + 1][lane + 1] + sq[r + 1][lane + 1]);
        const size_t m = (size_t)i * TV_NP + mcol(j);
        gb[m] = gv;
        g2 = fma((double)gv, (double)gv, g2);
        if (WITH_D) {
            const double dv = (double)sx[r + 1][lane + 1] - (double)__ldg(xprev + base + m);
            d2 = fma(dv, dv, d2);
        }
    }
    double* pb = part + (size_t)blockIdx.z * 2 * TV_TILES;
    const int tile = blockIdx.y * (TV_NP / TV_T) + blockIdx.x;
    g2 = block_sum_256(g2, red);
    if (tid == 0) pb[tile] = g2;
    if (WITH_D) {
        d2 = block_sum_256(d2, red);
        if (tid == 0) pb[TV_TILES + tile] = d2;
    }
}

// mode 0: t = step for every slice; 1: t = alpha * sqrt(sum (x - xprev)^2), stored in tval[slice]; 2: t = tval[slice]
__global__ void __launch_bounds__(256)
tv_update_kernel(float* __restrict__ x, const float* __restrict__ g, const double* __restrict__ part, double* __restrict__ tval,
                 int mode, double step) {
    __shared__ double red[8];
    const int tid = threadIdx.x, b = blockIdx.y;
    const double* pb = part + (size_t)b * 2 * TV_TILES;
    const double gn = sqrt(block_sum_256(pb[tid], red));
    double t = step;
    if (mode == 1) {
        t = step * sqrt(block_sum_256(pb[TV_TILES + tid], red));
        if (blockIdx.x == 0 && tid == 0) tval[b] = t;
    } else if (mode == 2) {
        t = tval[b];
    }
    if (!(gn > 0.0)) return;
    const float s = (float)(t / gn);
    const size_t o = (size_t)b * TV_NP * TV_NP + (size_t)blockIdx.x * TV_UPD_PIX;
    float4* xb = reinterpret_cast<float4*>(x + o);
    const float4* gb = reinterpret_cast<const float4*>(g + o);
#pragma unroll
    for (int k = 0; k < TV_UPD_PIX / 4 / 256; ++k) {
        const int e = tid + 256 * k;
        float4 v = xb[e];
        const float4 d = __ldg(gb + e);
        v.x = fmaxf(0.f, fmaf(-s, d.x, v.x));
        v.y = fmaxf(0.f, fmaf(-s, d.y, v.y));
        v.z = fmaxf(0.f, fmaf(-s, d.z, v.z));
        v.w = fmaxf(0.f, fmaf(-s, d.w, v.w));
        xb[e] = v;
    }
}

size_t tv_scratch_bytes(int batch) {
    return (size_t)batch * (2 * (size_t)TV_NP * TV_NP * sizeof(float) + (2 * TV_TILES + 1) * sizeof(double));
}

int launch_tv(ipdm_fbp_plan* p, float* img, int batch, int flip, int steps, bool sweep, double alpha_or_step, float eps,
              cudaStream_t st) {
    const size_t plane = (size_t)batch * TV_NP * TV_NP;
    const float* xprev = p->tv.f32();
    float* g = p->tv.f32() + plane;
    double* part = reinterpret_cast<double*>(g + plane);
    double* tval = part + (size_t)batch * 2 * TV_TILES;
    const dim3 gg(TV_NP / TV_T, TV_NP / TV_T, batch), gu(TV_NP * TV_NP / TV_UPD_PIX, batch);
    const float eps2 = eps * eps;
    for (int s = 0; s < steps; ++s) {
        if (sweep && s == 0)
            tv_grad_kernel<true><<<gg, 256, 0, st>>>(img, xprev, g, part, eps2, flip);
        else
            tv_grad_kernel<false><<<gg, 256, 0, st>>>(img, nullptr, g, part, eps2, flip);
        tv_update_kernel<<<gu, 256, 0, st>>>(img, g, part, tval, sweep ? (s == 0 ? 1 : 2) : 0, alpha_or_step);
        count_launch(2);
        IPDM_CHECK_LAUNCH();
    }
    return IPDM_OK;
}

}  // namespace ipdm

using namespace ipdm;

extern "C" int ipdm_fbp_tv_descent(ipdm_fbp_plan* p, float* img, int batch, int flip, int steps, float step, float eps, void* stream) {
    IPDM_REQUIRE(p && img && batch > 0 && batch <= 65535, "ipdm_fbp_tv_descent: bad arguments");
    IPDM_REQUIRE(steps >= 0, "ipdm_fbp_tv_descent: steps must be >= 0, got %d", steps);
    IPDM_REQUIRE(std::isfinite(step) && step >= 0.f, "ipdm_fbp_tv_descent: step must be finite and >= 0, got %g", (double)step);
    IPDM_REQUIRE(std::isfinite(eps) && eps > 0.f, "ipdm_fbp_tv_descent: eps must be finite and > 0, got %g", (double)eps);
    IPDM_REQUIRE(((uintptr_t)img & 15) == 0, "ipdm_fbp_tv_descent: img must be 16-byte aligned");
    if (steps == 0) return IPDM_OK;
    IPDM_CHECK(p->tv.reserve(tv_scratch_bytes(batch)));
    return launch_tv(p, img, batch, flip, steps, false, (double)step, eps, (cudaStream_t)stream);
}
