// The roughness penalty of PWLS (sart.cu run_pwls) for sm_100a: an edge-preserving hyperbola on the 8-neighbourhood of every
// pixel, with its gradient and separable quadratic surrogate (SQS) curvature.
//
// R(x) = sum_j sum_{k in N+(j)} kappa_jk psi(x_j - x_k), N+ = right, down, down-left, down-right (each pair once), kappa = 1 for
// edge and 1/sqrt(2) for diagonal neighbours, psi(t) = delta^2 (sqrt(1 + (t / delta)^2) - 1), no terms outside the image.  With
// omega(t) = 1 / sqrt(1 + (t / delta)^2):
//   grad R_j = sum_{k in N(j)} kappa_jk (x_j - x_k) omega(x_j - x_k),   d^R_j = 2 sum_{k in N(j)} kappa_jk omega(x_j - x_k)
// over all 8 neighbours; the factor 2 is De Pierro's bound for a pairwise term (Erdogan & Fessler, Phys. Med. Biol. 44 (1999) 2835).
//
// Kernel  pwls_penalty_kernel  one CTA per 32 x 32 native tile and slice: stages x with a one-pixel halo (34 x 34) in shared
//         memory, then every thread sums the 8 neighbour terms of 4 pixels in a fixed native-frame order and writes grad R and d^R
//         in the image's own memory frame.  Column j of the native frame is memory column 511 - j when flip = 1 and all arithmetic
//         is indexed natively, so a flip = 1 result is the column mirror of the flip = 0 one, bit for bit.  No atomics.
//         Bound: HBM / L2 traffic (4 bytes read, 8 written per pixel).
#include "fbp_plan.cuh"

#include <cmath>
#include <cstdint>

namespace ipdm {

constexpr int PW_NP = IPDM_N_PIX;
constexpr int PW_T = 32;                            // tile edge

// x, grad, curv: [B][512][512] in the memory frame (column-flipped iff flip)
__global__ void __launch_bounds__(256)
pwls_penalty_kernel(const float* __restrict__ x, float* __restrict__ grad, float* __restrict__ curv, float inv_delta, int flip) {
    __shared__ float sx[PW_T + 2][PW_T + 3];       // native rows i0 - 1 .. i0 + 32, columns j0 - 1 .. j0 + 32
    const int tid = threadIdx.x, lane = tid & 31, wrp = tid >> 5;
    const int i0 = blockIdx.y * PW_T, j0 = blockIdx.x * PW_T;
    const size_t base = (size_t)blockIdx.z * PW_NP * PW_NP;
    const float* xb = x + base;
    auto mcol = [flip](int j) { return flip ? PW_NP - 1 - j : j; };
    for (int e = tid; e < (PW_T + 2) * (PW_T + 2); e += 256) {
        const int r = e / (PW_T + 2), c = e - r * (PW_T + 2);
        const int i = i0 - 1 + r, j = j0 - 1 + c;
        sx[r][c] = (i >= 0 && i < PW_NP && j >= 0 && j < PW_NP) ? __ldg(xb + (size_t)i * PW_NP + mcol(j)) : 0.f;
    }
    __syncthreads();
    const int j = j0 + lane;
#pragma unroll
    for (int q = 0; q < PW_T / 8; ++q) {
        const int r = wrp + 8 * q, i = i0 + r;
        const float xv = sx[r + 1][lane + 1];
        float g = 0.f, c = 0.f;
#pragma unroll
        for (int n = 0; n < 9; ++n) {              // neighbours in native row-major order, the centre skipped
            const int di = n / 3 - 1, dj = n % 3 - 1;
            if (n == 4) continue;
            const int ii = i + di, jj = j + dj;
            if (ii < 0 || ii >= PW_NP || jj < 0 || jj >= PW_NP) continue;
            const float t = xv - sx[r + 1 + di][lane + 1 + dj];
            const float u = t * inv_delta;
            float ko = rsqrtf(fmaf(u, u, 1.0f));   // kappa omega(t)
            if (di != 0 && dj != 0) ko *= 0.70710678118654752f;
            g = fmaf(ko, t, g);
            c += ko;
        }
        const size_t m = base + (size_t)i * PW_NP + mcol(j);
        grad[m] = g;
        curv[m] = 2.0f * c;
    }
}

int launch_pwls_penalty(const float* img, float* grad, float* curv, int batch, int flip, float delta, cudaStream_t st) {
    pwls_penalty_kernel<<<dim3(PW_NP / PW_T, PW_NP / PW_T, batch), 256, 0, st>>>(img, grad, curv, 1.0f / delta, flip);
    count_launch();
    IPDM_CHECK_LAUNCH();
    return IPDM_OK;
}

}  // namespace ipdm

using namespace ipdm;

extern "C" int ipdm_fbp_pwls_penalty(ipdm_fbp_plan* p, const float* img, float* grad, float* curv, int batch, int flip, float delta,
                                     void* stream) {
    IPDM_REQUIRE(p && img && grad && curv && grad != curv && img != grad && img != curv && batch > 0 && batch <= 65535,
                 "ipdm_fbp_pwls_penalty: bad arguments");
    IPDM_REQUIRE(std::isfinite(delta) && delta > 0.f, "ipdm_fbp_pwls_penalty: delta must be finite and > 0, got %g", (double)delta);
    return launch_pwls_penalty(img, grad, curv, batch, flip, delta, (cudaStream_t)stream);
}
