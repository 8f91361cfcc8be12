// Fan-beam FBP convertor for sm_100a: (flip + cosine weighting + ramp filter) -> backprojection.
// Replaces the reference's Recon/FBP_kernel.py (FBP.__init__ :27-67, convert :86-122,
// conv_pj/conv_kernel :125-143, fbp_cpu/fbp_kernel :146-184).
//
// Data layout in HBM: sinogram / filtered sinogram [B][2000][912] f32, image [B][512][512] f32.
//
// Kernel 1  fbp_filter_kernel   one CTA per sinogram row.  The row is weighted on load
//           (f32 product with D*cos(gamma), then the fp64 product with dtheta rounded to f32, as
//           FBP_kernel.py:104-105), split by detector parity into two zero-padded, bank-skewed
//           shared-memory sequences, and convolved with the 913 non-zero ramp taps (the even
//           taps of h_RL are exactly zero, :52-56): output parity c only sees inputs of parity
//           1-c plus the centre tap.  Each thread keeps 8 outputs in registers and slides a
//           15-value window, so a tap costs 1 LDS + 8 FFMA.  FP32 FMA bound (0.83 GFMA / slice).
// Kernel 2  fbp_backproject_kernel<PX>  one CTA per 32 x (8*PX) pixel tile and slice, looping
//           the 2000 views in ascending order (the reference's rounding sequence, one f32
//           accumulator per pixel).  Per 16-view chunk the CTA stages (cos,sin) and, for each
//           view, only the detector segment its tile can hit (cp.async, double buffered) in shared
//           memory; a lane gathers its two taps there.  atan is a degree-15 odd polynomial
//           (|s/c| <= 0.6 inside the image), s/c is a Newton-refined reciprocal.  Bound: FP32 issue
//           (about 33 instructions per pixel-view update, 524.3 M updates / slice), not HBM
//           (8.345 MB compulsory bytes / slice; SURVEY.md D5).
#include "fbp_plan.cuh"

#include <cmath>
#include <vector>

namespace ipdm {

constexpr int NV = IPDM_N_VIEWS, ND = IPDM_N_DET, NP = IPDM_N_PIX;
constexpr int NHALF = ND / 2;          // 456 samples per detector parity
constexpr int NTAP = 2 * NHALF - 1;    // 911 taps per parity class (d = -455..455)

// ------------------------------------------------------------------------------------------------
// tables: same expressions as FBP.__init__ (FBP_kernel.py:32-56), evaluated in fp64 on the host
// ------------------------------------------------------------------------------------------------
static void build_tables(FbpTables& t) {
    t.D = 59.5;
    t.da = 0.0010125;
    t.theta.resize(NV);
    for (int i = 0; i < NV; ++i) t.theta[i] = (0.0 + i * 0.18) / 180 * M_PI;            // np.arange(0, 360, .18)/180*pi
    t.nda.resize(ND);
    const double a0 = (-ND / 2.0 + 0.5 + 3.75) * t.da;
    for (int k = 0; k < ND; ++k) t.nda[k] = (float)(a0 + k * t.da);                      // np.arange(a0, ., da).astype(f32)
    t.h.assign(2 * ND - 1, 0.f);
    for (int i = 0; i < ND; ++i) {
        double ng = (double)(-ND + 1 + 2 * i) * t.da;                                    // np.arange(-N+1, N, 2) * da
        double s = std::sin(ng);
        t.h[2 * i] = (float)((-0.5 / (M_PI * M_PI) / (s * s)) * t.da);
    }
    t.h[ND - 1] = (float)((1.0 / 8 / (t.da * t.da)) * t.da);
    t.wcos.resize(ND);
    for (int k = 0; k < ND; ++k) t.wcos[k] = 59.5f * (float)std::cos((double)t.nda[k]);   // f32 * f32 (weak python float)
    t.dtheta = t.theta[1] - t.theta[0];
}

// ------------------------------------------------------------------------------------------------
// kernel 1: weighting + ramp filter
// ------------------------------------------------------------------------------------------------
constexpr int FILT_THREADS = 128;                 // warps 0,1: even outputs; warps 2,3: odd outputs
constexpr int SEQ_PAD = 464;                      // >= 455 + 8 zeros on either side of each parity sequence
constexpr int SEQ_LEN = SEQ_PAD + NHALF + SEQ_PAD;
__device__ __forceinline__ int skew(int a) { return a + (a >> 5); }
constexpr int SEQ_SMEM = SEQ_LEN + (SEQ_LEN >> 5) + 1;

__global__ void __launch_bounds__(FILT_THREADS)
fbp_filter_kernel(const float* __restrict__ sino, float* __restrict__ q, const float* __restrict__ wcos,
                  const float* __restrict__ htap, float h0, double dtheta, int flip) {
    __shared__ float seq[2][SEQ_SMEM];            // seq[p][skew(SEQ_PAD + j)] = weighted row[2j + p]
    __shared__ float taps[2][NTAP + 1];
    const size_t row = blockIdx.x;                // b * 2000 + v
    const float* src = sino + row * ND;
    float* dst = q + row * ND;
    const int tid = threadIdx.x;

    for (int i = tid; i < 2 * SEQ_SMEM; i += FILT_THREADS) (&seq[0][0])[i] = 0.f;
    for (int i = tid; i < 2 * NTAP; i += FILT_THREADS) taps[i / NTAP][i % NTAP] = htap[i];
    __syncthreads();
    for (int n = tid; n < ND; n += FILT_THREADS) {
        float a = src[flip ? ND - 1 - n : n];
        float w = __fmul_rn(a, wcos[n]);
        float v = (float)((double)w * dtheta);
        seq[n & 1][skew(SEQ_PAD + (n >> 1))] = v;
    }
    __syncthreads();

    const int c = tid >> 6;                       // output parity handled by this thread
    const int t = tid & 63;
    if (t >= NHALF / 8) return;                   // 57 threads x 8 outputs = 456
    const int i0 = t * 8;
    const float* s = seq[1 - c];                  // opposite-parity inputs
    const float* own = seq[c];
    const float* H = taps[c];
    float acc[8];
#pragma unroll
    for (int r = 0; r < 8; ++r) acc[r] = h0 * own[skew(SEQ_PAD + i0 + r)];

    // q[2i+c] += sum_d H_c[d] * s[i - d],  d = -455..455 ; processed in blocks of 8 taps.
    // The tap range is padded to 912 = 114 * 8 (the extra tap has weight taps[c][911], which is 0
    // by construction of the staging loop above: index 911 is never written -> initialise below).
    for (int db = 0; db < 114; ++db) {
        const int d0 = -455 + db * 8;
        float win[15];                            // s[i0 - d0 - 7 .. i0 - d0 + 7]
        const int base = SEQ_PAD + i0 - d0 - 7;
#pragma unroll
        for (int k = 0; k < 15; ++k) win[k] = s[skew(base + k)];
#pragma unroll
        for (int dd = 0; dd < 8; ++dd) {
            const float hv = (db * 8 + dd < NTAP) ? H[db * 8 + dd] : 0.f;
#pragma unroll
            for (int r = 0; r < 8; ++r) acc[r] = fmaf(hv, win[7 - dd + r], acc[r]);   // s[i0 + r - (d0 + dd)]
        }
    }
#pragma unroll
    for (int r = 0; r < 8; ++r) dst[2 * (i0 + r) + c] = acc[r];
}

// ------------------------------------------------------------------------------------------------
// kernel 2: pixel-driven backprojection
// ------------------------------------------------------------------------------------------------
constexpr int BP_VC = 16;                         // views per staged chunk
template <int PX> struct BpCfg { static constexpr int SEG = PX == 4 ? 160 : (PX == 2 ? 128 : 112); };

// detector coordinate u = (atan(s/c) - nda[0])/da + 0.5 and 1/L^2 for one pixel and view
__device__ __forceinline__ void ray_coords(float x, float y, float cs, float sn, float inv_da, float u_off,
                                           float& u, float& w) {
    const float s = fmaf(x, sn, y * cs);
    const float c = fmaf(x, cs, fmaf(-y, sn, 59.5f));
    float r = __frcp_rn(c);
    float t = s * r;
    t = fmaf(fmaf(-c, t, s), r, t);               // one Newton step: correctly rounded quotient in practice
    u = fmaf(atan_small(t), inv_da, u_off);
    w = __frcp_rn(fmaf(s, s, c * c));
}

template <int PX>
__global__ void __launch_bounds__(256)
fbp_backproject_kernel(const float* __restrict__ q, float* __restrict__ img, const float2* __restrict__ cs_tab,
                       float inv_da, float u_off, int flip) {
    constexpr int SEG = BpCfg<PX>::SEG;
    constexpr int TH = 8 * PX;
    __shared__ __align__(16) float seg[2][BP_VC][SEG];
    __shared__ int seg0[2][BP_VC];
    __shared__ float2 scs[2][BP_VC];

    const int tid = threadIdx.x, lane = tid & 31, wrp = tid >> 5;
    const int j = blockIdx.x * 32 + lane;                    // image column (native frame)
    const int i_base = blockIdx.y * TH + wrp;                // first image row of this thread
    const float* qb = q + (size_t)blockIdx.z * NV * ND;
    constexpr float dx = 42.0f / 512.0f;
    const float x = ((float)j - 255.5f) * dx;
    float y[PX], acc[PX];
#pragma unroll
    for (int p = 0; p < PX; ++p) { y[p] = (255.5f - (float)(i_base + 8 * p)) * dx; acc[p] = 0.f; }

    // tile corners (pixel centres) for the per-view detector segment
    const float xc0 = ((float)(blockIdx.x * 32) - 255.5f) * dx, xc1 = xc0 + 31 * dx;
    const float yc0 = (255.5f - (float)(blockIdx.y * TH)) * dx, yc1 = yc0 - (TH - 1) * dx;

    auto stage = [&](int chunk, int buf) {
        // (a) first BP_VC threads: view constants and segment start
        if (tid < BP_VC) {
            const int v = chunk * BP_VC + tid;
            const float2 c = cs_tab[v];
            float u, w, umin;
            ray_coords(xc0, yc0, c.x, c.y, inv_da, u_off, u, w); umin = u;
            ray_coords(xc1, yc0, c.x, c.y, inv_da, u_off, u, w); umin = fminf(umin, u);
            ray_coords(xc0, yc1, c.x, c.y, inv_da, u_off, u, w); umin = fminf(umin, u);
            ray_coords(xc1, yc1, c.x, c.y, inv_da, u_off, u, w); umin = fminf(umin, u);
            int k0 = ((int)floorf(umin) - 2) & ~3;           // 16-byte aligned start, one bin of slack
            k0 = max(0, min(k0, ND - SEG));
            seg0[buf][tid] = k0;
            scs[buf][tid] = c;
        }
    };
    auto copy = [&](int chunk, int buf) {
        // (b) all threads: 16-byte async copies of the segments
        for (int e = tid; e < BP_VC * (SEG / 4); e += 256) {
            const int vv = e / (SEG / 4), part = e % (SEG / 4);
            const float* g = qb + (size_t)(chunk * BP_VC + vv) * ND + seg0[buf][vv] + part * 4;
            const unsigned sa = (unsigned)__cvta_generic_to_shared(&seg[buf][vv][part * 4]);
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(sa), "l"(g) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };

    constexpr int NCHUNK = NV / BP_VC;
    stage(0, 0);
    __syncthreads();
    copy(0, 0);
    for (int ch = 0; ch < NCHUNK; ++ch) {
        const int buf = ch & 1;
        if (ch + 1 < NCHUNK) stage(ch + 1, buf ^ 1);
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();                                     // chunk ch landed; seg0/scs of ch+1 visible
        if (ch + 1 < NCHUNK) copy(ch + 1, buf ^ 1);
#pragma unroll 4
        for (int vv = 0; vv < BP_VC; ++vv) {
            const float2 c = scs[buf][vv];
            const int k0 = seg0[buf][vv];
            const float* sg = seg[buf][vv];
#pragma unroll
            for (int p = 0; p < PX; ++p) {
                float u, w;
                ray_coords(x, y[p], c.x, c.y, inv_da, u_off, u, w);
                const float kf = floorf(u);
                const int k = (int)kf;
                if (k > 0 && k < ND) {
                    const float lam = u - kf;
                    const int o = k - 1 - k0;
                    float q0, q1;
                    if ((unsigned)o < (unsigned)(SEG - 1)) { q0 = sg[o]; q1 = sg[o + 1]; }
                    else {                                   // outside the staged window: read HBM/L2 directly
                        const float* g = qb + (size_t)(ch * BP_VC + vv) * ND + k - 1;
                        q0 = __ldg(g); q1 = __ldg(g + 1);
                    }
                    acc[p] = fmaf(fmaf(lam, q1 - q0, q0), w, acc[p]);
                }
            }
        }
        __syncthreads();                                     // everyone done with buf before it is restaged
    }
    float* ob = img + (size_t)blockIdx.z * NP * NP;
    const int jo = flip ? NP - 1 - j : j;
#pragma unroll
    for (int p = 0; p < PX; ++p) ob[(size_t)(i_base + 8 * p) * NP + jo] = acc[p];
}

}  // namespace ipdm

using namespace ipdm;

extern "C" int ipdm_fbp_plan_create(ipdm_fbp_plan** out, int max_batch) {
    IPDM_REQUIRE(out != nullptr && max_batch >= 0, "ipdm_fbp_plan_create: bad arguments");
    ipdm_fbp_plan* p = new ipdm_fbp_plan();
    build_tables(p->host);
    const FbpTables& t = p->host;
    std::vector<float> htap(2 * NTAP);
    for (int c = 0; c < 2; ++c)
        for (int d = -455; d <= 455; ++d) htap[c * NTAP + d + 455] = t.h[2 * d + 2 * c - 1 + (ND - 1)];
    std::vector<float2> cs(NV);
    for (int v = 0; v < NV; ++v) cs[v] = make_float2((float)std::cos(t.theta[v]), (float)std::sin(t.theta[v]));
    std::vector<float2> ray(ND);
    for (int k = 0; k < ND; ++k) {
        const double a = (double)t.nda[k] + 0.5 * t.da;
        ray[k] = make_float2((float)std::cos(a), (float)std::sin(a));
    }
    p->h0 = t.h[ND - 1];
    p->inv_da = (float)(1.0 / t.da);
    p->u_off = (float)(0.5 - (double)t.nda[0] / t.da);
    p->dtheta = t.dtheta;
    IPDM_CHECK_CUDA(cudaMalloc(&p->d_wcos, ND * sizeof(float)));
    IPDM_CHECK_CUDA(cudaMalloc(&p->d_htap, 2 * NTAP * sizeof(float)));
    IPDM_CHECK_CUDA(cudaMalloc(&p->d_cs, NV * sizeof(float2)));
    IPDM_CHECK_CUDA(cudaMalloc(&p->d_ray, ND * sizeof(float2)));
    IPDM_CHECK_CUDA(cudaMemcpy(p->d_wcos, t.wcos.data(), ND * sizeof(float), cudaMemcpyHostToDevice));
    IPDM_CHECK_CUDA(cudaMemcpy(p->d_htap, htap.data(), 2 * NTAP * sizeof(float), cudaMemcpyHostToDevice));
    IPDM_CHECK_CUDA(cudaMemcpy(p->d_cs, cs.data(), NV * sizeof(float2), cudaMemcpyHostToDevice));
    IPDM_CHECK_CUDA(cudaMemcpy(p->d_ray, ray.data(), ND * sizeof(float2), cudaMemcpyHostToDevice));
    IPDM_CHECK(p->work.reserve(work_bytes(max_batch)));
    *out = p;
    return IPDM_OK;
}

extern "C" int ipdm_fbp_plan_destroy(ipdm_fbp_plan* p) {
    if (!p) return IPDM_OK;
    cudaFree(p->d_wcos); cudaFree(p->d_htap); cudaFree(p->d_cs); cudaFree(p->d_ray); cudaFree(p->d_rowsum);
    for (auto& kv : p->colsum) cudaFree(kv.second);
    for (GrowBuffer* b : {&p->work, &p->subset, &p->tv, &p->pwls}) b->release();
    delete p;
    return IPDM_OK;
}

extern "C" int ipdm_fbp_tables(const ipdm_fbp_plan* p, double* theta, float* nda, float* h_rl, float* wcos) {
    IPDM_REQUIRE(p != nullptr, "ipdm_fbp_tables: null plan");
    if (theta) std::copy(p->host.theta.begin(), p->host.theta.end(), theta);
    if (nda) std::copy(p->host.nda.begin(), p->host.nda.end(), nda);
    if (h_rl) std::copy(p->host.h.begin(), p->host.h.end(), h_rl);
    if (wcos) std::copy(p->host.wcos.begin(), p->host.wcos.end(), wcos);
    return IPDM_OK;
}

extern "C" int ipdm_fbp_filter(ipdm_fbp_plan* p, const float* sino, float* q, int batch, int flip, void* stream) {
    IPDM_REQUIRE(p && sino && q && batch > 0, "ipdm_fbp_filter: bad arguments");
    ProfScope prof(PROF_FBP_FILTER, (cudaStream_t)stream, 2.0 * 4 * batch * (double)NV * ND);
    fbp_filter_kernel<<<batch * NV, FILT_THREADS, 0, (cudaStream_t)stream>>>(sino, q, p->d_wcos, p->d_htap, p->h0,
                                                                             p->dtheta, flip);
    count_launch();
    IPDM_CHECK_LAUNCH();
    return IPDM_OK;
}

extern "C" int ipdm_fbp_backproject(ipdm_fbp_plan* p, const float* q, float* img, int batch, int flip, void* stream) {
    IPDM_REQUIRE(p && q && img && batch > 0, "ipdm_fbp_backproject: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    ProfScope prof(PROF_FBP_BACKPROJECT, st, 4.0 * batch * ((double)NV * ND + (double)NP * NP));   // compulsory bytes (8.345 MB / slice)
    // tile height: keep >= ~4 CTAs per SM in flight for small batches, fattest tile otherwise
    if (batch >= 4) {
        fbp_backproject_kernel<4><<<dim3(NP / 32, NP / 32, batch), 256, 0, st>>>(q, img, p->d_cs, p->inv_da, p->u_off, flip);
    } else if (batch >= 2) {
        fbp_backproject_kernel<2><<<dim3(NP / 32, NP / 16, batch), 256, 0, st>>>(q, img, p->d_cs, p->inv_da, p->u_off, flip);
    } else {
        fbp_backproject_kernel<1><<<dim3(NP / 32, NP / 8, batch), 256, 0, st>>>(q, img, p->d_cs, p->inv_da, p->u_off, flip);
    }
    count_launch();
    IPDM_CHECK_LAUNCH();
    return IPDM_OK;
}

extern "C" int ipdm_fbp_forward(ipdm_fbp_plan* p, const float* sino, float* img, int batch, int flip, void* stream) {
    IPDM_REQUIRE(p && sino && img && batch > 0, "ipdm_fbp_forward: bad arguments");
    IPDM_CHECK(p->work.reserve(work_bytes(batch)));
    IPDM_CHECK(ipdm_fbp_filter(p, sino, p->work.f32(), batch, flip, stream));
    return ipdm_fbp_backproject(p, p->work.f32(), img, batch, flip, stream);
}

extern "C" int ipdm_fbp_convert_host(ipdm_fbp_plan* p, const float* sino_host, float* img_host, int batch, int flip) {
    IPDM_REQUIRE(p && sino_host && img_host && batch > 0, "ipdm_fbp_convert_host: bad arguments");
    float *d_in = nullptr, *d_out = nullptr;
    const size_t nin = (size_t)batch * NV * ND * sizeof(float), nout = (size_t)batch * NP * NP * sizeof(float);
    IPDM_CHECK_CUDA(cudaMalloc(&d_in, nin));
    IPDM_CHECK_CUDA(cudaMalloc(&d_out, nout));
    int rc = IPDM_OK;
    if (cudaMemcpy(d_in, sino_host, nin, cudaMemcpyHostToDevice) != cudaSuccess) rc = IPDM_ERR_CUDA;
    if (rc == IPDM_OK) rc = ipdm_fbp_forward(p, d_in, d_out, batch, flip, nullptr);
    if (rc == IPDM_OK && cudaMemcpy(img_host, d_out, nout, cudaMemcpyDeviceToHost) != cudaSuccess) rc = IPDM_ERR_CUDA;
    if (rc == IPDM_ERR_CUDA) set_error("ipdm_fbp_convert_host: %s", cudaGetErrorString(cudaGetLastError()));
    cudaFree(d_in); cudaFree(d_out);
    return rc;
}
