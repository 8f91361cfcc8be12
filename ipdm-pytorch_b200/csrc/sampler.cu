// Guided partial-DDPM sampler kernels for sm_100a (HBM-bound elementwise / reduction work).
// Replaces the ATen / numba / numpy algebra of the reference's Model/model.py (q_sample :438-445,
// q_sample_inverse :447-450, std :489-490, p_mean_variance_condition :492-502, p_sample_condition
// :504-515, condition_lambda_ratio_cuda :328-351, delta-map :596-600) and
// Utils/train_test_utils.py (weight_lambda / *curv_init :831-865, tensor_sharpen :868-878).
//
// One reverse step is "reduce -> apply" (SURVEY.md Appendix A):
//   pass 1  moments of eps and d = x_t - sa*x0c per slice (fp64 accumulators, fixed order)  12 B/elem
//   [pass 2 only for a per-pixel lambda map: moments of m = (1-lam) a + lam b]            +12 B/elem
//   apply   x_{t-1} from x_t, x0c, eps, noise with the per-slice constants                 20 B/elem
// All loads/stores are 128-bit; per-slice constants live in a small device buffer so nothing
// returns to the host between steps.
#include "common.cuh"

#include <cmath>
#include <vector>

namespace ipdm {

// ------------------------------------------------------------------------------------------------
// Philox4x32-10 + Box-Muller (common.cuh): 4 normals per (seed, call, slice, quad index)
// ------------------------------------------------------------------------------------------------
// Device-resident part of the Philox key.  Kernel arguments are frozen when a CUDA graph is captured, so the per-run
// entropy lives here: ipdm_set_noise_epoch() updates it between replays (ordinary stream-ordered memcpy).
__device__ unsigned long long d_noise_epoch = 0ull;

__device__ __forceinline__ float4 philox_normal4(uint64_t seed, uint64_t call, uint32_t slice, uint32_t quad) {
    const unsigned long long ep = d_noise_epoch;
    return philox_normal4_keyed(quad, slice, (uint32_t)call, (uint32_t)(call >> 32),
                                (uint32_t)seed ^ (uint32_t)(ep * 0x9E3779B97F4A7C15ull >> 32), (uint32_t)(seed >> 32) ^ (uint32_t)ep);
}

// ------------------------------------------------------------------------------------------------
// workspace layout (per call; all offsets in bytes from workspace_dev)
// ------------------------------------------------------------------------------------------------
constexpr int MOM_BLOCKS = 296;                 // 2 CTAs per SM worth of partials per slice
constexpr int MOM_THREADS = 256;
struct SliceStats {                             // written by finalize kernels, read by apply
    float A, Bc, C0;                            // scalar-lambda: e~ = A*eps + Bc*d + C0
    float mu_e, inv_se, mu_d, inv_sd;           // map-lambda: a = (eps-mu_e)*inv_se, b = (d-mu_d)*inv_sd
    float mu_m, inv_sm;                         //             e~ = (m - mu_m)*inv_sm
    float pad[7];
};
static size_t ws_partials(int batch) { return (size_t)batch * MOM_BLOCKS * 5 * sizeof(double); }
static size_t ws_stats(int batch) { return (size_t)batch * sizeof(SliceStats); }
static size_t ws_hist(int batch) { return (size_t)batch * 2048 * sizeof(unsigned); }
static size_t ws_sel(int batch) { return (size_t)batch * 4 * sizeof(unsigned); }
static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

// ------------------------------------------------------------------------------------------------
// pass 1: five raw moments per slice
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void block_reduce5(double v[5], double* out) {
    __shared__ double sm[5][MOM_THREADS / 32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < 5; ++k) { v[k] = warp_sum(v[k]); if (lane == 0) sm[k][w] = v[k]; }
    __syncthreads();
    if (threadIdx.x < 5) {
        double s = 0;
        for (int i = 0; i < MOM_THREADS / 32; ++i) s += sm[threadIdx.x][i];
        out[threadIdx.x] = s;
    }
}

__global__ void __launch_bounds__(MOM_THREADS)
moments1_kernel(const float* __restrict__ xt, const float* __restrict__ x0c, const float* __restrict__ eps,
                double* __restrict__ partials, size_t n, float sa) {
    const int b = blockIdx.y;
    const float4* X = reinterpret_cast<const float4*>(xt + (size_t)b * n);
    const float4* G = reinterpret_cast<const float4*>(x0c + (size_t)b * n);
    const float4* E = reinterpret_cast<const float4*>(eps + (size_t)b * n);
    double v[5] = {0, 0, 0, 0, 0};
    const size_t nq = n / 4;
    for (size_t i = (size_t)blockIdx.x * MOM_THREADS + threadIdx.x; i < nq; i += (size_t)gridDim.x * MOM_THREADS) {
        const float4 x = ld_stream(X + i), g = ld_stream(G + i), e = ld_stream(E + i);
        const float d0 = x.x - sa * g.x, d1 = x.y - sa * g.y, d2 = x.z - sa * g.z, d3 = x.w - sa * g.w;
        float se = (e.x + e.y) + (e.z + e.w), sd = (d0 + d1) + (d2 + d3);
        float see = fmaf(e.x, e.x, e.y * e.y) + fmaf(e.z, e.z, e.w * e.w);
        float sdd = fmaf(d0, d0, d1 * d1) + fmaf(d2, d2, d3 * d3);
        float sed = fmaf(e.x, d0, e.y * d1) + fmaf(e.z, d2, e.w * d3);
        v[0] += se; v[1] += see; v[2] += sd; v[3] += sdd; v[4] += sed;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {                 // scalar tail (n % 4)
        for (size_t i = nq * 4; i < n; ++i) {
            const float e = eps[(size_t)b * n + i], d = xt[(size_t)b * n + i] - sa * x0c[(size_t)b * n + i];
            v[0] += e; v[1] += (double)e * e; v[2] += d; v[3] += (double)d * d; v[4] += (double)e * d;
        }
    }
    block_reduce5(v, partials + ((size_t)b * gridDim.x + blockIdx.x) * 5);
}

__global__ void finalize1_kernel(const double* __restrict__ partials, SliceStats* __restrict__ stats, int nblk,
                                 double n, float lam, int use_map) {
    const int b = blockIdx.x;
    __shared__ double s[5];
    if (threadIdx.x < 5) {
        double a = 0;
        for (int i = 0; i < nblk; ++i) a += partials[((size_t)b * nblk + i) * 5 + threadIdx.x];
        s[threadIdx.x] = a;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const double mu_e = s[0] / n, mu_d = s[2] / n;
        const double var_e = (s[1] - n * mu_e * mu_e) / (n - 1), var_d = (s[3] - n * mu_d * mu_d) / (n - 1);
        const double se = sqrt(var_e), sd = sqrt(var_d);
        const double rho = (s[4] - n * mu_e * mu_d) / (se * sd) / (n - 1);
        SliceStats o;
        o.mu_e = (float)mu_e; o.inv_se = (float)(1.0 / se); o.mu_d = (float)mu_d; o.inv_sd = (float)(1.0 / sd);
        o.mu_m = 0.f; o.inv_sm = 1.f;
        if (!use_map) {
            const double l = (double)lam;
            const double sm = sqrt((1 - l) * (1 - l) + l * l + 2 * l * (1 - l) * rho);
            const double A = (1 - l) / (se * sm), Bc = l / (sd * sm);
            o.A = (float)A; o.Bc = (float)Bc; o.C0 = (float)(-(A * mu_e + Bc * mu_d));
        } else { o.A = o.Bc = o.C0 = 0.f; }
        for (int k = 0; k < 7; ++k) o.pad[k] = 0.f;
        stats[b] = o;
    }
}

// ------------------------------------------------------------------------------------------------
// pass 2 (per-pixel lambda): moments of m = (1-lam) a + lam b
// ------------------------------------------------------------------------------------------------
// lambda-map cell of element i (row-major [h][w] field, cells of ks x ks): 32-bit arithmetic, shifts when ks is a power of two
__device__ __forceinline__ unsigned lam_cell(unsigned i, unsigned w, unsigned ks, int ks_shift, unsigned lw) {
    const unsigned yy = i / w, xx = i - yy * w;
    return ks_shift >= 0 ? (yy >> ks_shift) * lw + (xx >> ks_shift) : (yy / ks) * lw + xx / ks;
}

// VEC: w % 4 == 0 and ks % 4 == 0, so the four elements of a 128-bit vector share one lambda cell
template <bool VEC>
__global__ void __launch_bounds__(MOM_THREADS)
moments2_kernel(const float* __restrict__ xt, const float* __restrict__ x0c, const float* __restrict__ eps,
                const float* __restrict__ lam_map, const SliceStats* __restrict__ stats, double* __restrict__ partials,
                int h, int w, int ks, int ks_shift, int lw, int lh, float sa) {
    const int b = blockIdx.y;
    const unsigned n = (unsigned)h * (unsigned)w;
    const SliceStats st = stats[b];
    const float* X = xt + (size_t)b * n; const float* G = x0c + (size_t)b * n; const float* E = eps + (size_t)b * n;
    const float* L = lam_map + (size_t)b * lw * lh;
    double v[5] = {0, 0, 0, 0, 0};
    if (VEC) {
        const unsigned nq = n / 4;
        for (unsigned q = blockIdx.x * MOM_THREADS + threadIdx.x; q < nq; q += gridDim.x * MOM_THREADS) {
            const float4 x = ld_stream(reinterpret_cast<const float4*>(X) + q), g = ld_stream(reinterpret_cast<const float4*>(G) + q),
                         e = ld_stream(reinterpret_cast<const float4*>(E) + q);
            const float lam = __ldg(L + lam_cell(q * 4, (unsigned)w, (unsigned)ks, ks_shift, (unsigned)lw)), oml = 1.0f - lam;
            const float m0 = oml * ((e.x - st.mu_e) * st.inv_se) + lam * (((x.x - sa * g.x) - st.mu_d) * st.inv_sd);
            const float m1 = oml * ((e.y - st.mu_e) * st.inv_se) + lam * (((x.y - sa * g.y) - st.mu_d) * st.inv_sd);
            const float m2 = oml * ((e.z - st.mu_e) * st.inv_se) + lam * (((x.z - sa * g.z) - st.mu_d) * st.inv_sd);
            const float m3 = oml * ((e.w - st.mu_e) * st.inv_se) + lam * (((x.w - sa * g.w) - st.mu_d) * st.inv_sd);
            v[0] += (double)((m0 + m1) + (m2 + m3));
            v[1] += (double)(fmaf(m0, m0, m1 * m1) + fmaf(m2, m2, m3 * m3));
        }
    } else {
        for (unsigned i = blockIdx.x * MOM_THREADS + threadIdx.x; i < n; i += gridDim.x * MOM_THREADS) {
            const float lam = __ldg(L + lam_cell(i, (unsigned)w, (unsigned)ks, ks_shift, (unsigned)lw));
            const float a = (E[i] - st.mu_e) * st.inv_se;
            const float bb = ((X[i] - sa * G[i]) - st.mu_d) * st.inv_sd;
            const float m = (1.0f - lam) * a + lam * bb;
            v[0] += m; v[1] += (double)m * m;
        }
    }
    block_reduce5(v, partials + ((size_t)b * gridDim.x + blockIdx.x) * 5);
}

__global__ void finalize2_kernel(const double* __restrict__ partials, SliceStats* __restrict__ stats, int nblk, double n) {
    const int b = blockIdx.x;
    if (threadIdx.x == 0) {
        double s0 = 0, s1 = 0;
        for (int i = 0; i < nblk; ++i) { s0 += partials[((size_t)b * nblk + i) * 5]; s1 += partials[((size_t)b * nblk + i) * 5 + 1]; }
        const double mu = s0 / n, var = (s1 - n * mu * mu) / (n - 1);
        stats[b].mu_m = (float)mu;
        stats[b].inv_sm = (float)(1.0 / sqrt(var));
    }
}

// ------------------------------------------------------------------------------------------------
// apply
// ------------------------------------------------------------------------------------------------
struct StepCoef { float sa, s1ma, srec, srecm1, c1, c2, sigma, ce; };      // ce: coefficient of e~ itself (DDIM direction term; 0 for DDPM)

__device__ __forceinline__ float step_one(float x, float etil, const StepCoef& k, int clip, float nz) {
    float x0 = k.srec * x - k.srecm1 * etil;
    if (clip) x0 = fminf(fmaxf(x0, -1.0f), 1.0f);
    if (k.ce != 0.0f) return k.c1 * x0 + k.c2 * x + k.ce * etil + nz;          // DDIM: sqrt(abar_prev) x0 + dir * e~ (+ sigma * noise)
    return k.c1 * x0 + k.c2 * x + nz;
}

template <bool MAP>
__global__ void __launch_bounds__(256)
apply_kernel(const float* xt, const float* __restrict__ x0c, const float* __restrict__ eps,
             const float* __restrict__ noise, float* out, const SliceStats* __restrict__ stats,
             const float* __restrict__ lam_map, int h, int w, int ks, int ks_shift, int lw, int lh, StepCoef k, int clip,
             int t_nonzero, uint64_t seed, uint64_t call_id) {
    const int b = blockIdx.y;
    const size_t n = (size_t)h * w, nq = n / 4;
    const SliceStats st = stats[b];
    const size_t base = (size_t)b * n;
    const float* L = MAP ? lam_map + (size_t)b * lw * lh : nullptr;
    const bool vec_map_ok = (w % 4 == 0) && (ks % 4 == 0);
    for (size_t q = (size_t)blockIdx.x * 256 + threadIdx.x; q < nq; q += (size_t)gridDim.x * 256) {
        const float4 x = ld_stream(reinterpret_cast<const float4*>(xt + base) + q);
        const float4 g = ld_stream(reinterpret_cast<const float4*>(x0c + base) + q);
        const float4 e = ld_stream(reinterpret_cast<const float4*>(eps + base) + q);
        float4 nz = make_float4(0.f, 0.f, 0.f, 0.f);
        if (t_nonzero) {
            nz = noise ? ld_stream(reinterpret_cast<const float4*>(noise + base) + q) : philox_normal4(seed, call_id, b, (uint32_t)q);
            nz.x *= k.sigma; nz.y *= k.sigma; nz.z *= k.sigma; nz.w *= k.sigma;
        }
        const float xs[4] = {x.x, x.y, x.z, x.w}, gs[4] = {g.x, g.y, g.z, g.w}, es[4] = {e.x, e.y, e.z, e.w};
        const float ns[4] = {nz.x, nz.y, nz.z, nz.w};
        float o[4];
        float lam4[4] = {0.f, 0.f, 0.f, 0.f};
        if (MAP) {
            const unsigned i0 = (unsigned)q * 4u;                      // a slice holds < 2^31 elements: 32-bit row / column arithmetic
            if (vec_map_ok) {
                const float l = __ldg(L + lam_cell(i0, (unsigned)w, (unsigned)ks, ks_shift, (unsigned)lw));
                lam4[0] = lam4[1] = lam4[2] = lam4[3] = l;
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) lam4[j] = __ldg(L + lam_cell(i0 + j, (unsigned)w, (unsigned)ks, ks_shift, (unsigned)lw));
            }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float d = xs[j] - k.sa * gs[j];
            float etil;
            if (MAP) {
                const float a = (es[j] - st.mu_e) * st.inv_se, bb = (d - st.mu_d) * st.inv_sd;
                etil = (((1.0f - lam4[j]) * a + lam4[j] * bb) - st.mu_m) * st.inv_sm;
            } else {
                etil = fmaf(st.A, es[j], fmaf(st.Bc, d, st.C0));
            }
            o[j] = step_one(xs[j], etil, k, clip, ns[j]);
        }
        st_stream(reinterpret_cast<float4*>(out + base) + q, make_float4(o[0], o[1], o[2], o[3]));
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {                 // scalar tail
        for (size_t i = nq * 4; i < n; ++i) {
            const float x = xt[base + i], d = x - k.sa * x0c[base + i], e = eps[base + i];
            float etil;
            if (MAP) {
                const int yy = (int)(i / w), xx = (int)(i - (size_t)yy * w);
                const float l = L[(size_t)(yy / ks) * lw + xx / ks];
                const float a = (e - st.mu_e) * st.inv_se, bb = (d - st.mu_d) * st.inv_sd;
                etil = (((1.0f - l) * a + l * bb) - st.mu_m) * st.inv_sm;
            } else etil = fmaf(st.A, e, fmaf(st.Bc, d, st.C0));
            float nzv = 0.f;
            if (t_nonzero) {
                if (noise) nzv = noise[base + i] * k.sigma;
                else { const float4 r = philox_normal4(seed, call_id, b, (uint32_t)(i / 4)); const float rr[4] = {r.x, r.y, r.z, r.w}; nzv = rr[i & 3] * k.sigma; }
            }
            out[base + i] = step_one(x, etil, k, clip, nzv);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// small elementwise kernels
// ------------------------------------------------------------------------------------------------
// (no __restrict__: these three are used in place)
__global__ void lincomb_kernel(float* out, float a, const float* x, float b, const float* y, float c, const float* z, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        float r = __fadd_rn(__fmul_rn(a, x[i]), __fmul_rn(b, y[i]));
        if (z) r = __fadd_rn(r, __fmul_rn(c, z[i]));
        out[i] = r;
    }
}
__global__ void clamp_kernel(float* x, float lo, float hi, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        x[i] = fminf(fmaxf(x[i], lo), hi);
}
__global__ void qsample_kernel(const float* x, const float* noise, float* out, float a, float b, size_t n, uint64_t seed,
                               uint64_t call_id) {
    const int s = blockIdx.y;
    const size_t base = (size_t)s * n;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < (n + 3) / 4; i += (size_t)gridDim.x * blockDim.x) {
        float r[4];
        if (!noise) { const float4 t = philox_normal4(seed, call_id, s, (uint32_t)i); r[0] = t.x; r[1] = t.y; r[2] = t.z; r[3] = t.w; }
        for (int j = 0; j < 4; ++j) {
            const size_t e = i * 4 + j;
            if (e < n) {
                const float nz = noise ? noise[base + e] : r[j];
                out[base + e] = __fadd_rn(__fmul_rn(a, x[base + e]), __fmul_rn(b, nz));
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// median of |x - img| per slice: 3-pass radix select on the fp32 bit pattern (values are >= 0)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
select_hist_kernel(const float* __restrict__ x, const float* __restrict__ img, unsigned* __restrict__ hist,
                   const unsigned* __restrict__ sel, size_t n, int pass) {
    __shared__ unsigned sh[2048];
    const int b = blockIdx.y;
    for (int i = threadIdx.x; i < 2048; i += 256) sh[i] = 0;
    __syncthreads();
    const unsigned prefix = pass ? sel[b * 4 + 0] : 0u;
    const unsigned pmask = pass == 0 ? 0u : (pass == 1 ? 0xFFE00000u : 0xFFFFFC00u);
    const int shift = pass == 0 ? 21 : (pass == 1 ? 10 : 0);
    const unsigned bmask = pass == 2 ? 0x3FFu : 0x7FFu;
    const float* X = x + (size_t)b * n; const float* G = img ? img + (size_t)b * n : nullptr;
    for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (size_t)gridDim.x * 256) {
        const unsigned u = __float_as_uint(fabsf(G ? X[i] - G[i] : X[i]));
        if ((u & pmask) == prefix) atomicAdd(&sh[(u >> shift) & bmask], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 2048; i += 256) if (sh[i]) atomicAdd(&hist[(size_t)b * 2048 + i], sh[i]);
}
// sel[b] = {prefix bits, remaining rank, -, -}
__global__ void select_scan_kernel(unsigned* __restrict__ hist, unsigned* __restrict__ sel, size_t n, int pass) {
    const int b = blockIdx.x;
    if (threadIdx.x == 0) {
        unsigned rank = pass ? sel[b * 4 + 1] : (unsigned)((n - 1) / 2);   // torch.median: lower middle
        const int nb = pass == 2 ? 1024 : 2048;
        const int shift = pass == 0 ? 21 : (pass == 1 ? 10 : 0);
        unsigned prefix = pass ? sel[b * 4 + 0] : 0u;
        int bin = 0;
        for (; bin < nb; ++bin) {
            const unsigned c = hist[(size_t)b * 2048 + bin];
            if (rank < c) break;
            rank -= c;
        }
        sel[b * 4 + 0] = prefix | ((unsigned)bin << shift);
        sel[b * 4 + 1] = rank;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 2048; i += blockDim.x) hist[(size_t)b * 2048 + i] = 0;   // ready for the next pass
}

// piecewise polynomial lambda curve (weight_lambda, train_test_utils.py:831-839), fp64 Horner
struct CurveCoef { double f1[5], f2[3]; };
__host__ __device__ inline double curve_eval(const CurveCoef& c, float xf) {
    const double x = (double)xf;
    auto p1 = [&](double v) { return (((c.f1[0] * v + c.f1[1]) * v + c.f1[2]) * v + c.f1[3]) * v + c.f1[4]; };
    auto p2 = [&](double v) { return (c.f2[0] * v + c.f2[1]) * v + c.f2[2]; };
    if (xf < 1.0f) return p1(1.0);
    if (x <= 1.7) return p1(x);
    if (x <= 2.75) return p2(x);
    return p2(2.75);
}

__global__ void delta_map_kernel(const float* __restrict__ x, const float* __restrict__ img, const unsigned* __restrict__ sel,
                                 float* __restrict__ lam_exp, float* __restrict__ med_out, int h, int w, int ks,
                                 int lh, int lw, float amplitude, CurveCoef cc) {
    const int b = blockIdx.y;
    const float med = __uint_as_float(sel[b * 4 + 0]);
    if (med_out && blockIdx.x == 0 && threadIdx.x == 0) med_out[b] = med;
    const size_t n = (size_t)h * w;
    for (int cidx = blockIdx.x * blockDim.x + threadIdx.x; cidx < lh * lw; cidx += gridDim.x * blockDim.x) {
        const int cy = cidx / lw, cx = cidx - cy * lw;
        float s = 0.f;
        for (int dy = 0; dy < ks; ++dy)
            for (int dxx = 0; dxx < ks; ++dxx) {
                const size_t i = (size_t)b * n + (size_t)(cy * ks + dy) * w + cx * ks + dxx;
                s = __fadd_rn(s, __fsub_rn(fabsf(__fsub_rn(x[i], img[i])), med));
            }
        float d = s / (float)(ks * ks);
        d = d <= 0.f ? 0.f : d;
        const float e = expf(__fmul_rn(amplitude, d));
        lam_exp[(size_t)b * lh * lw + cidx] = (float)curve_eval(cc, e);
    }
}

// Adaptive schedule selection (model.py:596-613): max over the slice of exp(amplitude * relu(avg_pool(|x - img| - median))).  exp is monotone,
// so the maximum of the pooled relu map is reduced (as a uint bit pattern: the values are >= 0) and exponentiated once.
__global__ void delta_pool_max_kernel(const float* __restrict__ x, const float* __restrict__ img, const unsigned* __restrict__ sel,
                                      unsigned* __restrict__ dmax_bits, int h, int w, int ks, int lh, int lw) {
    const int b = blockIdx.y;
    const float med = __uint_as_float(sel[b * 4 + 0]);
    const size_t n = (size_t)h * w;
    float best = 0.f;
    for (int cidx = blockIdx.x * blockDim.x + threadIdx.x; cidx < lh * lw; cidx += gridDim.x * blockDim.x) {
        const int cy = cidx / lw, cx = cidx - cy * lw;
        float s = 0.f;
        for (int dy = 0; dy < ks; ++dy)
            for (int dxx = 0; dxx < ks; ++dxx) {
                const size_t i = (size_t)b * n + (size_t)(cy * ks + dy) * w + cx * ks + dxx;
                s = __fadd_rn(s, __fsub_rn(fabsf(__fsub_rn(x[i], img[i])), med));
            }
        const float d = s / (float)(ks * ks);
        best = fmaxf(best, d <= 0.f ? 0.f : d);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) best = fmaxf(best, __shfl_xor_sync(0xffffffffu, best, o));
    if ((threadIdx.x & 31) == 0) atomicMax(&dmax_bits[b], __float_as_uint(best));
}
__global__ void delta_exp_kernel(const unsigned* __restrict__ dmax_bits, float* __restrict__ out, int batch, float amplitude) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < batch) out[b] = expf(__fmul_rn(amplitude, __uint_as_float(dmax_bits[b])));
}

// Image-domain variant (model.py:591-595): delt = avg_pool(|miu2pixel(x) - miu2pixel(img)|); delt -= median(delt); relu; curve(exp(amp * delt)).
// Note the order: pool first, median of the POOLED map.  miu2pixel as Dataset/npz_data_loader.py:20-36 in fp32.
__device__ __forceinline__ float miu2pixel_dev(float mu) {
    const float w = 0.183f;
    const float hu = __fsub_rn(__fdiv_rn(__fmul_rn(__fsub_rn(mu, w), 1e3f), w), 24.f);
    const float p = __fdiv_rn(__fsub_rn(hu, -1024.f), 4096.f);
    return hu < -1024.f ? 0.f : (hu > 3072.f ? 1.f : p);
}

__global__ void pool_absdiff_pixel_kernel(const float* __restrict__ x, const float* __restrict__ img, float* __restrict__ pooled,
                                          int h, int w, int ks, int lh, int lw) {
    const int b = blockIdx.y;
    const size_t n = (size_t)h * w;
    for (int cidx = blockIdx.x * blockDim.x + threadIdx.x; cidx < lh * lw; cidx += gridDim.x * blockDim.x) {
        const int cy = cidx / lw, cx = cidx - cy * lw;
        float s = 0.f;
        for (int dy = 0; dy < ks; ++dy)
            for (int dxx = 0; dxx < ks; ++dxx) {
                const size_t i = (size_t)b * n + (size_t)(cy * ks + dy) * w + cx * ks + dxx;
                s = __fadd_rn(s, fabsf(__fsub_rn(miu2pixel_dev(x[i]), miu2pixel_dev(img[i]))));
            }
        pooled[(size_t)b * lh * lw + cidx] = s / (float)(ks * ks);
    }
}

__global__ void delta_map_pooled_kernel(const float* __restrict__ pooled, const unsigned* __restrict__ sel, float* __restrict__ lam_exp,
                                        float* __restrict__ med_out, int cells, float amplitude, CurveCoef cc) {
    const int b = blockIdx.y;
    const float med = __uint_as_float(sel[b * 4 + 0]);
    if (med_out && blockIdx.x == 0 && threadIdx.x == 0) med_out[b] = med;
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < cells; c += gridDim.x * blockDim.x) {
        float d = __fsub_rn(pooled[(size_t)b * cells + c], med);
        d = d <= 0.f ? 0.f : d;
        lam_exp[(size_t)b * cells + c] = (float)curve_eval(cc, expf(__fmul_rn(amplitude, d)));
    }
}

__global__ void lambda_step_kernel(const float* __restrict__ lam_exp, float* __restrict__ out, size_t n, double f0,
                                   double f1, double f2) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const double l = (double)lam_exp[i];
        const double a0 = pow(f0, l);
        const double a1 = pow(f1, l) / a0, a2 = pow(f2, l) / a0;
        const float I = (float)(1.0 - a2 / a1);
        out[i] = fminf(fmaxf(I, 0.05f), 0.99f);
    }
}

__global__ void sharpen_kernel(const float* __restrict__ in, float* __restrict__ out, int h, int w, float centre, float other) {
    const int b = blockIdx.z;
    const int xx = blockIdx.x * blockDim.x + threadIdx.x, yy = blockIdx.y * blockDim.y + threadIdx.y;
    if (xx >= w || yy >= h) return;
    const float* I = in + (size_t)b * h * w;
    float acc = 0.f;
#pragma unroll
    for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
        for (int dxx = -1; dxx <= 1; ++dxx) {
            const int y2 = yy + dy, x2 = xx + dxx;
            const float v = (y2 >= 0 && y2 < h && x2 >= 0 && x2 < w) ? I[(size_t)y2 * w + x2] : 0.f;
            acc = fmaf((dy == 0 && dxx == 0) ? centre : other, v, acc);
        }
    out[(size_t)b * h * w + (size_t)yy * w + xx] = acc;
}

static void polyfit(const std::vector<double>& x, const std::vector<double>& y, int deg, double* out) {
    // least squares through the normal equations of the scaled Vandermonde matrix solved by QR (Householder),
    // matching np.polyfit to ~1e-12 relative on these 7-8 point fits; coefficients highest power first.
    const int m = (int)x.size(), n = deg + 1;
    std::vector<double> A((size_t)m * n), b(y);
    for (int i = 0; i < m; ++i) { double p = 1; for (int j = n - 1; j >= 0; --j) { A[(size_t)i * n + j] = p; p *= x[i]; } }
    for (int k = 0; k < n; ++k) {
        double norm = 0; for (int i = k; i < m; ++i) norm += A[(size_t)i * n + k] * A[(size_t)i * n + k];
        norm = std::sqrt(norm);
        const double alpha = A[(size_t)k * n + k] > 0 ? -norm : norm;
        std::vector<double> v(m, 0.0);
        for (int i = k; i < m; ++i) v[i] = A[(size_t)i * n + k];
        v[k] -= alpha;
        double vn = 0; for (int i = k; i < m; ++i) vn += v[i] * v[i];
        if (vn == 0) continue;
        for (int j = k; j < n; ++j) {
            double d = 0; for (int i = k; i < m; ++i) d += v[i] * A[(size_t)i * n + j];
            d = 2 * d / vn; for (int i = k; i < m; ++i) A[(size_t)i * n + j] -= d * v[i];
        }
        double d = 0; for (int i = k; i < m; ++i) d += v[i] * b[i];
        d = 2 * d / vn; for (int i = k; i < m; ++i) b[i] -= d * v[i];
    }
    for (int k = n - 1; k >= 0; --k) {
        double s = b[k]; for (int j = k + 1; j < n; ++j) s -= A[(size_t)k * n + j] * out[j];
        out[k] = s / A[(size_t)k * n + k];
    }
}

static CurveCoef make_curve(int kind) {
    CurveCoef c;
    const std::vector<double> x1 = {1, 1.1, 1.2, 1.3, 1.4, 1.5, 1.6, 1.7};
    if (kind == 0) {   // proj_curv_init (train_test_utils.py:855-865)
        polyfit(x1, {20, 17.5, 15, 12, 8.5, 7.5, 5, 4}, 4, c.f1);
        polyfit({1.7, 1.8, 2.0, 2.2, 2.35, 2.5, 3, 3.5}, {4, 3, 2, 1, 0.5, 0.3, 0.1, 0.01}, 2, c.f2);
    } else {           // curve_init (:842-852)
        polyfit(x1, {20, 17.5, 15, 12, 8.5, 5, 2, 1}, 4, c.f1);
        polyfit({1.7, 1.8, 2.0, 2.2, 2.35, 2.5, 3}, {1, 0.7, 0.5, 0.3, 0.2, 0.1, 0.05}, 2, c.f2);
    }
    return c;
}

static int grid_for(size_t n, int threads) {
    long long g = (long long)((n + threads - 1) / threads);
    const long long cap = (long long)kNumSMs * 8;
    return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

}  // namespace ipdm

using namespace ipdm;

extern "C" int ipdm_set_noise_epoch(uint64_t epoch, void* stream) {
    static uint64_t staging[64];
    static int slot = 0;
    uint64_t* h = &staging[slot++ & 63];            // the copy is asynchronous: keep the source alive
    *h = epoch;
    IPDM_CHECK_CUDA(cudaMemcpyToSymbolAsync(d_noise_epoch, h, sizeof(uint64_t), 0, cudaMemcpyHostToDevice, (cudaStream_t)stream));
    return IPDM_OK;
}

extern "C" int ipdm_lincomb(float* out, float a, const float* x, float b, const float* y, float c, const float* z,
                            size_t n, void* stream) {
    IPDM_REQUIRE(out && x && y && n > 0, "ipdm_lincomb: bad arguments");
    lincomb_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(out, a, x, b, y, c, z, n);
    count_launch();
    IPDM_CHECK_LAUNCH();
    return IPDM_OK;
}

extern "C" int ipdm_clamp(float* x, float lo, float hi, size_t n, void* stream) {
    IPDM_REQUIRE(x && n > 0, "ipdm_clamp: bad arguments");
    clamp_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(x, lo, hi, n);
    count_launch();
    IPDM_CHECK_LAUNCH();
    return IPDM_OK;
}

extern "C" size_t ipdm_sampler_workspace_bytes(int batch, int h, int w) {
    (void)h; (void)w;
    return align256(ws_partials(batch)) + align256(ws_stats(batch)) + align256(ws_hist(batch)) + align256(ws_sel(batch));
}

namespace {
struct Ws { double* partials; SliceStats* stats; unsigned* hist; unsigned* sel; };
Ws carve(void* ws, int batch) {
    char* p = (char*)ws;
    Ws o;
    o.partials = (double*)p; p += align256(ws_partials(batch));
    o.stats = (SliceStats*)p; p += align256(ws_stats(batch));
    o.hist = (unsigned*)p; p += align256(ws_hist(batch));
    o.sel = (unsigned*)p;
    return o;
}
}  // namespace

static int sampler_step_impl(const float* x_t, const float* x0c, const float* eps, const float* noise, float* x_out,
                             int batch, int h, int w, const float coef7[7], float coef_e, float lam_scalar, const float* lam_map,
                             int ks, int clip, int t_nonzero, uint64_t seed, uint64_t call_id, void* workspace,
                             void* stream) {
    IPDM_REQUIRE(x_t && x0c && eps && x_out && coef7 && workspace && batch > 0 && h > 0 && w > 0, "ipdm_sampler_step: bad arguments");
    IPDM_REQUIRE(((uintptr_t)x_t | (uintptr_t)x0c | (uintptr_t)eps | (uintptr_t)x_out | (uintptr_t)noise) % 16 == 0,
                 "ipdm_sampler_step: buffers must be 16-byte aligned");
    const size_t n = (size_t)h * w;
    IPDM_REQUIRE(batch == 1 || n % 4 == 0, "ipdm_sampler_step: H*W must be a multiple of 4 for batch > 1");
    IPDM_REQUIRE(lam_map == nullptr || (ks > 0 && h % ks == 0 && w % ks == 0),
                 "ipdm_sampler_step: a lambda map is [B][H/ks][W/ks] (as ipdm_delta_lambda_map writes it): H and W must be multiples of ks");
    cudaStream_t st = (cudaStream_t)stream;
    ProfScope prof(PROF_SAMPLER, st, (lam_map ? 44.0 : 32.0) * batch * (double)h * w);        // algorithmic bytes (SURVEY 8d)
    Ws ws = carve(workspace, batch);
    StepCoef k{coef7[0], coef7[1], coef7[2], coef7[3], coef7[4], coef7[5], coef7[6], coef_e};
    const int nblk = (int)std::min<size_t>(MOM_BLOCKS, (n / 4 + MOM_THREADS - 1) / MOM_THREADS > 0 ? (n / 4 + MOM_THREADS - 1) / MOM_THREADS : 1);
    moments1_kernel<<<dim3(nblk, batch), MOM_THREADS, 0, st>>>(x_t, x0c, eps, ws.partials, n, k.sa);
    finalize1_kernel<<<batch, 32, 0, st>>>(ws.partials, ws.stats, nblk, (double)n, lam_scalar, lam_map != nullptr);
    count_launch(2);
    const int lw = lam_map ? w / ks : 0, lh = lam_map ? h / ks : 0;
    int ks_shift = -1;
    for (int sft = 0; sft < 16; ++sft) if (ks == (1 << sft)) ks_shift = sft;
    IPDM_REQUIRE(n < (1ull << 31), "ipdm_sampler_step: a slice may hold at most 2^31 elements");
    const int ablk = (int)std::min<size_t>((size_t)kNumSMs * 4, (n / 4 + 255) / 256 > 0 ? (n / 4 + 255) / 256 : 1);
    if (lam_map) {
        const int nblk2 = (int)std::min<size_t>(MOM_BLOCKS, (n + MOM_THREADS - 1) / MOM_THREADS);
        if (w % 4 == 0 && ks % 4 == 0 && n % 4 == 0)
            moments2_kernel<true><<<dim3(nblk, batch), MOM_THREADS, 0, st>>>(x_t, x0c, eps, lam_map, ws.stats, ws.partials, h, w, ks, ks_shift, lw, lh, k.sa);
        else
            moments2_kernel<false><<<dim3(nblk2, batch), MOM_THREADS, 0, st>>>(x_t, x0c, eps, lam_map, ws.stats, ws.partials, h, w, ks, ks_shift, lw, lh, k.sa);
        finalize2_kernel<<<batch, 32, 0, st>>>(ws.partials, ws.stats, (w % 4 == 0 && ks % 4 == 0 && n % 4 == 0) ? nblk : nblk2, (double)n);
        apply_kernel<true><<<dim3(ablk, batch), 256, 0, st>>>(x_t, x0c, eps, noise, x_out, ws.stats, lam_map, h, w, ks, ks_shift, lw, lh, k, clip, t_nonzero, seed, call_id);
        count_launch(3);
    } else {
        apply_kernel<false><<<dim3(ablk, batch), 256, 0, st>>>(x_t, x0c, eps, noise, x_out, ws.stats, nullptr, h, w, 1, 0, 0, 0, k, clip, t_nonzero, seed, call_id);
        count_launch();
    }
    IPDM_CHECK_LAUNCH();
    return IPDM_OK;
}

extern "C" int ipdm_sampler_step(const float* x_t, const float* x0c, const float* eps, const float* noise, float* x_out,
                                 int batch, int h, int w, const float coef7[7], float lam_scalar, const float* lam_map,
                                 int ks, int clip, int t_nonzero, uint64_t seed, uint64_t call_id, void* workspace,
                                 void* stream) {
    return sampler_step_impl(x_t, x0c, eps, noise, x_out, batch, h, w, coef7, 0.0f, lam_scalar, lam_map, ks, clip, t_nonzero, seed, call_id,
                             workspace, stream);
}

extern "C" int ipdm_sampler_step_ddim(const float* x_t, const float* x0c, const float* eps, const float* noise, float* x_out,
                                      int batch, int h, int w, const float coef8[8], float lam_scalar, int clip, int with_noise,
                                      uint64_t seed, uint64_t call_id, void* workspace, void* stream) {
    IPDM_REQUIRE(coef8, "ipdm_sampler_step_ddim: bad arguments");
    return sampler_step_impl(x_t, x0c, eps, noise, x_out, batch, h, w, coef8, coef8[7], lam_scalar, nullptr, 1, clip, with_noise, seed, call_id,
                             workspace, stream);
}

extern "C" int ipdm_q_sample(const float* x, const float* noise, float* out, float a, float b, size_t n_per_slice,
                             int batch, uint64_t seed, uint64_t call_id, void* stream) {
    IPDM_REQUIRE(x && out && n_per_slice > 0 && batch > 0, "ipdm_q_sample: bad arguments");
    qsample_kernel<<<dim3(grid_for((n_per_slice + 3) / 4, 256), batch), 256, 0, (cudaStream_t)stream>>>(x, noise, out, a, b, n_per_slice, seed, call_id);
    count_launch();
    IPDM_CHECK_LAUNCH();
    return IPDM_OK;
}

extern "C" int ipdm_delta_lambda_map(const float* x, const float* img, float* lam_exp_out, float* median_out, int batch,
                                     int h, int w, int ks, float amplitude, int curve_kind, void* workspace, void* stream) {
    IPDM_REQUIRE(x && img && lam_exp_out && workspace && batch > 0 && ks > 0, "ipdm_delta_lambda_map: bad arguments");
    IPDM_REQUIRE(h % ks == 0 && w % ks == 0, "ipdm_delta_lambda_map: H and W must be multiples of ks");
    cudaStream_t st = (cudaStream_t)stream;
    Ws ws = carve(workspace, batch);
    const size_t n = (size_t)h * w;
    IPDM_CHECK_CUDA(cudaMemsetAsync(ws.hist, 0, ws_hist(batch), st));
    const int g = (int)std::min<size_t>((size_t)kNumSMs * 2, (n + 255) / 256);
    for (int pass = 0; pass < 3; ++pass) {
        select_hist_kernel<<<dim3(g, batch), 256, 0, st>>>(x, img, ws.hist, ws.sel, n, pass);
        select_scan_kernel<<<batch, 256, 0, st>>>(ws.hist, ws.sel, n, pass);
    }
    const int lh = h / ks, lw = w / ks;                       // avg_pool2d floors (model.py:598)
    delta_map_kernel<<<dim3(ceil_div((long long)lh * lw, 256), batch), 256, 0, st>>>(x, img, ws.sel, lam_exp_out, median_out, h, w, ks, lh, lw, amplitude, make_curve(curve_kind));
    count_launch(7);
    IPDM_CHECK_LAUNCH();
    return IPDM_OK;
}

extern "C" int ipdm_delta_exp_max(const float* x, const float* img, float* max_out, int batch, int h, int w, int ks, float amplitude,
                                  void* workspace, void* stream) {
    IPDM_REQUIRE(x && img && max_out && workspace && batch > 0 && ks > 0, "ipdm_delta_exp_max: bad arguments");
    IPDM_REQUIRE(h % ks == 0 && w % ks == 0, "ipdm_delta_exp_max: H and W must be multiples of ks");
    cudaStream_t st = (cudaStream_t)stream;
    Ws ws = carve(workspace, batch);
    const size_t n = (size_t)h * w;
    IPDM_CHECK_CUDA(cudaMemsetAsync(ws.hist, 0, ws_hist(batch), st));
    const int g = (int)std::min<size_t>((size_t)kNumSMs * 2, (n + 255) / 256);
    for (int pass = 0; pass < 3; ++pass) {                                   // exact lower median of |x - img| per slice
        select_hist_kernel<<<dim3(g, batch), 256, 0, st>>>(x, img, ws.hist, ws.sel, n, pass);
        select_scan_kernel<<<batch, 256, 0, st>>>(ws.hist, ws.sel, n, pass);
    }
    const int lh = h / ks, lw = w / ks;
    unsigned* bits = ws.hist;                                                // the histogram is idle (zeroed by the last scan pass)
    delta_pool_max_kernel<<<dim3(std::min(ceil_div((long long)lh * lw, 256), kNumSMs * 4), batch), 256, 0, st>>>(x, img, ws.sel, bits, h, w, ks, lh, lw);
    delta_exp_kernel<<<ceil_div(batch, 128), 128, 0, st>>>(bits, max_out, batch, amplitude);
    count_launch(8);
    IPDM_CHECK_LAUNCH();
    IPDM_CHECK_CUDA(cudaMemsetAsync(ws.hist, 0, (size_t)batch * sizeof(unsigned), st));
    return IPDM_OK;
}

extern "C" int ipdm_delta_lambda_map_img(const float* x, const float* img, float* lam_exp_out, float* median_out, float* pooled_tmp,
                                         int batch, int h, int w, int ks, float amplitude, int curve_kind, void* workspace, void* stream) {
    IPDM_REQUIRE(x && img && lam_exp_out && pooled_tmp && workspace && batch > 0 && ks > 0, "ipdm_delta_lambda_map_img: bad arguments");
    IPDM_REQUIRE(h % ks == 0 && w % ks == 0, "ipdm_delta_lambda_map_img: H and W must be multiples of ks");
    cudaStream_t st = (cudaStream_t)stream;
    Ws ws = carve(workspace, batch);
    const int lh = h / ks, lw = w / ks, cells = lh * lw;
    const int gc = ceil_div((long long)cells, 256);
    pool_absdiff_pixel_kernel<<<dim3(gc, batch), 256, 0, st>>>(x, img, pooled_tmp, h, w, ks, lh, lw);
    IPDM_CHECK_CUDA(cudaMemsetAsync(ws.hist, 0, ws_hist(batch), st));
    const int g = (int)std::min<size_t>((size_t)kNumSMs * 2, (size_t)gc);
    for (int pass = 0; pass < 3; ++pass) {                               // exact lower median of the pooled map (values >= 0)
        select_hist_kernel<<<dim3(g, batch), 256, 0, st>>>(pooled_tmp, nullptr, ws.hist, ws.sel, (size_t)cells, pass);
        select_scan_kernel<<<batch, 256, 0, st>>>(ws.hist, ws.sel, (size_t)cells, pass);
    }
    delta_map_pooled_kernel<<<dim3(gc, batch), 256, 0, st>>>(pooled_tmp, ws.sel, lam_exp_out, median_out, cells, amplitude, make_curve(curve_kind));
    count_launch(8);
    IPDM_CHECK_LAUNCH();
    return IPDM_OK;
}

extern "C" int ipdm_lambda_step_map(const float* lam_exp, float* lam_out, size_t n, int i, int ts, void* stream) {
    IPDM_REQUIRE(lam_exp && lam_out && n > 0 && ts > 0 && i >= 0 && i < ts, "ipdm_lambda_step_map: bad arguments");
    const double s = 0.008;
    auto f = [&](int k) { double c = std::cos((((double)k / ts) + s) / (1 + s) * M_PI * 0.5); return c * c; };
    lambda_step_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(lam_exp, lam_out, n, f(0), f(i), f(i + 1));
    count_launch();
    IPDM_CHECK_LAUNCH();
    return IPDM_OK;
}

extern "C" int ipdm_lambda_curve_host(const float* x, float* y, size_t n, int curve_kind) {
    IPDM_REQUIRE(x && y && (curve_kind == 0 || curve_kind == 1), "ipdm_lambda_curve_host: bad arguments");
    const CurveCoef c = make_curve(curve_kind);
    for (size_t i = 0; i < n; ++i) y[i] = (float)curve_eval(c, x[i]);
    return IPDM_OK;
}

extern "C" int ipdm_sharpen3x3(const float* in, float* out, int batch, int h, int w, int N, void* stream) {
    IPDM_REQUIRE(in && out && batch > 0 && h > 0 && w > 0, "ipdm_sharpen3x3: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    if (N == -1) {
        if (in != out) IPDM_CHECK_CUDA(cudaMemcpyAsync(out, in, (size_t)batch * h * w * sizeof(float), cudaMemcpyDeviceToDevice, st));
        return IPDM_OK;
    }
    IPDM_REQUIRE(in != out, "ipdm_sharpen3x3: in-place is not supported");
    IPDM_REQUIRE(N != 16, "ipdm_sharpen3x3: N == 16 divides by zero");
    const float centre = (float)N / (float)(N - 16), other = -2.0f / (float)(N - 16);
    sharpen_kernel<<<dim3(ceil_div(w, 32), ceil_div(h, 8), batch), dim3(32, 8), 0, st>>>(in, out, h, w, centre, other);
    count_launch();
    IPDM_CHECK_LAUNCH();
    return IPDM_OK;
}

// ---- schedule tables (host, fp64): Model/model.py:366-372, 376-421 -------------------------------
namespace ipdm {
struct Schedule { std::vector<double> v[10]; };
static void build_schedule(int T, double p, Schedule& s) {
    std::vector<double> ac(T + 1);
    for (int i = 0; i <= T; ++i) {
        const double c = std::cos((((double)i / T) + 0.008) / 1.008 * M_PI * 0.5);
        ac[i] = std::pow(c * c, p);
    }
    const double a0 = ac[0];
    for (auto& a : ac) a /= a0;
    for (int k = 0; k < 10; ++k) s.v[k].resize(T);
    double cum = 1.0;
    for (int t = 0; t < T; ++t) {
        double beta = 1 - ac[t + 1] / ac[t];
        beta = beta < 0 ? 0 : (beta > 0.999 ? 0.999 : beta);
        const double alpha = 1.0 - beta, prev = cum;
        cum *= alpha;
        s.v[0][t] = beta; s.v[1][t] = cum; s.v[2][t] = std::sqrt(cum); s.v[3][t] = std::sqrt(1.0 - cum);
        s.v[4][t] = std::sqrt(1.0 / cum); s.v[5][t] = std::sqrt(1.0 / cum - 1);
        const double pv = beta * (1.0 - prev) / (1.0 - cum);
        s.v[6][t] = pv; s.v[7][t] = std::log(pv < 1e-20 ? 1e-20 : pv);
        s.v[8][t] = beta * std::sqrt(prev) / (1.0 - cum);
        s.v[9][t] = (1.0 - prev) * std::sqrt(alpha) / (1.0 - cum);
    }
}
int schedule_at(int T, double p, int t, double out[10]) {
    static int cT = -1; static double cp = 0; static Schedule cache;
    if (cT != T || cp != p) { build_schedule(T, p, cache); cT = T; cp = p; }
    for (int k = 0; k < 10; ++k) out[k] = cache.v[k][t];
    return IPDM_OK;
}
}  // namespace ipdm

extern "C" int ipdm_cosine_beta_schedule(int timesteps, double schedule_power, double* betas_out) {
    IPDM_REQUIRE(timesteps > 0 && betas_out, "ipdm_cosine_beta_schedule: bad arguments");
    Schedule s; build_schedule(timesteps, schedule_power, s);
    std::copy(s.v[0].begin(), s.v[0].end(), betas_out);
    return IPDM_OK;
}
extern "C" int ipdm_schedule_at(int timesteps, double schedule_power, int t, double out10[10]) {
    IPDM_REQUIRE(timesteps > 0 && t >= 0 && t < timesteps && out10, "ipdm_schedule_at: bad arguments");
    return schedule_at(timesteps, schedule_power, t, out10);
}
