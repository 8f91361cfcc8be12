// The FBP plan (geometry tables + workspace), shared by the convertor (fbp.cu) and the forward projector (project.cu).
#pragma once
#include "common.cuh"

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
};

namespace ipdm {
// grows plan->d_work to `batch` filtered sinograms (it is never shrunk)
int ensure_workspace(ipdm_fbp_plan* plan, int batch);
}  // namespace ipdm
