/*
 * libipdm_b200.so -- C ABI of the B200-native IPDM domain-progressive inference path.
 *
 * Drop-in boundary for the hot path of LFY1998/IPDM-PyTorch (paths below are relative to the
 * reference root).  The reference is pure Python: its "FFI" for this path is the set of Python
 * call sites listed next to each entry point; the host-side mirrors under ipdm-pytorch_b200/
 * (Recon/FBP_kernel.py, Model/model.py, Utils/train_test_utils.py) bind these symbols with
 * ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - every function returns IPDM_OK (0) or a negative IPDM_ERR_* code; the message of the last
 *     failure on the calling thread is returned by ipdm_last_error().  No exceptions cross.
 *   - `*_dev` pointers are device pointers owned by the caller (PyTorch); the library never
 *     frees or retains them past the call.  Handles own only their tables, packed weights and
 *     workspace.  `stream` is a cudaStream_t passed as void*; all work is enqueued on it and
 *     nothing synchronises with the host unless stated ("host" in the name).
 *   - images / sinograms are fp32, slice-major: sinogram [B][2000 views][912 detectors],
 *     image [B][512][512], generic fields [B][H][W].  All statistics are per slice (the
 *     reference only ever runs B = 1; see SURVEY.md D3).
 *   - handles are not thread-safe; one host thread per GPU.
 */
#ifndef IPDM_B200_H
#define IPDM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IPDM_OK 0
#define IPDM_ERR_ARG (-1)
#define IPDM_ERR_CUDA (-2)
#define IPDM_ERR_UNSUPPORTED (-3)
#define IPDM_ERR_ALLOC (-4)

#define IPDM_N_VIEWS 2000
#define IPDM_N_DET 912
#define IPDM_N_PIX 512

const char* ipdm_last_error(void);
int ipdm_abi_version(void);
/* number of kernels this library has launched since the last reset (bench.py: gpu_launches) */
unsigned long long ipdm_launch_count(void);
void ipdm_launch_count_reset(void);

/* Per-kernel-family profiler for bench.py: when enabled, every launch is bracketed by CUDA events on its
 * stream.  Families (index): 0 conv_tc other than family 8 (work = FLOPs issued), 1 attention (FLOPs), 2 conv_direct (bytes),
 * 3 groupnorm (bytes), 4 upsample (bytes), 5 fbp_filter (bytes), 6 fbp_backproject (compulsory bytes),
 * 7 sampler step (algorithmic bytes), 8 conv_halo_persistent_kernel, the dominant kernel (FLOPs issued).
 * collect() synchronises the device and sums per family. */
#define IPDM_PROF_KINDS 9
void ipdm_profile_enable(int on);
int ipdm_profile_collect(double ms_out[IPDM_PROF_KINDS], double work_out[IPDM_PROF_KINDS], long long launches_out[IPDM_PROF_KINDS]);
/* Mixed roofline of one FLOP-counted family (the tensor-core conv families record their algorithmic HBM bytes too):
 * roof_ms = sum over its launches of max(flops / peak_flops_per_s, bytes / peak_bytes_per_s), ms = their measured time. */
int ipdm_profile_roofline(int kind, double peak_flops_per_s, double peak_bytes_per_s, double* roof_ms_out, double* ms_out, double* bytes_out);

/* ------------------------------------------------------------------------------------------
 * Image-quality metrics on the device (SURVEY N1).  Replaces the skimage calls of
 * progressive_domain_denoiser.metric_calculate, Utils/train_test_utils.py:789-799
 * (compare_psnr(fdct, ld, data_range=1), compare_ssim(fdct, ld, win_size=11, data_range=1)) and the
 * unit conversion miu2pixel, Dataset/npz_data_loader.py:20-36.  Images are [batch][h][w] f32 in
 * "pixel" units; NaNs of the test image count as 0.5 (:792).  out_dev[b] = {PSNR dB, SSIM} (f64).
 * ---------------------------------------------------------------------------------------- */
size_t ipdm_metrics_workspace_bytes(int batch, int h, int w);
int ipdm_psnr_ssim(const float* test_dev, const float* ref_dev, int batch, int h, int w, int win_size, double* out_dev,
                   void* workspace_dev, void* stream);
/* pix = clip((HU(mu) - hu_lo) / (hu_hi - hu_lo), 0, 1), HU(mu) = (mu - 0.183) * 1e3 / 0.183 - 24; NaN -> 0.5 */
int ipdm_miu2pixel(const float* mu_dev, float* pix_dev, size_t n, float hu_lo, float hu_hi, void* stream);

/* ------------------------------------------------------------------------------------------
 * FBP convertor.  Replaces Recon/FBP_kernel.py: FBP.__init__ :27-67 (tables), FBP.convert
 * :86-122, conv_pj/conv_kernel :125-143 (ramp filter), fbp_cpu/fbp_kernel :146-184
 * (pixel-driven fan-beam backprojection).  Call site: Utils/train_test_utils.py:229, :465, :475.
 * ---------------------------------------------------------------------------------------- */
typedef struct ipdm_fbp_plan ipdm_fbp_plan;

int ipdm_fbp_plan_create(ipdm_fbp_plan** out, int max_batch);
int ipdm_fbp_plan_destroy(ipdm_fbp_plan* plan);
/* weighting (flip, D cos(gamma), dtheta) + ramp filter: sino [B,2000,912] -> q [B,2000,912] */
int ipdm_fbp_filter(ipdm_fbp_plan* plan, const float* sino_dev, float* q_dev, int batch, int flip, void* stream);
/* backprojection of filtered data: q [B,2000,912] -> img [B,512,512] (column-flipped iff flip) */
int ipdm_fbp_backproject(ipdm_fbp_plan* plan, const float* q_dev, float* img_dev, int batch, int flip, void* stream);
/* both stages, device to device; uses the plan's workspace (grown on demand, max_batch is pre-sized) */
int ipdm_fbp_forward(ipdm_fbp_plan* plan, const float* sino_dev, float* img_dev, int batch, int flip, void* stream);
/* FBP.convert semantics: HOST sinogram in, HOST image out (copies + sync inside) */
int ipdm_fbp_convert_host(ipdm_fbp_plan* plan, const float* sino_host, float* img_host, int batch, int flip);
/* host copies of the tables, for parity tests: theta[2000] f64, nda[912], h_RL[1823], wcos[912] */
int ipdm_fbp_tables(const ipdm_fbp_plan* plan, double* theta, float* nda, float* h_rl, float* wcos);
/* Forward projector in the plan's geometry (no counterpart in the reference; its projector is the Windows-only
 * TASART2DNSL0.pyd): mu image img [B,512,512] (1/cm) -> line integrals sino [B,2000,912], the rays the backprojector reads
 * (fan angle nda[k] + da/2), Joseph's method (one linearly interpolated sample per column or row crossed, fp32).
 * flip as for ipdm_fbp_forward: 1 = image in the convertor's output frame, sinogram in its input frame; 0 = both native.
 * Uses the plan's workspace (grown on demand). */
int ipdm_fbp_project(ipdm_fbp_plan* plan, const float* img_dev, float* sino_dev, int batch, int flip, void* stream);
/* Exact adjoint (transpose) of ipdm_fbp_project: sino [B,2000,912] -> img [B,512,512], img = A^T sino with A the fp32 matrix the
 * projector applies (the same weights, bit for bit) and the same flip frames.  Deterministic (no atomics), slice by slice. */
int ipdm_fbp_project_adjoint(ipdm_fbp_plan* plan, const float* sino_dev, float* img_dev, int batch, int flip, void* stream);
/* Ordered-subset SART convertor (replaces the SART core of the reference's Windows-only ART convertor TASART2DNSL0.pyd,
 * correction_kernel / update_kernel; not its NSL0-TV step): line integrals sino [B,2000,912] -> mu image img [B,512,512], frames
 * as for ipdm_fbp_forward.  Subset s = views v with v mod S = s, S = subsets dividing 2000; a sweep visits s_n = n p mod S,
 * p the integer in [1, S) coprime to S closest to 0.382 S (smaller on a tie; 1 when S <= 2).  x0 = 0; per subset
 * r = (b - A_s x) / R (0 where R = A 1 is 0), x <- max(0, x + relaxation * A_s^T r / C_s) where C_s = A_s^T 1 > 0.
 * iterations >= 1 sweeps, 0 < relaxation < 2, img must not alias sino.  R and C_s are built in the plan by the first call
 * for a given S (that call synchronises the stream and cannot be captured); later calls of the same or a smaller shape allocate
 * nothing and do not synchronise. */
int ipdm_fbp_sart(ipdm_fbp_plan* plan, const float* sino_dev, float* img_dev, int batch, int flip, int iterations, int subsets,
                  float relaxation, void* stream);

/* ------------------------------------------------------------------------------------------
 * Diffusion schedule.  Replaces Model/model.py: cosine_beta_schedule :366-372 and
 * GaussianDiffusion.__init__ :376-421 (fp64 tables), _extract :424-428.
 * ---------------------------------------------------------------------------------------- */
/* betas_out[timesteps] fp64 */
int ipdm_cosine_beta_schedule(int timesteps, double schedule_power, double* betas_out);
/* fp64 table values at index t, in this order: betas, alphas_cumprod, sqrt_alphas_cumprod,
 * sqrt_one_minus_alphas_cumprod, sqrt_recip_alphas_cumprod, sqrt_recipm1_alphas_cumprod,
 * posterior_variance, posterior_log_variance_clipped, posterior_mean_coef1, posterior_mean_coef2 */
int ipdm_schedule_at(int timesteps, double schedule_power, int t, double out10[10]);

/* ------------------------------------------------------------------------------------------
 * Sampler kernels.  Replace the ATen / numba / numpy algebra of Model/model.py:
 *   q_sample :438-445, q_sample_inverse :447-450, std :489-490,
 *   p_mean_variance_condition :492-502, p_sample_condition :504-515,
 *   condition_lambda_ratio_cuda :328-351 (+ clip :558, nearest upsample :559),
 *   the delta-map of guided_reverse_process :596-600, :614, blends :626-638, clamps :569-573,
 * and Utils/train_test_utils.py: weight_lambda/proj_curv_init :831-865, tensor_sharpen :868-878.
 * ---------------------------------------------------------------------------------------- */
/* out = a*x + b*y (+ c*z if z_dev != NULL), each product and sum rounded to fp32 (no FMA), n elements */
int ipdm_lincomb(float* out_dev, float a, const float* x_dev, float b, const float* y_dev, float c,
                 const float* z_dev, size_t n, void* stream);
int ipdm_clamp(float* x_dev, float lo, float hi, size_t n, void* stream); /* pass -INF / +INF to disable a side */

size_t ipdm_sampler_workspace_bytes(int batch, int h, int w);
/*
 * One guided reverse step t for B slices of H x W:
 *   c      = (x_t - sa*x0c)/s1ma,  e~ = S((1-lam) S(eps) + lam S(c)),  S = per-slice standardise (unbiased std)
 *   x0     = srec*x_t - srecm1*e~  (clamped to [-1,1] iff clip)
 *   x_out  = coef1*x0 + coef2*x_t + (t_nonzero ? sigma*noise : 0)
 * coef7 = {sa, s1ma, srec, srecm1, coef1, coef2, sigma} as fp32 (sigma = exp(0.5*posterior_log_variance)).
 * lam: scalar `lam_scalar`, or per-pixel map lam_map_dev [B][ceil(H/ks)][ceil(W/ks)] (nearest-upsampled by ks)
 * when lam_map_dev != NULL.  noise_dev == NULL draws N(0,1) from Philox4x32-10 keyed by (seed, call_id).
 * x_out_dev may alias x_t_dev.
 */
int ipdm_sampler_step(const float* x_t_dev, const float* x0c_dev, const float* eps_dev, const float* noise_dev,
                      float* x_out_dev, int batch, int h, int w, const float coef7[7], float lam_scalar,
                      const float* lam_map_dev, int ks, int clip, int t_nonzero, uint64_t seed, uint64_t call_id,
                      void* workspace_dev, void* stream);
/*
 * One guided DDIM step (sparse sampler, Model/model.py ddim_sample :654-720) with the same e~ and x0 as above:
 *   x_out = coef1*x0 + coef_e*e~ + (with_noise ? sigma*noise : 0)
 * coef8 = {sa, s1ma, srec, srecm1, coef1 = sqrt(abar_prev), coef2 = 0, sigma = ddim_eta*posterior_variance[t],
 *          coef_e = sqrt(1 - abar_prev - sigma_t(eta)^2)}; lam is the scalar condition_lambda of the iteration.
 */
int ipdm_sampler_step_ddim(const float* x_t_dev, const float* x0c_dev, const float* eps_dev, const float* noise_dev,
                           float* x_out_dev, int batch, int h, int w, const float coef8[8], float lam_scalar, int clip,
                           int with_noise, uint64_t seed, uint64_t call_id, void* workspace_dev, void* stream);
/* Device-resident half of the Philox key (default 0).  CUDA-graph replays reuse frozen kernel arguments, so callers
 * bump this epoch between replays to get fresh noise; it is an ordinary stream-ordered update. */
int ipdm_set_noise_epoch(uint64_t epoch, void* stream);
/* out = a*x + b*N(0,1) with caller noise or Philox (q_sample) */
int ipdm_q_sample(const float* x_dev, const float* noise_dev, float* out_dev, float a, float b, size_t n_per_slice,
                  int batch, uint64_t seed, uint64_t call_id, void* stream);
/* Dose-reduction noise of the reference's Utils/Low_dose_CT_simulate.py add_noise (:38-44) on line integrals p:
 *   out = p + sqrt((1-f) e^p (1 + (1+f) Ne e^p / (f N0)) / (f N0)) * n,  f = dose in (0, 1], Ne = 5.8, N0 = 1.4e5,
 * clamped at 0 iff clip.  n from noise_dev (same layout as sino) or, when noise_dev == NULL, from Philox4x32-10 keyed by
 * (seed, slice id, element / 4); slice_ids_dev_or_null [B] holds the slice ids (NULL: 0..B-1), so a slice's noise does not depend
 * on its position in the batch.  The device-resident noise epoch is not part of the key.  out_dev may alias sino_dev. */
int ipdm_low_dose_noise(const float* sino_dev, const float* noise_dev, float* out_dev, int batch, size_t n_per_slice, float dose,
                        int clip, uint64_t seed, const uint64_t* slice_ids_dev_or_null, void* stream);
/* Lambda-exponent map of the first proj iteration: relu(avgpool_ks(|x-img| - median)) -> exp(amp*.) -> curve.
 * curve_kind 0 = proj_curv_init, 1 = curve_init.  out [B][H/ks][W/ks].  median_out_dev (optional) [B]. */
int ipdm_delta_lambda_map(const float* x_dev, const float* img_dev, float* lam_exp_out_dev, float* median_out_dev,
                          int batch, int h, int w, int ks, float amplitude, int curve_kind, void* workspace_dev,
                          void* stream);
/* Image-domain variant (Model/model.py:591-595): avgpool_ks(|miu2pixel(x) - miu2pixel(img)|) - median(pooled map) -> relu ->
 * exp(amp*.) -> curve.  pooled_tmp_dev: scratch [B][H/ks][W/ks]. */
int ipdm_delta_lambda_map_img(const float* x_dev, const float* img_dev, float* lam_exp_out_dev, float* median_out_dev,
                              float* pooled_tmp_dev, int batch, int h, int w, int ks, float amplitude, int curve_kind,
                              void* workspace_dev, void* stream);
/* Adaptive schedule selection of the projection domain (Model/model.py:596-613, t_start=None): per slice
 * max_out[b] = max over the slice of exp(amp * relu(avgpool_ks(|x - img| - median(|x - img|)))), the quantity the reference compares
 * with 30 / 4.5 to pick [30,25,20] / [20,18,15] / [15,15,15].  One D2H read of B floats is the only host round trip of that branch. */
int ipdm_delta_exp_max(const float* x_dev, const float* img_dev, float* max_out_dev, int batch, int h, int w, int ks,
                       float amplitude, void* workspace_dev, void* stream);
/* per-step guidance map clip(1 - (abar(i+1)/abar(i))^Lambda, .05, .99), fp64 math, n cells */
int ipdm_lambda_step_map(const float* lam_exp_dev, float* lam_out_dev, size_t n, int i, int ts, void* stream);
/* host evaluation of the piecewise lambda curve (fp64 polyfit coefficients), for tests */
int ipdm_lambda_curve_host(const float* x, float* y, size_t n, int curve_kind);
/* 3x3 sharpen with zero padding, centre N, others -2, all divided by N-16; N == -1 copies */
int ipdm_sharpen3x3(const float* in_dev, float* out_dev, int batch, int h, int w, int N, void* stream);

/* ------------------------------------------------------------------------------------------
 * UNet noise predictor.  Replaces Model/model.py UNetModel :190-310 and its blocks :14-185.
 * Weights arrive as ONE host fp32 buffer holding the reference state_dict tensors in
 * state_dict order (time_embed.0.weight, time_embed.0.bias, ..., out.2.bias), each in its
 * PyTorch layout; the library repacks them for its kernels.
 * ---------------------------------------------------------------------------------------- */
typedef struct ipdm_unet ipdm_unet;

typedef struct ipdm_unet_config {
    int in_channels, model_channels, out_channels, num_res_blocks, num_heads;
    int n_mult;               /* len(channel_mult), <= 8 */
    double channel_mult[8];
    int n_attn;               /* len(attention_resolutions), <= 8 */
    int attention_resolutions[8];
    int precision;            /* IPDM_PREC_* */
    int max_t;                /* time embeddings are precomputed for t in [0, max_t) */
} ipdm_unet_config;

#define IPDM_PREC_TF32 0   /* fp32 activations, tcgen05 kind::tf32 contractions, fp32 accumulate (reference GPU default) */
#define IPDM_PREC_BF16 1   /* bf16 operands (GroupNorm-apply / upsample outputs, weights) for tcgen05 kind::f16 in the 3x3 convs and
                              qkv; fp32 residual stream, accumulators, norm statistics, attention and sampler state */
#define IPDM_PREC_FP32 2   /* fp32 activations, 3xTF32 split contractions (fp32-accurate) */

int ipdm_unet_create(ipdm_unet** out, const ipdm_unet_config* cfg, const float* weights_host, size_t n_weights);
int ipdm_unet_destroy(ipdm_unet* net);
/* number of fp32 values ipdm_unet_create expects for this config (== sum of state_dict numels) */
long long ipdm_unet_param_count(const ipdm_unet_config* cfg);
/* eps[B,out_ch,H,W] = UNet(x[B,in_ch,H,W], t) for one integer timestep shared by the batch (model.py:564) */
int ipdm_unet_forward(ipdm_unet* net, const float* x_dev, int t, float* eps_dev, int batch, int h, int w, void* stream);
/* algorithmic FLOPs (2*MAC; convs, 1x1, attention QK^T + PV) of one forward at this shape */
double ipdm_unet_flops(const ipdm_unet* net, int batch, int h, int w);

/* ------------------------------------------------------------------------------------------
 * Guided partial reverse process and the progressive pipeline.  Replace
 * GaussianDiffusion.guided_reverse_process (Model/model.py:517-642, explicit t_start branches) and
 * progressive_domain_denoiser.{proj_denoiser,img_denoiser,progressive_denoiser}
 * (Utils/train_test_utils.py:421-567).  Everything is enqueued on `stream`; no host round trip.
 * ---------------------------------------------------------------------------------------- */
typedef struct ipdm_guided_params {
    int mode;                 /* 0 = proj, 1 = img */
    int n_iters;              /* len(t_start) <= 8 */
    int t_start[8];
    int clip;
    double lambda_ratio;      /* schedule_power of the scalar cosine lambda (proj iteration 0) */
    double eta;
    int constant_guidance_set;/* 0: adaptive lambda (proj), 1: constant */
    double constant_guidance;
    int kernel_size;
    double amplitude;
    int curve_kind;           /* 0 proj, 1 img */
    int timesteps;            /* 1000 */
    double schedule_power;    /* 5 proj, 1 img */
    uint64_t seed;            /* Philox key when noise_dev == NULL */
} ipdm_guided_params;

/* noise draws consumed by one guided process: sum(t_start) + n_iters */
int ipdm_guided_noise_count(const ipdm_guided_params* p);
size_t ipdm_guided_workspace_bytes(const ipdm_guided_params* p, int batch, int h, int w);
/*
 * img_dev [B,H,W]; ldct_dev [B,H,W] (img mode; may be NULL in proj mode);
 * noise_dev: NULL or tape [noise_count][B][H][W] in the reference's randn_like order;
 * iters_out_dev [n_iters + 1][B][H][W]: the result of every iteration, then the mean of the last two
 * (only n_iters entries are written when n_iters == 1).
 */
int ipdm_guided_process(ipdm_unet* net, const ipdm_guided_params* p, const float* img_dev, const float* ldct_dev,
                        const float* noise_dev, float* iters_out_dev, int batch, int h, int w, void* workspace_dev,
                        void* stream);
/*
 * Continuation of the adaptive-schedule branch (Model/model.py:582-613, 629-630): the probing iteration (t_start = 20) has been run
 * with ipdm_guided_process (n_iters = 1) and its lambda-exponent map built with ipdm_delta_lambda_map[_img]; this call runs the
 * iterations of the schedule the host picked (p->t_start, p->eta; n_iters >= 2) as iterations 1, 2, ... of the SAME process: x restarts
 * from img, every step uses the per-pixel lambda map of lam_exp_dev [B][H/ks][W/ks], the guidance blend follows every iteration.
 * noise_dev (optional) points at the first draw of the continuation; call_base = number of draws already consumed (keeps the
 * Philox call ids of the two halves apart).  iters_out_dev [n_iters + 1][B][H][W] as for ipdm_guided_process.
 */
int ipdm_guided_process_resume(ipdm_unet* net, const ipdm_guided_params* p, const float* img_dev, const float* ldct_dev,
                               const float* noise_dev, const float* lam_exp_dev, uint64_t call_base, float* iters_out_dev,
                               int batch, int h, int w, void* workspace_dev, void* stream);

/* ------------------------------------------------------------------------------------------
 * Single-kernel entry points used by the per-kernel parity tests (tests/test_unet_kernels_gpu.py).
 * Tensors are NHWC fp32 device buffers with an explicit channel stride (cs >= c, pad channels 0);
 * weights / affine parameters are HOST arrays in PyTorch layout.  They replace nothing in the
 * reference; they expose the building blocks of ipdm_unet_forward one at a time:
 *   conv        nn.Conv2d 3x3 / 1x1, stride 1 / 2, over a virtual concat of two sources
 *               (Model/model.py:101,113,117,142,143,165,180,306); use_tc: 0 CUDA-core path, 1 tcgen05 kind::tf32,
 *               2 tcgen05 3xTF32 (fp32-accurate), 3 tcgen05 kind::f16 with bf16 operands (src0 is then a bf16 NHWC tensor
 *               with a channel stride that is a multiple of 64, single source), 4 thin tcgen05 path (C_in <= 32, C_out 8 / 16,
 *               src0 channel stride 8 / 16 / 32, single source, stride 1);
 *               the direct path can fuse GroupNorm+SiLU on load and a nearest upsample (:168).
 *   groupnorm   norm_layer(C) statistics -> per-(slice, channel) scale/shift (+ optional apply, +SiLU) (:82-90)
 *   attention   AttentionBlock core (:148-153) from q,k in NHWC [B,T,3C] and v transposed [B,heads,d,t_pad]
 * ---------------------------------------------------------------------------------------- */
int ipdm_debug_conv(const float* src0_dev, int c0, int cs0, const float* src1_dev, int c1, int cs1, int n, int h, int w,
                    const float* w_host, const float* bias_host, int cout, int k, int stride, int upsample_h, int upsample_w,
                    const float* norm_scale_dev, const float* norm_shift_dev, const float* res_dev, int res_cs, float* out_dev,
                    int out_cs, int use_tc, void* stream);
/* average milliseconds of one tensor-core conv launch at the given shape (mode as use_tc above; variant: 0 auto,
 * 1 one-tile-per-CTA, 2 halo-reuse, 3 persistent, 4 persistent halo-reuse); buffers are allocated and freed inside */
int ipdm_debug_conv_time(int c0, int c1, int n, int h, int w, int cout, int k, int stride, int mode, int variant, int with_res,
                         int iters, float* ms_out, double* flops_out);
int ipdm_debug_groupnorm(const float* src0_dev, int c0, int cs0, const float* src1_dev, int c1, int cs1, int n, int h, int w,
                         const float* gamma_host, const float* beta_host, int act_silu, float* scale_out_dev,
                         float* shift_out_dev, float* out_dev, int out_cs, void* stream);
/* qk_lo_dev / vt_lo_dev: NULL (tf32 mode: qk, vt are used as they are) or the tf32 "lo" parts for the 3xTF32 fp32 mode */
int ipdm_debug_attention(const float* qk_dev, const float* vt_dev, const float* qk_lo_dev, const float* vt_lo_dev, float* out_dev,
                         int batch, int T, int t_pad, int heads, int C, void* stream);
/* the bf16 operand mode of the same kernel: qk_dev [B][T][3C] and vt_dev [B][heads][64][t_pad] hold bf16, t_pad % 8 == 0 */
int ipdm_debug_attention_bf16(const void* qk_dev, const void* vt_dev, float* out_dev, int batch, int T, int t_pad, int heads, int C,
                              void* stream);
/* Host-only: the width-folded weights of a thin layer ([tap][f*C_out][f*(c0+c1)], tf32-rounded, + the masks of the structurally non-zero
 * 8-column k-steps) and the four-phase weights of an Upsample conv ([phase 4][tap 9][C_out][round_up(C_in, 32)]) -- the two weight
 * transformations behind ConvTcDesc::fold / phase_up, exposed so that the CPU tests can check them against torch convolutions.
 * out == NULL returns the dimensions only; fold_out == 0 means the shape has no folded form. */
int ipdm_debug_fold_pack(const float* w_host, int cout, int c0, int c1, int k, float* out, unsigned long long* masks_out,
                         int* fold_out, int* n_out, int* k_out);
int ipdm_debug_phase_pack(const float* w_host, int cout, int cin, float* out, int* k_out);
int ipdm_debug_upsample(const float* src_dev, int n, int hs, int ws, int cs, float* dst_dev, int hd, int wd, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* IPDM_B200_H */
