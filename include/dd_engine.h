/*
 * dd_engine.h — C ABI of libddengine.so: the B200-native (sm_100a) DiffusionDepth hot path.
 *
 * The reference (duanyiqun/DiffusionDepth @ e1ca9d5) has no FFI on this path; these entry points
 * are what a binding for it would bind.  Each one names the reference interface it replaces:
 *
 *   dd_create / dd_destroy        <- construction of `ScheduledCNNRefine` + `CNNDDIMPipiline` +
 *                                    `DeepDepthTransformWithUpsampling` inside the head ctor
 *                                    (src/model/head/ddim_depth_estimate_res_swin_addHAHI.py:45-49,
 *                                     src/model/head/ddim_depth_estimate_res.py:36-40)
 *   dd_set_weight / dd_finalize_weights
 *                                 <- `load_state_dict(ckpt['net'])` for the keys under
 *                                    `depth_head.model.*` and `depth_head.depth_transform.*`
 *                                    (src/main.py:418-432; key layout SURVEY.md Appendix A)
 *   dd_set_schedule               <- `DDIMScheduler.set_timesteps` + the per-step scalar algebra of
 *                                    `DDIMScheduler.step` (src/model/diffusers/schedulers/
 *                                    scheduling_ddim.py:215-229, 285-326) collapsed to
 *                                    x_{t-1} = c_x * x_t + c_eps * eps
 *   dd_denoise_decode             <- `CNNDDIMPipiline.__call__` (head :254-303) = T x
 *                                    {`ScheduledCNNRefine.forward` (:361-382 / res.py:324-344),
 *                                    `DDIMScheduler.step`} followed by
 *                                    `DeepDepthTransformWithUpsampling.inv_t`
 *                                    (src/model/ops/depth_transform.py:33-35)
 *   dd_set_schedule_eta / dd_denoise_decode_stochastic
 *                                 <- the same pipeline with `eta > 0` (head :254-303 `eta=`; scheduling_ddim.py:
 *                                    313-350): x_{t-1} = c_x * x_t + c_eps * eps + sigma_t * z_t
 *   dd_denoiser_forward           <- one bare `ScheduledCNNRefine.forward(noisy, t, cond, ...)` call
 *                                    (the operator `ddim_loss` invokes, head :207-223)
 *   dd_decode                     <- `depth_transform.inv_t(latent)` alone (the *Vis heads call it
 *                                    per step, ..._swin_addHAHI_vis.py)
 *
 * Conventions (inherited from the reference, SURVEY.md §8b): every tensor is fp32, NCHW, contiguous,
 * resident on the engine's CUDA device; no autograd.  Ownership: the caller (PyTorch's allocator)
 * owns every buffer including the workspace; the engine borrows raw pointers for the duration of a
 * call and owns only its pre-packed weights / descriptors / CUDA graph.  Calls are enqueued on the
 * given stream and return without synchronising.  One handle per (process, device); a handle is not
 * re-entrant.  Errors: int status (0 = ok), never an exception across the ABI; text via
 * dd_last_error() (thread-local).  There is NO CPU path: dd_create fails if no sm_100 device is present.
 */
#ifndef DD_ENGINE_H_
#define DD_ENGINE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DD_ABI_VERSION 1

typedef struct dd_engine* dd_handle;

enum dd_status {
  DD_OK = 0,
  DD_ERR_INVALID = 1,     /* bad argument / shape / missing weight */
  DD_ERR_CUDA = 2,        /* a CUDA runtime or driver call failed */
  DD_ERR_UNSUPPORTED = 3, /* no sm_100 device, unsupported shape */
  DD_ERR_RANGE = 4        /* an activation left the fp16 split's range (see DESIGN.md "Numerics") */
};

enum dd_variant {
  DD_VARIANT_RES = 0,  /* DDIMDepthEstimate_Res: cond at latent resolution, no upsample_fuse */
  DD_VARIANT_SWIN = 1  /* DDIMDepthEstimate_Swin_ADDHAHI: cond upsampled (bilinear, align_corners)
                          to the latent grid, then convA/convB */
};

enum dd_flags {
  DD_FLAG_CUDA_GRAPH = 1 << 0, /* capture the T-step loop once and replay it */
  DD_FLAG_SIMT_CONV = 1 << 1,  /* debug: fp32 CUDA-core convolutions instead of tcgen05 */
  DD_FLAG_CHECK_RANGE = 1 << 2,/* after the call, sync and report DD_ERR_RANGE if the split overflowed */
  DD_FLAG_HALO_CONV = 1 << 3,  /* loop convs on the row-halo-reuse kernel (16x8 tiles, 2.7x less activation traffic) */
  DD_FLAG_SWAP_NARROW = 1 << 4, /* Cout <= 64 convs on the swapped-operand kernel (weights as A, 256 pixels as N) */
  DD_FLAG_PAIR_WIDE = 1 << 5,   /* Cout = 256 convs on CTA pairs (cluster of 2, tcgen05 cta_group::2, M = 256) */
  DD_FLAG_STEP_DECODE = 1 << 6, /* reserve workspace for dd_denoise_decode_steps (T decoded maps; the *Vis heads) */
  DD_FLAG_FP8_CORR = 1 << 7,    /* Swin variant, with HALO_CONV | PAIR_WIDE: the Cout = 256 convs (convA, convB 256->256 and
                                   noise_embedding.3 64->256) compute the correction
                                   products of the split (x_lo * w_hi, x_hi * w_lo) as e4m3 MMAs (kind::f8f6f4, K = 32) and
                                   only hi * hi in fp16: 2 pass-equivalents instead of 3, ~1.5x on the dominant kernel.
                                   Error per product ~2^-15 instead of ~2^-22 (DESIGN.md "Numerics": max |dz| 3.4e-4 on
                                   BASELINE config 3, tolerance 1e-3); activations must stay below 112 in magnitude
                                   (DD_ERR_RANGE otherwise).  Off = the exact 3-pass fp16 split everywhere. */
  DD_FLAG_STOCHASTIC = 1 << 8   /* stochastic DDIM (eta > 0): reserve the step-noise and per-step-latent workspace regions
                                   (2 x T*B*16*h*w fp32) for dd_denoise_decode_stochastic; dd_denoise_decode /
                                   dd_denoise_decode_steps then fail with DD_ERR_INVALID (they have no step noise) */
};

typedef struct dd_config {
  int32_t abi_version;          /* must be DD_ABI_VERSION */
  int32_t variant;              /* enum dd_variant */
  int32_t batch;                /* images per call on this device */
  int32_t latent_h, latent_w;   /* h = ceil(H/2), w = ceil(W/2): shape of depth_transform.t(gt) */
  int32_t cond_h, cond_w;       /* spatial size of the FPN condition map x (256 channels) */
  int32_t num_inference_steps;  /* T */
  int32_t device;               /* CUDA ordinal */
  int32_t flags;                /* enum dd_flags */
} dd_config;

/* Fixed by the reference architecture (head ctor): 16 latent channels, 256 condition channels,
 * GroupNorm(4, C), time_embedding rows = 1280. */
#define DD_LATENT_C 16
#define DD_COND_C 256
#define DD_TIME_ROWS 1280

int dd_abi_version(void);
const char* dd_last_error(void);

int dd_create(const dd_config* cfg, dd_handle* out);
int dd_destroy(dd_handle h);

/* Register one parameter/buffer by its reference state_dict key relative to `depth_head.`
 * (e.g. "model.noise_embedding.0.weight", "depth_transform.conv_inv_transform.1.running_var").
 * `dev_ptr` is a device fp32 pointer in the reference's own layout/shape; it is read during the next
 * dd_finalize_weights only, which then forgets every registered pointer (a re-pack registers all keys again).
 * Unknown keys are rejected (DD_ERR_INVALID). */
int dd_set_weight(dd_handle h, const char* name, const float* dev_ptr, const int64_t* shape, int32_t ndim);

/* Pre-pack: fold eval-BatchNorm into the decoder, repack conv weights tap-major, split them into
 * scaled fp16 hi/lo planes for the 3-pass tensor-core product.  Fails listing any missing key. */
int dd_finalize_weights(dd_handle h, void* cuda_stream);

/* Per-step timesteps (descending, as DDIMScheduler.set_timesteps produces) and the collapsed DDIM
 * coefficients; n must equal num_inference_steps. */
int dd_set_schedule(dd_handle h, const int64_t* timesteps, const double* c_x, const double* c_eps, int32_t n);

/* Stochastic DDIM: as dd_set_schedule, plus the per-step noise scale sigma_t = eta * sqrt(variance)
 * (reference scheduling_ddim.py:313-315, formula (16)); c_eps then is sqrt(1 - a_prev - sigma^2) - sqrt(a_prev (1 - a_t)
 * / a_t) (:321-326).  Every sigma must be >= 0.  Used by dd_denoise_decode_stochastic (dd_set_schedule leaves sigma = 0). */
int dd_set_schedule_eta(dd_handle h, const int64_t* timesteps, const double* c_x, const double* c_eps,
                        const double* sigma, int32_t n);

/* Optional: also run the step-invariant condition producers natively — HAHI neck (attention gates off, as
 * the shipped heads configure it: src/model/necks/hahi.py:165-276) and the FPN (head :112-122) — on the same
 * 3-pass tensor-core path.  Call before dd_finalize_weights; additionally register the reference keys
 * `hahineck.*` (only if has_neck), `conv_lateral.*`, `conv_up.*`.  Pyramid levels may be anything up to 2x their
 * coarser neighbour (an exact 2x pyramid makes the FPN's adaptive_avg_pool2d the identity; otherwise it is a real
 * resample kernel).  Channel counts: any positive multiples of 8 (Swin 192..1536, ResNet 64..512, MPViT 128/216/288/288);
 * partial 64-channel K chunks and partial N tiles are completed with zeros by TMA's out-of-bounds fill. */
typedef struct dd_producer_config {
  int32_t num_levels;   /* 2..4 */
  int32_t channels[4];  /* backbone feature channels, finest level first */
  int32_t heights[4];
  int32_t widths[4];
  int32_t has_neck;     /* 1: *HAHI heads (HAHIHeteroNeck in front of the FPN), 0: Res heads and Swin_ADD */
} dd_producer_config;
int dd_enable_producers(dd_handle h, const dd_producer_config* pc);

/* feats[i]: device fp32 NCHW [B, channels[i], heights[i], widths[i]] (the backbone's outputs).  Builds the
 * (feats may be NULL right after dd_run_backbone.)  256-channel condition map inside the workspace; a following dd_denoise_decode(cond = NULL, ...) consumes it.
 * cond_out (nullable): also write it as NCHW [B,256,cond_h,cond_w]. */
int dd_build_condition(dd_handle h, const float* const* feats, float* cond_out, void* workspace,
                       size_t workspace_bytes, void* cuda_stream);

/* Optional: also run the Swin backbone natively (reference src/model/backbone/swin.py:756-777): patch embed,
 * LayerNorms, QKV / proj / FFN / patch-merging Linears on the 3-pass tensor-core GEMM path, 7x7 (shifted-)window
 * attention with relative-position bias and the finite -100 mask, per-stage output norms written straight into the
 * neck's (or, without a neck, the FPN's) input planes.  Requires dd_enable_producers(4 levels) with matching geometry; register the
 * reference keys of `depth_backbone.*` as "backbone.<key>" (the int64 `relative_position_index` buffers are not
 * needed).  Instantiated for Swin-L (embed_dims 192, head_dim 32, window 7). */
enum dd_backbone_kind {
  DD_BACKBONE_SWIN = 1,   /* SwinTransformer (reference backbone/swin.py) */
  DD_BACKBONE_RESNET = 2, /* ResNetForMMBEV with BasicBlocks, no stem (reference backbone/mmbev_resnet.py:124-187): depths[] =
                             blocks per stage, channels 64/128/256/512, every stage stride 2; needs
                             dd_enable_producers(4 levels, has_neck = 0); embed_dims / num_heads / window ignored */
  DD_BACKBONE_MPVIT = 3   /* MPViT (reference backbone/mpvit.py:601-730; tiny / xsmall / small / base factories :743-870):
                             full-resolution stem, then 4 x { chained depthwise-separable patch embeddings (first one
                             stride 2), a conv path + one factorised-attention encoder per embedding, 1x1 aggregate }.
                             depths[] = encoder layers per stage, mp_dims[] = stage widths (multiples of 8, <= 512; stage
                             s outputs mp_dims[s + 1], the last one mp_dims[3]), mp_paths[] = embeddings per stage (<= 3),
                             mlp_ratio; 8 heads, crpe windows {3: 2, 5: 3, 7: 3} heads.  Outputs at 1/2 .. 1/16 of the image;
                             needs dd_enable_producers(4 levels) with those sizes and channels */
};
typedef struct dd_backbone_config {
  int32_t kind;        /* enum dd_backbone_kind */
  int32_t embed_dims;  /* 192 */
  int32_t depths[4];   /* 2, 2, 18, 2 */
  int32_t num_heads[4];/* 6, 12, 24, 48 */
  int32_t window;      /* 7 */
  int32_t height, width; /* input image size */
  int32_t mp_dims[4];  /* DD_BACKBONE_MPVIT only: 64, 128, 216, 288 (mpvit_small) */
  int32_t mp_paths[4]; /* 2, 3, 3, 3 */
  int32_t mlp_ratio;   /* 4 */
} dd_backbone_config;
int dd_enable_backbone(dd_handle h, const dd_backbone_config* bc);

/* rgb: device fp32 NCHW [B,3,height,width].  Leaves the four stage outputs in the workspace for a following
 * dd_build_condition(feats = NULL, ...); feats_out (nullable array of 4 nullable pointers) also receives them as
 * fp32 NCHW [B, C_s, H_s, W_s]. */
int dd_run_backbone(dd_handle h, const float* rgb, float* const* feats_out, void* workspace, size_t workspace_bytes,
                    void* cuda_stream);

size_t dd_workspace_bytes(dd_handle h);

/* cond [B,256,cond_h,cond_w], noise [B,16,h,w] -> latent_out [B,16,h,w] (nullable),
 * logit_out [B,1,2h,2w] (nullable; the decoder's pre-sigmoid z), depth_out [B,1,2h,2w].
 * cond may be NULL right after dd_build_condition. */
int dd_denoise_decode(dd_handle h, const float* cond, const float* noise, float* latent_out, float* logit_out,
                      float* depth_out, void* workspace, size_t workspace_bytes, void* cuda_stream);

/* The *Vis heads' variant (reference src/model/head/ddim_depth_estimate_res_swin_addHAHI_vis.py:130-149, pipeline
 * :289-304 `image_list`): same loop, and `inv_t` of the latent after EVERY step, all inside the captured graph.
 * depth_steps_out [T][B,1,2h,2w] (slice T-1 is the final `pred`); latent_out / logit_out (nullable) refer to the
 * final step.  Needs DD_FLAG_STEP_DECODE at dd_create. */
int dd_denoise_decode_steps(dd_handle h, const float* cond, const float* noise, float* latent_out, float* logit_out,
                            float* depth_steps_out, void* workspace, size_t workspace_bytes, void* cuda_stream);

/* `CNNDDIMPipiline.__call__(..., eta > 0)` (head :254-303; the step's `variance_noise`, scheduling_ddim.py:329-350):
 * the same loop with x <- c_x x + c_eps eps + sigma_t z_t.  step_noise: NCHW [T][B][16][h][w], z of step i in slice i
 * (the i-th `variance_noise` draw of the reference loop); it is staged into the workspace before the (captured) loop runs.
 * latent_steps_out (nullable): NCHW [T][B][16][h][w], the latent after every step (the *Vis pipelines' `image_list`);
 * depth_steps_out (nullable, needs DD_FLAG_STEP_DECODE) as in dd_denoise_decode_steps; at least one of depth_out /
 * depth_steps_out.  Needs DD_FLAG_STOCHASTIC.  With every sigma = 0 the outputs equal dd_denoise_decode's bit for bit. */
int dd_denoise_decode_stochastic(dd_handle h, const float* cond, const float* noise, const float* step_noise,
                                 float* latent_out, float* latent_steps_out, float* logit_out, float* depth_out,
                                 float* depth_steps_out, void* workspace, size_t workspace_bytes, void* cuda_stream);

/* eps = ScheduledCNNRefine(noisy, t, cond): noisy [B,16,h,w], t[b] int64 host array (one per image),
 * eps_out [B,16,h,w]. */
int dd_denoiser_forward(dd_handle h, const float* cond, const float* noisy, const int64_t* t_host, float* eps_out,
                        void* workspace, size_t workspace_bytes, void* cuda_stream);

/* depth = inv_t(latent): latent [B,16,h,w] -> logit_out (nullable), depth_out [B,1,2h,2w]. */
int dd_decode(dd_handle h, const float* latent, float* logit_out, float* depth_out, void* workspace,
              size_t workspace_bytes, void* cuda_stream);

/* latent = depth_transform.t(depth) (reference src/model/ops/depth_transform.py:29-31): depth [B,1,height,width] ->
 * latent_out [B,16,ceil(height/2),ceil(width/2)].  Needs the optional keys `depth_transform.conv_transform.*`. */
int dd_encode(dd_handle h, const float* depth, int32_t height, int32_t width, float* latent_out, void* cuda_stream);

/* Synchronise `cuda_stream` and report DD_ERR_RANGE if any activation left the fp16 split's range since the
 * last hot-path call started (DD_OK otherwise).  The hot-path calls themselves never synchronise unless
 * DD_FLAG_CHECK_RANGE is set. */
int dd_poll_status(dd_handle h, void* cuda_stream);

/* Number of kernel launches the last forward (dd_run_backbone .. dd_denoise_decode) enqueued; graph nodes count
 * individually. */
int64_t dd_last_launch_count(dd_handle h);

/* Standalone layer entry used by the parity tests and the roofline bench: one 3x3/s1/p1 convolution
 * + bias on the engine's tensor-core (or SIMT, per flags) path.
 * x [B,Cin,H,W], w [Cout,Cin,3,3], b [Cout] -> y [B,Cout,H,W]; all device fp32 NCHW. */
int dd_conv3x3(dd_handle h, const float* x, const float* w, const float* b, float* y, int32_t batch, int32_t cin,
               int32_t cout, int32_t height, int32_t width, void* workspace, size_t workspace_bytes,
               void* cuda_stream);
size_t dd_conv3x3_workspace_bytes(int32_t batch, int32_t cin, int32_t cout, int32_t height, int32_t width);

/* Time the dominant kernel (convA-shaped 256->256 3x3 on the engine's latent grid) `iters` times with
 * CUDA events on `cuda_stream`; returns average milliseconds per launch in *ms_out. */
int dd_bench_conv(dd_handle h, int32_t cin, int32_t cout, int32_t iters, float* ms_out, void* workspace,
                  size_t workspace_bytes, void* cuda_stream);

/* Tuning aid: average milliseconds per launch of the GEMM-mode kernel (tokens [M,K] x weights [N,K]^T) on
 * synthetic operands.  mode 0: fp32 out, 1: fp32 out + residual add, 2: GELU -> fp16 planes, 3: no output. */
int dd_bench_gemm(dd_handle h, int32_t M, int32_t K, int32_t N, int32_t mode, int32_t iters, float* ms_out);

#ifdef __cplusplus
}
#endif
#endif /* DD_ENGINE_H_ */
