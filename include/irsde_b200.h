/*
 * irsde_b200 - C ABI of the B200-native IR-SDE / Denoising-SDE reverse-diffusion sampler.
 *
 * The reference (Algolzw/image-restoration-sde @ 2598d73) is pure Python and has no FFI; the
 * calls below are what a binding for its hot path would bind.  Each entry point cites the
 * reference interface it replaces (paths relative to the reference checkout).
 *
 * Conventions
 *   - every function returns 0 on success or a negative irsde_status; the message for the last
 *     failure is available from irsde_last_error(ctx) (ctx may be NULL for create failures);
 *   - nothing throws across the ABI; one context per device; a context is not thread-safe;
 *   - image tensors are raw DEVICE pointers to dense fp32 NCHW data ([B,C,H,W], the layout
 *     the reference's torch tensors have); `stream` is a cudaStream_t passed as void*
 *     (torch.cuda.current_stream().cuda_stream);
 *   - weights are copied/repacked by the library; the caller keeps ownership of its buffers.
 */
#ifndef IRSDE_B200_H
#define IRSDE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct irsde_ctx irsde_ctx;

typedef enum {
  IRSDE_OK = 0,
  IRSDE_ERR_INVALID = -1,     /* bad argument / shape */
  IRSDE_ERR_CUDA = -2,        /* CUDA runtime / driver error */
  IRSDE_ERR_STATE = -3,       /* call order (weights / schedule missing) */
  IRSDE_ERR_UNSUPPORTED = -4  /* configuration this build cannot run */
} irsde_status;

/* score-network variant */
#define IRSDE_NET_CONDITIONAL 0 /* codes/config/deraining/models/modules/DenoisingUNet_arch.py:19-134 */
#define IRSDE_NET_DENOISING 1   /* codes/config/denoising-sde/models/modules/DenoisingUNet_arch.py:19-133 */

/* numerics mode */
#define IRSDE_PREC_FP32 0 /* parity mode: fp32 storage + fp32 FMA everywhere                     */
#define IRSDE_PREC_BF16 1 /* perf mode: bf16 activations/weights, tcgen05 MMA, fp32 accumulate,  */
                          /* fp32 sampler state                                                   */
#define IRSDE_PREC_FP32X3 2 /* fp32-accurate tensor-core mode: fp32 storage; every conv is three   */
                            /* tcgen05.mma.kind::tf32 passes over hi/lo split operands            */
                            /* (hi*hi + lo*hi + hi*lo, fp32 accumulate in TMEM): meets the 1e-3    */
                            /* bound of the fp32 mode on the tensor cores                          */

/* sampler */
#define IRSDE_MODE_SDE 0       /* IRSDE.reverse_sde        codes/utils/sde_utils.py:252-266 */
#define IRSDE_MODE_ODE 1       /* IRSDE.reverse_ode        codes/utils/sde_utils.py:268-282 */
#define IRSDE_MODE_POSTERIOR 2 /* IRSDE.reverse_posterior  codes/utils/sde_utils.py:284-299 */
#define IRSDE_MODE_DSDE_SDE 3  /* DenoisingSDE.reverse_sde codes/utils/sde_utils.py:483-500 */
#define IRSDE_MODE_DSDE_ODE 4  /* DenoisingSDE.reverse_ode codes/utils/sde_utils.py:502-522 */
#define IRSDE_NUM_MODES 5
#define IRSDE_NUM_COEF 8 /* floats per timestep in a coefficient table */

typedef struct {
  int32_t in_nc;     /* image channels (ConditionalUNet in_nc)  */
  int32_t out_nc;    /* output channels                          */
  int32_t nf;        /* base width                               */
  int32_t depth;     /* number of levels                         */
  int32_t variant;   /* IRSDE_NET_*                              */
  int32_t precision; /* IRSDE_PREC_*                             */
  int32_t device;    /* CUDA device ordinal                      */
  int32_t flags;     /* IRSDE_FLAG_* (0 = defaults)              */
} irsde_config;
/* flags (all three config structs): bf16 storage through the fp32-FMA SIMT conv engine instead of tcgen05 - a debugging
 * aid that separates storage rounding from tensor-core issues; never the product path. */
#define IRSDE_FLAG_FORCE_SIMT 1

/* Refusion score network: ConditionalNAFNet(img_channel, width, middle_blk_num, enc_blk_nums, dec_blk_nums)
 * (codes/config/deraining/models/modules/DenoisingNAFNet_arch.py:87-143); latent != 0 selects the latent
 * variant whose last conv sees x + intro(x) (codes/config/latent-dehazing/models/modules/DenoisingNAFNet_arch.py:176). */
typedef struct {
  int32_t img_channel;
  int32_t width;
  int32_t middle_blk_num;
  int32_t n_levels;          /* len(enc_blk_nums) == len(dec_blk_nums), <= 8 */
  int32_t enc_blk_nums[8];
  int32_t dec_blk_nums[8];
  int32_t latent;
  int32_t precision;         /* IRSDE_PREC_* */
  int32_t device;
  int32_t flags;             /* IRSDE_FLAG_* */
} irsde_nafnet_config;

/* Refusion latent autoencoder: UNet(in_ch, out_ch, ch, ch_mult, embed_dim)
 * (codes/config/latent-dehazing/models/modules/UNet_arch.py:17-57). */
typedef struct {
  int32_t in_ch, out_ch, ch;
  int32_t n_levels;      /* len(ch_mult) <= 8 */
  int32_t ch_mult[8];
  int32_t embed_dim;
  int32_t precision;     /* IRSDE_PREC_* */
  int32_t device;
  int32_t flags;         /* IRSDE_FLAG_* */
} irsde_latent_unet_config;

/* Replaces `ConditionalUNet(in_nc,out_nc,nf,depth)` + `.to(device)`
 * (DenoisingUNet_arch.py:20, models/denoising_model.py:36). */
int irsde_create(const irsde_config* cfg, irsde_ctx** out);
/* The latent-task variant `ConditionalUNet(in_nc, out_nc, nf, ch_mult=[1,2,4,4])`
 * (codes/config/latent-dehazing/models/modules/DenoisingUNet_arch.py:17-20,51-56,70): level i has nf*[1,ch_mult...][i]
 * channels and depth = len(ch_mult) (cfg->depth is ignored). */
int irsde_create_ch_mult(const irsde_config* cfg, const int32_t* ch_mult, int32_t n_levels, irsde_ctx** out);
/* Same context type, ConditionalNAFNet architecture; every other entry point (load_tensor, noise_fn, reverse, ...)
 * is shared.  Replaces `ConditionalNAFNet(...)` + `.to(device)` (DenoisingNAFNet_arch.py:89). */
int irsde_create_nafnet(const irsde_nafnet_config* cfg, irsde_ctx** out);
/* ConditionalNAFNet of codes/config/latent-bokeh (models/modules/DenoisingNAFNet_arch.py:92-200): time + camera-conditioned
 * blocks, plain ending(x); cfg->latent must be 0.  State-dict names: time_mlp.0/.2 and cam_mlp.0/.2 at the top, time_mlp.1 and
 * cam_mlp.1 in every block.  Every run (noise_fn, reverse, trace_forward) needs irsde_set_lens first (IRSDE_ERR_STATE). */
int irsde_create_nafnet_lens(const irsde_nafnet_config* cfg, irsde_ctx** out);
/* lens: HOST [n][3] = (src_lens, tgt_lens, disparity) per image as the dataset yields them; n = 1 (shared) or the B of the
 * following noise_fn / reverse / trace_forward calls (else those return IRSDE_ERR_INVALID).  Computes the per-image camera
 * rows on the device (cam_mlp, then every block's cam_mlp.1): once per call, not per step.  Drains the device before it
 * re-writes the rows, so a chain already enqueued keeps the lens it was started with.  IRSDE_ERR_INVALID on a context that
 * is not a lens network. */
int irsde_set_lens(irsde_ctx* ctx, const float* lens, int32_t n, void* stream);
void irsde_destroy(irsde_ctx* ctx);
const char* irsde_last_error(const irsde_ctx* ctx);
/* "irsde_b200 <version> sm_100a" */
const char* irsde_version(void);

/* Latent autoencoder context (same weight-loading entry points).  encode replaces `UNet.encode(x) -> (z, h)`
 * (UNet_arch.py:59-76): z is fp32 [B, embed_dim, lat_h, lat_w] (irsde_latent_shape); the skip list h stays inside the
 * context.  decode replaces `UNet.decode(z, h)` (UNet_arch.py:78-91) and uses the skips of the last encode with the
 * same (B, H, W); out is fp32 [B, out_ch, H, W]. */
int irsde_create_latent_unet(const irsde_latent_unet_config* cfg, irsde_ctx** out);
int irsde_latent_shape(irsde_ctx* ctx, int32_t H, int32_t W, int32_t* lat_h, int32_t* lat_w);
int irsde_latent_encode(irsde_ctx* ctx, const float* x, float* z, int32_t B, int32_t H, int32_t W, void* stream);
int irsde_latent_decode(irsde_ctx* ctx, const float* z, float* out, int32_t B, int32_t H, int32_t W, void* stream);

/* Replaces `load_state_dict` (models/base_model.py:92-105): one call per state-dict entry,
 * `name` and `shape` exactly as in the reference state dict; `data` is fp32, host or device. */
int irsde_load_tensor(irsde_ctx* ctx, const char* name, const void* data, int32_t ndim, const int64_t* shape);
/* Check that every tensor of the architecture was loaded and repack for the kernels. */
int irsde_finalize_weights(irsde_ctx* ctx);

/* Replaces `IRSDE.__init__/_initialize` / `DenoisingSDE._initialize` results
 * (sde_utils.py:132-149, :419-426): host arrays of length T+1, index 0 unused. */
int irsde_set_schedule(irsde_ctx* ctx, const float* thetas, const float* sigmas, const float* thetas_cumsum,
                       const float* sigma_bars, float dt, float max_sigma, int32_t T);
/* Optional: override the per-timestep scalars of one mode ([T+1][IRSDE_NUM_COEF] host floats)
 * with values computed by the caller in the reference's own op order (see DESIGN.md). */
int irsde_set_coeffs(irsde_ctx* ctx, int32_t mode, const float* table, int32_t T);

/* Replaces `IRSDE.noise_fn` -> `ConditionalUNet.forward(xt, cond, time)`
 * (sde_utils.py:192-194, DenoisingUNet_arch.py:85-134).  `times` is a HOST array of n_times
 * values (1 = shared by the batch, B = per image); `mu` is ignored for IRSDE_NET_DENOISING. */
int irsde_noise_fn(irsde_ctx* ctx, const float* x, const float* mu, const float* times, int32_t n_times, float* out,
                   int32_t B, int32_t H, int32_t W, void* stream);

/* Replaces `reverse_sde_step / reverse_ode_step / reverse_posterior_step`
 * (sde_utils.py:44-48,219-223,450-462): one fused elementwise update over n floats.
 * z may be NULL for the ODE modes.  out may alias x. */
int irsde_step(irsde_ctx* ctx, int32_t mode, const float* x, const float* mu, const float* noise, const float* z,
               int32_t t, float* out, int64_t n, void* stream);

/* Replaces the whole loop `for t in reversed(range(1, T+1))` of reverse_sde/ode/posterior
 * (sde_utils.py:252-299, :483-522): network forward + update for t = T..1.
 * z: [T][B*C*H*W] pre-drawn N(0,1) in loop order (first slice used at t=T), or NULL to draw
 * in-kernel (Philox4x32-10, seeded with `seed`).  use_graph != 0 replays one captured step graph. */
int irsde_reverse(irsde_ctx* ctx, int32_t mode, const float* xT, const float* mu, const float* z, float* x0,
                  int32_t B, int32_t H, int32_t W, int32_t T, uint64_t seed, int32_t use_graph, void* stream);

/* x_T = mu + N(0,1)*max_sigma on the device (sde_utils.py:360-361) with the library's Philox; the n floats are
 * treated as ONE image (uid = the ctx's image base). */
int irsde_noise_state(irsde_ctx* ctx, const float* mu, float* out, int64_t n, uint64_t seed, void* stream);
/* Same for a batch [B][image_elems]: image b is drawn with uid = image base + b. */
int irsde_noise_state_images(irsde_ctx* ctx, const float* mu, float* out, int32_t B, int64_t image_elems, uint64_t seed,
                             void* stream);
/* Training-time state sampler `IRSDE.generate_random_states` (sde_utils.py:343-358; train.py:236): one fused pass
 * x_t = noise * sigma_bar[t_b] + (mu + (x0 - mu) * w[b]) with per-image scalars w[b] = exp(-thetas_cumsum[t_b] dt) and
 * sigma_bar[b] (device arrays of B floats); bit-identical to the reference's torch expression.  Stateless (no ctx). */
int irsde_random_states(const float* x0, const float* mu, const float* noise, const float* w, const float* sigma_bar, float* out,
                        int32_t B, int64_t image_elems, void* stream);

/* The in-kernel Philox (irsde_reverse with z == NULL, irsde_noise_state*) is keyed by
 * (seed, image uid, timestep, element index inside the image), uid = image base + position in the batch.
 * An image's noise therefore does not depend on the batch it is processed in, its position, or the rank that
 * owns it: set the base to the global index of the shard's / batch's first image (default 0) and batched,
 * sharded and one-at-a-time runs give bit-identical images (SURVEY.md 8 a-16 xi, e, f-2). */
int irsde_set_image_base(irsde_ctx* ctx, uint64_t first_image_uid);
/* Explicit uids for the next batch (n host values, n == B of the following calls), e.g. when a batch is assembled from
 * same-sized images that are not consecutive in the dataset.  irsde_set_image_base() returns to base + position. */
int irsde_set_image_uids(irsde_ctx* ctx, const uint64_t* uids, int32_t n, void* stream);

/* Instrumented pass: between begin/end every op of the launch plan is bracketed by CUDA events on the
 * launching stream (graph replay is bypassed).  end() synchronises and returns, per op category
 * (0 tcgen05 conv, 1 SIMT conv, 2 LayerNorm, 3 attention, 4 misc, 5 update), the summed device time in
 * ms, the executed conv flops and the number of ops.  ncat must be >= 6. */
int irsde_profile_begin(irsde_ctx* ctx);
int irsde_profile_end(irsde_ctx* ctx, double* ms, double* flops, int64_t* launches, int32_t ncat);
/* Same, plus bytes[cat] = the ops' ALGORITHMIC HBM bytes (each op's inputs + outputs + its weights once; DESIGN.md 4):
 * the numerator of the HBM roofline of the memory-bound kernels. */
int irsde_profile_end_bytes(irsde_ctx* ctx, double* ms, double* flops, int64_t* launches, double* bytes, int32_t ncat);

/* Kernel launches issued by this context since creation (for bench.py's gpu_launches). */
int64_t irsde_launch_count(const irsde_ctx* ctx);
/* Bytes of device memory held by the context (weights + workspaces). */
int64_t irsde_device_bytes(const irsde_ctx* ctx);

/* ---- standalone operator entry points (unit-test / micro-benchmark surface) -------------- */
/* Generic NHWC convolution through the engine selected by `engine` (0 = fp32 SIMT implicit
 * GEMM, 1 = tcgen05 bf16 tap-GEMM, 2 = tcgen05 fp32x3 tap-GEMM: fp32 in/out, 3 x kind::tf32 MMA).  Input/weights/output are fp32 device buffers:
 * x [B,Cin,H,W], w [Cout,Cin,KH,KW] (nn.Conv2d layout, module_util.py:96,101,105), y
 * [B,Cout,Ho,Wo]; the call repacks to the engine's layout, runs, and unpacks. */
int irsde_conv2d(irsde_ctx* ctx, int32_t engine, const float* x, const float* w, const float* bias, float* y,
                 int32_t B, int32_t Cin, int32_t H, int32_t W, int32_t Cout, int32_t KH, int32_t KW, int32_t stride,
                 int32_t pad, int32_t upsample, int32_t silu, void* stream);

/* Same with the tensor-core engine's fused epilogues (engine must be 1 when any is used):
 *   residual  fp32 [B,Cout,Ho,Wo] added after the activation (ResBlock `h + res_conv(x)`, module_util.py:146), or NULL;
 *   IRSDE_CONV_QSOFTMAX     1x1 conv whose first 128 output channels are LinearAttention's q: softmax over each
 *                           32-channel head times 32^-0.5 (module_util.py:168,171);
 *   IRSDE_CONV_W_PER_IMAGE  w is [B,Cout,Cin]: image b is multiplied by its own matrix (LinearAttention's second einsum
 *                           + to_out re-associated, module_util.py:176-178). */
#define IRSDE_CONV_QSOFTMAX 1
#define IRSDE_CONV_W_PER_IMAGE 2
int irsde_conv2d_ex(irsde_ctx* ctx, int32_t engine, const float* x, const float* w, const float* bias, const float* residual,
                    float* y, int32_t B, int32_t Cin, int32_t H, int32_t W, int32_t Cout, int32_t KH, int32_t KW,
                    int32_t stride, int32_t pad, int32_t upsample, int32_t silu, int32_t flags, void* stream);

/* ---- launch-plan introspection (parity instrumentation: per-layer comparison with the oracle) ----
 * The network forward for a (B,H,W) input is a fixed list of ops.  irsde_plan_num_ops returns its length (or a negative
 * irsde_status); irsde_plan_op_info gives op `op`'s label (the state-dict name of the weight it applies, e.g.
 * "downs.0.0.block1.proj.weight 256x256 k3 ...") and dims = {C, H, W of the NHWC view it writes (C == 0: none),
 * category as in irsde_profile_end}; irsde_trace_forward runs ops 0..op of `irsde_noise_fn(x, mu, times)` and writes
 * op `op`'s output as fp32 [B,C,H,W] to `dump` (device). */
int32_t irsde_plan_num_ops(irsde_ctx* ctx, int32_t B, int32_t H, int32_t W);
int irsde_plan_op_info(irsde_ctx* ctx, int32_t B, int32_t H, int32_t W, int32_t op, char* label, int32_t label_cap,
                       int32_t* dims /* [4] */);
int irsde_trace_forward(irsde_ctx* ctx, const float* x, const float* mu, const float* times, int32_t n_times, int32_t B,
                        int32_t H, int32_t W, int32_t op, float* dump, void* stream);

/* Drop every cached (B,H,W) launch plan (activation workspaces, TMA descriptors, step graphs).  The cache is also
 * bounded on its own: least-recently-used plans are evicted beyond IRSDE_PLAN_CACHE_MB (default 24576) megabytes or
 * IRSDE_PLAN_CACHE_MAX (default 8) entries, so looping over variable-size images (codes/config/<task>/test.py:96-130,
 * batch 1 at native resolution) does not grow device memory without limit. */
int irsde_trim(irsde_ctx* ctx);

/* ---- multi-GPU plumbing (one process per GPU; SURVEY.md 8 b, e) ------------------------------------------------
 * Replaces DataParallel's per-step replicate / scatter / gather (models/denoising_model.py:41-42) with the two
 * collectives the path needs.  NCCL is dlopen()ed on first use (IRSDE_NCCL_LIB overrides the soname) so single-GPU users
 * keep a library without an NCCL dependency; ranks exchange the 128-byte id out of band (rank 0 creates it).
 * irsde_broadcast_weights: every rank has loaded a state dict of the same names/shapes; the fp32 tensors are replaced
 * by rank `src`'s in one NCCL group and repacked (irsde_finalize_weights is called inside).
 * irsde_gather: rank r contributes counts[r] floats (its slice of x0 in the contiguous batch partition, which may be
 * ragged); x_all receives all slices in rank order = batch order, on every rank. */
int irsde_comm_unique_id(void* id128);
int irsde_comm_init(irsde_ctx* ctx, const void* id128, int32_t rank, int32_t nranks);
int irsde_broadcast_weights(irsde_ctx* ctx, int32_t src, void* stream);
int irsde_gather(irsde_ctx* ctx, const float* x_local, float* x_all, const int64_t* counts /* [nranks] */, void* stream);

/* ---- image conversion and full-reference metrics on the device (SURVEY.md section 8 f-3) -------------------
 * Stateless (no ctx): errors are reported through the return code and irsde_last_error(NULL).
 * Replaces util.tensor2img (codes/utils/img_utils.py:136-163), img2tensor / read_img's "/255." (:171-180,
 * codes/data/util.py:72), calculate_psnr (:182-190) and ssim / calculate_ssim (:193-234).  All pointers are
 * device pointers.  Images are uint8 [B][H][W][C] (BGR when C == 3, the cv2 order), tensors fp32 [B][C][H][W] RGB. */
int irsde_tensor2img_u8(const float* chw, uint8_t* hwc, int32_t B, int32_t C, int32_t H, int32_t W, double lo, double hi,
                        void* stream);
int irsde_img2tensor_u8(const uint8_t* hwc, float* chw, int32_t B, int32_t C, int32_t H, int32_t W, void* stream);
/* sums[b] = sum over the crop-bordered region of (a - b)^2, exact; PSNR = 20 log10(255 / sqrt(sums / n)). */
int irsde_sqerr_u8(const uint8_t* a, const uint8_t* b, int32_t B, int32_t H, int32_t W, int32_t C, int32_t crop,
                   uint64_t* sums, void* stream);
/* number of doubles irsde_ssim_u8 needs as workspace */
int64_t irsde_ssim_workspace(int32_t B, int32_t H, int32_t W, int32_t C, int32_t crop);
/* ssim[b] = mean SSIM of the crop-bordered images (11x11 Gaussian window, valid region), fp64 */
int irsde_ssim_u8(const uint8_t* a, const uint8_t* b, int32_t B, int32_t H, int32_t W, int32_t C, int32_t crop,
                  double* workspace, double* ssim, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* IRSDE_B200_H */
