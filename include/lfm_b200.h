/* lfm_b200.h - C ABI of liblfm_b200.so: the B200-native latent flow-matching sampling path.
 *
 * Drop-in boundary for the sampling hot path of VinAIResearch/LFM.  The reference has no native code and
 * therefore no FFI of its own; each entry point below replaces a Python call site of the reference (cited as
 * reference-file:line) and is bound from Python with ctypes (see INTEGRATION.md for the stub a reference
 * maintainer would add).  Plain C: pointers, sizes, int status codes.  No torch types, no C++ exceptions.
 *
 * Conventions
 *  - All tensor pointers are DEVICE pointers on the ctx's device unless the name ends in _host.
 *  - Tensors use the reference's dtype and layout: latents/velocities fp32 NCHW contiguous [B, C, H, W];
 *    labels int64 [B]; times fp32.
 *  - The library BORROWS caller buffers for the duration of a call; it owns its weight copy and workspace.
 *  - Work is stream-ordered on `stream` (a cudaStream_t passed as void*; NULL = the legacy default stream).
 *  - Return value: 0 = ok, non-zero = error; lfm_last_error(ctx) (or lfm_last_error(NULL) for create
 *    failures) returns a message.  A ctx is bound to one device and is not thread-safe.
 */
#ifndef LFM_B200_H
#define LFM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct lfm_ctx lfm_ctx;

enum { LFM_ARCH_DIT = 0, LFM_ARCH_UNET = 1 };
enum { LFM_DTYPE_F32 = 0 };
enum { LFM_METHOD_EULER = 0, LFM_METHOD_HEUN = 1, LFM_METHOD_MIDPOINT = 2, LFM_METHOD_RK4 = 3 };
/* bits of lfm_sample_fixed's `t_as_vector` argument */
enum { LFM_FIXED_T_VECTOR = 1, LFM_FIXED_PERTURB = 2 };
/* torchdiffeq's adaptive Runge-Kutta pairs (test_flow_latent.py:27 ADAPTIVE_SOLVER; dopri8 is not implemented) */
enum { LFM_ADAPTIVE_DOPRI5 = 0, LFM_ADAPTIVE_BOSH3 = 1, LFM_ADAPTIVE_HEUN = 2 };

/* Constructor arguments of the reference network (models/DiT.py:157-169, selected by
 * models/__init__.py:12-17 create_network).  image side = grid * patch. */
typedef struct lfm_model_desc {
    int32_t arch;            /* LFM_ARCH_DIT */
    int32_t img_resolution;  /* latent side, e.g. 32 */
    int32_t patch_size;      /* 2 */
    int32_t in_channels;     /* 4 */
    int32_t hidden_size;     /* D; multiple of 128; heads * 64 */
    int32_t depth;           /* L */
    int32_t num_heads;       /* H; head_dim must be 64 */
    int32_t mlp_hidden;      /* int(hidden_size * mlp_ratio) */
    int32_t table_rows;      /* y_embedder rows = num_classes + (label_dropout > 0) (models/DiT.py:79-81) */
} lfm_model_desc;

/* Constructor arguments of the reference ADM network (models/guided_diffusion/unet.py:407-428 as called by
 * get_flow_model, models/__init__.py:46-68).  Only the configuration the LFM presets use is implemented:
 * use_scale_shift_norm = True, resblock_updown = False, conv_resample = True, legacy attention order, dims = 2. */
typedef struct lfm_unet_desc {
    int32_t image_size;                /* latent side (config.image_size // 8), e.g. 64 */
    int32_t in_channels;               /* 4 */
    int32_t model_channels;            /* nf, multiple of 128 */
    int32_t out_channels;              /* 4 */
    int32_t num_res_blocks;
    int32_t n_attn_res;                /* number of entries used in attention_resolutions */
    int32_t attention_resolutions[8];  /* DOWNSAMPLE RATES at which attention is applied (unet.py:482) */
    int32_t n_mult;                    /* number of entries used in channel_mult */
    int32_t channel_mult[8];
    int32_t num_heads;
    int32_t num_head_channels;         /* -1: use num_heads */
    int32_t num_classes;               /* 0: unconditional; > 0: label_emb rows (y is then required) */
} lfm_unet_desc;

/* Constructor arguments of the reference EDM-style ADM network DhariwalUNet (models/EDM.py:716-735 as called by
 * get_edm_network, models/EDM.py:906-921, for `--model_type adm` without `--use_origin_adm`: the ffhq_adm / bed_adm /
 * imnet_adm presets).  channel_mult_emb = 4, channels_per_head = 64, augment_dim = 0, use_context = False. */
typedef struct lfm_edm_desc {
    int32_t img_resolution;       /* latent side (config.image_size // config.f), e.g. 32 */
    int32_t in_channels;          /* 4 */
    int32_t out_channels;         /* 4 */
    int32_t label_dim;            /* 0: unconditional; > 0: one-hot width of map_label */
    int32_t model_channels;       /* nf, multiple of 128 */
    int32_t n_mult;               /* number of entries used in channel_mult */
    int32_t channel_mult[8];
    int32_t num_blocks;           /* residual blocks per resolution (config.num_res_blocks) */
    int32_t n_attn_res;           /* number of entries used in attn_resolutions */
    int32_t attn_resolutions[8];  /* feature-map RESOLUTIONS with self-attention (EDM.py:788) */
} lfm_edm_desc;

/* Decoder half of the Stable-Diffusion AutoencoderKL the reference loads with
 * AutoencoderKL.from_pretrained(args.pretrained_autoencoder_ckpt) (test_flow_latent.py:131, test_flow_latent_ddp.py:57;
 * "stabilityai/sd-vae-ft-mse": block_out_channels (128, 256, 512, 512), layers_per_block 2, norm_num_groups 32,
 * latent_channels 4, out_channels 3).  diffusers is a third-party dependency outside /root/reference: the architecture
 * is restated in oracle/vae.py (parity unpinned). */
typedef struct lfm_vae_desc {
    int32_t latent_size;            /* latent side = image_size // 8: 16, 32 (256 x 256 images; the LFM presets), 64 (512 x 512) */
    int32_t latent_channels;        /* 4 */
    int32_t out_channels;           /* 3 */
    int32_t n_blocks;               /* number of entries used in block_out_channels */
    int32_t block_out_channels[8];  /* encoder order, e.g. 128, 256, 512, 512 (the decoder walks it backwards) */
    int32_t layers_per_block;       /* 2 => 3 ResnetBlock2D per decoder up-block */
    int32_t norm_num_groups;        /* 32 */
} lfm_vae_desc;

typedef struct lfm_ode_stats {
    int64_t nfe;       /* network evaluations */
    int64_t accepted;  /* dopri5 accepted steps */
    int64_t rejected;  /* dopri5 rejected steps */
} lfm_ode_stats;

/* models/__init__.py:6-17 create_network(config) -> nn.Module.  Creates an empty context on `device`. */
int lfm_create(const lfm_model_desc* desc, int device, lfm_ctx** out);

/* models/__init__.py:20-70 get_flow_model(config) -> UNetModel (config.use_origin_adm).  The same
 * lfm_set_param / lfm_finalize / lfm_forward / lfm_sample_* entry points then operate on the UNet
 * (model(t, x, y) = UNetModel.forward, unet.py:613-655; it has no forward_with_cfg: cfg_scale must be <= 1). */
int lfm_create_unet(const lfm_unet_desc* desc, int device, lfm_ctx** out);

/* models/__init__.py:10-11 create_network(config) -> get_edm_network(config) -> DhariwalUNet (EDM.py:906-921).
 * The same lfm_set_param / lfm_finalize / lfm_forward / lfm_sample_* entry points then operate on it:
 * model(t, x, y) = DhariwalUNet.forward (EDM.py:812-845; y may be NULL even for a class-conditional net: the label
 * term is then skipped, :823) and cfg_scale > 1 = forward_with_cfg (EDM.py:847-861: the labels of the second half of
 * the batch are DROPPED - pass label_dim there, or anything: rows [B/2, B) of y are ignored).
 * State-dict keys as in the reference, including the constant `*.resample_filter` buffers of the up/down blocks
 * (accepted and checked to be 0.25). */
int lfm_create_edm(const lfm_edm_desc* desc, int device, lfm_ctx** out);

/* AutoencoderKL.from_pretrained(...) (test_flow_latent.py:131): a context for the DECODER.  lfm_set_param takes the
 * `decoder.*` and `post_quant_conv.*` entries of the diffusers state dict (attention projections under their current
 * names to_q / to_k / to_v / to_out.0); lfm_finalize(max_batch) sizes the workspace for max_batch images per call. */
int lfm_create_vae(const lfm_vae_desc* desc, int device, lfm_ctx** out);

/* first_stage_model.decode(z).sample (test_flow_latent.py:193, test_flow_latent_ddp.py:110; the caller divides the
 * latents by scale_factor as the reference does) and, optionally, the post-processing of the generation loop
 * (test_flow_latent_ddp.py:131-135) fused into the decoder's last kernel:
 *   z:       [B, 4, s, s] fp32 NCHW (device)
 *   out_f32: [B, 3, 8s, 8s] fp32 NCHW `sample`, or NULL
 *   out_u8:  [B, 8s, 8s, 3] uint8 = (clamp((sample + 1) / 2, 0, 1) * 255).permute(0, 2, 3, 1).to(uint8), or NULL */
int lfm_decode(lfm_ctx* ctx, const float* z, int B, float* out_f32, uint8_t* out_u8, void* stream);

/* nn.Module.load_state_dict (test_flow_latent.py:142): one call per state-dict entry, `key` exactly as in the
 * reference state_dict (SURVEY.md 8(b)); `ptr` may be a host or a device pointer (fp32).  The data is copied
 * (GEMM weights are repacked to bf16).  Unknown key or wrong shape -> error (strict=True behaviour). */
int lfm_set_param(lfm_ctx* ctx, const char* key, const void* ptr, int dtype, const int64_t* shape, int ndim);

/* After all parameters are set: checks that none is missing (strict), allocates the activation workspace for
 * up to `max_batch` network rows (2x images under CFG) and builds the TMA descriptors. */
int lfm_finalize(lfm_ctx* ctx, int max_batch);

/* model(t, x, y) / model.forward_with_cfg(t, x, y, cfg_scale)  (models/DiT.py:252-272, 274-290).
 *   t: [t_numel] fp32, t_numel == 1 (0-d t, broadcast) or B.   x, v_out: [B, C, H, W].   y: [B] int64 or NULL
 *   (NULL = the table's last row, models/DiT.py:259-260).
 *   cfg_scale <= 1: v_out = DiT(t, x, y).
 *   cfg_scale  > 1: forward_with_cfg - B must be even, rows [B/2, B) of y hold the null class; the first half
 *   of x is evaluated with both label halves and v_out = cat[g, g], g = u + s (c - u).
 *   Labels are validated by the caller (the Python mirror raises like nn.Embedding / one_hot would); on the device an
 *   out-of-range label is clamped to the table, never read out of bounds. */
int lfm_forward(lfm_ctx* ctx, const float* t, int t_numel, const float* x, const int64_t* y, int B, float cfg_scale,
                float* v_out, void* stream);

/* Fixed-step integration of dx/dt = v(t, x) over the nodes t_grid[0..n_grid) (device or host pointer, fp32):
 *   LFM_METHOD_EULER  x += v(t_i, x) (t_{i+1} - t_i)                sampler/karras_sample.py:86-118 and
 *                                                                   torchdiffeq fixed-grid euler (test_flow_latent.py:61-73)
 *   LFM_METHOD_HEUN   predictor + trapezoid corrector for intervals i < heun_corrector_limit, Euler beyond
 *                                                                   sampler/karras_sample.py:122-161
 *   LFM_METHOD_MIDPOINT / LFM_METHOD_RK4   torchdiffeq's fixed-grid midpoint and rk4 (3/8 rule) step functions
 *                                                                   (test_flow_latent.py:61-73 with --method midpoint|rk4)
 *   t_as_vector: bit 0 (LFM_FIXED_T_VECTOR): 0 = the model sees a 0-d t (torchdiffeq), 1 = a [B] vector (Karras samplers);
 *   bit 1 (LFM_FIXED_PERTURB): torchdiffeq options["perturb"] = True (test_flow_latent.py:44-48,64): the first evaluation of
 *   every step sees t one fp32 ulp past the node, rk4's last one one ulp before the next node.
 *   x_inout: [B_img, C, H, W] latents, updated in place.  y: labels, [B_img] (cfg_scale <= 1) or [2*B_img]
 *   (cfg_scale > 1: conditional labels then null labels; a 2*B_img-row network batch is evaluated per NFE).
 *   The whole trajectory runs from a captured CUDA graph; no host synchronisation between steps. */
int lfm_sample_fixed(lfm_ctx* ctx, int method, float* x_inout, const float* t_grid_host, int n_grid, int t_as_vector,
                     int heun_corrector_limit, const int64_t* y, int B_img, float cfg_scale, lfm_ode_stats* stats,
                     void* stream);

/* Adaptive Dormand-Prince 5(4) from t0 down to t1 with torchdiffeq's controller (rtol/atol, RMS norm over the
 * whole batch, fp64 time, dense output at t1)        test_flow_latent.py:42-76 with --method dopri5. */
int lfm_sample_dopri5(lfm_ctx* ctx, float* x_inout, double t0, double t1, double rtol, double atol, const int64_t* y,
                      int B_img, float cfg_scale, lfm_ode_stats* stats, void* stream);

/* The same controller with another embedded pair: --method dopri5 | bosh3 | adaptive_heun (test_flow_latent.py:27,61-73;
 * torchdiffeq rk_common.RKAdaptiveStepsizeODESolver: initial step with order - 1, step factor with order, y1 / f1 / dense
 * output as in its _runge_kutta_step / _interp_fit).  lfm_sample_dopri5 == lfm_sample_adaptive(LFM_ADAPTIVE_DOPRI5). */
int lfm_sample_adaptive(lfm_ctx* ctx, int method, float* x_inout, double t0, double t1, double rtol, double atol,
                        const int64_t* y, int B_img, float cfg_scale, lfm_ode_stats* stats, void* stream);

const char* lfm_last_error(const lfm_ctx* ctx);
void lfm_destroy(lfm_ctx* ctx);

/* Number of kernels the library has launched on this ctx since creation (bench.py's gpu_launches). */
int64_t lfm_launch_count(const lfm_ctx* ctx);

/* ---- kernel-level entry points used by the parity tests (tests/test_gpu_parity.py) ------------------- */
/* C = A[M,K] W[N,K]^T with epilogue `epi` (0 bias->bf16, 1 bias+gelu->bf16, 2 gated residual fp32, 3 bias->fp32).
 * a, w: bf16 device pointers.  block_n: 128 / 256 (one CTA per tile) or 512 (CTA-pair kernel, 256 x 256 tile). */
int lfm_dbg_gemm(const void* a_bf16, const void* w_bf16, const float* bias, void* out, const float* gate,
                 int gate_stride, int rows_per_sample, int M, int N, int K, int epi, int block_n, void* stream);
/* softmax(q k^T / 8) v on a [B*256, 3*D] bf16 qkv buffer -> out [B*256, D] bf16.  variant: 3 = persistent single-TMEM-read kernel (default), 2 = persistent two-pass, 0 = P in TMEM,
 * 1 = P through shared memory.  dbg_s (optional) receives the raw S = q k^T as fp32 [B, H, 256, 256]. */
int lfm_dbg_attention(const void* qkv_bf16, void* out_bf16, int B, int H, int variant, float* dbg_s, void* stream);
/* The mma.sync attention kernels of the DiT geometries the tcgen05 kernel does not cover (16 / 64 tokens: whole sequence in registers;
 * other multiples of 64, e.g. 256 / 1024: keys streamed in chunks of 64).  qkv [B*T, 3*H*ch] bf16 with HEAD-MAJOR features
 * (head * 3 ch + {q,k,v} * ch + c), ch = 64 or 80 (head_dim 72 zero-padded), scale head_dim^-1/2 -> out [B*T, H*ch] bf16. */
int lfm_dbg_attention_mma(const void* qkv_bf16, void* out_bf16, int B, int H, int T, int ch, int head_dim, void* stream);
/* Intermediate activations of the last lfm_forward (fp32 token stream [B*T, D] after all blocks). */
int lfm_dbg_tokens(lfm_ctx* ctx, float* out, int B);

#ifdef __cplusplus
}
#endif
#endif /* LFM_B200_H */
