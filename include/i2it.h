/* libi2it — C ABI of the B200-native one-step image-translation path
 *
 *     VAE.encode -> one SD-Turbo UNet step (t = 999) -> DDPM closed form -> VAE.decode
 *
 * This is the boundary the reference's Python wrappers would bind (via ctypes; see INTEGRATION.md) in
 * place of the four diffusers calls at
 *     /root/reference/src/pix2pix_turbo.py:198-203   (deterministic)   and :204-218 (stochastic)
 *     /root/reference/src/cyclegan_turbo.py:199-207  (forward_with_networks)
 * i.e.  vae.encode(x).latent_dist.sample()*sf ; unet(z, 999, text).sample ; sched.step(...).prev_sample ;
 *       vae.decode(x0/sf).sample.clamp(-1,1)
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types cross this header.
 *   - every function returns 0 on success, non-zero on failure; i2it_last_error() gives the message.
 *     Nothing throws across the ABI.
 *   - the caller owns inputs, outputs and the CUDA stream; the library owns folded weights + workspace.
 *   - a handle is NOT thread-safe: one handle per (device, stream).  Work is enqueued asynchronously on
 *     the caller's stream (the caller synchronises), except where noted.
 *   - activations at the boundary are NCHW contiguous in the handle's dtype (fp16 or bf16), exactly what
 *     the reference passes to / receives from vae.encode / vae.decode after `.half()`.
 */
#ifndef I2IT_H
#define I2IT_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct i2it_handle i2it_handle;

enum { I2IT_F16 = 0, I2IT_BF16 = 1, I2IT_F32 = 2 };
enum { I2IT_PIX2PIX = 0, I2IT_CYCLEGAN = 1 };
enum { I2IT_A2B = 0, I2IT_B2A = 1 };
/* uint8 input transforms of i2it_forward_u8 (what the reference CLIs do on the host before the forward) */
enum { I2IT_IN_UNIT = 0,        /* F.to_tensor(img): u8/255                       src/inference_paired.py:50      */
       I2IT_IN_NORMALIZE = 1,   /* ToTensor + Normalize([0.5],[0.5])              src/inference_unpaired.py:45-47 */
       I2IT_IN_SKETCH = 2 };    /* (F.to_tensor(img) < 0.5).float()               src/inference_paired.py:56-57   */

/* Network hyper-parameters (HF config.json of stabilityai/sd-turbo; i2it_default_config fills them in). */
typedef struct i2it_config {
  int dtype;                 /* I2IT_F16 | I2IT_BF16 : activation + weight dtype, fp32 accumulation        */
  int model_kind;            /* I2IT_PIX2PIX | I2IT_CYCLEGAN                                               */
  int device;                /* CUDA device ordinal                                                        */
  int unet_channels[4];      /* 320, 640, 1280, 1280                                                       */
  int unet_heads[4];         /* 5, 10, 20, 20 (head_dim is 64 everywhere)                                  */
  int cross_dim;             /* 1024                                                                       */
  int temb_dim;              /* 1280                                                                       */
  int vae_channels[4];       /* 128, 256, 512, 512                                                         */
  float scaling_factor;      /* 0.18215                                                                    */
  int keep_stages;           /* 1: keep named intermediate tensors readable via i2it_read_stage (tests)    */
  int use_cuda_graph;        /* 1: replay the forward as one CUDA graph when shapes and pointers repeat    */
  int text_heads;            /* CLIP text tower: attention heads (16; head_dim must be 64); 0 = hidden/64  */
  int text_act;              /* CLIP text tower MLP activation: 0 = gelu (SD-Turbo), 1 = quick_gelu        */
} i2it_config;

/* Fill `cfg` with the SD-Turbo configuration. */
int i2it_default_config(i2it_config* cfg);

/* Create / destroy an engine.  Replaces AutoencoderKL/UNet2DConditionModel construction
 * (/root/reference/src/pix2pix_turbo.py:36-45; cyclegan_turbo.py:115-124). */
int i2it_create(const i2it_config* cfg, i2it_handle** out);
void i2it_destroy(i2it_handle* h);
const char* i2it_last_error(const i2it_handle* h);   /* h may be NULL: last error of a failed create */

/* Register one tensor of the state dict.  `key` is "<model>.<diffusers key>" with model in
 * {unet, vae, vae_b2a}; peft spellings ("X.base_layer.weight", "X.lora_A.<adapter>.weight",
 * "X.lora_B.<adapter>.weight") are accepted as-is.  `data` may be a host or device pointer
 * (is_device); dtype is I2IT_F32/F16/BF16.  The engine keeps an fp32 device copy (synchronous).
 * Replaces load_state_dict at /root/reference/src/pix2pix_turbo.py:66-78, cyclegan_turbo.py:162-190. */
int i2it_set_weight(i2it_handle* h, const char* key, const void* data, const int64_t* shape, int ndim,
                    int dtype, int is_device);

/* LoRA scale (lora_alpha / r) of an adapter name ("default", "vae_skip", "default_encoder", ...);
 * replaces peft LoraConfig scaling (/root/reference/src/pix2pix_turbo.py:141-151, cyclegan_turbo.py:66-72). */
int i2it_set_adapter_scale(i2it_handle* h, const char* adapter, float alpha_over_r);

/* Fold LoRA into the base weights (W' = W + s*w*B@A in fp32, one rounding), blend TwinConv
 * (W = (1-r) W_pre + r W_cur), scale the skip convs by gamma, fold the t=999 time embedding into
 * conv1 biases, re-lay out for the kernels.  Callable again when the runtime weights change
 * (stochastic mode: unet.set_adapters(["default"],[r]), set_weights_and_activate_adapters(vae,...,[r]),
 * decoder.gamma = r, conv_in.r = r  — /root/reference/src/pix2pix_turbo.py:206-217).
 * lora_weight_* multiply the adapter scales of the UNet / VAE adapters; twin_r < 0 means "no TwinConv blend
 * requested" (error if the state dict has a TwinConv). */
int i2it_finalize_weights(i2it_handle* h, float lora_weight_unet, float lora_weight_vae, float skip_gamma,
                          float twin_r);

/* Bytes of device workspace the engine holds for a (batch, H, W) forward (builds the plan if needed). */
int i2it_workspace_bytes(i2it_handle* h, int batch, int H, int W, size_t* bytes);

/* The fused hot path.  All pointers are DEVICE pointers in the handle dtype, NCHW contiguous:
 *   x        [batch, 3, H, W]          control image / input image (fed to the VAE as is)
 *   text_emb [text_batch, 77, cross]   CLIP hidden states (text_batch is 1 or batch)
 *   eps      [batch, 4, H/8, W/8]      the posterior noise of latent_dist.sample()
 *   noise_map[batch, 4, H/8, W/8]      nullable; non-NULL selects the stochastic blend with r
 *   out      [batch, 3, H, W]          clamp(-1,1) image
 *   out_latent [batch, 4, H/8, W/8]    nullable; x_denoised (the "output latents")
 * direction selects vae (A2B) or vae_b2a (B2A) for I2IT_CYCLEGAN; ignored for I2IT_PIX2PIX.
 * text_emb may be NULL: the cross-attention K / V^T cached by the last i2it_set_text(…, text_batch) are used (one prompt,
 * many images: the reference re-projects the 77 text tokens in all 16 cross-attention layers on every forward).
 * The DDPM step follows the wrapper the handle was created for: fp32 with one rounding for I2IT_PIX2PIX
 * (src/pix2pix_turbo.py:162,200-201: 1-D timesteps), three activation-dtype roundings for I2IT_CYCLEGAN
 * (src/cyclegan_turbo.py:205: 0-dim timestep).
 * H and W must be multiples of 64.  `stream` is a cudaStream_t. */
int i2it_forward(i2it_handle* h, const void* x, const void* text_emb, int text_batch, const void* eps,
                 const void* noise_map, float r, void* out, void* out_latent, int batch, int H, int W,
                 int direction, void* stream);

/* Project and cache the cross-attention operands of a prompt: K = to_k(text_emb), V^T = to_v(text_emb)^T for every
 * transformer block (32 small launches, enqueued on `stream`).  text_emb [text_batch, 77, cross] device pointer in the
 * handle dtype; it is consumed before the call returns control to the stream order (the caller may reuse the buffer after
 * the stream reaches this point).  Must be called again after i2it_finalize_weights (the projections carry the LoRA scale).
 * Replaces the per-forward `attn2.to_k / attn2.to_v` calls under unet(...) at /root/reference/src/pix2pix_turbo.py:199. */
int i2it_set_text(i2it_handle* h, const void* text_emb, int text_batch, void* stream);

/* The CLIP text tower on the engine (SURVEY.md section 8f #1): tokens [batch, 77] int32 (device) -> last_hidden_state
 * [batch, 77, hidden] (device, handle dtype), i.e. `self.text_encoder(tokens)[0]` of /root/reference/src/pix2pix_turbo.py:190-196
 * and cyclegan_turbo.py:251-253.  Needs the "text_encoder.<transformers CLIPTextModel key>" tensors registered with
 * i2it_set_weight.  Enqueued on `stream` (no CUDA graph: a prompt is encoded once and cached by the caller). */
int i2it_encode_text(i2it_handle* h, const int32_t* tokens, int batch, void* out, void* stream);

/* i2it_forward with a uint8 HWC boundary: x_u8_hwc [batch, H, W, 3] and out_u8_hwc [batch, H, W, 3] are device pointers.
 * Input transform `in_mode` (I2IT_IN_*) and the output `ToPILImage()(out*0.5+0.5)` (src/inference_paired.py:72,
 * src/inference_unpaired.py:53; three activation-dtype roundings then truncation to uint8) are fused into the first /
 * a trailing kernel, so a caller moves 3 bytes per pixel each way instead of 2 x 3 x sizeof(half). */
int i2it_forward_u8(i2it_handle* h, const void* x_u8_hwc, int in_mode, const void* text_emb, int text_batch,
                    const void* eps, const void* noise_map, float r, void* out_u8_hwc, void* out_latent, int batch,
                    int H, int W, int direction, void* stream);

/* cv2.Canny(img, low_threshold, high_threshold) (apertureSize 3, L1 gradient) of each RGB image, replicated to three
 * channels: np.array(canny_from_pil(img)) of the reference's src/image_prep.py:6-12, bit for bit.  x_u8_hwc, out_u8_hwc:
 * [batch, H, W, 3] uint8 device pointers; any H, W >= 1 with batch*H*W < 2^31.  Values {0, 255}.  Thresholds are floored and
 * ordered as cv2 does; non-finite ones are rejected.  Four launches enqueued on `stream` (not part of the forward's CUDA
 * graph); needs no weights.  The workspace (6 bytes per pixel) is owned by the handle and grown on demand.  The output
 * feeds i2it_forward_u8(..., I2IT_IN_UNIT, ...) as is. */
int i2it_canny_u8(i2it_handle* h, const void* x_u8_hwc, int batch, int H, int W, float low_threshold,
                  float high_threshold, void* out_u8_hwc, void* stream);

/* Number of kernel launches one forward of this shape issues (for bench accounting): the plan the last forward used if it
 * has this shape, else the plan with the text embedding passed inline. */
int i2it_launch_count(i2it_handle* h, int batch, int H, int W, int direction, int* launches);

/* Kernel launches spent on weight preparation (LoRA fold / TwinConv / re-layout / time embedding) since the handle was
 * created: a job table makes this 4-5 per finalize+plan instead of one to four per tensor. */
int i2it_prep_launch_count(i2it_handle* h, int* launches);

/* Host-side check of the division-free tile decode the GEMM kernels use (csrc/tapgemm.cuh: make_magic / fast_div): returns the
 * quotient the device computes for x / d (magic made for dividends <= max_dividend, 32-bit high multiply), or -1 when the host
 * would refuse that tile space.  No GPU needed: lets the CPU test suite pin the index arithmetic bit for bit. */
long long i2it_debug_fast_div(long long max_dividend, int d, int x);

/* Per-launch device timing of the plan the LAST forward used: runs it `reps` more times with CUDA events around
 * every launch and writes a JSON array [{"i","kind","ms","flops","bytes","shape"}...] (algorithmic flops/bytes per
 * launch) into `json`.  Synchronous.  This is what bench.py's roofline numbers are computed from. */
int i2it_profile(i2it_handle* h, int reps, char* json, size_t cap, void* stream);

/* Named intermediate tensors of the LAST forward (needs cfg.keep_stages): copies the stage as fp32 NCHW
 * into dst (device pointer) and reports its dims.  Synchronous.  Names: "skip0".."skip3", "moments",
 * "latent", "model_pred", "dec_in", "pre_out"... (see DESIGN.md). */
int i2it_read_stage(i2it_handle* h, const char* name, float* dst, size_t dst_elems, int dims[4]);

/* ---- diagnostic single-op entry points (used by tests/ to check each kernel against the oracle) ----
 * Activations NHWC with pixel stride ld (elements); weights fp32 device pointers in PyTorch layout.
 * All are synchronous on `stream`. */
int i2it_op_conv2d(i2it_handle* h, const void* x, int N, int H, int W, int Cin, int ldx, const float* w,
                   const float* bias, int Cout, int ksize, int stride, int asym_pad, const void* residual,
                   int ldr, int act, void* out, int ldo, int out_fp32, void* stream);
int i2it_op_group_norm(i2it_handle* h, const void* x, int N, int HW, int C, int ldx, const float* gamma,
                       const float* beta, float eps, int silu, void* out, int ldo, void* stream);
int i2it_op_layer_norm(i2it_handle* h, const void* x, int rows, int C, int ldx, const float* gamma,
                       const float* beta, float eps, void* out, int ldo, void* stream);
/* q [B,Nq,heads*d] (ldq), k [B,Nk,heads*d] (ldk), vt [B, heads*d, ldv] (V transposed), out [B,Nq,heads*d] */
int i2it_op_attention(i2it_handle* h, const void* q, int ldq, const void* k, int ldk, const void* vt, int ldv,
                      int B, int Nq, int Nk, int heads, int d, int kv_batch, void* out, int ldo, void* stream);
int i2it_op_upsample2x(i2it_handle* h, const void* x, int N, int H, int W, int C, void* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* I2IT_H */
