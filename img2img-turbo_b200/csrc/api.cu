// extern "C" boundary of libi2it (see include/i2it.h).  Nothing throws across it.
#include "engine.cuh"
#include "canny.cuh"

using namespace i2it;

struct i2it_handle {
  Engine* eng = nullptr;
};
static thread_local std::string g_create_error;

#define API_BEGIN(h)                                            \
  if (!(h) || !(h)->eng) return 1;                              \
  Engine& E = *(h)->eng;                                        \
  try {                                                         \
    I2IT_CUDA(cudaSetDevice(E.cfg.device));
#define API_END                                                 \
    return 0;                                                   \
  } catch (const std::exception& ex) {                          \
    E.last_error = ex.what();                                   \
    cudaGetLastError();                                         \
    return 2;                                                   \
  } catch (...) {                                               \
    E.last_error = "unknown C++ exception";                     \
    return 3;                                                   \
  }

extern "C" {

int i2it_default_config(i2it_config* c) {
  if (!c) return 1;
  std::memset(c, 0, sizeof *c);
  c->dtype = I2IT_BF16;
  c->model_kind = I2IT_PIX2PIX;
  c->device = 0;
  const int uc[4] = {320, 640, 1280, 1280}, uh[4] = {5, 10, 20, 20}, vc[4] = {128, 256, 512, 512};
  for (int i = 0; i < 4; ++i) { c->unet_channels[i] = uc[i]; c->unet_heads[i] = uh[i]; c->vae_channels[i] = vc[i]; }
  c->cross_dim = 1024;
  c->temb_dim = 1280;
  c->scaling_factor = 0.18215f;
  c->keep_stages = 0;
  c->use_cuda_graph = 1;
  c->text_heads = 16;
  c->text_act = 0;
  return 0;
}

int i2it_create(const i2it_config* cfg, i2it_handle** out) {
  if (!cfg || !out) return 1;
  try {
    i2it_handle* h = new i2it_handle();
    h->eng = new Engine(*cfg);
    *out = h;
    return 0;
  } catch (const std::exception& ex) {
    g_create_error = ex.what();
    cudaGetLastError();
    return 2;
  }
}

void i2it_destroy(i2it_handle* h) {
  if (!h) return;
  try { delete h->eng; } catch (...) {}
  delete h;
}

const char* i2it_last_error(const i2it_handle* h) {
  if (!h || !h->eng) return g_create_error.c_str();
  return h->eng->last_error.c_str();
}

int i2it_set_weight(i2it_handle* h, const char* key, const void* data, const int64_t* shape, int ndim, int dtype,
                    int is_device) {
  API_BEGIN(h)
  I2IT_CHECK(key && data && shape && ndim > 0 && ndim <= 4, "i2it_set_weight: bad arguments");
  E.set_weight(key, data, shape, ndim, dtype, is_device != 0);
  API_END
}

int i2it_set_adapter_scale(i2it_handle* h, const char* adapter, float s) {
  API_BEGIN(h)
  I2IT_CHECK(adapter != nullptr, "null adapter name");
  E.set_adapter_scale(adapter, s);
  API_END
}

int i2it_finalize_weights(i2it_handle* h, float lw_unet, float lw_vae, float skip_gamma, float twin_r) {
  API_BEGIN(h)
  E.finalize(lw_unet, lw_vae, skip_gamma, twin_r);
  API_END
}

int i2it_workspace_bytes(i2it_handle* h, int batch, int H, int W, size_t* bytes) {
  API_BEGIN(h)
  I2IT_CHECK(bytes != nullptr, "null out pointer");
  Plan* P = E.plan_for(batch, H, W, I2IT_A2B, 1);
  *bytes = P->pool.total;
  API_END
}

int i2it_forward(i2it_handle* h, const void* x, const void* text_emb, int text_batch, const void* eps,
                 const void* noise_map, float r, void* out, void* out_latent, int batch, int H, int W, int direction,
                 void* stream) {
  API_BEGIN(h)
  IO io;
  std::memset(&io, 0, sizeof io);
  io.x = x; io.text = text_emb; io.eps = eps; io.noise = noise_map; io.r = r; io.out = out; io.out_latent = out_latent;
  E.check_device_error();
  E.forward(io, batch, H, W, direction, text_batch, static_cast<cudaStream_t>(stream));
  API_END
}

int i2it_set_text(i2it_handle* h, const void* text_emb, int text_batch, void* stream) {
  API_BEGIN(h)
  E.check_device_error();
  E.set_text(text_emb, text_batch, static_cast<cudaStream_t>(stream));
  API_END
}

int i2it_encode_text(i2it_handle* h, const int32_t* tokens, int batch, void* out, void* stream) {
  API_BEGIN(h)
  E.check_device_error();
  E.encode_text(reinterpret_cast<const int*>(tokens), batch, out, static_cast<cudaStream_t>(stream));
  API_END
}

int i2it_forward_u8(i2it_handle* h, const void* x_u8_hwc, int in_mode, const void* text_emb, int text_batch, const void* eps,
                    const void* noise_map, float r, void* out_u8_hwc, void* out_latent, int batch, int H, int W, int direction,
                    void* stream) {
  API_BEGIN(h)
  I2IT_CHECK(in_mode >= 0 && in_mode <= 2, "i2it_forward_u8: in_mode must be I2IT_IN_UNIT, I2IT_IN_NORMALIZE or I2IT_IN_SKETCH");
  I2IT_CHECK(x_u8_hwc && out_u8_hwc, "i2it_forward_u8: null image pointer");
  IO io;
  std::memset(&io, 0, sizeof io);
  io.x_u8 = x_u8_hwc; io.in_mode = in_mode; io.text = text_emb; io.eps = eps; io.noise = noise_map; io.r = r;
  io.out_u8 = out_u8_hwc; io.out_latent = out_latent;
  E.check_device_error();
  E.forward(io, batch, H, W, direction, text_batch, static_cast<cudaStream_t>(stream));
  API_END
}

int i2it_canny_u8(i2it_handle* h, const void* x_u8_hwc, int batch, int H, int W, float low_threshold, float high_threshold,
                  void* out_u8_hwc, void* stream) {
  API_BEGIN(h)
  I2IT_CHECK(x_u8_hwc && out_u8_hwc, "i2it_canny_u8: null image pointer");
  I2IT_CHECK(batch > 0 && H > 0 && W > 0, "i2it_canny_u8: batch, H and W must be positive");
  const long long n = static_cast<long long>(batch) * H * W;
  I2IT_CHECK(n < (1ll << 31), "i2it_canny_u8: batch*H*W must be below 2^31 (int32 labels)");
  I2IT_CHECK(std::isfinite(low_threshold) && std::isfinite(high_threshold), "i2it_canny_u8: thresholds must be finite");
  void* ws = E.canny_workspace(canny_workspace_bytes(n));
  launch_canny(static_cast<const uint8_t*>(x_u8_hwc), batch, H, W, low_threshold, high_threshold,
               static_cast<uint8_t*>(out_u8_hwc), ws, static_cast<cudaStream_t>(stream));
  API_END
}

long long i2it_debug_fast_div(long long max_dividend, int d, int x) {
  const uint32_t m = i2it::make_magic(max_dividend, d);              // the host function launch_gemm uses
  if (m == 0) return -1;
  if (d == 1) return x;                                              // fast_div selects x for d == 1
  return static_cast<long long>((static_cast<unsigned long long>(static_cast<uint32_t>(x)) * m) >> 32);   // == __umulhi(x, m)
}

int i2it_prep_launch_count(i2it_handle* h, int* launches) {
  API_BEGIN(h)
  I2IT_CHECK(launches != nullptr, "null out pointer");
  *launches = E.prep_launches_;
  API_END
}

int i2it_launch_count(i2it_handle* h, int batch, int H, int W, int direction, int* launches) {
  API_BEGIN(h)
  I2IT_CHECK(launches != nullptr, "null out pointer");
  Plan* P = E.last_plan();
  const bool match = P && P->key.size() >= 4 && P->key[0] == batch && P->key[1] == H && P->key[2] == W && P->key[3] == direction;
  if (!match) P = E.plan_for(batch, H, W, direction, 1);
  *launches = static_cast<int>(P->ops.size());
  API_END
}

int i2it_profile(i2it_handle* h, int reps, char* json, size_t cap, void* stream) {
  API_BEGIN(h)
  I2IT_CHECK(json != nullptr && cap > 2 && reps > 0, "i2it_profile: bad arguments");
  const std::string js = E.profile_json(reps, static_cast<cudaStream_t>(stream));
  I2IT_CHECK(js.size() + 1 <= cap, "i2it_profile: buffer too small (" + std::to_string(js.size() + 1) + " bytes needed)");
  std::memcpy(json, js.c_str(), js.size() + 1);
  API_END
}

int i2it_read_stage(i2it_handle* h, const char* name, float* dst, size_t dst_elems, int dims[4]) {
  API_BEGIN(h)
  E.read_stage(name, dst, dst_elems, dims);
  API_END
}

// ------------------------------------------------------------------------------------------------
// diagnostic single-op entry points
// ------------------------------------------------------------------------------------------------
static void run_plan(Engine& E, Plan& P, cudaStream_t st) {
  E.flush_prep();
  I2IT_CUDA(cudaDeviceSynchronize());
  for (auto& op : P.ops) op(st);
  cudaError_t e = cudaStreamSynchronize(st);
  E.check_device_error();
  I2IT_CUDA(e);
  I2IT_CUDA(cudaGetLastError());
}

static Act view(const void* p, int N, int H, int W, int C, int ld) {
  Act a;
  a.p = reinterpret_cast<uint16_t*>(const_cast<void*>(p));
  a.N = N; a.H = H; a.W = W; a.C = C; a.ld = ld;
  return a;
}

int i2it_op_conv2d(i2it_handle* h, const void* x, int N, int H, int W, int Cin, int ldx, const float* w,
                   const float* bias, int Cout, int ksize, int stride, int asym_pad, const void* residual, int ldr,
                   int act, void* out, int ldo, int out_fp32, void* stream) {
  API_BEGIN(h)
  const int64_t wshape[4] = {Cout, Cin, ksize, ksize};
  E.set_weight("__op.conv.weight", w, wshape, 4, I2IT_F32, true);
  if (bias) { const int64_t bshape[1] = {Cout}; E.set_weight("__op.conv.bias", bias, bshape, 1, I2IT_F32, true); }
  E.finalize(1.f, 1.f, 1.f, -1.f);
  {
    Plan P;
    PW pw = E.prep("__op.conv", {"__op.conv"}, act == TG_ACT_GEGLU);
    ConvOpts o;
    o.ksize = ksize; o.stride = stride; o.asym = asym_pad != 0; o.act = act; o.out_fp32 = out_fp32 != 0;
    const int Ho = H / stride, Wo = W / stride;
    Act xin = view(x, N, H, W, Cin, ldx);
    Act res = view(residual, N, Ho, Wo, Cout, ldr);
    if (residual) o.res = &res;
    Act ov = view(out, N, Ho, Wo, (act == TG_ACT_GEGLU) ? Cout / 2 : Cout, ldo);
    o.out = &ov;
    E.conv(P, xin, pw, o);
    run_plan(E, P, static_cast<cudaStream_t>(stream));
  }
  API_END
}

int i2it_op_group_norm(i2it_handle* h, const void* x, int N, int HW, int C, int ldx, const float* gamma,
                       const float* beta, float eps, int silu, void* out, int ldo, void* stream) {
  API_BEGIN(h)
  {
    Plan P;
    NormW nw; nw.g = gamma; nw.b = beta; nw.C = C;
    Act y = E.group_norm(P, view(x, N, 1, HW, C, ldx), nw, eps, silu != 0);
    E.copy_channels(P, y, view(out, N, 1, HW, C, ldo));
    run_plan(E, P, static_cast<cudaStream_t>(stream));
  }
  API_END
}

int i2it_op_layer_norm(i2it_handle* h, const void* x, int rows, int C, int ldx, const float* gamma, const float* beta,
                       float eps, void* out, int ldo, void* stream) {
  API_BEGIN(h)
  (void)eps;
  {
    Plan P;
    NormW nw; nw.g = gamma; nw.b = beta; nw.C = C;
    Act y = E.layer_norm(P, view(x, 1, 1, rows, C, ldx), nw);
    E.copy_channels(P, y, view(out, 1, 1, rows, C, ldo));
    run_plan(E, P, static_cast<cudaStream_t>(stream));
  }
  API_END
}

int i2it_op_attention(i2it_handle* h, const void* q, int ldq, const void* k, int ldk, const void* vt, int ldv, int B,
                      int Nq, int Nk, int heads, int d, int kv_batch, void* out, int ldo, void* stream) {
  API_BEGIN(h)
  {
    Plan P;
    const int C = heads * d;
    Act o = E.attention(P, view(q, B, 1, Nq, C, ldq), view(k, kv_batch, 1, Nk, C, ldk), view(vt, kv_batch, 1, C, ldv, ldv), B,
                        Nq, Nk, heads, d, kv_batch);
    E.copy_channels(P, o, view(out, B, 1, Nq, C, ldo));
    run_plan(E, P, static_cast<cudaStream_t>(stream));
  }
  API_END
}

int i2it_op_upsample2x(i2it_handle* h, const void* x, int N, int H, int W, int C, void* out, void* stream) {
  API_BEGIN(h)
  {
    Plan P;
    Act y = E.upsample2x(P, view(x, N, H, W, C, C));
    E.copy_channels(P, y, view(out, N, 2 * H, 2 * W, C, C));
    run_plan(E, P, static_cast<cudaStream_t>(stream));
  }
  API_END
}

}  // extern "C"
