// Engine implementation: weight store + load-time fold, op builders, executor.  The model graph lives in model.cu.
#include "engine.cuh"

#include <algorithm>
#include <cstdlib>

#include <nvtx3/nvToolsExt.h>   // header-only: ranges show up under Nsight tools, no-ops otherwise

namespace i2it {

static inline int ceil_div(long long a, long long b) { return static_cast<int>((a + b - 1) / b); }
static inline int round_up(int a, int b) { return (a + b - 1) / b * b; }
static inline int pow2ceil(int v) { int p = 1; while (p < v) p <<= 1; return p; }

#define DISPATCH_T(dt, ...)                                   \
  do {                                                        \
    if ((dt) == DT_BF16) { using T = __nv_bfloat16; __VA_ARGS__; } \
    else { using T = __half; __VA_ARGS__; }                   \
  } while (0)

// ---------------------------------------------------------------------------------------------
// TMA
// ---------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    I2IT_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q));
    I2IT_CHECK(q == cudaDriverEntryPointSuccess && p != nullptr, "cuTensorMapEncodeTiled unavailable in this driver");
    fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

CUtensorMap encode_tmap(const TmapSpec& s, int dtype) {
  CUtensorMap m;
  cuuint64_t dims[5], strides[4];
  cuuint32_t box[5], es[5] = {1, 1, 1, 1, 1};
  for (int i = 0; i < 5; ++i) { dims[i] = s.dim[i]; box[i] = s.box[i]; }
  for (int i = 0; i < 4; ++i) strides[i] = s.stride[i];
  const CUtensorMapDataType dt = (dtype == DT_BF16) ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  CUresult r = encode_fn()(&m, dt, 5, const_cast<void*>(s.base), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char buf[512];
    snprintf(buf, sizeof buf,
             "cuTensorMapEncodeTiled failed (%d): base=%p dim=(%llu,%llu,%llu,%llu,%llu) stride=(%llu,%llu,%llu,%llu) "
             "box=(%u,%u,%u,%u,%u)", static_cast<int>(r), s.base, (unsigned long long)dims[0], (unsigned long long)dims[1],
             (unsigned long long)dims[2], (unsigned long long)dims[3], (unsigned long long)dims[4],
             (unsigned long long)strides[0], (unsigned long long)strides[1], (unsigned long long)strides[2],
             (unsigned long long)strides[3], box[0], box[1], box[2], box[3], box[4]);
    throw Error(buf);
  }
  return m;
}

// ---------------------------------------------------------------------------------------------
// pool
// ---------------------------------------------------------------------------------------------
Pool::~Pool() {
  for (auto& b : blocks) cudaFree(b.first);
}
void* Pool::get(size_t bytes, size_t* actual) {
  bytes = (bytes + 511) / 512 * 512;
  auto it = free_.lower_bound(bytes);
  if (it != free_.end() && it->first <= bytes + bytes / 2 + (1u << 20)) {
    void* p = it->second;
    *actual = it->first;
    free_.erase(it);
    return p;
  }
  void* p = nullptr;
  I2IT_CUDA(cudaMalloc(&p, bytes));
  blocks.emplace_back(p, bytes);
  total += bytes;
  *actual = bytes;
  return p;
}

void* Pool::get_fresh(size_t bytes) {
  bytes = (bytes + 511) / 512 * 512;
  void* p = nullptr;
  I2IT_CUDA(cudaMalloc(&p, bytes));
  blocks.emplace_back(p, bytes);
  total += bytes;
  return p;
}

// ---------------------------------------------------------------------------------------------
// engine basics
// ---------------------------------------------------------------------------------------------
__global__ void cvt16_to_f32_kernel(const uint16_t* s, float* d, long long n, int is_bf16) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (is_bf16) d[i] = __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(s)[i]);
  else d[i] = __half2float(reinterpret_cast<const __half*>(s)[i]);
}

Engine::Engine(const i2it_config& c) : cfg(c), dtype(c.dtype) {
  I2IT_CHECK(c.dtype == DT_F16 || c.dtype == DT_BF16, "dtype must be I2IT_F16 or I2IT_BF16");
  I2IT_CUDA(cudaSetDevice(c.device));
  cudaDeviceProp prop;
  I2IT_CUDA(cudaGetDeviceProperties(&prop, c.device));
  I2IT_CHECK(prop.major == 10, "libi2it is built for sm_100a (B200) only; found compute capability " +
                                   std::to_string(prop.major) + "." + std::to_string(prop.minor));
  num_sms = prop.multiProcessorCount;
  I2IT_CUDA(cudaFuncSetAttribute(tapgemm_kernel<__half, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TG_SMEM));
  I2IT_CUDA(cudaFuncSetAttribute(tapgemm_kernel<__half, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TG_SMEM));
  I2IT_CUDA(cudaFuncSetAttribute(tapgemm_kernel<__nv_bfloat16, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TG_SMEM));
  I2IT_CUDA(cudaFuncSetAttribute(tapgemm_kernel<__nv_bfloat16, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TG_SMEM));
  I2IT_CUDA(cudaFuncSetAttribute(flash_attn_kernel<__half>, cudaFuncAttributeMaxDynamicSharedMemorySize, FA_SMEM));
  I2IT_CUDA(cudaFuncSetAttribute(flash_attn_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, FA_SMEM));
  use_pair = std::getenv("I2IT_NO_PAIR") == nullptr;
#ifdef I2IT_TRACE_BUILD
  trace_on = std::getenv("I2IT_TRACE") != nullptr;
#endif
  use_tmaout = std::getenv("I2IT_NO_TMAOUT") == nullptr;   // TMA-store epilogue (per-thread stores otherwise)
  sync_each = std::getenv("I2IT_SYNC_EACH") != nullptr;    // eager path: synchronise after every launch and name the one that faults
  use_lean = std::getenv("I2IT_NO_LEAN") == nullptr;       // compile-time-stripped epilogue for the plain (no activation) TMA-store launches
  use_gnepi = std::getenv("I2IT_NO_GNEPI") == nullptr;     // GroupNorm statistics in the producing GEMM's epilogue
  use_splitk = std::getenv("I2IT_NO_SPLITK") == nullptr;   // split-K for the 8x8 1280-channel convs
  use_halo = std::getenv("I2IT_NO_HALO") == nullptr;   // 3x3 convs: one halo tile per k-chunk instead of nine shifted A boxes
  I2IT_CUDA(cudaFuncSetAttribute(tapgemm2_kernel<__half, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TG2_SMEM));
  I2IT_CUDA(cudaFuncSetAttribute(tapgemm2_kernel<__half, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TG2_SMEM));
  I2IT_CUDA(cudaFuncSetAttribute(tapgemm2_kernel<__nv_bfloat16, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TG2_SMEM));
  I2IT_CUDA(cudaFuncSetAttribute(tapgemm2_kernel<__nv_bfloat16, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TG2_SMEM));
  int* h = nullptr;
  I2IT_CUDA(cudaHostAlloc(&h, sizeof(int), cudaHostAllocMapped));
  *h = 0;
  I2IT_CUDA(cudaHostGetDevicePointer(&d_err, h, 0));
  err_host_ = h;
  I2IT_CUDA(cudaStreamCreateWithFlags(&gstream_, cudaStreamNonBlocking));
  I2IT_CUDA(cudaEventCreateWithFlags(&ev_in_, cudaEventDisableTiming));
  I2IT_CUDA(cudaEventCreateWithFlags(&ev_out_, cudaEventDisableTiming));
  encode_fn();
}

Engine::~Engine() {
  plans_.clear();
  textkv_.clear();
  textenc_.clear();
  free_prepared();
  for (auto& kv : w_) cudaFree(kv.second.d);
  if (canny_ws_) cudaFree(canny_ws_);
  if (err_host_) cudaFreeHost(err_host_);
  if (gstream_) cudaStreamDestroy(gstream_);
  if (ev_in_) cudaEventDestroy(ev_in_);
  if (ev_out_) cudaEventDestroy(ev_out_);
}

void Engine::check_device_error() {
  if (err_host_ && *err_host_ != 0) {
    const int code = *err_host_;
    throw Error("tapgemm watchdog tripped (pipeline stage code " + std::to_string(code) +
                ": 1=producer/empty 2=mma/tmem_empty 3=mma/full 4=epilogue/tmem_full)");
  }
}

void* Engine::canny_workspace(size_t bytes) {
  if (bytes > canny_ws_bytes_) {
    if (canny_ws_) I2IT_CUDA(cudaFree(canny_ws_));     // cudaFree waits for the device: no launch still uses the old buffer
    canny_ws_ = nullptr;
    canny_ws_bytes_ = 0;
    I2IT_CUDA(cudaMalloc(&canny_ws_, bytes));
    canny_ws_bytes_ = bytes;
  }
  return canny_ws_;
}

void* Engine::dmalloc(size_t bytes) {
  void* p = nullptr;
  I2IT_CUDA(cudaMalloc(&p, std::max<size_t>(bytes, 16)));
  prep_allocs_.push_back(p);
  return p;
}

void Engine::free_prepared() {
  for (void* p : prep_allocs_) cudaFree(p);
  prep_allocs_.clear();
  prepared_.clear();
  prepared_f32_.clear();
  emb_act_ = nullptr;
  pending_jobs_.clear();
  pending_blocks_ = 0;
  for (auto& g : pending_gemv_) g.clear();
}

void Engine::set_weight(const std::string& key_in, const void* data, const int64_t* shape, int ndim, int dt, bool is_dev) {
  std::string key = key_in;
  const std::string bl = ".base_layer.";
  const size_t pos = key.find(bl);
  if (pos != std::string::npos) key = key.substr(0, pos) + "." + key.substr(pos + bl.size());
  WT t;
  t.numel = 1;
  for (int i = 0; i < ndim; ++i) { t.shape.push_back(shape[i]); t.numel *= shape[i]; }
  I2IT_CHECK(t.numel > 0, "empty tensor for key " + key);
  I2IT_CUDA(cudaMalloc(&t.d, t.numel * sizeof(float)));
  if (dt == DT_F32) {
    I2IT_CUDA(cudaMemcpy(t.d, data, t.numel * sizeof(float), is_dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice));
  } else {
    I2IT_CHECK(dt == DT_F16 || dt == DT_BF16, "unsupported weight dtype");
    uint16_t* tmp = nullptr;
    I2IT_CUDA(cudaMalloc(&tmp, t.numel * 2));
    I2IT_CUDA(cudaMemcpy(tmp, data, t.numel * 2, is_dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice));
    cvt16_to_f32_kernel<<<ceil_div(t.numel, 256), 256>>>(tmp, t.d, t.numel, dt == DT_BF16);
    I2IT_CUDA(cudaDeviceSynchronize());
    cudaFree(tmp);
  }
  auto it = w_.find(key);
  if (it != w_.end()) { cudaFree(it->second.d); w_.erase(it); }
  w_.emplace(key, std::move(t));
  finalized_ = false;
}

bool Engine::has(const std::string& key) const { return w_.count(key) != 0; }

const WT& Engine::raw(const std::string& name, const char* what) const {
  auto it = w_.find(name + "." + what);
  I2IT_CHECK(it != w_.end(), "missing weight '" + name + "." + what + "'");
  return it->second;
}

float Engine::adapter_weight(const std::string& name, const std::string& adapter) const {
  auto it = adapter_scale_.find(adapter);
  I2IT_CHECK(it != adapter_scale_.end(), "no scale registered for LoRA adapter '" + adapter + "' (layer " + name + ")");
  const bool is_unet = name.rfind("unet.", 0) == 0;
  return it->second * (is_unet ? lw_unet_ : lw_vae_);
}

void Engine::finalize(float lw_unet, float lw_vae, float skip_gamma, float twin_r) {
  I2IT_CUDA(cudaDeviceSynchronize());
  lw_unet_ = lw_unet; lw_vae_ = lw_vae; skip_gamma_ = skip_gamma; twin_r_ = twin_r;
  plans_.clear();
  textkv_.clear();                 // cached cross-attention operands were projected with the old (LoRA-scaled) weights
  textenc_.clear();
  last_plan_ = nullptr;
  free_prepared();
  finalized_ = true;
}

// Fold recipe of a layer: c0*W (+ c1*W_other) + sum_adapters s_a * B_a @ A_a — filled into a job, evaluated on device
void Engine::fill_fold(PrepJob& j, const std::string& name, float c0, const std::string& other, float c1) {
  const WT& w = raw(name, "weight");
  j.w0 = w.d; j.c0 = c0; j.w1 = nullptr; j.c1 = 0.f; j.n_adapters = 0;
  if (!other.empty()) {
    const WT& o = raw(other, "weight");
    I2IT_CHECK(o.numel == w.numel, "TwinConv shapes differ");
    j.w1 = o.d; j.c1 = c1;
  }
  const std::string pre = name + ".lora_A.";
  std::vector<std::string> adapters;
  for (const auto& kv : w_)
    if (kv.first.compare(0, pre.size(), pre) == 0) {
      const std::string rest = kv.first.substr(pre.size());            // "<adapter>.weight"
      adapters.push_back(rest.substr(0, rest.rfind('.')));
    }
  std::sort(adapters.begin(), adapters.end());                          // fixed summation order
  for (const auto& adapter : adapters) {
    const float s = adapter_weight(name, adapter);
    if (s == 0.f) continue;
    const WT& A = w_.at(pre + adapter + ".weight");
    auto itb = w_.find(name + ".lora_B." + adapter + ".weight");
    I2IT_CHECK(itb != w_.end(), "lora_A without lora_B for " + name);
    const WT& Bm = itb->second;
    const int rank = static_cast<int>(A.shape[0]);
    const long long inner = A.numel / rank;
    I2IT_CHECK(Bm.shape[0] * inner == w.numel && Bm.shape[1] == rank, "LoRA shape mismatch at " + name);
    I2IT_CHECK(j.n_adapters < PREP_MAX_ADAPTERS, "too many LoRA adapters on " + name);
    j.A[j.n_adapters] = A.d; j.B[j.n_adapters] = Bm.d; j.s[j.n_adapters] = s; j.rank[j.n_adapters] = rank;
    ++j.n_adapters;
  }
}

void Engine::push_job(PrepJob& j) {
  if (j.n <= 0) return;
  j.block0 = pending_blocks_;
  pending_blocks_ += (j.n + PREP_ELEMS_PER_BLOCK - 1) / PREP_ELEMS_PER_BLOCK;
  pending_jobs_.push_back(j);
}

void Engine::push_bias_job(float* out, const float* b, const float* add, int cout, int row_off, int half, float c0,
                           const float* b1, float c1) {
  PrepJob j;
  std::memset(&j, 0, sizeof j);
  j.mode = PREP_BIAS; j.out = out; j.bias = b; j.bias_add = add; j.cout = cout; j.row_off = row_off; j.interleave_half = half;
  j.c0 = c0; j.w1 = b1; j.c1 = c1;
  j.n = cout;
  push_job(j);
}

// Runs every pending preparation job: <= 3 GEMV launches (time embedding chain) + ONE fold/re-layout launch.
void Engine::flush_prep() {
  for (int st = 0; st < 3; ++st) {
    auto& g = pending_gemv_[st];
    if (g.empty()) continue;
    int warps = 0;
    for (auto& j : g) { j.warp0 = warps; warps += j.out; }
    GemvJob* d = static_cast<GemvJob*>(dmalloc(g.size() * sizeof(GemvJob)));
    I2IT_CUDA(cudaMemcpy(d, g.data(), g.size() * sizeof(GemvJob), cudaMemcpyHostToDevice));
    gemv_jobs_kernel<<<ceil_div(warps * 32ll, 256), 256>>>(d, static_cast<int>(g.size()));
    I2IT_CUDA(cudaGetLastError());
    prep_launches_ += 1;
    g.clear();
  }
  if (!pending_jobs_.empty()) {
    PrepJob* d = static_cast<PrepJob*>(dmalloc(pending_jobs_.size() * sizeof(PrepJob)));
    I2IT_CUDA(cudaMemcpy(d, pending_jobs_.data(), pending_jobs_.size() * sizeof(PrepJob), cudaMemcpyHostToDevice));
    I2IT_CHECK(pending_blocks_ < (1ll << 31), "weight preparation: too many blocks for one launch");
    DISPATCH_T(dtype, (prep_jobs_kernel<T><<<static_cast<unsigned>(pending_blocks_), 256>>>(d, static_cast<int>(pending_jobs_.size()))));
    I2IT_CUDA(cudaGetLastError());
    prep_launches_ += 1;
    pending_jobs_.clear();
    pending_blocks_ = 0;
  }
}

PW Engine::prep(const std::string& cache_key, const std::vector<std::string>& names, bool geglu, float scale,
                const float* bias_add) {
  auto it = prepared_.find(cache_key);
  if (it != prepared_.end()) return it->second;
  I2IT_CHECK(finalized_, "i2it_finalize_weights must be called before a forward");
  PW pw;
  const WT& w0 = raw(names[0], "weight");
  pw.cin = static_cast<int>(w0.shape[1]);
  pw.taps = (w0.shape.size() == 4) ? static_cast<int>(w0.shape[2] * w0.shape[3]) : 1;
  pw.cin_pad = round_up(pw.cin, 8);
  bool any_bias = bias_add != nullptr;
  for (const auto& n : names) {
    const WT& w = raw(n, "weight");
    I2IT_CHECK(static_cast<int>(w.shape[1]) == pw.cin, "fused projection with different input widths: " + n);
    pw.rows += static_cast<int>(w.shape[0]);
    any_bias = any_bias || has(n + ".bias");
  }
  I2IT_CHECK(!geglu || names.size() == 1, "GEGLU interleave applies to a single projection");
  const size_t wbytes = static_cast<size_t>(pw.taps) * pw.rows * pw.cin_pad * 2;
  pw.w = static_cast<uint16_t*>(dmalloc(wbytes));
  if (any_bias) pw.bias = static_cast<float*>(dmalloc(pw.rows * sizeof(float)));
  int row_off = 0;
  for (const auto& n : names) {
    const int cout = static_cast<int>(raw(n, "weight").shape[0]);
    const int half = geglu ? cout / 2 : 0;
    PrepJob j;
    std::memset(&j, 0, sizeof j);
    fill_fold(j, n);
    j.mode = PREP_STORE; j.out = pw.w; j.cout = cout; j.cin = pw.cin; j.taps = pw.taps; j.cin_pad = pw.cin_pad;
    j.rows_total = pw.rows; j.row_off = row_off; j.interleave_half = half; j.scale = scale;
    j.n = static_cast<long long>(cout) * pw.cin_pad * pw.taps;
    push_job(j);
    if (pw.bias) push_bias_job(pw.bias, has(n + ".bias") ? raw(n, "bias").d : nullptr, bias_add, cout, row_off, half);
    row_off += cout;
  }
  prepared_[cache_key] = pw;
  return pw;
}

PW Engine::prep_twin(const std::string& pre, const std::string& cur, float r) {
  const std::string key = pre + "|twin";
  auto it = prepared_.find(key);
  if (it != prepared_.end()) return it->second;
  I2IT_CHECK(r >= 0.f, "the state dict has a TwinConv conv_in but no blend ratio r was given (deterministic forward on a "
                       "sketch_to_image_stochastic model is undefined in the reference too)");
  PW pw;
  const WT& w0 = raw(pre, "weight");
  pw.rows = static_cast<int>(w0.shape[0]);
  pw.cin = static_cast<int>(w0.shape[1]);
  pw.taps = static_cast<int>(w0.shape[2] * w0.shape[3]);
  pw.cin_pad = round_up(pw.cin, 8);
  pw.w = static_cast<uint16_t*>(dmalloc(static_cast<size_t>(pw.taps) * pw.rows * pw.cin_pad * 2));
  pw.bias = static_cast<float*>(dmalloc(pw.rows * sizeof(float)));
  PrepJob j;
  std::memset(&j, 0, sizeof j);
  fill_fold(j, pre, 1.f - r, cur, r);                       // W = (1-r) W_pre + r W_cur   (pix2pix_turbo.py:23-26)
  j.mode = PREP_STORE; j.out = pw.w; j.cout = pw.rows; j.cin = pw.cin; j.taps = pw.taps; j.cin_pad = pw.cin_pad;
  j.rows_total = pw.rows; j.scale = 1.f;
  j.n = static_cast<long long>(pw.rows) * pw.cin_pad * pw.taps;
  push_job(j);
  push_bias_job(pw.bias, raw(pre, "bias").d, nullptr, pw.rows, 0, 0, 1.f - r, raw(cur, "bias").d, r);   // (1-r) b_pre + r b_cur
  prepared_[key] = pw;
  return pw;
}

PW Engine::prep_im2col3(const std::string& name) {
  const std::string key = name + "|im2col";
  auto it = prepared_.find(key);
  if (it != prepared_.end()) return it->second;
  const WT& w0 = raw(name, "weight");
  I2IT_CHECK(w0.shape.size() == 4 && w0.shape[1] == 3 && w0.shape[2] == 3 && w0.shape[3] == 3, "prep_im2col3: expects [Cout,3,3,3]");
  PW pw;
  pw.rows = static_cast<int>(w0.shape[0]); pw.cin = 32; pw.cin_pad = 32; pw.taps = 1;
  pw.w = static_cast<uint16_t*>(dmalloc(static_cast<size_t>(pw.rows) * 32 * 2));
  pw.bias = static_cast<float*>(dmalloc(pw.rows * sizeof(float)));
  PrepJob j;
  std::memset(&j, 0, sizeof j);
  fill_fold(j, name);
  j.mode = PREP_IM2COL3; j.out = pw.w; j.cout = pw.rows; j.cin = 3; j.taps = 9; j.scale = 1.f;
  j.n = static_cast<long long>(pw.rows) * 32;
  push_job(j);
  push_bias_job(pw.bias, raw(name, "bias").d, nullptr, pw.rows, 0, 0);
  prepared_[key] = pw;
  return pw;
}

PW Engine::prep_subpixel(const std::string& name) {
  const std::string key = name + "|subpixel";
  auto it = prepared_.find(key);
  if (it != prepared_.end()) return it->second;
  const WT& w0 = raw(name, "weight");
  I2IT_CHECK(w0.shape.size() == 4 && w0.shape[2] == 3 && w0.shape[3] == 3, "prep_subpixel: expects a 3x3 conv");
  PW pw;
  pw.rows = static_cast<int>(w0.shape[0]); pw.cin = static_cast<int>(w0.shape[1]); pw.cin_pad = round_up(pw.cin, 8); pw.taps = 16;
  const long long total = 16ll * pw.rows * pw.cin_pad;
  pw.w = static_cast<uint16_t*>(dmalloc(static_cast<size_t>(total) * 2));
  pw.bias = static_cast<float*>(dmalloc(pw.rows * sizeof(float)));
  PrepJob j;
  std::memset(&j, 0, sizeof j);
  fill_fold(j, name);
  j.mode = PREP_SUBPIXEL; j.out = pw.w; j.cout = pw.rows; j.cin = pw.cin; j.taps = 9; j.cin_pad = pw.cin_pad; j.scale = 1.f;
  j.n = total;
  push_job(j);
  push_bias_job(pw.bias, raw(name, "bias").d, nullptr, pw.rows, 0, 0);
  prepared_[key] = pw;
  return pw;
}

// nearest-2x upsample + conv3x3 (+ optional folded 1x1 second source at output resolution) as four parity-phase launches
Act Engine::conv_up2x(Plan& P, const Act& x, const PW& wsub, const Act* x2, const PW* w2, bool gn_out) {
  Act out = alloc_act(P, x.N, 2 * x.H, 2 * x.W, wsub.rows);
  for (int ph = 0; ph < 4; ++ph) {
    ConvOpts o;
    o.subpixel_phase = ph;
    o.out = &out;
    o.x2 = x2; o.w2 = w2;
    o.gn_out = gn_out;
    o.gn_share = out.gn;                 // phase 0 creates the partial buffer, phases 1..3 fill their slot ranges
    Act y = conv(P, x, wsub, o);
    out.gn = y.gn;
  }
  return out;
}

NormW Engine::norm(const std::string& name) {
  NormW n;
  const WT& g = raw(name, "weight");
  n.g = g.d;
  n.b = raw(name, "bias").d;
  n.C = static_cast<int>(g.numel);
  return n;
}

const float* Engine::temb_bias(const std::string& p) {
  const std::string key = p + "|temb";
  auto it = prepared_f32_.find(key);
  if (it != prepared_f32_.end()) return it->second;
  const int T = cfg.temb_dim, C0 = cfg.unet_channels[0];
  auto gemv = [&](int stage, const std::string& name, const float* x, float* y, int out, int in, int silu) {
    PrepJob f;
    std::memset(&f, 0, sizeof f);
    fill_fold(f, name);
    GemvJob g;
    std::memset(&g, 0, sizeof g);
    g.w = f.w0; g.b = raw(name, "bias").d; g.x = x; g.y = y; g.out = out; g.in = in; g.silu_out = silu;
    g.n_adapters = f.n_adapters;
    for (int a = 0; a < f.n_adapters; ++a) { g.A[a] = f.A[a]; g.B[a] = f.B[a]; g.s[a] = f.s[a]; g.rank[a] = f.rank[a]; }
    pending_gemv_[stage].push_back(g);
  };
  if (!emb_act_) {
    // Timesteps(flip_sin_to_cos=True, freq_shift=0) at t = 999, then TimestepEmbedding, then the SiLU every resnet applies
    std::vector<float> te(C0);
    const int half = C0 / 2;
    for (int i = 0; i < half; ++i) {
      const float f = expf(-logf(10000.f) * static_cast<float>(i) / static_cast<float>(half));
      te[i] = cosf(999.f * f);
      te[half + i] = sinf(999.f * f);
    }
    float* d_te = static_cast<float*>(dmalloc(C0 * sizeof(float)));
    float* d_h = static_cast<float*>(dmalloc(T * sizeof(float)));
    emb_act_ = static_cast<float*>(dmalloc(T * sizeof(float)));
    I2IT_CUDA(cudaMemcpy(d_te, te.data(), C0 * sizeof(float), cudaMemcpyHostToDevice));
    gemv(0, "unet.time_embedding.linear_1", d_te, d_h, T, C0, 1);
    gemv(1, "unet.time_embedding.linear_2", d_h, emb_act_, T, T, 1);
  }
  const WT& w = raw(p + ".time_emb_proj", "weight");
  const int cout = static_cast<int>(w.shape[0]);
  float* out = static_cast<float*>(dmalloc(cout * sizeof(float)));
  gemv(2, p + ".time_emb_proj", emb_act_, out, cout, T, 0);
  prepared_f32_[key] = out;
  return out;
}

// ---------------------------------------------------------------------------------------------
// op builders
// ---------------------------------------------------------------------------------------------
std::shared_ptr<void> Engine::alloc_raw(Plan& P, size_t bytes) {
  size_t actual = 0;
  void* p = P.pool.get(bytes, &actual);
  Pool* pool = &P.pool;
  return std::shared_ptr<void>(p, [pool, actual](void* q) { pool->put(q, actual); });
}

Act Engine::alloc_act(Plan& P, int N, int H, int W, int C, int ld, bool zero_persistent) {
  Act a;
  a.N = N; a.H = H; a.W = W; a.C = C; a.ld = ld ? ld : C;
  const size_t bytes = static_cast<size_t>(N) * H * W * a.ld * 2;
  if (zero_persistent) {
    // A recycled block would be dirtied at RUN time by the earlier ops that used it (the memset below runs once, at
    // build time), so padded small-channel tensors get their own allocation for the plan's lifetime.
    void* p = P.pool.get_fresh(bytes);
    I2IT_CUDA(cudaMemset(p, 0, bytes));
    a.hold = std::shared_ptr<void>(p, [](void*) {});
    a.p = static_cast<uint16_t*>(p);
    return a;
  }
  a.hold = alloc_raw(P, bytes);
  a.p = static_cast<uint16_t*>(a.hold.get());
  return a;
}

int Engine::pick_bn(long long m_tiles, int N, int step) const {
  if (N <= 16) return 16;
  static const int cand_any[] = {256, 224, 192, 160, 128, 112, 96, 80, 64, 48, 32, 16};
  static const int cand_64[] = {256, 192, 128, 64};
  static const int cand_128[] = {256, 128};
  const int* cand = step == 128 ? cand_128 : (step == 64 ? cand_64 : cand_any);
  const int ncand = step == 128 ? 2 : (step == 64 ? 4 : 12);
  int best = cand[ncand - 1];
  double best_cost = 1e30;
  for (int i = 0; i < ncand; ++i) {
    const int bn = cand[i];
    if (bn > round_up(N, step > 0 ? step : 16)) continue;
    const long long tiles = m_tiles * ceil_div(N, bn);
    const long long waves = (tiles + num_sms - 1) / num_sms;
    // a tile's time is bounded by its L2->SMEM traffic (A 128 rows + B bn rows per k-step) as much as by the MMA (bn)
    const double cost = static_cast<double>(waves) * (128 + bn);
    if (cost < best_cost - 1e-9) { best_cost = cost; best = bn; }
  }
  return best;
}

// The TMA-store epilogue handles 16-bit row-major outputs whose channel count and tile width are whole 64-column rounds (128
// accumulator columns for GEGLU) with 16-byte aligned rows; everything else keeps per-thread stores.
bool Engine::tma_eligible(const TapGemmParams& p, bool out_from_io) const {
  if (!use_tmaout || out_from_io || p.out_fp32 || p.ocol != 1 || p.bias_mode == TG_BIAS_ROW || p.out == nullptr) return false;
  const int acols = (p.act == TG_ACT_GEGLU) ? 128 : 64;
  if (p.N % acols != 0 || p.BN % acols != 0) return false;
  if (reinterpret_cast<uintptr_t>(p.out) % 16 != 0) return false;
  for (int d = 0; d < 4; ++d)
    if (p.ext[d] > 1 && (p.ostride[d] * 2) % 16 != 0) return false;
  if (p.res) {
    if (p.rcol != 1 || reinterpret_cast<uintptr_t>(p.res) % 16 != 0 || p.act == TG_ACT_GEGLU) return false;
    for (int d = 0; d < 4; ++d)
      if (p.ext[d] > 1 && (p.rstride[d] * 2) % 16 != 0) return false;
  }
  return true;
}

static void fill_strides(TmapSpec& s);

void Engine::launch_gemm(Plan& P, const TmapSpec& sa, TmapSpec sb, const TapGemmParams& p_in, bool out_from_io,
                         const char* kind, double k_valid, double bytes, const TmapSpec* sa2p, const TmapSpec* sb2p,
                         const TmapSpec* shalo) {
  TapGemmParams p = p_in;
  for (int t = 0; t < p.num_taps; ++t)
    if (p.tap_kc[t] == 0) p.tap_kc[t] = p.kchunks;          // single-source callers only set kchunks
  if (p.nprim == 0) p.nprim = p.num_taps;
  const long long m_tiles = 1ll * p.tdim[0] * p.tdim[1] * p.tdim[2] * p.tdim[3];
  const long long total_tiles = m_tiles * p.n_tiles * (p.ksplit > 1 ? p.ksplit : 1);
  // CTA-pair kernel: weights/B shared by every M tile (no per-tile B batch coordinates), enough tiles to fill the chip twice
  const bool pair = use_pair && p.ksplit <= 1 && p.b_mul[0] == 0 && p.b_mul[1] == 0 && p.b_mul[2] == 0 && (p.BN % 32) == 0 &&
                    total_tiles >= 2ll * num_sms && m_tiles >= 2;
  TmapSpec sb2 = sb2p ? *sb2p : sb;
  if (pair) { sb.box[1] = p.BN / 2; sb2.box[1] = p.BN / 2; p.idesc = make_idesc2(dtype, p.BN); }
  p.halo = (pair && shalo != nullptr && use_halo) ? 1 : 0;
  p.tma_out = tma_eligible(p, out_from_io) ? 1 : 0;
  {  // smem ring geometry: B stage = the real (half) tile rounded to the 1024-byte swizzle atom, as many stages as fit
    const int brows = pair ? p.BN / 2 : p.BN;
    p.b_stage = (brows * TG_BK * 2 + 1023) / 1024 * 1024;
    const int budget = pair ? (p.halo ? TG2_DATA_BYTES - TG2_HALO_REGION : TG2_DATA_BYTES) : TG_STAGES * (TG_A_STAGE + TG_B_STAGE);
    const int per = (p.halo ? 0 : TG_A_STAGE) + p.b_stage;
    p.stages = std::max(2, std::min(TG_MAX_STAGES, budget / per));
  }
  const CUtensorMap ta = encode_tmap(sa, dtype), tb = encode_tmap(sb, dtype);
  const CUtensorMap th = p.halo ? encode_tmap(*shalo, dtype) : ta;
  const CUtensorMap ta2 = sa2p ? encode_tmap(*sa2p, dtype) : ta, tb2 = sb2p ? encode_tmap(sb2, dtype) : tb;
  const int dt = dtype;
  Plan* plan = &P;
  const double m_valid = 1.0 * p.ext[0] * p.ext[1] * p.ext[2] * p.ext[3];
  int grid;
  if (pair) {
    const long long pairs = ((m_tiles + 1) / 2) * p.n_tiles;
    grid = 2 * static_cast<int>(std::min<long long>(pairs, num_sms / 2));
  } else {
    grid = static_cast<int>(std::min<long long>(total_tiles, num_sms));
  }
  char shp[160];
  snprintf(shp, sizeof shp, "M=%.0f N=%d K=%.0f taps=%d BN=%d tiles=%lld grid=%d st=%d%s%s%s", m_valid, p.N, k_valid, p.num_taps, p.BN,
           total_tiles, grid, p.stages, pair ? (p.halo ? " pair halo" : " pair") : "", p.tma_out ? " tma" : "",
           (p.gn_part && p.tma_out) ? " gn" : "");
  // TMA-store epilogue: the output tensor map has the tile's row dims (extents = logical extents, so ragged edges are clipped
  // by the hardware) and a box of 64 columns x the 32 rows one epilogue warp owns
  if (!p.tma_out) p.gn_part = nullptr;
  CUtensorMap to = ta;
  if (p.tma_out) {
    TmapSpec so;
    so.base = p.out;
    so.dim[0] = (p.act == TG_ACT_GEGLU) ? p.N / 2 : p.N;
    int left = 32;
    for (int d = 0; d < 4; ++d) {
      so.dim[d + 1] = static_cast<uint64_t>(std::max(1, p.ext[d]));
      so.stride[d] = static_cast<uint64_t>(p.ostride[d]) * 2ull;
      const int sb = std::min(p.box[d], left);
      so.box[d + 1] = static_cast<uint32_t>(sb);
      left /= sb;
    }
    I2IT_CHECK(left == 1, "TMA-store box: the tile's row box does not factor into 32-row warp boxes");
    so.box[0] = 64;
    fill_strides(so);
    to = encode_tmap(so, dtype);
  }
  p.trace = nullptr;
  if (trace_on) {   // diagnostic timeline (I2IT_TRACE=1): 16 clock64 stamps per CTA, dumped to stderr after each forward
    p.trace = static_cast<unsigned long long*>(dmalloc(static_cast<size_t>(grid) * 16 * sizeof(unsigned long long)));
    I2IT_CUDA(cudaMemset(p.trace, 0, static_cast<size_t>(grid) * 16 * sizeof(unsigned long long)));
    P.traces.push_back({p.trace, grid, std::string(kind) + " " + shp});
  }
  {  // division-free tile decode (see fast_div): dividends are tile indices (pair kernel: up to 2 * m-tile index + 1)
    const long long maxd = std::max<long long>(total_tiles, 2 * m_tiles + 2) + grid;
    p.magic[0] = make_magic(maxd, p.n_tiles);
    for (int d = 0; d < 4; ++d) p.magic[d + 1] = make_magic(maxd, p.tdim[d]);
    for (int d = 0; d < 5; ++d) I2IT_CHECK(p.magic[d] != 0, "tapgemm: tile space too large for the division-free tile decode");
    p.gn_shift = 0;
    while ((1 << p.gn_shift) < p.gn_red) ++p.gn_shift;
  }
  const bool lean = use_lean && p.tma_out && p.act == TG_ACT_NONE;      // the epilogue variant without activation / direct-store code
  if (pair) {
    add_op(P, [ta, tb, ta2, tb2, th, to, p, grid, dt, out_from_io, plan, lean](cudaStream_t st) {
      TapGemmParams q = p;
      if (out_from_io) q.out = plan->io.out;
      if (lean) { DISPATCH_T(dt, (launch_k(tapgemm2_kernel<T, true>, dim3(grid), dim3(TG_THREADS), TG2_SMEM, st, 2, ta, tb, ta2, tb2, th, to, q))); }
      else { DISPATCH_T(dt, (launch_k(tapgemm2_kernel<T, false>, dim3(grid), dim3(TG_THREADS), TG2_SMEM, st, 2, ta, tb, ta2, tb2, th, to, q))); }
    }, kind, 2.0 * m_valid * p.N * k_valid, bytes, shp);
  } else {
    add_op(P, [ta, tb, ta2, tb2, to, p, grid, dt, out_from_io, plan, lean](cudaStream_t st) {
      TapGemmParams q = p;
      if (out_from_io) q.out = plan->io.out;
      if (lean) { DISPATCH_T(dt, (launch_k(tapgemm_kernel<T, true>, dim3(grid), dim3(TG_THREADS), TG_SMEM, st, 0, ta, tb, ta2, tb2, to, q))); }
      else { DISPATCH_T(dt, (launch_k(tapgemm_kernel<T, false>, dim3(grid), dim3(TG_THREADS), TG_SMEM, st, 0, ta, tb, ta2, tb2, to, q))); }
    }, kind, 2.0 * m_valid * p.N * k_valid, bytes, shp);
  }
}

static void fill_strides(TmapSpec& s) {
  // size-1 dims still need a legal (16-byte multiple) stride
  for (int i = 0; i < 4; ++i)
    if (s.stride[i] == 0 || (s.stride[i] % 16) != 0) s.stride[i] = 16;
}

Act Engine::conv(Plan& P, const Act& x, const PW& w, const ConvOpts& o_in) {
  if (o_in.stride == 2 && ((x.H | x.W) & 1)) {
    // odd-sized map (latent of an image that is a multiple of 8 but not of 64): the right / bottom zero padding is materialised
    // once so that the 5-D parity view stays a plain box; Ho = ceil(H/2) as F.conv2d(stride=2, padding=1) gives
    return conv(P, pad_even(P, x), w, o_in);
  }
  const ConvOpts& o = o_in;
  const bool sub = o.subpixel_phase >= 0;
  const int k = o.ksize, taps = sub ? 4 : k * k;
  I2IT_CHECK(sub ? (w.taps == 16 && k == 3 && o.stride == 1 && o.out && !o.res && !o.to_io_out_nchw) : (w.taps == taps),
             "conv: weight taps mismatch");
  I2IT_CHECK(x.C == w.cin || x.C == w.cin_pad, "conv: input channels " + std::to_string(x.C) + " vs weight " +
                                                  std::to_string(w.cin));
  I2IT_CHECK(x.ld % 8 == 0, "conv: pixel stride must be a multiple of 8 elements");
  const int Ho = x.H / o.stride, Wo = x.W / o.stride;
  const int gemm_n = w.rows;
  const int outc = (o.act == TG_ACT_GEGLU) ? gemm_n / 2 : gemm_n;

  Act out;
  if (o.out) {
    out = *o.out;
  } else if (!o.to_io_out_nchw) {
    I2IT_CHECK(!o.out_fp32, "conv: fp32 output needs an explicit out view");
    const int ld = round_up(outc, 8);
    const bool small = (outc % 8) != 0;
    out = alloc_act(P, x.N, Ho, Wo, small ? ld : outc, ld, small);
  }

  TmapSpec sa, sb;
  TapGemmParams p;
  std::memset(&p, 0, sizeof p);
  int tw, th, tn;
  const long long ldo = o.to_io_out_nchw ? 0 : out.ld;
  // halo mode (CTA-pair kernel): 8 x 16 output tiles whose nine taps share one halo tile per k-chunk
  const bool want_halo = use_halo && use_pair && o.stride == 1 && k == 3 && !sub && !o.x2 && !o.to_io_out_nchw && x.H >= 16 &&
                         x.W >= 8 && x.C % 64 == 0;
  if (o.stride == 1) {
    tw = (x.H == 1) ? std::min(128, pow2ceil(x.W)) : std::min(o.to_io_out_nchw ? 32 : 16, pow2ceil(x.W));
    th = std::min(128 / tw, pow2ceil(x.H));
    tn = 128 / (tw * th);
    if (want_halo) { tw = 8; th = 16; tn = 1; }
    sa.base = x.p;
    sa.dim[0] = x.C; sa.dim[1] = x.W; sa.dim[2] = x.H; sa.dim[3] = x.N; sa.dim[4] = 1;
    sa.stride[0] = x.ld * 2ull; sa.stride[1] = 2ull * x.W * x.ld; sa.stride[2] = 2ull * x.H * x.W * x.ld;
    sa.stride[3] = sa.stride[2];
    sa.box[0] = 64; sa.box[1] = tw; sa.box[2] = th; sa.box[3] = tn; sa.box[4] = 1;
    p.tdim[0] = ceil_div(x.W, tw); p.tdim[1] = ceil_div(x.H, th); p.tdim[2] = ceil_div(x.N, tn); p.tdim[3] = 1;
    p.box[0] = tw; p.box[1] = th; p.box[2] = tn; p.box[3] = 1;
    p.ext[0] = Wo; p.ext[1] = Ho; p.ext[2] = x.N; p.ext[3] = 1;
    p.a_mul[0] = tw; p.a_mul[1] = th; p.a_mul[2] = tn; p.a_mul[3] = 0;
    const int pad = k / 2;
    if (sub) {
      // output parity (py,px): 2x2 taps at low-res offsets (ty-1+py, tx-1+px); output pixel (2y+py, 2x+px)
      const int py = o.subpixel_phase >> 1, px = o.subpixel_phase & 1;
      for (int ty = 0; ty < 2; ++ty)
        for (int tx = 0; tx < 2; ++tx) {
          const int t = ty * 2 + tx;
          p.tap_a[t][0] = 0; p.tap_a[t][1] = tx - 1 + px; p.tap_a[t][2] = ty - 1 + py; p.tap_a[t][3] = 0; p.tap_a[t][4] = 0;
          p.tap_b[t][0] = 0; p.tap_b[t][1] = o.subpixel_phase * 4 + t; p.tap_b[t][2] = 0; p.tap_b[t][3] = 0;
        }
      p.ostride[0] = 2 * ldo; p.ostride[1] = 2ll * (2 * Wo) * ldo;
      p.ostride[2] = 4ll * Ho * Wo * ldo; p.ostride[3] = 0;
    } else {
      for (int ky = 0; ky < k; ++ky)
        for (int kx = 0; kx < k; ++kx) {
          const int t = ky * k + kx;
          p.tap_a[t][0] = 0; p.tap_a[t][1] = kx - pad; p.tap_a[t][2] = ky - pad; p.tap_a[t][3] = 0; p.tap_a[t][4] = 0;
          p.tap_b[t][0] = 0; p.tap_b[t][1] = t; p.tap_b[t][2] = 0; p.tap_b[t][3] = 0;
        }
      p.ostride[0] = ldo; p.ostride[1] = static_cast<long long>(Wo) * ldo;
      p.ostride[2] = static_cast<long long>(Ho) * Wo * ldo; p.ostride[3] = 0;
    }
    p.kchunks = ceil_div(x.C, 64);
  } else {
    I2IT_CHECK(o.stride == 2 && k == 3, "conv: only 3x3 stride-2 is on the path");
    I2IT_CHECK(x.ld % 8 == 0 && x.C % 64 == 0 && x.H % 2 == 0 && x.W % 2 == 0, "conv s2: needs NHWC with ld%8==0, C%64==0, even H/W");
    tw = std::min(16, pow2ceil(Wo));
    th = std::min(128 / tw, pow2ceil(Ho));
    tn = 128 / (tw * th);
    const unsigned long long C = x.C, LD = x.ld;
    // 5-D view (px*ld + c, xo, py, yo, n) of the NHWC input (pixel pitch ld >= C: the input may be a channel slice of a concat
    // buffer): a stride-2 tap is a plain box in this view.  dim 0 spans the C channels of the even pixel, the gap, and the C
    // channels of the odd pixel; boxes only ever start at c or ld + c with c + 64 <= C.
    sa.base = x.p;
    sa.dim[0] = LD + C; sa.dim[1] = Wo; sa.dim[2] = 2; sa.dim[3] = Ho; sa.dim[4] = x.N;
    sa.stride[0] = 2 * LD * 2; sa.stride[1] = x.W * LD * 2; sa.stride[2] = 2ull * x.W * LD * 2; sa.stride[3] = 1ull * x.H * x.W * LD * 2;
    sa.box[0] = 64; sa.box[1] = tw; sa.box[2] = 1; sa.box[3] = th; sa.box[4] = tn;
    p.tdim[0] = ceil_div(Wo, tw); p.tdim[1] = 1; p.tdim[2] = ceil_div(Ho, th); p.tdim[3] = ceil_div(x.N, tn);
    p.box[0] = tw; p.box[1] = 1; p.box[2] = th; p.box[3] = tn;
    p.ext[0] = Wo; p.ext[1] = 1; p.ext[2] = Ho; p.ext[3] = x.N;
    p.a_mul[0] = tw; p.a_mul[1] = 0; p.a_mul[2] = th; p.a_mul[3] = tn;
    const int padl = o.asym ? 0 : 1;
    for (int ky = 0; ky < 3; ++ky)
      for (int kx = 0; kx < 3; ++kx) {
        const int t = ky * 3 + kx;
        const int ex = kx - padl, ey = ky - padl;
        const int px = ex & 1, py = ey & 1;
        const int ox = (ex - px) / 2, oy = (ey - py) / 2;
        p.tap_a[t][0] = px * x.ld; p.tap_a[t][1] = ox; p.tap_a[t][2] = py; p.tap_a[t][3] = oy; p.tap_a[t][4] = 0;
        p.tap_b[t][0] = 0; p.tap_b[t][1] = t; p.tap_b[t][2] = 0; p.tap_b[t][3] = 0;
      }
    p.ostride[0] = ldo; p.ostride[1] = 0; p.ostride[2] = static_cast<long long>(Wo) * ldo;
    p.ostride[3] = static_cast<long long>(Ho) * Wo * ldo;
    p.kchunks = x.C / 64;
  }
  fill_strides(sa);

  sb.base = w.w;
  sb.dim[0] = w.cin_pad; sb.dim[1] = w.rows; sb.dim[2] = w.taps; sb.dim[3] = 1; sb.dim[4] = 1;
  sb.stride[0] = w.cin_pad * 2ull; sb.stride[1] = 2ull * w.rows * w.cin_pad; sb.stride[2] = 2ull * w.taps * w.rows * w.cin_pad;
  sb.stride[3] = sb.stride[2];
  fill_strides(sb);

  const long long m_tiles = 1ll * p.tdim[0] * p.tdim[1] * p.tdim[2] * p.tdim[3];
  p.N = gemm_n;
  {
    // whole 64-column store rounds (128 accumulator columns for GEGLU) when the output can take the TMA-store epilogue
    const int acols = (o.act == TG_ACT_GEGLU) ? 128 : 64;
    const bool rounds = use_tmaout && !o.to_io_out_nchw && !o.out_fp32 && gemm_n % acols == 0 && (ldo % 8) == 0;
    p.BN = pick_bn(m_tiles, gemm_n, rounds ? acols : 0);
  }
  p.n_tiles = ceil_div(gemm_n, p.BN);
  sb.box[0] = 64; sb.box[1] = p.BN; sb.box[2] = 1; sb.box[3] = 1; sb.box[4] = 1;
  p.num_taps = taps;
  p.nprim = taps;
  p.idesc = make_idesc(dtype, p.BN);
  p.ocol = 1;
  p.out_fp32 = o.out_fp32 ? 1 : 0;
  if (o.to_io_out_nchw) {
    p.out = nullptr;                                   // patched from IO at launch
    const long long hw = static_cast<long long>(Ho) * Wo;
    p.ostride[0] = 1; p.ostride[1] = Wo; p.ostride[2] = hw * outc; p.ostride[3] = 0;
    p.ocol = hw;
  } else if (sub) {
    const int py = o.subpixel_phase >> 1, px = o.subpixel_phase & 1;
    p.out = out.p + (static_cast<long long>(py) * (2 * Wo) + px) * ldo;
  } else {
    p.out = out.p;
  }
  if (o.res) {
    I2IT_CHECK(o.stride == 1, "conv: residual only on stride-1 convs");
    p.res = o.res->p;
    const long long ldr = o.res->ld;
    p.rstride[0] = ldr; p.rstride[1] = static_cast<long long>(Wo) * ldr; p.rstride[2] = static_cast<long long>(Ho) * Wo * ldr;
    p.rcol = 1;
  }
  p.bias = w.bias;
  p.bias_mode = (o.bias_mode >= 0) ? o.bias_mode : (w.bias ? TG_BIAS_COL : TG_BIAS_NONE);
  if (!w.bias) p.bias_mode = TG_BIAS_NONE;
  p.alpha = o.alpha;
  p.act = o.act;
  p.err = d_err;

  // GroupNorm statistics of the output in this GEMM's epilogue (the consumer is a GroupNorm): needs the TMA-store path, a
  // 32-group channel count, and m-tiles that never straddle two images (so a 32-row slot belongs to one image)
  if ((o.gn_out || o.gn_share) && use_gnepi && outc % 64 == 0 && tma_eligible(p, o.to_io_out_nchw) && o.act != TG_ACT_GEGLU) {
    long long mt_img = 0;                 // m-tiles per image
    int images = x.N;
    if (o.gn_rows_per_image > 0) {        // flattened token matrix: 128-row tiles
      if (o.gn_rows_per_image % 128 == 0 && x.rows() % o.gn_rows_per_image == 0) {
        mt_img = o.gn_rows_per_image / 128;
        images = static_cast<int>(x.rows() / o.gn_rows_per_image);
      }
    } else if (tn == 1) {
      mt_img = (o.stride == 1) ? 1ll * p.tdim[0] * p.tdim[1] : 1ll * p.tdim[0] * p.tdim[2];
    }
    if (mt_img > 0) {
      const int cgrp = outc / 32;
      const int red = (cgrp == 4 || cgrp == 8 || cgrp == 16) ? cgrp : 2;
      std::shared_ptr<GnPart> g = o.gn_share;
      if (!g) {
        g = std::make_shared<GnPart>();
        g->red = red; g->C = outc; g->images = images; g->phases = sub ? 4 : 1;
        g->slots_per_image = static_cast<int>(mt_img * 4);
        g->hold = alloc_raw(P, static_cast<size_t>(g->phases) * images * g->slots_per_image * (outc / red) * 2 * sizeof(float));
        g->buf = static_cast<float*>(g->hold.get());
      }
      I2IT_CHECK(g->C == outc && g->slots_per_image == mt_img * 4 && g->images == images, "conv: shared GroupNorm partials mismatch");
      p.gn_part = g->buf;
      p.gn_red = g->red;
      p.gn_slot0 = sub ? o.subpixel_phase * images * g->slots_per_image : 0;
      p.gn_mtiles = static_cast<int>(mt_img * images);
      out.gn = g;
    }
  }

  // split-K for the 8x8 / 1280-channel convs (M = 64 rows per image): with K = 11.5k..23k and 4 m-tiles per batch of 8 the
  // launch had 80-108 weight-bandwidth-bound CTAs; five K ranges per tile write fp32 partials that splitk_reduce sums in a fixed
  // order.  The decision and the ranges depend on the layer only (never on the batch): batch-invariant bits.
  const bool splitk = use_splitk && !sub && k == 3 && o.stride == 1 && !o.to_io_out_nchw && !o.out_fp32 && o.act == TG_ACT_NONE &&
                      x.H * x.W <= 64 && p.kchunks * taps >= 180 && p.kchunks % 5 == 0 && gemm_n >= 640 && gemm_n % 8 == 0;
  std::shared_ptr<void> sk_hold;
  const Act* sk_res = nullptr;
  const float* sk_bias = nullptr;
  if (splitk) {
    const int S = 5;                      // kchunks is 20 or 40 here: equal shares
    const long long Mrows = 1ll * x.N * Ho * Wo;
    sk_hold = alloc_raw(P, static_cast<size_t>(S) * Mrows * gemm_n * sizeof(float));
    p.ksplit = S;
    p.kc_per = ceil_div(p.kchunks, S);
    p.split_ostride = Mrows * gemm_n;
    p.out = sk_hold.get();
    p.out_fp32 = 1;
    p.ostride[0] = gemm_n; p.ostride[1] = 1ll * Wo * gemm_n; p.ostride[2] = 1ll * Ho * Wo * gemm_n; p.ostride[3] = 0;
    sk_res = o.res; sk_bias = (p.bias_mode == TG_BIAS_COL) ? p.bias : nullptr;
    p.res = nullptr; p.bias = nullptr; p.bias_mode = TG_BIAS_NONE;
    p.gn_part = nullptr; out.gn = nullptr;
    p.BN = 256;
    p.n_tiles = ceil_div(gemm_n, p.BN);
    sb.box[1] = p.BN;
    p.idesc = make_idesc(dtype, p.BN);
  }

  TmapSpec sa2, sb2;
  double k2 = 0;
  if (o.x2) {
    // extra 1x1 "tap" over a second activation tensor with the same spatial geometry as the output
    I2IT_CHECK(o.w2 && o.stride == 1 && o.w2->taps == 1 && o.w2->rows == w.rows, "conv: bad second source");
    const int sm = sub ? 2 : 1;     // sub-pixel: the second source lives at OUTPUT resolution, sampled at this parity
    I2IT_CHECK(o.x2->N == x.N && o.x2->H == sm * Ho && o.x2->W == sm * Wo && (o.x2->C == o.w2->cin || o.x2->C == o.w2->cin_pad),
               "conv: second source shape mismatch");
    I2IT_CHECK(taps + 1 <= TG_MAX_TAPS, "conv: too many taps");
    sa2 = sa;
    sa2.base = o.x2->p;
    sa2.dim[0] = o.x2->C;
    sa2.stride[0] = o.x2->ld * 2ull; sa2.stride[1] = 2ull * o.x2->W * o.x2->ld; sa2.stride[2] = 2ull * o.x2->H * o.x2->W * o.x2->ld;
    sa2.stride[3] = sa2.stride[2];
    if (sub) {
      const int py = o.subpixel_phase >> 1, px = o.subpixel_phase & 1;
      sa2.base = o.x2->p + (static_cast<long long>(py) * o.x2->W + px) * o.x2->ld;
      sa2.stride[0] = 2ull * o.x2->ld * 2; sa2.stride[1] = 2ull * 2 * o.x2->W * o.x2->ld;   // every other pixel / row
    }
    fill_strides(sa2);
    sb2.base = o.w2->w;
    sb2.dim[0] = o.w2->cin_pad; sb2.dim[1] = o.w2->rows;
    sb2.stride[0] = o.w2->cin_pad * 2ull; sb2.stride[1] = 2ull * o.w2->rows * o.w2->cin_pad; sb2.stride[2] = sb2.stride[1];
    sb2.stride[3] = sb2.stride[1];
    sb2.box[0] = 64; sb2.box[1] = p.BN;
    fill_strides(sb2);
    for (int t = 0; t < taps; ++t) { p.tap_src[t] = 0; p.tap_kc[t] = p.kchunks; }
    const int t2 = taps;
    for (int d = 0; d < 5; ++d) p.tap_a[t2][d] = 0;
    for (int d = 0; d < 4; ++d) p.tap_b[t2][d] = 0;
    p.tap_src[t2] = 1;
    p.tap_kc[t2] = ceil_div(o.x2->C, 64);
    p.num_taps = taps + 1;
    k2 = o.w2->cin;
  }
  {
    const double m_valid = 1.0 * x.N * Ho * Wo, k_valid = 1.0 * taps * w.cin + k2;
    const double bytes = 2.0 * (1.0 * x.N * x.H * x.W * w.cin + m_valid * outc * (o.out_fp32 ? 2 : 1) + 1.0 * gemm_n * k_valid +
                                (o.res ? m_valid * outc : 0) + m_valid * k2);
    const char* kind = sub ? "tapgemm:conv_up2x" : (k == 3) ? (o.stride == 2 ? "tapgemm:conv3x3s2" : "tapgemm:conv3x3") : "tapgemm:linear";
    TmapSpec sh = sa;
    sh.box[1] = TG2_HALO_W; sh.box[2] = TG2_HALO_H; sh.box[3] = 1;
    launch_gemm(P, sa, sb, p, o.to_io_out_nchw, kind, k_valid, bytes, o.x2 ? &sa2 : nullptr, o.x2 ? &sb2 : nullptr,
                want_halo ? &sh : nullptr);
  }
  if (splitk) {
    const float* part = static_cast<const float*>(sk_hold.get());
    const long long Mrows = 1ll * x.N * Ho * Wo, total = Mrows * (gemm_n / 8), sstride = p.split_ostride;
    const uint16_t* rp = sk_res ? sk_res->p : nullptr;
    uint16_t* op = out.p;
    const int ldr = sk_res ? sk_res->ld : 0, ldo2 = out.ld, S = p.ksplit, dt = dtype, Nn = gemm_n;
    const float* bb = sk_bias;
    add_op(P, [=](cudaStream_t st) {
      DISPATCH_T(dt, (launch_k(splitk_reduce_kernel<T>, dim3(ceil_div(total, 256)), dim3(256), 0, st, 0, part, S, sstride, bb,
                               reinterpret_cast<const T*>(rp), ldr, reinterpret_cast<T*>(op), ldo2, Nn, total)));
    }, "splitk_reduce", 0, 4.0 * S * Mrows * gemm_n + 4.0 * Mrows * gemm_n);
  }
  return out;
}

Act Engine::linear(Plan& P, const Act& x, const PW& w, const Act* res, int act, bool gn_out, const Act* out) {
  ConvOpts o;
  o.ksize = 1;
  o.act = act;
  o.gn_out = gn_out;
  o.gn_rows_per_image = static_cast<long long>(x.H) * x.W;
  Act xr = x.as_rows(), rr, orows;
  if (res) { rr = res->as_rows(); o.res = &rr; }
  if (out) { orows = out->as_rows(); o.out = &orows; }
  Act y = conv(P, xr, w, o);
  y.N = x.N; y.H = x.H; y.W = x.W;
  return y;
}

// One ticket counter per image, shared by every GroupNorm launch of a plan: launches are stream-ordered and each one leaves
// the counters at zero (the block that draws the last ticket re-arms it), so graph replays start clean.
int* Engine::gn_counters(Plan& P, int images) {
  I2IT_CHECK(images <= 4096, "group_norm: batch too large for the ticket array");
  if (!P.gn_counter) {
    P.gn_counter = static_cast<int*>(P.pool.get_fresh(4096 * sizeof(int)));
    I2IT_CUDA(cudaMemset(P.gn_counter, 0, 4096 * sizeof(int)));
  }
  return P.gn_counter;
}

Act Engine::group_norm(Plan& P, const Act& x, const NormW& nw, float eps, bool silu) {
  I2IT_CHECK(x.C == nw.C && x.C % 32 == 0 && x.C % 8 == 0, "group_norm: bad channel count " + std::to_string(x.C));
  const int C = x.C, HW = x.H * x.W, cg = C / 32, vecs = C / 8;
  I2IT_CHECK(vecs <= 1024, "group_norm: too many channels");
  // about 128 threads per CTA and at most 512 CTAs per image: the best of the r01 sweep
  const int rows = std::max(1, 128 / vecs), threads = vecs * rows;
  const int chunks = std::max(1, std::min(512, ceil_div(HW, rows * 4)));
  // statistics pass over the tensor (no epilogue partials available): at most 64 chunk partials per image
  const int schunks = std::min(chunks, 64), spix = ceil_div(HW, schunks);
  const int pix = ceil_div(HW, chunks);
  I2IT_CHECK(chunks <= 1024, "group_norm: too many chunks");
  auto partial = alloc_raw(P, static_cast<size_t>(x.N) * 64 * 32 * sizeof(double) * 2);   // [N][<=64 chunks][32] double2 (or float2)
  auto stats = alloc_raw(P, static_cast<size_t>(x.N) * 64 * sizeof(float));
  Act y = alloc_act(P, x.N, x.H, x.W, C);
  float* d_part = static_cast<float*>(partial.get());
  float* d_stats = static_cast<float*>(stats.get());
  int* d_counter = gn_counters(P, x.N);                // zeroed once at build time; every launch leaves it at zero again
  const uint16_t* xp = x.p;
  uint16_t* yp = y.p;
  const long long ximg = x.img(), yimg = y.img();
  const int ldx = x.ld, ldy = y.ld, N = x.N, dt = dtype, isilu = silu ? 1 : 0;
  const float* g = nw.g;
  const float* b = nw.b;
  const double inv_count = 1.0 / (static_cast<double>(HW) * cg);
  if (x.gn && use_gnepi && x.gn->C == C && x.gn->images == N) {
    // the producer's epilogue already summed the tensor: reduce its per-slot partials (no pass over the tensor itself)
    const GnPart gp = *x.gn;
    const float* pb = gp.buf;
    const int per_row = C / gp.red, epg = cg / gp.red;
    I2IT_CHECK(per_row <= 640, "group_norm: too many partial entries per slot");
    const int nch = std::max(1, std::min(64, gp.slots_per_image / 16));
    const int e_lanes = std::min(256, pow2ceil(per_row));
    double2* p2 = reinterpret_cast<double2*>(d_part);
    add_op(P, [=](cudaStream_t st) {
      launch_k(gn_part_reduce_kernel, dim3(nch, N), dim3(256), 0, st, 0, pb, gp.phases, gp.images, gp.slots_per_image, per_row, epg,
               e_lanes, p2, d_counter, inv_count, eps, d_stats);
    }, "gn_final_part", 0, 8.0 * gp.phases * N * gp.slots_per_image * per_row);
  } else {
    add_op(P, [=](cudaStream_t st) {
      DISPATCH_T(dt, (launch_k(gn_stats_kernel<T>, dim3(schunks, N), dim3(threads), static_cast<size_t>(rows) * 2 * C * sizeof(float), st, 0,
                               reinterpret_cast<const T*>(xp), ximg, ldx, C, HW, cg, spix, d_part, d_counter, inv_count, eps, d_stats)));
    }, "gn_stats", 0, 2.0 * N * HW * C);
  }
  add_op(P, [=](cudaStream_t st) {
    DISPATCH_T(dt, (launch_k(gn_apply_kernel<T>, dim3(chunks, N), dim3(threads), 0, st, 0,
                       reinterpret_cast<const T*>(xp), ximg, ldx, reinterpret_cast<T*>(yp), yimg, ldy, C, HW, cg, pix,
                       d_stats, g, b, isilu)));
  }, "gn_apply", 0, 4.0 * N * HW * C);
  return y;     // (y carries no statistics: it is a different tensor)
}

Act Engine::layer_norm(Plan& P, const Act& x, const NormW& nw, bool to_io_out) {
  I2IT_CHECK(x.C == nw.C && x.C % 8 == 0 && x.C <= 1280, "layer_norm: C must be a multiple of 8 and <= 1280");
  Act y = to_io_out ? x : alloc_act(P, x.N, x.H, x.W, x.C);       // to_io_out: dense rows straight into the caller's buffer
  const long long rows = x.rows();
  const uint16_t* xp = x.p;
  uint16_t* yp = to_io_out ? nullptr : y.p;
  const int ldx = x.ld, ldy = to_io_out ? x.C : y.ld, C = x.C, dt = dtype;
  const float* g = nw.g;
  const float* b = nw.b;
  Plan* plan = &P;
  add_op(P, [=](cudaStream_t st) {
    uint16_t* dst = yp ? yp : static_cast<uint16_t*>(plan->io.out);
    DISPATCH_T(dt, (launch_k(layernorm_kernel<T>, dim3(ceil_div(rows * 32, 256)), dim3(256), 0, st, 0,
                       reinterpret_cast<const T*>(xp), ldx, reinterpret_cast<T*>(dst), ldy, static_cast<int>(rows), C, g, b,
                       1e-5f)));
  }, "layernorm", 0, 4.0 * rows * C);
  return y;
}

Act Engine::upsample_to(Plan& P, const Act& x, int Ho, int Wo) {
  Act y = alloc_act(P, x.N, Ho, Wo, x.C);
  const long long total = static_cast<long long>(x.N) * Ho * Wo * (x.C / 8);
  const uint16_t* xp = x.p;
  uint16_t* yp = y.p;
  const int ldx = x.ld, ldy = y.ld, H = x.H, W = x.W, C = x.C, dt = dtype;
  const float sh = static_cast<float>(H) / static_cast<float>(Ho), sw = static_cast<float>(W) / static_cast<float>(Wo);
  const double N_ = x.N;
  add_op(P, [=](cudaStream_t st) {
    DISPATCH_T(dt, (launch_k(upsample_nearest_kernel<T>, dim3(ceil_div(total, 256)), dim3(256), 0, st, 0, reinterpret_cast<const T*>(xp),
                             ldx, reinterpret_cast<T*>(yp), ldy, H, W, Ho, Wo, sh, sw, C, total)));
  }, "upsample_nearest", 0, 2.0 * N_ * C * (1.0 * H * W + 1.0 * Ho * Wo));
  return y;
}

Act Engine::pad_even(Plan& P, const Act& x) {
  const int H2 = x.H + (x.H & 1), W2 = x.W + (x.W & 1);
  if (H2 == x.H && W2 == x.W && x.ld == x.C) return x;
  Act y = alloc_act(P, x.N, H2, W2, x.C);
  const long long total = static_cast<long long>(x.N) * H2 * W2 * (x.C / 8);
  const uint16_t* xp = x.p;
  uint16_t* yp = y.p;
  const int ldx = x.ld, H = x.H, W = x.W, C = x.C, dt = dtype;
  add_op(P, [=](cudaStream_t st) {
    DISPATCH_T(dt, (launch_k(pad_copy_kernel<T>, dim3(ceil_div(total, 256)), dim3(256), 0, st, 0, reinterpret_cast<const T*>(xp), ldx,
                             reinterpret_cast<T*>(yp), H, W, H2, W2, C, total)));
  }, "pad_even", 0, 4.0 * total * 8);
  return y;
}

void Engine::copy_channels(Plan& P, const Act& src, const Act& dst) {
  I2IT_CHECK(src.C == dst.C && src.rows() == dst.rows() && src.C % 8 == 0, "copy_channels: shape mismatch");
  const long long total = src.rows() * (src.C / 8);
  const uint16_t* xp = src.p;
  uint16_t* yp = dst.p;
  const int ldx = src.ld, ldy = dst.ld, C = src.C, dt = dtype;
  add_op(P, [=](cudaStream_t st) {
    DISPATCH_T(dt, (launch_k(copy2d_kernel<T>, dim3(ceil_div(total, 256)), dim3(256), 0, st, 0, reinterpret_cast<const T*>(xp), ldx,
                                                                         reinterpret_cast<T*>(yp), ldy, C, total)));
  }, "concat_copy", 0, 4.0 * total * 8);
}

Act Engine::vt_proj(Plan& P, const Act& x, int B, int ntok, const PW& wv) {
  I2IT_CHECK(x.rows() == static_cast<long long>(B) * ntok, "vt_proj: token count mismatch");
  I2IT_CHECK(x.C == wv.cin || x.C == wv.cin_pad, "vt_proj: width mismatch");
  const int C = wv.rows, ldv = round_up(ntok, 8);
  Act vt = alloc_act(P, B, 1, C, ldv, ldv);      // [B][C rows][ldv]; "C" field carries the padded token count
  TmapSpec sa, sb;
  TapGemmParams p;
  std::memset(&p, 0, sizeof p);
  sa.base = wv.w;
  sa.dim[0] = wv.cin_pad; sa.dim[1] = C;
  sa.stride[0] = wv.cin_pad * 2ull; sa.stride[1] = 2ull * C * wv.cin_pad; sa.stride[2] = sa.stride[1]; sa.stride[3] = sa.stride[1];
  sa.box[0] = 64; sa.box[1] = 128;
  fill_strides(sa);
  sb.base = x.p;
  sb.dim[0] = x.C; sb.dim[1] = ntok; sb.dim[2] = 1; sb.dim[3] = B; sb.dim[4] = 1;
  sb.stride[0] = x.ld * 2ull; sb.stride[1] = 2ull * ntok * x.ld; sb.stride[2] = 2ull * ntok * x.ld; sb.stride[3] = sb.stride[2];
  fill_strides(sb);
  p.tdim[0] = ceil_div(C, 128); p.tdim[1] = 1; p.tdim[2] = B; p.tdim[3] = 1;
  p.box[0] = 128; p.box[1] = 1; p.box[2] = 1; p.box[3] = 1;
  p.ext[0] = C; p.ext[1] = 1; p.ext[2] = B; p.ext[3] = 1;
  p.a_mul[0] = 128;
  p.b_mul[0] = 0; p.b_mul[1] = 1; p.b_mul[2] = 0;
  const long long m_tiles = 1ll * p.tdim[0] * B;
  p.N = ntok;
  p.BN = pick_bn(m_tiles, ntok, false);
  p.n_tiles = ceil_div(ntok, p.BN);
  sb.box[0] = 64; sb.box[1] = p.BN;
  p.num_taps = 1;
  p.kchunks = ceil_div(x.C, 64);
  p.idesc = make_idesc(dtype, p.BN);
  p.out = vt.p;
  p.ostride[0] = ldv; p.ostride[1] = 0; p.ostride[2] = static_cast<long long>(C) * ldv; p.ostride[3] = 0;
  p.ocol = 1;
  p.bias = wv.bias;
  p.bias_mode = wv.bias ? TG_BIAS_ROW : TG_BIAS_NONE;
  p.alpha = 1.f;
  p.err = d_err;
  launch_gemm(P, sa, sb, p, false, "tapgemm:vt",
              wv.cin, 2.0 * (1.0 * C * wv.cin + 1.0 * B * ntok * wv.cin + 1.0 * B * C * ntok));
  return vt;
}

Act Engine::attention(Plan& P, const Act& q, const Act& k, const Act& vt, int B, int Nq, int Nk, int heads, int d,
                      int kv_batch) {
  if (d == FA_D) return flash_attention(P, q, k, vt, B, Nq, Nk, heads, kv_batch);
  I2IT_CHECK(d % 64 == 0 && (d <= 256 || d % 256 == 0), "attention: head dim must be a multiple of 64");

  I2IT_CHECK(kv_batch == B || kv_batch == 1, "attention: kv batch must be 1 or B");
  const int C = heads * d, lds = round_up(Nk, 8);
  const long long rows = static_cast<long long>(B) * heads * Nq;
  auto sbuf = alloc_raw(P, static_cast<size_t>(rows) * lds * sizeof(float));
  auto pbuf = alloc_raw(P, static_cast<size_t>(rows) * lds * 2);
  float* S = static_cast<float*>(sbuf.get());
  uint16_t* Pm = static_cast<uint16_t*>(pbuf.get());
  Act out = alloc_act(P, B, 1, Nq, C);
  const int kvb = (kv_batch == B) ? 1 : 0;

  {  // S = alpha * Q K^T   (fp32 logits)
    TmapSpec sa, sb;
    TapGemmParams p;
    std::memset(&p, 0, sizeof p);
    sa.base = q.p;
    sa.dim[0] = d; sa.dim[1] = Nq; sa.dim[2] = heads; sa.dim[3] = B;
    sa.stride[0] = q.ld * 2ull; sa.stride[1] = d * 2ull; sa.stride[2] = 2ull * Nq * q.ld; sa.stride[3] = sa.stride[2];
    sa.box[0] = 64; sa.box[1] = 128;
    fill_strides(sa);
    sb.base = k.p;
    sb.dim[0] = d; sb.dim[1] = Nk; sb.dim[2] = heads; sb.dim[3] = kv_batch;
    sb.stride[0] = k.ld * 2ull; sb.stride[1] = d * 2ull; sb.stride[2] = 2ull * Nk * k.ld; sb.stride[3] = sb.stride[2];
    fill_strides(sb);
    p.tdim[0] = ceil_div(Nq, 128); p.tdim[1] = heads; p.tdim[2] = B; p.tdim[3] = 1;
    p.box[0] = 128; p.box[1] = 1; p.box[2] = 1; p.box[3] = 1;
    p.ext[0] = Nq; p.ext[1] = heads; p.ext[2] = B; p.ext[3] = 1;
    p.a_mul[0] = 128; p.a_mul[1] = 1; p.a_mul[2] = 1;
    p.b_mul[0] = 1; p.b_mul[1] = kvb; p.b_mul[2] = 0;
    const long long m_tiles = 1ll * p.tdim[0] * heads * B;
    p.N = Nk;
    p.BN = pick_bn(m_tiles, Nk, false);
    p.n_tiles = ceil_div(Nk, p.BN);
    sb.box[0] = 64; sb.box[1] = p.BN;
    p.num_taps = 1;
    p.kchunks = d / 64;
    p.idesc = make_idesc(dtype, p.BN);
    p.out = S;
    p.out_fp32 = 1;
    p.ostride[0] = lds; p.ostride[1] = static_cast<long long>(Nq) * lds; p.ostride[2] = static_cast<long long>(heads) * Nq * lds;
    p.ocol = 1;
    p.alpha = 1.0f / sqrtf(static_cast<float>(d));
    p.err = d_err;
    launch_gemm(P, sa, sb, p, false, "tapgemm:attn_qk", d,
                2.0 * B * heads * (1.0 * Nq * d + 1.0 * Nk * d) + 4.0 * rows * Nk);
  }
  {  // P = softmax(S)
    const int dt = dtype;
    if (Nk > 4096) {
      add_op(P, [=](cudaStream_t st) {
        DISPATCH_T(dt, (launch_k(softmax_long_kernel<T>, dim3(static_cast<unsigned>(rows)), dim3(256), 0, st, 0, S, lds, reinterpret_cast<T*>(Pm),
                                                                                          lds, Nk, lds)));
      }, "softmax", 0, 6.0 * rows * Nk);
    } else if (Nk > 1024) {
      add_op(P, [=](cudaStream_t st) {
        DISPATCH_T(dt, (launch_k(softmax_kernel<T, 128>, dim3(static_cast<unsigned>(rows)), dim3(128), 0, st, 0, S, lds, reinterpret_cast<T*>(Pm), lds,
                                                                                          rows, Nk, lds)));
      }, "softmax", 0, 6.0 * rows * Nk);
    } else {
      add_op(P, [=](cudaStream_t st) {
        DISPATCH_T(dt, (launch_k(softmax_kernel<T, 32>, dim3(static_cast<unsigned>((rows + 3) / 4)), dim3(128), 0, st, 0,
                           S, lds, reinterpret_cast<T*>(Pm), lds, rows, Nk, lds)));
      }, "softmax", 0, 6.0 * rows * Nk);
    }
  }
  {  // O = P V   (V given transposed: [kvB][C][ldv])
    TmapSpec sa, sb;
    TapGemmParams p;
    std::memset(&p, 0, sizeof p);
    sa.base = Pm;
    sa.dim[0] = Nk; sa.dim[1] = Nq; sa.dim[2] = heads; sa.dim[3] = B;
    sa.stride[0] = lds * 2ull; sa.stride[1] = 2ull * Nq * lds; sa.stride[2] = 2ull * heads * Nq * lds; sa.stride[3] = sa.stride[2];
    sa.box[0] = 64; sa.box[1] = 128;
    fill_strides(sa);
    const int ldv = vt.ld;
    sb.base = vt.p;
    sb.dim[0] = Nk; sb.dim[1] = d; sb.dim[2] = heads; sb.dim[3] = kv_batch;
    sb.stride[0] = ldv * 2ull; sb.stride[1] = 2ull * d * ldv; sb.stride[2] = 2ull * C * ldv; sb.stride[3] = sb.stride[2];
    fill_strides(sb);
    p.tdim[0] = ceil_div(Nq, 128); p.tdim[1] = heads; p.tdim[2] = B; p.tdim[3] = 1;
    p.box[0] = 128; p.box[1] = 1; p.box[2] = 1; p.box[3] = 1;
    p.ext[0] = Nq; p.ext[1] = heads; p.ext[2] = B; p.ext[3] = 1;
    p.a_mul[0] = 128; p.a_mul[1] = 1; p.a_mul[2] = 1;
    p.b_mul[0] = 1; p.b_mul[1] = kvb; p.b_mul[2] = 0;
    const long long m_tiles = 1ll * p.tdim[0] * heads * B;
    p.N = d;
    p.BN = std::min(d, 256);
    p.n_tiles = ceil_div(d, p.BN);
    sb.box[0] = 64; sb.box[1] = p.BN;
    p.num_taps = 1;
    p.kchunks = ceil_div(Nk, 64);
    p.idesc = make_idesc(dtype, p.BN);
    p.out = out.p;
    p.ostride[0] = out.ld; p.ostride[1] = d; p.ostride[2] = static_cast<long long>(Nq) * out.ld;
    p.ocol = 1;
    p.alpha = 1.f;
    p.err = d_err;
    launch_gemm(P, sa, sb, p, false, "tapgemm:attn_pv", Nk,
                2.0 * (1.0 * rows * Nk + 1.0 * B * heads * Nk * d + 1.0 * rows * d));
  }
  return out;
}

Act Engine::flash_attention(Plan& P, const Act& q, const Act& k, const Act& vt, int B, int Nq, int Nk, int heads, int kv_batch,
                            bool causal) {
  I2IT_CHECK(kv_batch == B || kv_batch == 1, "attention: kv batch must be 1 or B");
  const int d = FA_D, C = heads * d;
  Act out = alloc_act(P, B, 1, Nq, C);
  TmapSpec sq, sk, sv;
  sq.base = q.p;
  sq.dim[0] = d; sq.dim[1] = Nq; sq.dim[2] = heads; sq.dim[3] = B;
  sq.stride[0] = q.ld * 2ull; sq.stride[1] = d * 2ull; sq.stride[2] = 2ull * Nq * q.ld; sq.stride[3] = sq.stride[2];
  sq.box[0] = 64; sq.box[1] = FA_BM;
  fill_strides(sq);
  sk.base = k.p;
  sk.dim[0] = d; sk.dim[1] = Nk; sk.dim[2] = heads; sk.dim[3] = kv_batch;
  sk.stride[0] = k.ld * 2ull; sk.stride[1] = d * 2ull; sk.stride[2] = 2ull * Nk * k.ld; sk.stride[3] = sk.stride[2];
  sk.box[0] = 64; sk.box[1] = FA_BN;
  fill_strides(sk);
  const int ldv = vt.ld;
  sv.base = vt.p;
  sv.dim[0] = Nk; sv.dim[1] = d; sv.dim[2] = heads; sv.dim[3] = kv_batch;
  sv.stride[0] = ldv * 2ull; sv.stride[1] = 2ull * d * ldv; sv.stride[2] = 2ull * C * ldv; sv.stride[3] = sv.stride[2];
  sv.box[0] = FA_BN; sv.box[1] = d;
  fill_strides(sv);
  FlashParams fp;
  std::memset(&fp, 0, sizeof fp);
  fp.Nq = Nq; fp.Nk = Nk; fp.heads = heads; fp.B = B;
  fp.q_tiles = ceil_div(Nq, FA_BM);
  fp.kv_bmul = (kv_batch == B) ? 1 : 0;
  fp.scale_log2e = (1.0f / sqrtf(static_cast<float>(d))) * 1.4426950408889634f;
  fp.out = out.p;
  fp.ldo = out.ld;
  fp.idesc = make_idesc(dtype, FA_BN);
  fp.err = d_err;
  fp.causal = causal ? 1 : 0;
  const CUtensorMap tq = encode_tmap(sq, dtype), tk = encode_tmap(sk, dtype), tv = encode_tmap(sv, dtype);
  const int grid = fp.q_tiles * heads * B, dt = dtype;
  char shp[96];
  snprintf(shp, sizeof shp, "B=%d h=%d Nq=%d Nk=%d d=%d", B, heads, Nq, Nk, d);
  add_op(P, [=](cudaStream_t st) {
    DISPATCH_T(dt, (launch_k(flash_attn_kernel<T>, dim3(grid), dim3(FA_THREADS), FA_SMEM, st, 0, tq, tk, tv, fp)));
  }, "flash_attn", 4.0 * B * heads * Nq * Nk * d, 2.0 * (2.0 * B * Nq * C + 2.0 * kv_batch * Nk * C), shp);
  return out;
}

// ---------------------------------------------------------------------------------------------
// executor
// ---------------------------------------------------------------------------------------------
void Engine::set_text(const void* text, int text_batch, cudaStream_t st) {
  I2IT_CHECK(finalized_, "i2it_finalize_weights must be called before i2it_set_text");
  I2IT_CHECK(text != nullptr && text_batch > 0, "i2it_set_text: null text embedding");
  auto& slot = textkv_[text_batch];
  if (!slot) {
    slot.reset(new TextKV());
    slot->text_batch = text_batch;
    build_text_kv(*slot);
  }
  TextKV& T = *slot;
  T.plan.io.text = text;
  nvtxRangePushA("i2it:text_kv");
  for (auto& op : T.plan.ops) op(st);
  nvtxRangePop();
  I2IT_CUDA(cudaGetLastError());
  T.filled = true;
}

// CLIP text tower on the engine (SURVEY 8f #1; transformers models/clip/modeling_clip.py CLIPTextTransformer.forward): token +
// position embeddings, pre-LN transformer layers with CAUSAL self-attention (16 heads x 64 for SD-Turbo's OpenCLIP-H tower) and a
// GELU MLP, final LayerNorm -> last_hidden_state, i.e. `text_encoder(tokens)[0]` of /root/reference/src/pix2pix_turbo.py:190-196.
// Same kernels as the image path: tapgemm (fused q|k projection, V^T projection with row bias, GELU in the fc1 epilogue, residual
// adds in the out_proj / fc2 epilogues), flash_attn with the causal flag, layernorm.
void Engine::encode_text(const int* tokens, int batch, void* out, cudaStream_t st) {
  I2IT_CHECK(finalized_, "i2it_finalize_weights must be called before i2it_encode_text");
  I2IT_CHECK(tokens && out && batch > 0, "i2it_encode_text: bad arguments");
  I2IT_CHECK(has_text_encoder(), "no text_encoder.* weights were registered (i2it_set_weight)");
  auto& slot = textenc_[batch];
  if (!slot) {
    slot.reset(new Plan());
    Plan& P = *slot;
    const std::string te = "text_encoder.text_model";
    const WT& tok = raw(te + ".embeddings.token_embedding", "weight");
    const WT& pos = raw(te + ".embeddings.position_embedding", "weight");
    const int C = static_cast<int>(tok.shape[1]), vocab = static_cast<int>(tok.shape[0]), ntok = static_cast<int>(pos.shape[0]);
    I2IT_CHECK(C % 64 == 0 && C <= 1280, "text encoder width must be a multiple of 64 (64-wide heads) and <= 1280");
    const int heads = cfg.text_heads > 0 ? cfg.text_heads : C / 64;
    I2IT_CHECK(heads * 64 == C, "text encoder: head_dim must be 64");
    const int act = cfg.text_act == 1 ? TG_ACT_QUICKGELU : TG_ACT_GELU;
    int layers = 0;
    while (has(te + ".encoder.layers." + std::to_string(layers) + ".layer_norm1.weight")) ++layers;
    I2IT_CHECK(layers > 0, "text encoder: no layers found");
    Act x = alloc_act(P, batch, 1, ntok, C);
    {
      const long long total = static_cast<long long>(batch) * ntok * (C / 8);
      uint16_t* xp = x.p;
      const float* tp = tok.d;
      const float* pp = pos.d;
      const int dt = dtype;
      Plan* plan = &P;
      add_op(P, [=](cudaStream_t s2) {
        DISPATCH_T(dt, (launch_k(clip_embed_kernel<T>, dim3(ceil_div(total, 256)), dim3(256), 0, s2, 0,
                           reinterpret_cast<const int*>(plan->io.x), tp, pp, reinterpret_cast<T*>(xp), C, ntok, vocab, total)));
      }, "clip_embed", 0, 2.0 * total * 8 * 3);
    }
    for (int l = 0; l < layers; ++l) {
      const std::string L = te + ".encoder.layers." + std::to_string(l);
      Act n = layer_norm(P, x, norm(L + ".layer_norm1"));
      Act qk = linear(P, n, prep(L + ".qk", {L + ".self_attn.q_proj", L + ".self_attn.k_proj"}));
      Act vt = vt_proj(P, n, batch, ntok, prep(L + ".self_attn.v_proj", {L + ".self_attn.v_proj"}));
      Act a = flash_attention(P, qk.slice(0, C), qk.slice(C, C), vt, batch, ntok, ntok, heads, batch, /*causal=*/true);
      a.N = batch; a.H = 1; a.W = ntok;
      x = linear(P, a, prep(L + ".self_attn.out_proj", {L + ".self_attn.out_proj"}), &x);
      Act m = layer_norm(P, x, norm(L + ".layer_norm2"));
      Act h = linear(P, m, prep(L + ".mlp.fc1", {L + ".mlp.fc1"}), nullptr, act);
      x = linear(P, h, prep(L + ".mlp.fc2", {L + ".mlp.fc2"}), &x);
    }
    layer_norm(P, x, norm(te + ".final_layer_norm"), /*to_io_out=*/true);
    P.keep.push_back(x.hold);
    flush_prep();
    I2IT_CUDA(cudaDeviceSynchronize());
  }
  Plan& P = *slot;
  P.io.x = tokens;
  P.io.out = out;
  nvtxRangePushA("i2it:clip_text_encoder");
  for (auto& op : P.ops) op(st);
  nvtxRangePop();
  I2IT_CUDA(cudaGetLastError());
}

void Engine::forward(const IO& io_in, int B, int H, int W, int direction, int text_batch, cudaStream_t st) {
  I2IT_CHECK(H % 8 == 0 && W % 8 == 0 && H > 0 && W > 0, "H and W must be positive multiples of 8 (as the reference CLIs crop them)");
  I2IT_CHECK(B > 0 && (text_batch == 1 || text_batch == B), "text_batch must be 1 or batch");
  IO io = io_in;
  const int io_mode = (io.x_u8 ? IO_U8_IN : 0) | (io.out_u8 ? IO_U8_OUT : 0);
  I2IT_CHECK((io.x || io.x_u8) && io.eps && (io.out || io.out_u8), "null input/output pointer");
  const bool text_cached = io.text == nullptr;
  if (text_cached) {
    auto it = textkv_.find(text_batch);
    I2IT_CHECK(it != textkv_.end() && it->second->filled,
               "text_emb == NULL: call i2it_set_text first (and again after every i2it_finalize_weights)");
  }
  Plan* P = plan_for(B, H, W, direction, text_batch, text_cached, io_mode);
  if (io_mode & IO_U8_OUT) io.out = P->u8_out_tmp;
  P->io = io;
  last_plan_ = P;
  if (cfg.use_cuda_graph) {
    // replay on the engine's own stream, ordered after/before the caller's stream with events
    I2IT_CUDA(cudaEventRecord(ev_in_, st));
    I2IT_CUDA(cudaStreamWaitEvent(gstream_, ev_in_, 0));
    cudaGraphExec_t ge = nullptr;
    for (auto& g : P->graphs) if (g.first == io) ge = g.second;
    if (!ge) {
      // pointers are baked into the captured launches: one graph per distinct IO set (the torch allocator recycles blocks,
      // so a steady-state loop hits this cache)
      if (P->graphs.size() >= 8) { cudaGraphExecDestroy(P->graphs.front().second); P->graphs.erase(P->graphs.begin()); }
      cudaGraph_t g = nullptr;
      I2IT_CUDA(cudaStreamBeginCapture(gstream_, cudaStreamCaptureModeThreadLocal));
      for (auto& op : P->ops) op(gstream_);
      I2IT_CUDA(cudaStreamEndCapture(gstream_, &g));
      I2IT_CUDA(cudaGraphInstantiate(&ge, g, 0));
      cudaGraphDestroy(g);
      P->graphs.emplace_back(io, ge);
    }
    nvtxRangePushA("i2it:forward(graph)");
    I2IT_CUDA(cudaGraphLaunch(ge, gstream_));
    nvtxRangePop();
    I2IT_CUDA(cudaEventRecord(ev_out_, gstream_));
    I2IT_CUDA(cudaStreamWaitEvent(st, ev_out_, 0));
  } else {
    size_t next_range = 0;
    bool open = false;
    for (size_t i = 0; i < P->ops.size(); ++i) {
      if (next_range < P->ranges.size() && P->ranges[next_range].first == i) {   // NVTX: vae_encode / unet / ddpm_step / vae_decode
        if (open) nvtxRangePop();
        nvtxRangePushA((std::string("i2it:") + P->ranges[next_range].second).c_str());
        open = true;
        ++next_range;
      }
      P->ops[i](st);
      if (sync_each) {   // I2IT_SYNC_EACH=1 (debugging): attribute an asynchronous fault to the launch that caused it
        const cudaError_t e = cudaStreamSynchronize(st);
        if (e != cudaSuccess)
          throw Error("launch " + std::to_string(i) + " (" + P->meta[i].kind + " " + P->meta[i].shape + "): " + cudaGetErrorString(e));
      }
    }
    if (open) nvtxRangePop();
    I2IT_CUDA(cudaGetLastError());
  }
  if (trace_on) dump_trace(*P, st);
}

// I2IT_TRACE=1: per GEMM launch, the median over CTAs of each phase stamp relative to the CTA's entry stamp (SM cycles).
// slots: 1 prologue done | 2 first tile's loads issued | 3 all loads issued | 4 first operands landed | 5 first tile's MMAs
// issued | 6 all MMAs issued | 7 first bias slice staged | 8 first accumulator ready | 9 first tile stored | 10 all tiles
// stored | 11 CTA joined | 12 TMEM freed
void Engine::dump_trace(Plan& P, cudaStream_t st) {
  I2IT_CUDA(cudaStreamSynchronize(st));
  I2IT_CUDA(cudaStreamSynchronize(gstream_));
  int idx = 0;
  for (auto& t : P.traces) {
    std::vector<unsigned long long> h(static_cast<size_t>(t.grid) * 16);
    I2IT_CUDA(cudaMemcpy(h.data(), t.buf, h.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    std::string line = "TRACE " + std::to_string(idx++) + " " + t.what + " |";
    for (int sl = 1; sl <= 12; ++sl) {
      std::vector<long long> d;
      for (int c = 0; c < t.grid; ++c)
        if (h[c * 16 + sl] && h[c * 16]) d.push_back(static_cast<long long>(h[c * 16 + sl] - h[c * 16]));
      if (d.empty()) { line += " -"; continue; }
      std::sort(d.begin(), d.end());
      line += " " + std::to_string(d[d.size() / 2]);
      if (sl == 12) line += " max " + std::to_string(d.back());
    }
    fprintf(stderr, "%s\n", line.c_str());
  }
}

// Per-launch device timing of the last forward's plan (CUDA events around every op, `reps` passes, averaged).
std::string Engine::profile_json(int reps, cudaStream_t st) {
  I2IT_CHECK(last_plan_ != nullptr, "profile: run a forward first");
  Plan& P = *last_plan_;
  const size_t n = P.ops.size();
  std::vector<cudaEvent_t> ev(n + 1);
  for (auto& e : ev) I2IT_CUDA(cudaEventCreate(&e));
  std::vector<double> ms(n, 0.0);
  for (int r = 0; r < reps; ++r) {
    I2IT_CUDA(cudaEventRecord(ev[0], st));
    for (size_t i = 0; i < n; ++i) { P.ops[i](st); I2IT_CUDA(cudaEventRecord(ev[i + 1], st)); }
    I2IT_CUDA(cudaStreamSynchronize(st));
    for (size_t i = 0; i < n; ++i) { float t = 0; I2IT_CUDA(cudaEventElapsedTime(&t, ev[i], ev[i + 1])); ms[i] += t / reps; }
  }
  for (auto& e : ev) cudaEventDestroy(e);
  std::string js = "[";
  char buf[512];
  for (size_t i = 0; i < n; ++i) {
    const OpMeta& m = P.meta[i];
    snprintf(buf, sizeof buf, "%s{\"i\":%zu,\"kind\":\"%s\",\"ms\":%.6f,\"flops\":%.6g,\"bytes\":%.6g,\"shape\":\"%s\"}", i ? "," : "", i,
             m.kind.c_str(), ms[i], m.flops, m.bytes, m.shape.c_str());
    js += buf;
  }
  return js + "]";
}

__global__ void stage_to_nchw_f32_kernel(const uint16_t* x, int ld, int C, long long HW, long long total, float* out,
                                         int is_bf16) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;   // over N*C*HW (NCHW order)
  if (i >= total) return;
  const long long p = i % HW;
  const long long r = i / HW;
  const int c = static_cast<int>(r % C);
  const long long n = r / C;
  const uint16_t v = x[(n * HW + p) * ld + c];
  out[i] = is_bf16 ? __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(&v))
                   : __half2float(*reinterpret_cast<const __half*>(&v));
}

void Engine::read_stage(const std::string& name_in, float* dst, size_t dst_elems, int dims[4]) {
  I2IT_CHECK(last_plan_ != nullptr, "no forward has run yet");
  // "name@i" selects image i of the stage (large-batch stages do not fit a test's scratch buffer)
  std::string name = name_in;
  int pick = -1;
  const size_t at = name.find('@');
  if (at != std::string::npos) { pick = atoi(name.c_str() + at + 1); name = name.substr(0, at); }
  auto it = last_plan_->stages.find(name);
  I2IT_CHECK(it != last_plan_->stages.end(), "unknown stage '" + name + "' (was keep_stages set?)");
  const Act& a = it->second;
  I2IT_CHECK(pick < a.N, "read_stage: image index out of range");
  const int n = pick >= 0 ? 1 : a.N;
  dims[0] = n; dims[1] = a.C; dims[2] = a.H; dims[3] = a.W;
  const long long HW = static_cast<long long>(a.H) * a.W, total = HW * a.C * n;
  I2IT_CHECK(static_cast<size_t>(total) <= dst_elems, "read_stage: destination too small");
  I2IT_CUDA(cudaDeviceSynchronize());
  const uint16_t* src = a.p + (pick >= 0 ? static_cast<long long>(pick) * a.img() : 0);
  stage_to_nchw_f32_kernel<<<ceil_div(total, 256), 256>>>(src, a.ld, a.C, HW, total, dst, dtype == DT_BF16);
  I2IT_CUDA(cudaDeviceSynchronize());
}

}  // namespace i2it
