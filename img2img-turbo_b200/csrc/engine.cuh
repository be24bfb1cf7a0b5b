// Engine: weight store, load-time fold, plan builder (the model graph) and executor behind the C ABI.
#pragma once
#include <cmath>
#include <cstring>
#include <functional>
#include <map>
#include <memory>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/i2it.h"
#include "kernels.cuh"
#include "prep.cuh"
#include "tapgemm.cuh"
#include "flash.cuh"
#include "tapgemm2.cuh"

namespace i2it {

// ---------------------------------------------------------------------------------------------
// TMA tensor-map encoding (driver entry point fetched through the runtime: no libcuda link dependency)
// ---------------------------------------------------------------------------------------------
struct TmapSpec {
  const void* base = nullptr;
  uint64_t dim[5] = {1, 1, 1, 1, 1};
  uint64_t stride[4] = {16, 16, 16, 16};   // bytes, dims 1..4
  uint32_t box[5] = {1, 1, 1, 1, 1};
};
CUtensorMap encode_tmap(const TmapSpec& s, int dtype);

// ---------------------------------------------------------------------------------------------
// workspace pool (plan-build time only; execution never allocates)
// ---------------------------------------------------------------------------------------------
struct Pool {
  std::vector<std::pair<void*, size_t>> blocks;
  std::multimap<size_t, void*> free_;
  size_t total = 0;
  ~Pool();
  void* get(size_t bytes, size_t* actual);
  void* get_fresh(size_t bytes);   // never recycled (zero-padded small-channel tensors must stay clean at run time)
  void put(void* p, size_t bytes) { free_.emplace(bytes, p); }
};

// GroupNorm partial statistics written by the epilogue of the GEMM that PRODUCED a tensor (see TapGemmParams::gn_part):
// [phases][images][slots_per_image][C / red] x (sum, sum of squares), fp32
struct GnPart {
  std::shared_ptr<void> hold;
  float* buf = nullptr;
  int red = 2, slots_per_image = 0, C = 0, phases = 1, images = 0;
};

struct Act {                       // NHWC view, 2-byte elements
  std::shared_ptr<void> hold;
  uint16_t* p = nullptr;
  int N = 0, H = 0, W = 0, C = 0, ld = 0;
  std::shared_ptr<GnPart> gn;      // statistics of this (whole) tensor, if its producer computed them
  long long img() const { return static_cast<long long>(H) * W * ld; }
  long long rows() const { return static_cast<long long>(N) * H * W; }
  Act as_rows() const { Act a = *this; a.W = static_cast<int>(rows()); a.N = 1; a.H = 1; return a; }
  Act slice(int c0, int c) const { Act a = *this; a.p = p + c0; a.C = c; a.gn = nullptr; return a; }
};

struct PW {                        // prepared (folded, re-laid-out) weight: [taps][rows][cin_pad] + fp32 bias
  uint16_t* w = nullptr;
  float* bias = nullptr;
  int rows = 0, cin = 0, cin_pad = 0, taps = 1;
};
// ---- kernel launch for plan ops: `cluster` > 0 adds a (cluster,1,1) cluster dimension
template <typename... KA, typename... A>
inline void launch_k(void (*kern)(KA...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, int cluster, A&&... args) {
  cudaLaunchConfig_t cfg;
  std::memset(&cfg, 0, sizeof cfg);
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  unsigned n = 0;
  if (cluster > 0) {
    at[n].id = cudaLaunchAttributeClusterDimension;
    at[n].val.clusterDim.x = cluster; at[n].val.clusterDim.y = 1; at[n].val.clusterDim.z = 1;
    ++n;
  }
  cfg.attrs = at; cfg.numAttrs = n;
  cudaLaunchKernelEx(&cfg, kern, std::forward<A>(args)...);
}

struct NormW { const float* g = nullptr; const float* b = nullptr; int C = 0; };

struct IO {
  const void* x = nullptr; const void* text = nullptr; const void* eps = nullptr; const void* noise = nullptr;
  float r = 1.f; void* out = nullptr; void* out_latent = nullptr;
  const void* x_u8 = nullptr; void* out_u8 = nullptr;   // uint8 HWC boundary (i2it_forward_u8): x / out then point at internal buffers
  int in_mode = 0;                                      // u8 input transform (see pack_input_im2col_u8_kernel)
  int pad_ = 0;
  bool operator==(const IO& o) const { return std::memcmp(this, &o, sizeof(IO)) == 0; }
};
enum IoMode : int { IO_U8_IN = 1, IO_U8_OUT = 2 };

struct OpMeta {                  // bookkeeping for i2it_profile / bench roofline accounting
  std::string kind;              // "tapgemm:conv3x3", "gn_apply", ...
  double flops = 0, bytes = 0;   // ALGORITHMIC work of the launch (2*M*N*K; unique bytes in + out + weights)
  std::string shape;
};

struct Plan {
  Pool pool;                                           // declared first: destroyed last
  std::vector<std::function<void(cudaStream_t)>> ops;  // one kernel launch each
  std::vector<OpMeta> meta;                            // parallel to ops
  std::map<std::string, Act> stages;
  struct Trace { unsigned long long* buf; int grid; std::string what; };
  std::vector<Trace> traces;                           // I2IT_TRACE=1 only
  std::vector<std::shared_ptr<void>> keep;
  std::vector<int> key;                                // (B, H, W, direction, text_batch, text_cached, io_mode)
  void* u8_out_tmp = nullptr;                          // NCHW image the last conv writes when the caller wants uint8 HWC
  int* gn_counter = nullptr;                           // per-image tickets of the GroupNorm last-block reductions (zero between launches)
  std::vector<std::pair<size_t, const char*>> ranges;  // (first op index, name): NVTX stage ranges of the eager path
  IO io;
  std::vector<std::pair<IO, cudaGraphExec_t>> graphs;  // small cache: one instantiated graph per distinct IO pointer set
  ~Plan() { for (auto& g : graphs) cudaGraphExecDestroy(g.second); }
};

struct ConvOpts {
  int ksize = 3, stride = 1;
  bool asym = false;             // VAE Downsample2D: F.pad(0,1,0,1) then pad-0 stride-2 conv
  const Act* res = nullptr;
  int act = TG_ACT_NONE;
  const Act* out = nullptr;      // write into this view instead of allocating
  bool out_fp32 = false;
  float alpha = 1.f;
  bool to_io_out_nchw = false;   // final image: write NCHW straight into IO.out
  int bias_mode = -1;            // -1: column bias iff the weight has one
  // second source folded into the same accumulator: out = conv(x) + conv1x1(x2)   (resnet conv_shortcut, decoder skip convs)
  const Act* x2 = nullptr;
  const PW* w2 = nullptr;
  int subpixel_phase = -1;       // >=0: this launch is parity phase (py*2+px) of a fused nearest-2x-upsample + 3x3 conv
  bool gn_out = false;           // the consumer of the output is a GroupNorm: take its statistics in this GEMM's epilogue
  std::shared_ptr<GnPart> gn_share;   // sub-pixel phases 1..3 add to the partial buffer phase 0 created
  long long gn_rows_per_image = 0;    // linear(): rows per image of the flattened token matrix (0: spatial conv)
};

struct WT {                      // raw fp32 tensor of the state dict, on device
  float* d = nullptr;
  std::vector<int64_t> shape;
  long long numel = 0;
};

// cached cross-attention operands of one prompt batch: K [tb*77, C] and V^T [tb][C][80] per transformer block
struct TextKV {
  Plan plan;                                   // declared first: its pool outlives the Acts below
  Act text;
  std::map<std::string, std::pair<Act, Act>> kv;   // transformer-block prefix -> (K, V^T)
  int text_batch = 0;
  bool filled = false;
};

class Engine {
 public:
  explicit Engine(const i2it_config& c);
  ~Engine();
  i2it_config cfg;
  int dtype, num_sms;
  std::string last_error;

  void set_weight(const std::string& key, const void* data, const int64_t* shape, int ndim, int dt, bool is_dev);
  void set_adapter_scale(const std::string& a, float s) { adapter_scale_[a] = s; }
  void finalize(float lw_unet, float lw_vae, float skip_gamma, float twin_r);
  Plan* plan_for(int B, int H, int W, int direction, int text_batch, bool text_cached = false, int io_mode = 0);
  void forward(const IO& io, int B, int H, int W, int direction, int text_batch, cudaStream_t st);
  // cross-attention K / V^T of the prompt, computed once per prompt (i2it_set_text) instead of once per forward
  void set_text(const void* text, int text_batch, cudaStream_t st);
  // CLIP text tower (SURVEY 8f #1): tokens [batch, 77] int32 -> last_hidden_state [batch, 77, hidden] in the handle dtype
  void encode_text(const int* tokens, int batch, void* out, cudaStream_t st);
  bool has_text_encoder() const { return has("text_encoder.text_model.embeddings.token_embedding.weight"); }
  Plan* last_plan() const { return last_plan_; }
  void* canny_workspace(size_t bytes);                            // i2it_canny_u8 scratch, grown on demand
  void read_stage(const std::string& name, float* dst, size_t dst_elems, int dims[4]);

  // ---- op builders (append launches to a plan) ----
  Act alloc_act(Plan& P, int N, int H, int W, int C, int ld = 0, bool zero_persistent = false);
  std::shared_ptr<void> alloc_raw(Plan& P, size_t bytes);
  Act conv(Plan& P, const Act& x, const PW& w, const ConvOpts& o);
  Act linear(Plan& P, const Act& x, const PW& w, const Act* res = nullptr, int act = TG_ACT_NONE, bool gn_out = false,
             const Act* out = nullptr);
  Act group_norm(Plan& P, const Act& x, const NormW& nw, float eps, bool silu);
  int* gn_counters(Plan& P, int images);
  Act layer_norm(Plan& P, const Act& x, const NormW& nw, bool to_io_out = false);
  Act upsample2x(Plan& P, const Act& x) { return upsample_to(P, x, 2 * x.H, 2 * x.W); }
  Act upsample_to(Plan& P, const Act& x, int Ho, int Wo);          // F.interpolate(size=(Ho,Wo), mode="nearest")
  Act pad_even(Plan& P, const Act& x);                               // zero-padded copy with even H and W
  void copy_channels(Plan& P, const Act& src, const Act& dst_slice);
  // V^T[b] = Wv X[b]^T (+ row bias): returns [B][C][ldv] as an Act with N=B,H=1,W=C,ld=ldv (C field = Ntok)
  Act vt_proj(Plan& P, const Act& x_tokens, int B, int ntok, const PW& wv);
  // attention core on projected operands; q/k are column slices of token matrices; returns [B*Nq, heads*d]
  Act attention(Plan& P, const Act& q, const Act& k, const Act& vt, int B, int Nq, int Nk, int heads, int d,
                int kv_batch);
  Act flash_attention(Plan& P, const Act& q, const Act& k, const Act& vt, int B, int Nq, int Nk, int heads, int kv_batch,
                      bool causal = false);

  // ---- weights ----
  bool has(const std::string& key) const;
  const WT& raw(const std::string& name, const char* what) const;   // accepts X.what or X.base_layer.what
  PW prep(const std::string& cache_key, const std::vector<std::string>& names, bool geglu = false,
          float scale = 1.f, const float* bias_add = nullptr);
  PW prep_twin(const std::string& pre, const std::string& cur, float r);
  PW prep_im2col3(const std::string& name);
  PW prep_subpixel(const std::string& name);                       // 16 pre-summed 2x2 taps for upsample2x+conv3x3
  Act conv_up2x(Plan& P, const Act& x, const PW& wsub, const Act* x2, const PW* w2, bool gn_out = false);                        // 3x3 conv over 3 channels as a K=32 single-tap GEMM
  NormW norm(const std::string& name);
  const float* temb_bias(const std::string& resnet_prefix);          // time_emb_proj(silu(emb)) at t=999
  void free_prepared();
  void flush_prep();                                                // run all pending preparation jobs (4-5 launches)
  int prep_launches_ = 0;

  // ---- model graph ----
  Act build_vae_encoder(Plan& P, const std::string& vp, int B, int H, int W, std::vector<Act>& skips, bool u8_in = false);
  Act build_unet(Plan& P, const Act& z, int text_batch, bool text_cached);
  void build_text_kv(struct TextKV& T);
  std::vector<std::string> xformer_prefixes() const;
  void build_vae_decoder(Plan& P, const std::string& vp, const Act& dec_in, std::vector<Act>& skips);
  Act vae_resnet(Plan& P, const std::string& p, const Act& x, const Act* skip = nullptr, const PW* skip_w = nullptr,
                 bool gn_next = true);
  Act vae_attn(Plan& P, const std::string& p, const Act& x);
  // `out`: write the block's output into this view (a channel slice of a pre-allocated concat buffer) instead of a new tensor
  Act unet_resnet(Plan& P, const std::string& p, const Act& x, bool gn_next = false, const Act* out = nullptr);
  Act unet_xformer(Plan& P, const std::string& p, const Act& x, int heads, int text_batch, bool gn_next = false,
                   const Act* out = nullptr);
  void mark(Plan& P, const std::string& name, const Act& a) { if (cfg.keep_stages) P.stages[name] = a; }

  template <typename F> void add_op(Plan& P, F&& f, const char* kind = "misc", double flops = 0, double bytes = 0,
                                    const std::string& shape = "") {
    P.ops.emplace_back(std::forward<F>(f));
    OpMeta m; m.kind = kind; m.flops = flops; m.bytes = bytes; m.shape = shape;
    P.meta.push_back(m);
  }
  // encodes the tensor maps and appends the launch; picks the CTA-pair kernel (tapgemm2) for big conv/linear layers
  void launch_gemm(Plan& P, const TmapSpec& sa, TmapSpec sb, const TapGemmParams& p, bool out_from_io, const char* kind,
                   double k_valid, double bytes, const TmapSpec* sa2 = nullptr, const TmapSpec* sb2 = nullptr,
                   const TmapSpec* shalo = nullptr);
  bool use_pair = true, use_halo = true, trace_on = false, use_tmaout = true, use_gnepi = true, use_splitk = true, use_lean = true, sync_each = false;
  bool tma_eligible(const TapGemmParams& p, bool out_from_io) const;
  std::string profile_json(int reps, cudaStream_t st);
  void dump_trace(Plan& P, cudaStream_t st);
  int pick_bn(long long m_tiles, int N, int step) const;   // step 64 / 128: BN restricted to multiples (TMA-store rounds)

  int* d_err = nullptr;      // device alias of a mapped host word written by the tapgemm watchdog
  int* err_host_ = nullptr;
  cudaStream_t gstream_ = nullptr;          // graphs are captured/replayed here (capture is illegal on the legacy stream)
  cudaEvent_t ev_in_ = nullptr, ev_out_ = nullptr;
  void check_device_error();

 private:
  std::unordered_map<std::string, WT> w_;
  std::unordered_map<std::string, float> adapter_scale_;
  float lw_unet_ = 1.f, lw_vae_ = 1.f, skip_gamma_ = 1.f, twin_r_ = -1.f;
  bool finalized_ = false;
  std::unordered_map<std::string, PW> prepared_;
  std::unordered_map<std::string, float*> prepared_f32_;
  std::vector<void*> prep_allocs_;
  float* emb_act_ = nullptr;
  std::vector<PrepJob> pending_jobs_;
  std::vector<GemvJob> pending_gemv_[3];
  long long pending_blocks_ = 0;
  void fill_fold(PrepJob& j, const std::string& name, float c0 = 1.f, const std::string& other = "", float c1 = 0.f);
  void push_job(PrepJob& j);
  void push_bias_job(float* out, const float* b, const float* add, int cout, int row_off, int half, float c0 = 1.f,
                     const float* b1 = nullptr, float c1 = 0.f);
  std::map<int, std::unique_ptr<struct TextKV>> textkv_;   // by text_batch
  std::map<int, std::unique_ptr<Plan>> textenc_;            // CLIP text tower plans, by batch
  std::map<std::vector<int>, std::unique_ptr<Plan>> plans_;
  Plan* last_plan_ = nullptr;
  void* canny_ws_ = nullptr;
  size_t canny_ws_bytes_ = 0;
  Act text_;                     // staged text embedding while a UNet plan is being built
  TextKV* text_kv_ = nullptr;    // ... or the cached cross-attention operands (text_emb == NULL forwards)

  float adapter_weight(const std::string& name, const std::string& adapter) const;
  void* dmalloc(size_t bytes);
};

}  // namespace i2it
