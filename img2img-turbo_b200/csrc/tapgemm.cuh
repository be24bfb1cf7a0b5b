// tapgemm: the one tensor-core kernel of the path.
//
//   D[m, n] = act( alpha * sum_{tap t} sum_k A_t[m, k] * B_t[n, k]  + bias ) + residual
//
// A_t is a TMA *box* of the activation tensor shifted by the tap's spatial offset, so a 3x3 /
// stride-2 / 1x1 convolution, a linear layer and the attention GEMMs (Q K^T, P V, V^T = W X^T)
// are all the same implicit GEMM.  Zero padding, ragged edges and channel padding come from TMA
// out-of-bounds zero fill, never from materialised copies.
//
// sm_100a structure (one persistent CTA per SM, 192 threads):
//   warp 8        : TMA producer   cp.async.bulk.tensor.5d -> 128B-swizzled smem ring (4 stages)
//   warp 9        : MMA issuer     tcgen05.mma.cta_group::1.kind::f16, M=128, N=BN<=256, K=16
//                                  accumulators in TMEM (2 stages x 256 fp32 columns)
//   warps 0..7    : epilogue       tcgen05.ld 32x32b -> bias/residual/GEGLU/clamp -> global
//   mbarriers     : full/empty per smem stage, tmem_full/tmem_empty per accumulator stage
//
// Replaces (reference call sites): every nn.Conv2d / nn.Linear / SDPA matmul under
// vae.encode / unet(...) / vae.decode at /root/reference/src/pix2pix_turbo.py:198-203, which
// dispatch to cuDNN implicit GEMM, cuBLAS and flash/mem-efficient SDPA in the reference stack.
#pragma once
#include "common.cuh"

namespace i2it {

constexpr int TG_BM = 128;             // rows per tile (= TMEM lanes)
constexpr int TG_BK = 64;              // K elements per stage (= 128 B = one swizzle atom)
constexpr int TG_STAGES = 4;            // stages when the B tile is the full 32 KiB; smaller tiles get more (<= TG_MAX_STAGES)
constexpr int TG_MAX_STAGES = 16;      // small B tiles (BN <= 128) need more stages for the same lookahead in TIME
constexpr int TG_MAX_TAPS = 16;
constexpr int TG_A_STAGE = TG_BM * TG_BK * 2;    // 16 KiB
constexpr int TG_B_STAGE = 256 * TG_BK * 2;      // 32 KiB (BN <= 256)
constexpr int TG_EPI_WARPS = 8;        // TG_EPI_GROUPS warps per TMEM lane quarter: they take the 32-column rounds in turn
constexpr int TG_EPI_GROUPS = TG_EPI_WARPS / 4;
constexpr int TG_EPI_RPW = 8 / TG_EPI_GROUPS;      // rounds per warp at BN = 256
constexpr int TG_BAR_BYTES = 512;
constexpr int TG_BIAS_BYTES = 2 * 256 * 4;       // per-tile bias slice, double-buffered like the accumulators
// Epilogue store staging: each epilogue warp owns ONE TMA box = 32 rows x 64 output columns (128-byte rows, SWIZZLE_128B: the
// 16-byte chunk c of row r lives at r*128 + ((c ^ (r & 7)) << 4)).  A thread holds one accumulator ROW, so direct stores touch 32
// different lines per instruction (r01 trace: ~6000 cycles of LSU transactions per 128x160 tile, the limiter of every
// K <= ~1152 GEMM).  Through the box the thread writes its row with conflict-free st.shared.v4 and ONE elected lane hands the
// 4 KB box to the TMA unit (cp.async.bulk.tensor...global.shared::cta = UTMASTG), which writes full lines and clips ragged edges.
// The residual takes the same road in reverse: coalesced 16-byte global loads (4 rows x 128 B per instruction), transposed
// through the box, added in place.
constexpr int TG_OSTG_WARP = 32 * 128;
constexpr int TG_OSTG_BYTES = TG_EPI_WARPS * TG_OSTG_WARP;
// manual 1024-byte alignment slack of the dynamic smem base: 512 B are budgeted (a full 1 KB would put the CTA over the
// 227 KB limit) and the kernels trap with an error word if the runtime base needs more (it is 1 KB aligned in practice).
constexpr int TG_ALIGN_PAD = 512;
constexpr int TG_SMEM = TG_STAGES * (TG_A_STAGE + TG_B_STAGE) + TG_BAR_BYTES + TG_BIAS_BYTES + TG_OSTG_BYTES + TG_ALIGN_PAD;
// + TMA producer warp + MMA issuer warp.  Register reallocation (setmaxnreg) was tried: with two idle warps completing the third
// warpgroup the epilogue warpgroups can grow to 224 registers while the control warps drop to 64, but ptxas then spills the
// control roles' hoisted parameter loads (0.5..5 KB of spill traffic depending on the split), so it is compiled out
// (TG_REGS_EPI = 0); the epilogue fits in the 168 registers a 10-warp CTA gets with ~40 B of spills per round.
constexpr int TG_REGS_EPI = 0, TG_REGS_CTRL = 64;
constexpr int TG_THREADS = (TG_EPI_WARPS + (TG_REGS_EPI > 0 ? 4 : 2)) * 32;
constexpr int TG_ACC_COLS = 256;       // TMEM columns per accumulator stage

enum TgAct : int { TG_ACT_NONE = 0, TG_ACT_CLAMP1 = 1, TG_ACT_GEGLU = 2, TG_ACT_GELU = 3, TG_ACT_QUICKGELU = 4 };   // 3, 4: CLIP MLP
enum TgBias : int { TG_BIAS_NONE = 0, TG_BIAS_COL = 1, TG_BIAS_ROW = 2 };

struct TapGemmParams {
  // ---- tile space: 4 "row" dims d1..d4 of the A tensor map (d0 is K) ----
  int tdim[4];     // tiles per dim
  int box[4];      // A box extent per dim, prod == 128; row r of a tile = j1 + box0*(j2 + box1*(j3 + box2*j4))
  int ext[4];      // logical extent per dim: row valid iff t*box + j < ext
  int a_mul[4];    // A coordinate(d) = t_d * a_mul[d] + tap_a[tap][d+1]
  int b_mul[3];    // B coordinate(2..4) = t_{2..4} * b_mul + tap_b[tap][1..3]
  int n_tiles, BN, N;
  int num_taps, kchunks;   // kchunks: default K chunks per tap (tap_kc overrides per tap)
  int tap_src[TG_MAX_TAPS]; // 0: (tmA, tmB)   1: (tmA2, tmB2) — a second activation tensor folded into the same accumulator
  int tap_kc[TG_MAX_TAPS];  // K chunks (of 64) for this tap
  int nprim;                // the first nprim taps share kchunks and are walked k-chunk-outer / tap-inner (same
                            // accumulation order in every kernel variant => bit-identical results); the rest follow
  int stages, b_stage;      // smem ring: number of stages and bytes per B stage (sized to the actual tile, <= TG_MAX_STAGES)
  int halo;                 // pair kernel only: 3x3 taps read shifted views of ONE halo tile per k-chunk
  int tap_a[TG_MAX_TAPS][5];
  int tap_b[TG_MAX_TAPS][4];
  uint32_t idesc;
  // ---- epilogue ----
  void* out;
  long long ostride[4];   // elements
  long long ocol;         // element stride between consecutive output columns (1 = contiguous)
  int out_fp32;
  const void* res;        // optional residual, element type == activation type
  long long rstride[4];
  long long rcol;
  const float* bias;
  int bias_mode;
  float alpha;
  int act;
  int* err;               // device error word (watchdog)
  int tma_out;            // 1: 64-column rounds are staged in smem and stored by TMA (I2IT_NO_TMAOUT=1 -> 0: per-thread stores)
  // GroupNorm statistics of the OUTPUT tensor, taken from the staged (rounded) tile: per 32-row slot and per `gn_red` columns,
  // (sum, sum of squares) -> gn_part[(slot0 + m_tile*4 + quarter) * (N/gn_red) + col/gn_red][2]; nullptr = off
  float* gn_part;
  // split-K (1-CTA kernel only): the primary taps' k-chunks are divided over `ksplit` tiles that write fp32 partials
  // `split_ostride` elements apart (splitk_reduce_kernel sums them in a fixed order); secondary taps go with split 0
  int ksplit, kc_per;
  long long split_ostride;
  int gn_red, gn_slot0, gn_mtiles;   // gn_mtiles: m-tiles of the launch (the pair kernel's odd tail tile has no slot)
  int gn_shift;                      // log2(gn_red)
  // tile decode without integer division: magic[i] = floor(2^32 / d_i) + 1 for d = (n_tiles, tdim[0..3]); exact while
  // tile * d < 2^32 (the host refuses larger tile spaces)
  uint32_t magic[5];
  unsigned long long* trace;   // optional (I2IT_TRACE=1): 16 %clock64 stamps per CTA at the phase boundaries, else nullptr
};

// ------------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  return ok;
}
__device__ __forceinline__ uint64_t globaltimer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
// Bounded wait: a protocol bug must surface as a trapped launch with an error word, never as a hung GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int* err, int code) {
  if (mbar_try_wait(bar, parity)) return;
  const uint64_t t0 = globaltimer_ns();
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 0x3ff) == 0 && globaltimer_ns() - t0 > 4000000000ull) {
      if (err) atomicExch(err, code);
      __threadfence_system();
      __trap();
    }
  }
}
__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1,
                                            int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
// TMA store of one box from shared memory (async proxy): the writer threads fence (fence.proxy.async) and sync first
__device__ __forceinline__ void tma_store_5d(const CUtensorMap* tm, uint32_t src, int c0, int c1, int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5, %6}], [%1];"
      ::"l"(reinterpret_cast<uint64_t>(tm)), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// one lane of a fully converged warp (warp-uniform control flow keeps descriptors/addresses in uniform registers)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// register reallocation between warpgroups (all four warps of a warpgroup execute the same instruction)
template <int N> __device__ __forceinline__ void reg_inc() { if (N >= 24) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N >= 24 ? N : 24)); }
template <int N> __device__ __forceinline__ void reg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }

// K-major, 128B-swizzled operand tile: rows of 128 B, 8-row groups 1024 B apart (SBO), start address
// advanced by 32 B per UMMA_K=16 step inside the swizzle atom.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr) {
  uint64_t d = static_cast<uint64_t>((saddr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(1024 >> 4) << 32;   // stride byte offset between 8-row core-matrix groups
  d |= static_cast<uint64_t>(1) << 46;           // descriptor version (sm_100)
  d |= static_cast<uint64_t>(2) << 61;           // SWIZZLE_128B
  return d;
}

// host: instruction descriptor for kind::f16 (A,B fp16 or bf16 K-major, D fp32), M=128, N=bn
inline uint32_t make_idesc(int dtype, int bn) {
  uint32_t fmt = (dtype == DT_BF16) ? 1u : 0u;
  return (1u << 4) | (fmt << 7) | (fmt << 10) | (static_cast<uint32_t>(bn >> 3) << 17) | ((128u >> 4) << 24);
}

__device__ __forceinline__ void sts16(uint32_t saddr, const uint4& u) {
  asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(saddr), "r"(u.x), "r"(u.y), "r"(u.z), "r"(u.w) : "memory");
}
__device__ __forceinline__ uint4 lds16(uint32_t saddr) {
  uint4 u;
  asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(u.x), "=r"(u.y), "=r"(u.z), "=r"(u.w) : "r"(saddr) : "memory");
  return u;
}

// timeline stamp for the diagnostic trace (build with `make TRACE=1`, run with I2IT_TRACE=1; one thread per role writes;
// cycles are per-SM, compare within a CTA only)
__device__ __forceinline__ void tg_stamp(const TapGemmParams& p, int slot) {
#ifdef I2IT_TRACE_BUILD   // `make TRACE=1`: even a never-taken stamp in the issue loops costs ~2 % of a step, so it is compiled out by default
  if (p.trace) p.trace[blockIdx.x * 16 + slot] = static_cast<unsigned long long>(clock64());
#endif
}

struct TileCoord {
  int nt, t[4], split;
};
// x / d with the host's magic number (one IMAD.HI instead of ~20 instructions; the tile loops of all three roles decode a tile
// per iteration and the r02g profile charged 137 of the epilogue's 1460 instructions per tile to these divisions)
__device__ __forceinline__ int fast_div(int x, int d, uint32_t magic) {
  const int q = static_cast<int>(__umulhi(static_cast<uint32_t>(x), magic));      // branch-free: one IMAD.HI + one select
  return d == 1 ? x : q;
}
__device__ __forceinline__ TileCoord decode_tile(const TapGemmParams& p, int tile) {
  TileCoord c;
  int r = fast_div(tile, p.n_tiles, p.magic[0]), q;
  c.nt = tile - r * p.n_tiles;
  q = fast_div(r, p.tdim[0], p.magic[1]); c.t[0] = r - q * p.tdim[0]; r = q;
  q = fast_div(r, p.tdim[1], p.magic[2]); c.t[1] = r - q * p.tdim[1]; r = q;
  q = fast_div(r, p.tdim[2], p.magic[3]); c.t[2] = r - q * p.tdim[2]; r = q;
  q = fast_div(r, p.tdim[3], p.magic[4]); c.t[3] = r - q * p.tdim[3];
  c.split = q;                                   // 0 unless ksplit > 1 (slowest index)
  return c;
}
inline uint32_t make_magic(long long max_dividend, int d) {   // host; 0 = the tile space is too large for the 32-bit magic (caller raises)
  if (d <= 1) return 1u;                                        // unused (fast_div selects x for d == 1)
  if (max_dividend * d >= (1ll << 32)) return 0u;
  return static_cast<uint32_t>((1ull << 32) / static_cast<unsigned>(d)) + 1u;
}

// One 16-column chunk of one accumulator row: alpha, bias, (GEGLU), residual, clamp, single rounding, store.
template <typename T>
__device__ __forceinline__ void epilogue_chunk(const TapGemmParams& p, const uint32_t (&raw)[16], int col0, long long obase,
                                               long long rbase, float rbias, const float* sbias, bool rfast, const uint4& r0,
                                               const uint4& r1) {
  float v[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(raw[i]) * p.alpha;
  if (p.bias_mode == TG_BIAS_COL) {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] += sbias[i];   // smem broadcast; columns >= N hold 0 (staged once per tile)
  } else if (p.bias_mode == TG_BIAS_ROW) {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] += rbias;
  }
  const bool full = (col0 + 16 <= p.N);
  if (p.act == TG_ACT_GEGLU) {
    // interleaved columns (2j, 2j+1) = (h_j, gate_j) -> out column j = h * gelu(gate)
    float o[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) o[i] = v[2 * i] * gelu_erf_f(v[2 * i + 1]);
    T* optr = reinterpret_cast<T*>(p.out) + obase + (col0 >> 1);
    if (p.res) {
      const T* rptr = reinterpret_cast<const T*>(p.res) + rbase + (col0 >> 1);
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] += Elem<T>::to_f(rptr[i]);
    }
    if (full && ((reinterpret_cast<uintptr_t>(optr) & 15) == 0)) {
      uint4 u;
      u.x = Elem<T>::pack(o[0], o[1]); u.y = Elem<T>::pack(o[2], o[3]);
      u.z = Elem<T>::pack(o[4], o[5]); u.w = Elem<T>::pack(o[6], o[7]);
      st16(optr, u);
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i) if (col0 + 2 * i + 1 < p.N) optr[i] = Elem<T>::from_f(o[i]);
    }
    return;
  }
  if (p.act == TG_ACT_GELU) {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = gelu_erf_f(v[i]);
  } else if (p.act == TG_ACT_QUICKGELU) {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = quick_gelu_f(v[i]);
  }
  if (p.res) {
    if (rfast) {
      const uint32_t ru[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float2 f = Elem<T>::unpack(ru[i]);
        v[2 * i] += f.x; v[2 * i + 1] += f.y;
      }
    } else {
      const T* rptr = reinterpret_cast<const T*>(p.res) + rbase + col0 * p.rcol;
#pragma unroll
      for (int i = 0; i < 16; ++i) if (col0 + i < p.N) v[i] += Elem<T>::to_f(rptr[i * p.rcol]);
    }
  }
  if (p.act == TG_ACT_CLAMP1) {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = fminf(fmaxf(v[i], -1.0f), 1.0f);
  }
  if (p.out_fp32) {
    float* optr = reinterpret_cast<float*>(p.out) + obase + col0 * p.ocol;
    if (full && p.ocol == 1 && ((reinterpret_cast<uintptr_t>(optr) & 15) == 0)) {
#pragma unroll
      for (int i = 0; i < 4; ++i)
        *reinterpret_cast<float4*>(optr + 4 * i) = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
    } else {
#pragma unroll
      for (int i = 0; i < 16; ++i) if (col0 + i < p.N) optr[i * p.ocol] = v[i];
    }
  } else {
    T* optr = reinterpret_cast<T*>(p.out) + obase + col0 * p.ocol;
    if (full && p.ocol == 1 && ((reinterpret_cast<uintptr_t>(optr) & 15) == 0)) {
      uint4 u0, u1;
      u0.x = Elem<T>::pack(v[0], v[1]);   u0.y = Elem<T>::pack(v[2], v[3]);
      u0.z = Elem<T>::pack(v[4], v[5]);   u0.w = Elem<T>::pack(v[6], v[7]);
      u1.x = Elem<T>::pack(v[8], v[9]);   u1.y = Elem<T>::pack(v[10], v[11]);
      u1.z = Elem<T>::pack(v[12], v[13]); u1.w = Elem<T>::pack(v[14], v[15]);
      st16(optr, u0);
      st16(optr + 8, u1);
    } else {
#pragma unroll
      for (int i = 0; i < 16; ++i) if (col0 + i < p.N) optr[i * p.ocol] = Elem<T>::from_f(v[i]);
    }
  }
}

// The whole epilogue of one output tile for one thread (= one accumulator row).  Shared by the 1-CTA and the 2-CTA kernels.
// Caller signals tmem_empty afterwards.  Two paths, chosen per launch on the host:
//   * tma_out: 64-column rounds -> this warp's swizzled 4 KB box in smem -> one TMA store per round (see TG_OSTG_WARP);
//     the residual is fetched with coalesced loads before the accumulator wait and added from the box; optional GroupNorm
//     statistics of the rounded output come from the box as well;
//   * direct: each thread stores its own row (fp32 logits, NCHW image, row-bias V^T, channel counts that are not multiples of 64).
// LEAN (compile time): the launch takes the TMA-store path with no activation (every conv / linear of the path except the GEGLU,
// GELU and clamp epilogues) -> the activation branches, the GEGLU rounds and the whole direct path are not compiled in; half the
// code, fewer instruction-cache misses (17 % of the r02g stall samples were no_inst).
template <typename T, bool LEAN>
__device__ __forceinline__ void epilogue_tile(const TapGemmParams& p, const CUtensorMap* tmO, const TileCoord& c, int m_tile,
                                              int row, int warp, int j1, int j2, int j3, int j4, int acc, int aphase,
                                              uint32_t tmem_base, float* s_bias, uint32_t ostg_base, uint32_t tfull_bar_addr,
                                              bool stage_bias, bool stamp = false) {
  const int lane = threadIdx.x & 31;
  const uint32_t ostg_warp = ostg_base + warp * TG_OSTG_WARP;   // this warp's store box, 1024-byte aligned
  const int grp = warp >> 2;                     // which of the two warps sharing this TMEM lane quarter
  const int g1 = c.t[0] * p.box[0] + j1, g2 = c.t[1] * p.box[1] + j2, g3 = c.t[2] * p.box[2] + j3,
            g4 = c.t[3] * p.box[3] + j4;
  const bool row_ok = (g1 < p.ext[0]) && (g2 < p.ext[1]) && (g3 < p.ext[2]) && (g4 < p.ext[3]);
  const long long rbase = p.res ? g1 * p.rstride[0] + g2 * p.rstride[1] + g3 * p.rstride[2] + g4 * p.rstride[3] : 0;
  const int n0 = c.nt * p.BN;

  // stage this tile's bias slice in smem once (a per-chunk global load here stalled the whole epilogue: r01 ncu)
  // (a launch with a single n-tile stages its one slice into both buffers during the first two tiles and then skips this and the
  // barrier: 110 tiles per CTA in the 512x512 convs)
  float* sb = s_bias + acc * 256;
  if (stage_bias) {      // no column bias: zeros, so the rounds add unconditionally (one FFMA: alpha * acc + bias)
    for (int cc = warp * 32 + (threadIdx.x & 31); cc < p.BN; cc += TG_EPI_WARPS * 32)
      sb[cc] = (p.bias_mode == TG_BIAS_COL && n0 + cc < p.N) ? p.bias[n0 + cc] : 0.f;
    asm volatile("bar.sync 1, %0;" ::"n"(TG_EPI_WARPS * 32) : "memory");   // the epilogue warps only
  }
  if (stamp) tg_stamp(p, 7);
  const uint32_t taddr = tmem_base + (static_cast<uint32_t>((warp & 3) * 32) << 16) + acc * TG_ACC_COLS;
  const bool geglu = !LEAN && p.act == TG_ACT_GEGLU;

  if (LEAN || p.tma_out) {
    // ================= TMA-store path: rounds of 64 OUTPUT columns (64 accumulator columns, 128 for GEGLU) =================
    const int acols = geglu ? 128 : 64;                       // accumulator columns per round
    const int nrounds = p.BN >> (geglu ? 7 : 6);              // host guarantees BN % acols == 0 and N % acols == 0
    const bool res_on = p.res != nullptr && !geglu;
    // Residual prefetch: independent of the accumulator, so it is requested BEFORE the accumulator wait and its latency
    // overlaps the mainloop.  Instruction i loads rows 4i..4i+3 of the warp's 32 (8 lanes x 16 B = one full 128-byte row
    // segment each) -> 4 fully used lines per instruction instead of 32 half-used sectors.
    uint4 rq[8];
    const int lrow = lane >> 3, lch = lane & 7;
    auto load_res = [&](int r) {                             // this warp's residual box of round r -> registers
      const int colg = n0 + 64 * r;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int src_row = 4 * i + lrow;
        const long long rb = __shfl_sync(0xffffffffu, rbase, src_row);
        const int ok = __shfl_sync(0xffffffffu, static_cast<int>(row_ok), src_row);
        rq[i] = make_uint4(0u, 0u, 0u, 0u);
        if (ok && r < nrounds && colg < p.N)
          rq[i] = ld_nc16(reinterpret_cast<const T*>(p.res) + rb + colg + lch * 8);
      }
    };
    if (res_on) load_res(grp);
    mbar_wait(tfull_bar_addr, aphase, p.err, 4);
    tc_fence_after();
    if (stamp) tg_stamp(p, 8);
    const int sw = lane & 7;
#pragma unroll
    for (int k = 0; k < TG_EPI_RPW / 2; ++k) {
      const int r = grp + TG_EPI_GROUPS * k;
      if (r >= nrounds) break;                               // warp-uniform
      const int c0 = acols * r;                              // accumulator column of this round inside the tile
      if (n0 + c0 >= p.N) break;                             // whole round beyond N (last n-tile): nothing to store
      // the previous TMA store out of this box must have finished READING it
      const uint32_t my_row = ostg_warp + lane * 128;
      if (lane == 0) bulk_wait_read0();
      __syncwarp();
      if (res_on) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int rr = 4 * i + lrow;
          sts16(ostg_warp + rr * 128 + ((lch ^ (rr & 7)) << 4), rq[i]);
        }
        __syncwarp();
        if (r + TG_EPI_GROUPS < nrounds) load_res(r + TG_EPI_GROUPS);   // next round's residual: in flight during this round's math
      }
      const int nq = geglu ? 4 : 2;
      // 32 accumulator columns per step, software-pipelined: the TMEM load of step q+1 is in flight during the math of step q
      // (tcgen05.wait::ld waits for ALL outstanding loads, so the next load is issued right after the wait)
      uint32_t xa0[16], xa1[16], xb0[16], xb1[16];       // two 32-column register buffers
      auto step = [&](int q, const uint32_t (&raw0)[16], const uint32_t (&raw1)[16]) {
        const uint32_t sbq_s = smem_u32(sb + c0 + 32 * q);      // 16-byte aligned: the bias slice comes in as ld.shared.v4
        const float* sbq = sb + c0 + 32 * q;
        if (geglu) {
          // interleaved accumulator columns (2j, 2j+1) = (h_j, gate_j) -> output column j = h * gelu(gate): 32 -> 16 columns
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const uint32_t* raw = h ? raw1 : raw0;
            float o[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float hv = __uint_as_float(raw[2 * i]) * p.alpha + sbq[16 * h + 2 * i];
              const float gv = __uint_as_float(raw[2 * i + 1]) * p.alpha + sbq[16 * h + 2 * i + 1];
              o[i] = hv * gelu_erf_f(gv);
            }
            uint4 u;
            u.x = Elem<T>::pack(o[0], o[1]); u.y = Elem<T>::pack(o[2], o[3]);
            u.z = Elem<T>::pack(o[4], o[5]); u.w = Elem<T>::pack(o[6], o[7]);
            sts16(my_row + (((2 * q + h) ^ sw) << 4), u);
          }
        } else {
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const uint32_t* raw = h ? raw1 : raw0;
            float v[16];
#pragma unroll
            for (int i4 = 0; i4 < 4; ++i4) {               // v = alpha * acc + bias (zeros staged when there is no column bias)
              const uint4 bq = lds16(sbq_s + (16 * h + 4 * i4) * 4);
              v[4 * i4] = fmaf(__uint_as_float(raw[4 * i4]), p.alpha, __uint_as_float(bq.x));
              v[4 * i4 + 1] = fmaf(__uint_as_float(raw[4 * i4 + 1]), p.alpha, __uint_as_float(bq.y));
              v[4 * i4 + 2] = fmaf(__uint_as_float(raw[4 * i4 + 2]), p.alpha, __uint_as_float(bq.z));
              v[4 * i4 + 3] = fmaf(__uint_as_float(raw[4 * i4 + 3]), p.alpha, __uint_as_float(bq.w));
            }
            if (!LEAN) {
              if (p.act == TG_ACT_GELU) {
#pragma unroll
                for (int i = 0; i < 16; ++i) v[i] = gelu_erf_f(v[i]);
              } else if (p.act == TG_ACT_QUICKGELU) {
#pragma unroll
                for (int i = 0; i < 16; ++i) v[i] = quick_gelu_f(v[i]);
              }
            }
            const uint32_t a0 = my_row + (((4 * q + 2 * h) ^ sw) << 4), a1 = my_row + (((4 * q + 2 * h + 1) ^ sw) << 4);
            if (res_on) {
              const uint4 r0 = lds16(a0), r1 = lds16(a1);
              const uint32_t ru[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const float2 f = Elem<T>::unpack(ru[i]);
                v[2 * i] += f.x; v[2 * i + 1] += f.y;
              }
            }
            if (!LEAN && p.act == TG_ACT_CLAMP1) {
#pragma unroll
              for (int i = 0; i < 16; ++i) v[i] = fminf(fmaxf(v[i], -1.0f), 1.0f);
            }
            uint4 u0, u1;
            u0.x = Elem<T>::pack(v[0], v[1]);   u0.y = Elem<T>::pack(v[2], v[3]);
            u0.z = Elem<T>::pack(v[4], v[5]);   u0.w = Elem<T>::pack(v[6], v[7]);
            u1.x = Elem<T>::pack(v[8], v[9]);   u1.y = Elem<T>::pack(v[10], v[11]);
            u1.z = Elem<T>::pack(v[12], v[13]); u1.w = Elem<T>::pack(v[14], v[15]);
            if (p.gn_part && !row_ok) u0 = u1 = make_uint4(0u, 0u, 0u, 0u);   // clipped by the TMA store; keeps the statistics clean
            sts16(a0, u0);
            sts16(a1, u1);
          }
        }
      };
      tc_ld16(taddr + c0, xa0); tc_ld16(taddr + c0 + 16, xa1);
      tc_wait_ld();
      tc_ld16(taddr + c0 + 32, xb0); tc_ld16(taddr + c0 + 48, xb1);
      step(0, xa0, xa1);
      tc_wait_ld();
      if (!LEAN && nq > 2) { tc_ld16(taddr + c0 + 64, xa0); tc_ld16(taddr + c0 + 80, xa1); }   // warp-uniform (GEGLU rounds)
      step(1, xb0, xb1);
      if (!LEAN && nq > 2) {
        tc_wait_ld();
        tc_ld16(taddr + c0 + 96, xb0); tc_ld16(taddr + c0 + 112, xb1);
        step(2, xa0, xa1);
        tc_wait_ld();
        step(3, xb0, xb1);
      }
      fence_async_smem();                                    // generic-proxy writes -> visible to the TMA unit
      __syncwarp();
      const int ocol0 = geglu ? ((n0 + c0) >> 1) : (n0 + c0);
      if (lane == 0) {                                       // lane 0 holds the box origin: its own row coordinates
        tma_store_5d(tmO, ostg_warp, ocol0, g1, g2, g3, g4);
        bulk_commit();
      }
      if (p.gn_part) {
        // GroupNorm statistics of the tensor just produced, from the ROUNDED values in the box (what the next layer's GroupNorm
        // sees; rows outside the tensor were written as zeros).  Lane (rg, ch) = (lane >> 3, lane & 7) reads the 16-byte chunk
        // ch (8 output columns) of rows rg, rg+4, ..., rg+28: eight independent conflict-free ld.shared.v4 (a quarter warp
        // covers one 128-byte row), per-column-pair sums in registers, then the four row groups are combined by two shuffle
        // steps and lanes 0..7 write one (sum, sum of squares) entry per gn_red columns.  Fixed order, no atomics.
        const int rg = lane >> 3, ch = lane & 7;
        uint4 w[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int rr = 4 * i + rg;
          w[i] = lds16(ostg_warp + rr * 128 + ((ch ^ (rr & 7)) << 4));
        }
        float s2[4] = {0.f, 0.f, 0.f, 0.f}, q2[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const uint32_t ww[4] = {w[i].x, w[i].y, w[i].z, w[i].w};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float2 f = Elem<T>::unpack(ww[j]);
            s2[j] += f.x + f.y;
            q2[j] = fmaf(f.x, f.x, fmaf(f.y, f.y, q2[j]));
          }
        }
        const int red = p.gn_red;                            // 2, 4, 8 or 16 columns per entry (warp-uniform)
        if (red >= 4) { s2[0] += s2[1]; q2[0] += q2[1]; s2[2] += s2[3]; q2[2] += q2[3]; }
        if (red >= 8) { s2[0] += s2[2]; q2[0] += q2[2]; }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if ((red >= 4 && (j & 1)) || (red >= 8 && j)) continue;   // folded above
          s2[j] += __shfl_xor_sync(0xffffffffu, s2[j], 8);  q2[j] += __shfl_xor_sync(0xffffffffu, q2[j], 8);
          s2[j] += __shfl_xor_sync(0xffffffffu, s2[j], 16); q2[j] += __shfl_xor_sync(0xffffffffu, q2[j], 16);
        }
        if (red == 16) { s2[0] += __shfl_xor_sync(0xffffffffu, s2[0], 1); q2[0] += __shfl_xor_sync(0xffffffffu, q2[0], 1); }
        if (rg == 0 && m_tile < p.gn_mtiles) {               // slots without a valid row still get their zeros
          const int per_row = p.N >> p.gn_shift;
          const long long slot = p.gn_slot0 + static_cast<long long>(m_tile) * 4 + (warp & 3);
          float2* dst = reinterpret_cast<float2*>(p.gn_part) + slot * per_row + ((ocol0 + 8 * ch) >> p.gn_shift);
          if (red == 2) {
            reinterpret_cast<float4*>(dst)[0] = make_float4(s2[0], q2[0], s2[1], q2[1]);
            reinterpret_cast<float4*>(dst)[1] = make_float4(s2[2], q2[2], s2[3], q2[3]);
          } else if (red == 4) {
            *reinterpret_cast<float4*>(dst) = make_float4(s2[0], q2[0], s2[2], q2[2]);
          } else if (red == 8 || (ch & 1) == 0) {
            *dst = make_float2(s2[0], q2[0]);
          }
        }
      }
    }
    return;
  }

  if constexpr (LEAN) return;
  // ================= direct path =================
  const long long obase = g1 * p.ostride[0] + g2 * p.ostride[1] + g3 * p.ostride[2] + g4 * p.ostride[3] + c.split * p.split_ostride;
  const float rbias = (p.bias_mode == TG_BIAS_ROW && row_ok) ? p.bias[g1] : 0.0f;
  // Residual reads do not depend on the accumulator: this thread's WHOLE residual slice (its row x the 32-column rounds
  // r = grp, grp+2, ...; <= 256 B) is requested before the accumulator wait, so global-load latency overlaps the mainloop.
  const int nrounds = (p.BN + 31) >> 5;
  const bool res_on = p.res != nullptr && row_ok && p.rcol == 1 && !geglu;
  uint4 rq[TG_EPI_RPW][4];
  bool fast[TG_EPI_RPW];
#pragma unroll
  for (int i = 0; i < TG_EPI_RPW; ++i) {
    const int r = grp + TG_EPI_GROUPS * i;
    fast[i] = false;
    if (res_on && r < nrounds) {
      const int colg = n0 + 32 * r;
      const int nch = min(2, (p.BN - 32 * r) >> 4);
      const T* rgrp = reinterpret_cast<const T*>(p.res) + rbase + colg;
      if (colg + 16 * nch <= p.N && (reinterpret_cast<uintptr_t>(rgrp) & 15) == 0) {
        rq[i][0] = ld_nc16(rgrp); rq[i][1] = ld_nc16(rgrp + 8);
        if (nch == 2) { rq[i][2] = ld_nc16(rgrp + 16); rq[i][3] = ld_nc16(rgrp + 24); }
        fast[i] = true;
      }
    }
  }

  mbar_wait(tfull_bar_addr, aphase, p.err, 4);
  tc_fence_after();
  if (stamp) tg_stamp(p, 8);

#pragma unroll
  for (int i = 0; i < TG_EPI_RPW; ++i) {
    const int r = grp + TG_EPI_GROUPS * i;
    if (r >= nrounds) break;                     // warp-uniform
    const int c0 = 32 * r;
    const int nch = min(2, (p.BN - c0) >> 4);
    uint32_t raw0[16], raw1[16];
    __syncwarp();                                // tcgen05.ld is .sync.aligned: reconverge after the guarded stores
    tc_ld16(taddr + c0, raw0);
    if (nch == 2) tc_ld16(taddr + c0 + 16, raw1);
    tc_wait_ld();
    const int col0 = n0 + c0;
    if (row_ok) {
      if (col0 < p.N) epilogue_chunk<T>(p, raw0, col0, obase, rbase, rbias, sb + c0, fast[i], rq[i][0], rq[i][1]);
      if (nch == 2 && col0 + 16 < p.N)
        epilogue_chunk<T>(p, raw1, col0 + 16, obase, rbase, rbias, sb + c0 + 16, fast[i], rq[i][2], rq[i][3]);
    }
  }
}

template <typename T, bool LEAN>
__global__ void __launch_bounds__(TG_THREADS, 1)
tapgemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmA2, const __grid_constant__ CUtensorMap tmB2,
               const __grid_constant__ CUtensorMap tmO, const __grid_constant__ TapGemmParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  if (TG_ALIGN_PAD < 1024 && base - smem_u32(smem_raw) > static_cast<uint32_t>(TG_ALIGN_PAD)) {
    if (threadIdx.x == 0 && p.err) { atomicExch(p.err, 90); __threadfence_system(); }
    __trap();
  }
  const int NS = p.stages;
  const uint32_t BST = static_cast<uint32_t>(p.b_stage);
  const uint32_t sA = base;
  const uint32_t sB = base + NS * TG_A_STAGE;
  const uint32_t ostg = base + TG_STAGES * (TG_A_STAGE + TG_B_STAGE);   // epilogue store boxes (1024-byte aligned)
  const uint32_t bars = ostg + TG_OSTG_BYTES;
  auto full_bar = [&](int s) { return bars + 8u * s; };
  auto empty_bar = [&](int s) { return bars + 8u * (TG_MAX_STAGES + s); };
  auto tfull_bar = [&](int a) { return bars + 8u * (2 * TG_MAX_STAGES + a); };
  auto tempty_bar = [&](int a) { return bars + 8u * (2 * TG_MAX_STAGES + 2 + a); };
  const uint32_t tmem_slot = bars + 8u * (2 * TG_MAX_STAGES + 4);
  float* const s_bias = reinterpret_cast<float*>(smem_raw + (bars - smem_u32(smem_raw)) + TG_BAR_BYTES);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) tg_stamp(p, 0);
  const int nsplit = p.ksplit > 1 ? p.ksplit : 1;
  const int total_tiles = p.n_tiles * p.tdim[0] * p.tdim[1] * p.tdim[2] * p.tdim[3] * nsplit;
  int steps = 0, sec_steps = 0;
  for (int t = 0; t < p.num_taps; ++t) steps += p.tap_kc[t];
  for (int t = p.nprim; t < p.num_taps; ++t) sec_steps += p.tap_kc[t];

  if (warp == TG_EPI_WARPS && lane == 0) {
    for (int s = 0; s < NS; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), TG_EPI_WARPS); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmB)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA2)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmB2)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmO)) : "memory");
  }
  if (warp == TG_EPI_WARPS + 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(tmem_slot) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (threadIdx.x == 0) tg_stamp(p, 1);
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot) : "memory");
  if (TG_REGS_EPI > 0) { if (warp >= TG_EPI_WARPS) reg_dec<TG_REGS_CTRL>(); else reg_inc<TG_REGS_EPI>(); }

  if (warp == TG_EPI_WARPS) {
    // ================================ TMA producer (whole warp runs the loop, one elected lane issues) ==========
    // (the single-thread form of the CTA-pair kernel is NOT used here: with it this kernel faulted sporadically in the
    // timeline-stamp build — different launches each time, clean under compute-sanitizer — so it keeps the round-1 form)
    int stage = 0, phase = 0;
    const uint32_t tx_bytes = TG_A_STAGE + static_cast<uint32_t>(p.BN) * (TG_BK * 2);
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      const TileCoord c = decode_tile(p, tile);
      const int a1 = c.t[0] * p.a_mul[0], a2 = c.t[1] * p.a_mul[1], a3 = c.t[2] * p.a_mul[2],
                a4 = c.t[3] * p.a_mul[3];
      const int b2 = c.t[1] * p.b_mul[0], b3 = c.t[2] * p.b_mul[1], b4 = c.t[3] * p.b_mul[2];
      const int n0 = c.nt * p.BN;
      auto load_step = [&](int t, int kc) {
        const CUtensorMap* ta = p.tap_src[t] ? &tmA2 : &tmA;
        const CUtensorMap* tb = p.tap_src[t] ? &tmB2 : &tmB;
        mbar_wait(empty_bar(stage), phase ^ 1, p.err, 1);
        if (elect_one()) {
          mbar_expect_tx(full_bar(stage), tx_bytes);
          tma_load_5d(sA + stage * TG_A_STAGE, ta, full_bar(stage), kc * TG_BK + p.tap_a[t][0],
                      a1 + p.tap_a[t][1], a2 + p.tap_a[t][2], a3 + p.tap_a[t][3], a4 + p.tap_a[t][4]);
          tma_load_5d(sB + stage * BST, tb, full_bar(stage), kc * TG_BK + p.tap_b[t][0], n0,
                      b2 + p.tap_b[t][1], b3 + p.tap_b[t][2], b4 + p.tap_b[t][3]);
        }
        __syncwarp();
        if (++stage == NS) { stage = 0; phase ^= 1; }
      };
      const int kc0 = nsplit > 1 ? c.split * p.kc_per : 0, kc1 = nsplit > 1 ? min(p.kchunks, kc0 + p.kc_per) : p.kchunks;
      for (int kc = kc0; kc < kc1; ++kc)
        for (int t = 0; t < p.nprim; ++t) load_step(t, kc);
      if (c.split == 0)
        for (int t = p.nprim; t < p.num_taps; ++t)
          for (int kc = 0; kc < p.tap_kc[t]; ++kc) load_step(t, kc);
      if (tile == static_cast<int>(blockIdx.x) && lane == 0) tg_stamp(p, 2);   // first tile's loads all issued
    }
    if (lane == 0) tg_stamp(p, 3);
  } else if (warp == TG_EPI_WARPS + 1) {
    // ================================ MMA issuer (warp-uniform loop, elected lane issues) ================================
    int stage = 0, phase = 0, iter = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++iter) {
      const int acc = iter & 1, aphase = (iter >> 1) & 1;
      mbar_wait(tempty_bar(acc), aphase ^ 1, p.err, 2);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc * TG_ACC_COLS;
      int tsteps = steps;
      if (nsplit > 1) {                                                         // this tile's share of the K loop
        const int split = tile / (total_tiles / nsplit);
        const int kc0 = split * p.kc_per, kc1 = min(p.kchunks, kc0 + p.kc_per);
        tsteps = (kc1 - kc0) * p.nprim + (split == 0 ? sec_steps : 0);
      }
      for (int s = 0; s < tsteps; ++s) {
        mbar_wait(full_bar(stage), phase, p.err, 3);
        tc_fence_after();
        if (iter == 0 && s == 0 && lane == 0) tg_stamp(p, 4);                   // first operands landed
        if (elect_one()) {
          const uint64_t adesc = umma_desc_sw128(sA + stage * TG_A_STAGE);
          const uint64_t bdesc = umma_desc_sw128(sB + stage * BST);
#pragma unroll
          for (int k = 0; k < TG_BK / 16; ++k)
            tc_mma_f16(d_tmem, adesc + 2 * k, bdesc + 2 * k, p.idesc, (s > 0 || k > 0) ? 1u : 0u);
          tc_commit(empty_bar(stage));               // frees the smem slot when these MMAs retire
          if (s == tsteps - 1) tc_commit(tfull_bar(acc));  // accumulator complete -> epilogue
        }
        __syncwarp();
        if (++stage == NS) { stage = 0; phase ^= 1; }
      }
      if (iter == 0 && lane == 0) tg_stamp(p, 5);                               // first tile fully issued
    }
    if (lane == 0) tg_stamp(p, 6);
  } else if (warp < TG_EPI_WARPS) {
    // ================================ epilogue (warps 0..7) ================================
    const int row = (warp & 3) * 32 + lane;
    int rr = row;
    const int j1 = rr % p.box[0]; rr /= p.box[0];
    const int j2 = rr % p.box[1]; rr /= p.box[1];
    const int j3 = rr % p.box[2];
    const int j4 = rr / p.box[2];
    int iter = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++iter) {
      const int acc = iter & 1, aphase = (iter >> 1) & 1;
      const TileCoord c = decode_tile(p, tile);
      epilogue_tile<T, LEAN>(p, &tmO, c, fast_div(tile, p.n_tiles, p.magic[0]), row, warp, j1, j2, j3, j4, acc, aphase, tmem_base, s_bias, ostg,
                       tfull_bar(acc), p.n_tiles > 1 || iter < 2, iter == 0 && threadIdx.x == 0);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(acc));
      if (iter == 0 && threadIdx.x == 0) tg_stamp(p, 9);                        // first tile stored
    }
    if (p.tma_out && lane == 0) bulk_wait_all();      // the store boxes live in this CTA's shared memory
    if (threadIdx.x == 0) tg_stamp(p, 10);
  }

  tc_fence_before();
  __syncthreads();
  if (threadIdx.x == 0) tg_stamp(p, 11);
  if (warp == TG_EPI_WARPS + 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
    if (lane == 0) tg_stamp(p, 12);
  }
}

}  // namespace i2it
