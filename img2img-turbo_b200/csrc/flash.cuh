// flash_attn_kernel: fused softmax(Q K^T * scale) V for head_dim 64 (all UNet self/cross attention of the path).
//
// Replaces, per attention layer, the three launches  S = QK^T (fp32 logits to HBM) -> softmax -> O = PV  — i.e. what the
// reference gets from F.scaled_dot_product_attention / xformers FMHA (diffusers AttnProcessor2_0; call sites under
// /root/reference/src/pix2pix_turbo.py:199 and /root/reference/src/inference_unpaired.py:36).
//
// One CTA = one 128-row Q tile of one (batch, head); 192 threads:
//   warp 4 lane 0 : TMA producer   Q once; (K_j [64 keys x 64], V^T_j [64 d x 64 keys]) through a 3-stage ring
//   warp 5 lane 0 : MMA issuer     S_j = Q K_j^T (4 x tcgen05.mma M128 N64 K16) -> TMEM S buffer j&1
//                                  PV_j = P_j V_j  (4 x tcgen05.mma, A = P_j staged in swizzled smem) -> TMEM cols [128,192)
//                                  QK_{j+1} is issued as soon as the softmax warps have pulled S_j out of TMEM
//   warps 0..3    : one Q row per thread: S_j is pulled out of TMEM ONCE (64 registers), online softmax in fp32 with a LAZY
//                   reference maximum, P_j -> bf16/fp16 smem tile; O stays in TMEM (PV accumulates across KV steps) and is only
//                   rescaled (tcgen05.ld -> mul -> tcgen05.st) when a row's maximum grows by more than 2^8; final O / l written once.
//                   Round 1 read S twice and the PV tile once per step: 96 KB of TMEM reads per step at 64 B/clk/SM made the
//                   kernel TMEM-read bound (25 % tensor pipe); this version reads 32 KB per step.
// 2 CTAs per SM (80 KB smem, 256 TMEM columns each: S double-buffered + PV) so one CTA's MMAs overlap the other's exponentials.
#pragma once
#include "tapgemm.cuh"

namespace i2it {

constexpr int FA_BM = 128, FA_BN = 64, FA_D = 64, FA_STAGES = 3;
constexpr int FA_Q_BYTES = FA_BM * FA_D * 2;            // 16 KiB
constexpr int FA_KV_DATA = 2 * FA_BN * FA_D * 2;        // K 8 KiB + V^T 8 KiB (what TMA writes per stage)
// The PV product runs with N = 80: rows 64..79 of every V^T stage are constant — row 64 all ones, the rest zero — so column 64
// of the O accumulator is the row sum l = sum_k P[m,k] of the ROUNDED probabilities (the same values the numerator uses); the
// softmax threads no longer add 64 values per row and step (they are the critical path: MUFU + issue slots, profiles/r02g_flash*).
constexpr int FA_PV_N = 80;
constexpr int FA_KV_STAGE = FA_KV_DATA + (FA_PV_N - FA_D) * FA_BN * 2;   // + 2 KiB of constant rows
constexpr int FA_P_BYTES = FA_BM * FA_BN * 2;           // 16 KiB
constexpr int FA_SMEM = FA_Q_BYTES + FA_STAGES * FA_KV_STAGE + 2 * FA_P_BYTES + 256 + 1024;   // P is double-buffered
constexpr int FA_THREADS = 192;

struct FlashParams {
  int Nq, Nk, heads, B, q_tiles, kv_bmul;   // kv_bmul: 1 if K/V are per batch item, 0 if one K/V set is shared (text)
  float scale_log2e;                        // softmax scale * log2(e)
  void* out;                                // [B*Nq, ldo] tokens, head h at columns [64h, 64h+64)
  long long ldo;
  uint32_t idesc;                           // M=128, N=64 (both GEMMs)
  int causal;                               // 1: key j attends only to queries i >= j (CLIP text tower); KV tiles past the diagonal are skipped
  int* err;
};

__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tc_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]),
        "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]),
        "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tc_ld1(uint32_t taddr, uint32_t (&r)[1]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r[0]) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tc_st1(uint32_t taddr, const uint32_t (&r)[1]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x1.b32 [%0], {%1};" ::"r"(taddr), "r"(r[0]) : "memory");
}
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float fmax3(float a, float b, float c) {
  float r;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}
__device__ __forceinline__ void sts16(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

template <typename T>
__global__ void __launch_bounds__(FA_THREADS, 2)
flash_attn_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                  const __grid_constant__ CUtensorMap tmVt, const __grid_constant__ FlashParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sQ = base;
  const uint32_t sKV = base + FA_Q_BYTES;
  const uint32_t sP = sKV + FA_STAGES * FA_KV_STAGE;
  const uint32_t bars = sP + 2 * FA_P_BYTES;
  const uint32_t q_full = bars;
  auto kv_full = [&](int s) { return bars + 8u * (1 + s); };
  auto kv_empty = [&](int s) { return bars + 8u * (1 + FA_STAGES + s); };
  // S is double-buffered in TMEM; each buffer has its own full/free barrier so no waiter can fall two phases behind
  const uint32_t s_full0 = bars + 8u * (1 + 2 * FA_STAGES);
  auto s_full = [&](int u) { return s_full0 + 8u * u; };
  auto s_free = [&](int u) { return s_full0 + 16u + 8u * u; };
  // P_j goes to smem buffer j&1 and PV_j signals pv_done(j&1): the softmax of step j+1 no longer waits for PV_j (only the
  // buffer's previous user PV_{j-1}... i.e. step j-2's product, and a rescale of O still waits for everything issued so far)
  auto p_full = [&](int u) { return s_full0 + 32 + 8u * u; };
  auto pv_done = [&](int u) { return s_full0 + 48 + 8u * u; };
  const uint32_t tmem_slot = s_full0 + 64;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int qt = blockIdx.x % p.q_tiles;
  const int h = (blockIdx.x / p.q_tiles) % p.heads;
  const int b = blockIdx.x / (p.q_tiles * p.heads);
  int nkv = (p.Nk + FA_BN - 1) / FA_BN;
  if (p.causal) nkv = min(nkv, (qt * FA_BM + FA_BM + FA_BN - 1) / FA_BN);   // same value in all three roles

  if (warp == 4 && lane == 0) {
    mbar_init(q_full, 1);
    for (int s = 0; s < FA_STAGES; ++s) { mbar_init(kv_full(s), 1); mbar_init(kv_empty(s), 1); }
    for (int u = 0; u < 2; ++u) { mbar_init(s_full(u), 1); mbar_init(s_free(u), 4); }
    for (int u = 0; u < 2; ++u) { mbar_init(p_full(u), 4); mbar_init(pv_done(u), 1); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmQ)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmK)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmVt)) : "memory");
  }
  if (warp < 4) {
    // constant rows 64..79 of each stage's V^T tile (128-byte rows; all 16-byte chunks of a row are equal, so the 128B swizzle
    // does not matter): row 64 = ones in the activation dtype, rows 65..79 = zeros
    const uint32_t one2 = Elem<T>::pack(1.0f, 1.0f);
    for (int i = threadIdx.x; i < FA_STAGES * (FA_PV_N - FA_D) * 8; i += 128) {
      const int st = i / ((FA_PV_N - FA_D) * 8), r = (i / 8) % (FA_PV_N - FA_D), ch = i & 7;
      const uint32_t v = (r == 0) ? one2 : 0u;
      sts16(sKV + st * FA_KV_STAGE + FA_KV_DATA + r * 128 + ch * 16, v, v, v, v);
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 5) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;" ::"r"(tmem_slot) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot) : "memory");
  const uint32_t tS0 = tmem_base, tPV = tmem_base + 128;   // S buffers at columns [0,64) and [64,128)

  if (warp == 4) {
    // producer: warp-uniform loop, one elected lane issues the TMA
    if (elect_one()) {
      mbar_expect_tx(q_full, FA_Q_BYTES);
      tma_load_5d(sQ, &tmQ, q_full, 0, qt * FA_BM, h, b, 0);
    }
    __syncwarp();
    for (int j = 0; j < nkv; ++j) {
      const int s = j % FA_STAGES;
      mbar_wait(kv_empty(s), ((j / FA_STAGES) & 1) ^ 1, p.err, 11);
      if (elect_one()) {
        mbar_expect_tx(kv_full(s), FA_KV_DATA);
        tma_load_5d(sKV + s * FA_KV_STAGE, &tmK, kv_full(s), 0, j * FA_BN, h, b * p.kv_bmul, 0);
        tma_load_5d(sKV + s * FA_KV_STAGE + FA_BN * FA_D * 2, &tmVt, kv_full(s), j * FA_BN, 0, h, b * p.kv_bmul, 0);
      }
      __syncwarp();
    }
  } else if (warp == 5) {
    // MMA issuer: warp-uniform loop, one elected lane issues tcgen05.mma / commit
    mbar_wait(q_full, 0, p.err, 12);
    const uint64_t qdesc = umma_desc_sw128(sQ);
    const uint32_t idesc_pv = (p.idesc & ~(0x3Fu << 17)) | (static_cast<uint32_t>(FA_PV_N >> 3) << 17);   // same shape, N = 80
    auto issue_qk = [&](int j) {
      const int s = j % FA_STAGES;
      mbar_wait(kv_full(s), (j / FA_STAGES) & 1, p.err, 13);
      tc_fence_after();
      if (elect_one()) {
        const uint64_t kdesc = umma_desc_sw128(sKV + s * FA_KV_STAGE);
#pragma unroll
        for (int k = 0; k < FA_D / 16; ++k)
          tc_mma_f16(tS0 + 64 * (j & 1), qdesc + 2 * k, kdesc + 2 * k, p.idesc, k > 0 ? 1u : 0u);
        tc_commit(s_full(j & 1));
      }
      __syncwarp();
    };
    issue_qk(0);
    for (int j = 0; j < nkv; ++j) {
      if (j + 1 < nkv) {
        // S buffer (j+1)&1 was last read by softmax iteration j-1: QK_{j+1} overlaps the exponentials of iteration j
        if (j >= 1) { mbar_wait(s_free((j + 1) & 1), ((j - 1) >> 1) & 1, p.err, 14); tc_fence_after(); }
        issue_qk(j + 1);
      }
      mbar_wait(p_full(j & 1), (j >> 1) & 1, p.err, 15);   // P_j is in smem buffer j&1 (and any rescale of O is complete)
      tc_fence_after();
      const int s = j % FA_STAGES;
      if (elect_one()) {
        const uint64_t vdesc = umma_desc_sw128(sKV + s * FA_KV_STAGE + FA_BN * FA_D * 2);
        const uint64_t pdesc = umma_desc_sw128(sP + (j & 1) * FA_P_BYTES);
#pragma unroll
        for (int k = 0; k < FA_BN / 16; ++k)                 // O accumulates in TMEM across the KV steps
          tc_mma_f16(tPV, pdesc + 2 * k, vdesc + 2 * k, idesc_pv, (j > 0 || k > 0) ? 1u : 0u);
        tc_commit(pv_done(j & 1));
        tc_commit(kv_empty(s));                     // K_j and V_j are free once everything issued so far retires
      }
      __syncwarp();
    }
  } else {
    // ---------------- softmax / output warps: thread = Q row ----------------
    const int row = warp * 32 + lane;
    const uint32_t lane_off = static_cast<uint32_t>(warp * 32) << 16;
    const int qpos = qt * FA_BM + row;
    const int klim = p.causal ? min(p.Nk, qpos + 1) : p.Nk;     // keys [0, klim) are visible to this row
    const float sc = p.scale_log2e;
    constexpr float TAU = 8.0f;                                  // lazy rescale: P <= 2^8 relative to the reference maximum
    float m = -INFINITY;                                         // reference maximum (raw logit units) of this row
    for (int j = 0; j < nkv; ++j) {
      mbar_wait(s_full(j & 1), (j >> 1) & 1, p.err, 16);
      tc_fence_after();
      const uint32_t tS = tS0 + 64 * (j & 1);
      const int kbase = j * FA_BN;
      // element-wise masking only where needed (warp-uniform): the last KV tile, or causal tiles that reach this warp's diagonal
      const bool ragged = (kbase + FA_BN > p.Nk) || (p.causal && kbase + FA_BN - 1 > qt * FA_BM + warp * 32);
      // S_j leaves TMEM once: 64 fp32 logits per row in registers; the buffer goes back to the MMA warp right away
      uint32_t raw[64];
      {
        uint32_t (&r0)[32] = *reinterpret_cast<uint32_t (*)[32]>(&raw[0]);
        uint32_t (&r1)[32] = *reinterpret_cast<uint32_t (*)[32]>(&raw[32]);
        tc_ld32(tS + lane_off, r0);
        tc_ld32(tS + lane_off + 32, r1);
        tc_wait_ld();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(s_free(j & 1));
      float mx = -INFINITY;
      if (ragged) {
#pragma unroll
        for (int i = 0; i < 64; ++i)
          if (kbase + i < klim) mx = fmaxf(mx, __uint_as_float(raw[i]));
      } else {
        // four independent chains of 3-input maxima (FMNMX3): 34 instructions instead of a 64-deep dependent chain
        float m4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int c4 = 0; c4 < 4; ++c4)
            m4[c4] = fmax3(m4[c4], __uint_as_float(raw[16 * c4 + 2 * i]), __uint_as_float(raw[16 * c4 + 2 * i + 1]));
        mx = fmax3(fmaxf(m4[0], m4[1]), m4[2], m4[3]);
      }
      const bool grow = (fmaxf(m, mx) - m) * sc > TAU;          // first tile: m = -inf -> true
      if (j == 0) {
        m = mx;
      } else if (__any_sync(0xffffffffu, grow)) {
        // some row of this warp outgrew its reference maximum: rescale the warp's 32 O rows in TMEM (factor 1 for the others).
        // Every PV issued so far must have landed first: PV_{j-1} is the last one (MMAs retire in order).
        mbar_wait(pv_done((j - 1) & 1), ((j - 1) >> 1) & 1, p.err, 17);
        tc_fence_after();
        const float m_new = grow ? fmaxf(m, mx) : m;
        const float factor = fast_exp2((m - m_new) * sc);
        uint32_t o[32];
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          tc_ld32(tPV + lane_off + half * 32, o);
          tc_wait_ld();
#pragma unroll
          for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * factor);
          tc_st32(tPV + lane_off + half * 32, o);
        }
        {                                                     // ... and the row-sum column
          uint32_t lcol[1];
          tc_ld1(tPV + lane_off + FA_D, lcol);
          tc_wait_ld();
          lcol[0] = __float_as_uint(__uint_as_float(lcol[0]) * factor);
          tc_st1(tPV + lane_off + FA_D, lcol);
        }
        tc_wait_st();
        m = m_new;
      }
      // P buffer j&1 was last read by PV_{j-2}
      if (j >= 2) mbar_wait(pv_done(j & 1), ((j - 2) >> 1) & 1, p.err, 19);
      const uint32_t sPj = sP + (j & 1) * FA_P_BYTES;
      const float neg_ms = -m * sc;
      // p = exp2(s*scale - m*scale) (one FFMA + one MUFU per element), pack to 16 bit, write the
      // swizzled K-major P tile
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        uint32_t pk[16];
        if (ragged) {
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const int k0 = kbase + half * 32 + 2 * i;
            const float p0 = (k0 < klim) ? fast_exp2(fmaf(__uint_as_float(raw[half * 32 + 2 * i]), sc, neg_ms)) : 0.f;
            const float p1 = (k0 + 1 < klim) ? fast_exp2(fmaf(__uint_as_float(raw[half * 32 + 2 * i + 1]), sc, neg_ms)) : 0.f;
            pk[i] = Elem<T>::pack(p0, p1);
          }
        } else {
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const float p0 = fast_exp2(fmaf(__uint_as_float(raw[half * 32 + 2 * i]), sc, neg_ms));
            const float p1 = fast_exp2(fmaf(__uint_as_float(raw[half * 32 + 2 * i + 1]), sc, neg_ms));
            pk[i] = Elem<T>::pack(p0, p1);
          }
        }
#pragma unroll
        for (int g = 0; g < 4; ++g) {               // 16-byte group g' = half*4+g holds keys 8g'..8g'+7 of this row
          const int gg = half * 4 + g;
          sts16(sPj + row * 128 + ((gg ^ (row & 7)) << 4), pk[4 * g], pk[4 * g + 1], pk[4 * g + 2], pk[4 * g + 3]);
        }
      }
      // P_j visible to the async proxy (and any O rescale complete) -> PV_j may start
      tc_fence_before();
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive(p_full(j & 1));
    }
    // last PV, then the only read of O
    mbar_wait(pv_done((nkv - 1) & 1), ((nkv - 1) >> 1) & 1, p.err, 18);
    tc_fence_after();
    const int q = qt * FA_BM + row;
    float inv;
    {
      uint32_t lcol[1];
      tc_ld1(tPV + lane_off + FA_D, lcol);
      tc_wait_ld();
      inv = 1.0f / __uint_as_float(lcol[0]);
    }
    T* optr = reinterpret_cast<T*>(p.out) + (static_cast<long long>(b) * p.Nq + q) * p.ldo + h * FA_D;
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      uint32_t o[32];
      tc_ld32(tPV + lane_off + half * 32, o);
      tc_wait_ld();
      if (q < p.Nq) {
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          uint4 u;
          u.x = Elem<T>::pack(__uint_as_float(o[8 * g]) * inv, __uint_as_float(o[8 * g + 1]) * inv);
          u.y = Elem<T>::pack(__uint_as_float(o[8 * g + 2]) * inv, __uint_as_float(o[8 * g + 3]) * inv);
          u.z = Elem<T>::pack(__uint_as_float(o[8 * g + 4]) * inv, __uint_as_float(o[8 * g + 5]) * inv);
          u.w = Elem<T>::pack(__uint_as_float(o[8 * g + 6]) * inv, __uint_as_float(o[8 * g + 7]) * inv);
          st16(optr + half * 32 + 8 * g, u);
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 5) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;" ::"r"(tmem_base) : "memory");
  }
}

}  // namespace i2it
