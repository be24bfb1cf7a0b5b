// tapgemm2: the CTA-pair (cta_group::2) version of tapgemm for the big layers.
//
// Two CTAs on the two SMs of a TPC form a cluster and compute a 256-row x BN tile together:
//   * each CTA TMA-loads ITS 128-row A tile and HALF of the B (weight) tile (BN/2 rows) into its own smem and signals the
//     leader's "full" mbarrier (cp.async.bulk.tensor...cta_group::2, barrier address with the peer bit cleared);
//   * the leader's elected lane issues tcgen05.mma.cta_group::2 (M = 256): the tensor cores of both SMs read A from their
//     own smem and B split across the pair, accumulating into each CTA's own TMEM (128 lanes each);
//   * tcgen05.commit...multicast::cluster releases the smem stage / publishes the accumulator in BOTH CTAs;
//   * both CTAs run the same epilogue on their own 128 rows and arrive (remotely for the peer) on the leader's tmem_empty.
// Per CTA and k-step this moves 16 KB (A) + BN*64 B (half of B) instead of 16 KB + BN*128 B, and an N=128 tile no longer
// starves the tensor pipe on shared-memory operand reads (M=256 x N=128 per instruction instead of 128 x 128).
#pragma once
#include "tapgemm.cuh"

namespace i2it {

constexpr int TG2_STAGES = 6;
constexpr int TG2_B_STAGE = 128 * TG_BK * 2;     // half of a BN<=256 weight tile: 16 KiB
// halo mode (3x3 stride-1 convs): ONE halo tile per k-chunk instead of nine shifted 128-row boxes.  Output tile = 8 wide x 16
// tall; the halo box is 18 rows x 16 pixels (8 + 2 halo + 6 unused), so every image row starts a 2048-byte group and a tap's
// view is "start + dy*2048 + dx*128" with SBO 2048 (swizzle phase from the absolute address, see umma_desc_halo).
constexpr int TG2_HALO_W = 16, TG2_HALO_H = 18;
constexpr int TG2_HALO_BYTES = TG2_HALO_H * TG2_HALO_W * TG_BK * 2;   // 36,864
constexpr int TG2_HALO_STAGES = 2;   // two 36 KB halo tiles (each serves nine taps) leave room for the 32 KB of epilogue store boxes
constexpr int TG2_HALO_REGION = TG2_HALO_STAGES * TG2_HALO_BYTES;
constexpr int TG2_DATA_BYTES = TG2_STAGES * (TG_A_STAGE + TG2_B_STAGE);   // 192 KB; halo mode: [halo region][B stages in the rest]
static_assert(TG2_HALO_REGION + 4 * TG2_B_STAGE <= TG2_DATA_BYTES, "halo region leaves fewer than four full B stages");
constexpr int TG2_SMEM = TG2_DATA_BYTES + TG_BAR_BYTES + TG_BIAS_BYTES + TG_OSTG_BYTES + TG_ALIGN_PAD;
static_assert(TG_SMEM <= 232448 && TG2_SMEM <= 232448, "dynamic shared memory per CTA exceeds the 227 KB limit");

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the barrier at the same smem offset in CTA `cta` of the cluster
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar, uint32_t cta) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}"
      ::"r"(bar), "r"(cta) : "memory");
}
__device__ __forceinline__ void tma_load_5d_2sm(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2,
                                                int c3, int c4) {
  // executed by both CTAs: data lands in the issuing CTA's smem, the transaction bytes on CTA0's barrier (mapa -> rank 0)
  asm volatile(
      "{\n\t.reg .b32 lb;\n\t"
      "mapa.shared::cluster.u32 lb, %2, 0;\n\t"
      "cp.async.bulk.tensor.5d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6, %7}], [lb];\n\t}"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
__device__ __forceinline__ void tc_mma_f16_2sm(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc_commit_2sm(uint32_t bar) {
  asm volatile(
      "{\n\t.reg .b16 m;\n\tmov.b16 m, 3;\n\t"
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], m;\n\t}"
      ::"r"(bar) : "memory");
}

// descriptor of a tap's view into the halo tile: rows of 128 B, 8-row groups 2048 B apart (one image row of the 16-pixel
// pitch).  The start address is dx rows past a 1024-byte swizzle-atom boundary; the tensor core derives the 128B-swizzle phase
// from the absolute shared-memory address bits (the same bits TMA used when it wrote the tile), so base_offset stays 0
// (measured: base_offset = dx reads the wrong chunks, 0 is bit-exact against the nine-box path).
__device__ __forceinline__ uint64_t umma_desc_halo(uint32_t saddr) {
  uint64_t d = static_cast<uint64_t>((saddr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(2048 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;           // SWIZZLE_128B
  return d;
}

// host: instruction descriptor for the pair MMA (M = 256)
inline uint32_t make_idesc2(int dtype, int bn) {
  uint32_t fmt = (dtype == DT_BF16) ? 1u : 0u;
  return (1u << 4) | (fmt << 7) | (fmt << 10) | (static_cast<uint32_t>(bn >> 3) << 17) | ((256u >> 4) << 24);
}

// tmB / tmB2 here are encoded with a box of BN/2 rows.  gridDim.x must be even (cluster dims (2,1,1)).
template <typename T, bool LEAN>
__global__ void __launch_bounds__(TG_THREADS, 1)
tapgemm2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                const __grid_constant__ CUtensorMap tmA2, const __grid_constant__ CUtensorMap tmB2,
                const __grid_constant__ CUtensorMap tmH, const __grid_constant__ CUtensorMap tmO,
                const __grid_constant__ TapGemmParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  if (TG_ALIGN_PAD < 1024 && base - smem_u32(smem_raw) > static_cast<uint32_t>(TG_ALIGN_PAD)) {
    if (threadIdx.x == 0 && p.err) { atomicExch(p.err, 90); __threadfence_system(); }
    __trap();
  }
  // normal mode: [A stages][B stages]; halo mode: [halo stages][B stages]
  const int NS = p.stages;                                  // host-chosen: B stage sized to the real half tile, <= TG_MAX_STAGES
  const uint32_t BST = static_cast<uint32_t>(p.b_stage);
  const uint32_t sA = base;
  const uint32_t sB = base + (p.halo ? TG2_HALO_REGION : NS * TG_A_STAGE);
  const uint32_t ostg = base + TG2_DATA_BYTES;                // epilogue store boxes (1024-byte aligned)
  const uint32_t bars = ostg + TG_OSTG_BYTES;
  auto full_bar = [&](int s) { return bars + 8u * s; };
  auto empty_bar = [&](int s) { return bars + 8u * (TG_MAX_STAGES + s); };
  auto tfull_bar = [&](int a) { return bars + 8u * (2 * TG_MAX_STAGES + a); };
  auto tempty_bar = [&](int a) { return bars + 8u * (2 * TG_MAX_STAGES + 2 + a); };
  const uint32_t tmem_slot = bars + 8u * (2 * TG_MAX_STAGES + 4);
  auto hfull_bar = [&](int s) { return bars + 8u * (2 * TG_MAX_STAGES + 6 + s); };
  auto hempty_bar = [&](int s) { return bars + 8u * (2 * TG_MAX_STAGES + 6 + TG2_HALO_STAGES + s); };
  float* const s_bias = reinterpret_cast<float*>(smem_raw + (bars - smem_u32(smem_raw)) + TG_BAR_BYTES);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) tg_stamp(p, 0);
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int m_tiles = p.tdim[0] * p.tdim[1] * p.tdim[2] * p.tdim[3];
  const int total_pairs = p.n_tiles * ((m_tiles + 1) >> 1);
  const int num_clusters = gridDim.x >> 1, cluster_id = blockIdx.x >> 1;
  int steps = 0;
  for (int t = 0; t < p.num_taps; ++t) steps += p.tap_kc[t];
  const int half_bn = p.BN >> 1;

  // pair tile -> this CTA's (n tile, m tile) coordinates
  auto decode_pair = [&](int pt) {
    TileCoord c;
    const int mp = fast_div(pt, p.n_tiles, p.magic[0]);
    c.nt = pt - mp * p.n_tiles;
    int r = 2 * mp + static_cast<int>(rank), q;
    q = fast_div(r, p.tdim[0], p.magic[1]); c.t[0] = r - q * p.tdim[0]; r = q;
    q = fast_div(r, p.tdim[1], p.magic[2]); c.t[1] = r - q * p.tdim[1]; r = q;
    q = fast_div(r, p.tdim[2], p.magic[3]); c.t[2] = r - q * p.tdim[2];
    c.t[3] = q;                               // may exceed tdim[3] for the odd tail: rows then fail the extent check
    c.split = 0;                              // split-K is a 1-CTA-kernel feature
    return c;
  };

  if (warp == TG_EPI_WARPS && lane == 0) {
    for (int s = 0; s < NS; ++s) { mbar_init(full_bar(s), 2); mbar_init(empty_bar(s), 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 2 * TG_EPI_WARPS); }
    for (int s = 0; s < TG2_HALO_STAGES; ++s) { mbar_init(hfull_bar(s), 2); mbar_init(hempty_bar(s), 1); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmB)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA2)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmB2)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmH)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmO)) : "memory");
  }
  cluster_sync_all();                                   // peer barriers initialised before any remote arrive / TMEM alloc
  if (warp == TG_EPI_WARPS + 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(tmem_slot) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (threadIdx.x == 0) tg_stamp(p, 1);
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot) : "memory");
  if (TG_REGS_EPI > 0) { if (warp >= TG_EPI_WARPS) reg_dec<TG_REGS_CTRL>(); else reg_inc<TG_REGS_EPI>(); }   // see TG_THREADS

  if (warp == TG_EPI_WARPS) {
    // ================================ TMA producer (both CTAs): ONE elected thread runs the whole loop =====================
    // (after the MMA issue loop was trimmed the r02i profile showed the MMA thread waiting for operands on 91 % of the steps of
    // the N = 128 halo convs: this loop — per-step elect, parameter-table lookups — had become the critical path)
    if (elect_one()) {
    int stage = 0, phase = 0, hs = 0, hphase = 0;
    const uint32_t b_bytes = static_cast<uint32_t>(half_bn) * (TG_BK * 2);
    const uint32_t tx_bytes = 2u * (TG_A_STAGE + b_bytes);                                         // both CTAs' bytes
    for (int pt = cluster_id; pt < total_pairs; pt += num_clusters) {
      const TileCoord c = decode_pair(pt);
      const int a1 = c.t[0] * p.a_mul[0], a2 = c.t[1] * p.a_mul[1], a3 = c.t[2] * p.a_mul[2], a4 = c.t[3] * p.a_mul[3];
      const int b2 = c.t[1] * p.b_mul[0], b3 = c.t[2] * p.b_mul[1], b4 = c.t[3] * p.b_mul[2];
      const int n0 = c.nt * p.BN + static_cast<int>(rank) * half_bn;
      auto load_step = [&](int t, int kc) {
        const CUtensorMap* ta = p.tap_src[t] ? &tmA2 : &tmA;
        const CUtensorMap* tb = p.tap_src[t] ? &tmB2 : &tmB;
        mbar_wait(empty_bar(stage), phase ^ 1, p.err, 21);
        {
          if (leader) mbar_expect_tx(full_bar(stage), tx_bytes);
          else mbar_arrive_cluster(full_bar(stage), 0);
          tma_load_5d_2sm(sA + stage * TG_A_STAGE, ta, full_bar(stage), kc * TG_BK + p.tap_a[t][0], a1 + p.tap_a[t][1],
                          a2 + p.tap_a[t][2], a3 + p.tap_a[t][3], a4 + p.tap_a[t][4]);
          tma_load_5d_2sm(sB + stage * BST, tb, full_bar(stage), kc * TG_BK + p.tap_b[t][0], n0,
                          b2 + p.tap_b[t][1], b3 + p.tap_b[t][2], b4 + p.tap_b[t][3]);
        }
        if (++stage == NS) { stage = 0; phase ^= 1; }
      };
      if (p.halo) {
        for (int kc = 0; kc < p.kchunks; ++kc) {
          // one halo tile (rows y0-1 .. y0+16, pixels x0-1 .. x0+14) serves all nine taps of this k-chunk
          mbar_wait(hempty_bar(hs), hphase ^ 1, p.err, 24);
          {
            if (leader) mbar_expect_tx(hfull_bar(hs), 2u * TG2_HALO_BYTES);
            else mbar_arrive_cluster(hfull_bar(hs), 0);
            tma_load_5d_2sm(sA + hs * TG2_HALO_BYTES, &tmH, hfull_bar(hs), kc * TG_BK, a1 - 1, a2 - 1, a3, a4);
          }
          if (++hs == TG2_HALO_STAGES) { hs = 0; hphase ^= 1; }
#pragma unroll
          for (int t = 0; t < 9; ++t) {                    // halo mode: 3x3 taps, weight tap t at B coordinate (kc*64, n0, t, 0, 0)
            mbar_wait(empty_bar(stage), phase ^ 1, p.err, 21);
            if (leader) mbar_expect_tx(full_bar(stage), 2u * b_bytes);
            else mbar_arrive_cluster(full_bar(stage), 0);
            tma_load_5d_2sm(sB + stage * BST, &tmB, full_bar(stage), kc * TG_BK, n0, t, 0, 0);
            if (++stage == NS) { stage = 0; phase ^= 1; }
          }
        }
      } else {
        for (int kc = 0; kc < p.kchunks; ++kc)
          for (int t = 0; t < p.nprim; ++t) load_step(t, kc);
        for (int t = p.nprim; t < p.num_taps; ++t)
          for (int kc = 0; kc < p.tap_kc[t]; ++kc) load_step(t, kc);
      }
      if (pt == cluster_id) tg_stamp(p, 2);   // first tile's loads all issued
    }
    tg_stamp(p, 3);
    }
    __syncwarp();
  } else if (warp == TG_EPI_WARPS + 1) {
    // ================================ MMA issuer (leader CTA only) ================================
    // ONE elected thread runs the whole issue loop (no per-step elect / reconvergence: the loop is the critical path of the
    // short-MMA launches, see the halo branch); the other lanes wait at the warp barrier below.
    if (leader && elect_one()) {
      int stage = 0, phase = 0, iter = 0, hs = 0, hphase = 0;
      for (int pt = cluster_id; pt < total_pairs; pt += num_clusters, ++iter) {
        const int acc = iter & 1, aphase = (iter >> 1) & 1;
        mbar_wait(tempty_bar(acc), aphase ^ 1, p.err, 22);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * TG_ACC_COLS;
        if (p.halo) {
          // The nine taps are unrolled with compile-time offsets into the halo tile (host order t = ky*3 + kx: tap t reads rows
          // shifted by t/3 image rows = 2048 B and t%3 pixels = 128 B).  The r02h profile showed this single-thread loop, not
          // operands or TMEM, bounding the N = 128 convs: ~90 instructions (parameter-table lookups, R2UR moves) per 4 MMAs
          // of 64 cycles each = 55 % tensor pipe.
          for (int kc = 0; kc < p.kchunks; ++kc) {
            mbar_wait(hfull_bar(hs), hphase, p.err, 25);
            const uint32_t a_base = sA + hs * TG2_HALO_BYTES;
            const bool last_kc = kc == p.kchunks - 1;
#pragma unroll
            for (int t = 0; t < 9; ++t) {
              mbar_wait(full_bar(stage), phase, p.err, 23);
              tc_fence_after();
              {
                const uint64_t adesc = umma_desc_halo(a_base + static_cast<uint32_t>(t / 3) * 2048u + static_cast<uint32_t>(t % 3) * 128u);
                const uint64_t bdesc = umma_desc_sw128(sB + stage * BST);
#pragma unroll
                for (int k = 0; k < TG_BK / 16; ++k)
                  tc_mma_f16_2sm(d_tmem, adesc + 2 * k, bdesc + 2 * k, p.idesc, (kc > 0 || t > 0 || k > 0) ? 1u : 0u);
                tc_commit_2sm(empty_bar(stage));
                if (t == 8) tc_commit_2sm(hempty_bar(hs));
                if (t == 8 && last_kc && steps == 9 * p.kchunks) tc_commit_2sm(tfull_bar(acc));
              }
              if (++stage == NS) { stage = 0; phase ^= 1; }
            }
            if (++hs == TG2_HALO_STAGES) { hs = 0; hphase ^= 1; }
          }
        } else {
          for (int s = 0; s < steps; ++s) {
            mbar_wait(full_bar(stage), phase, p.err, 23);
            tc_fence_after();
            if (iter == 0 && s == 0) tg_stamp(p, 4);               // first operands landed (both CTAs)
            {
              const uint64_t adesc = umma_desc_sw128(sA + stage * TG_A_STAGE);
              const uint64_t bdesc = umma_desc_sw128(sB + stage * BST);
#pragma unroll
              for (int k = 0; k < TG_BK / 16; ++k)
                tc_mma_f16_2sm(d_tmem, adesc + 2 * k, bdesc + 2 * k, p.idesc, (s > 0 || k > 0) ? 1u : 0u);
              tc_commit_2sm(empty_bar(stage));
              if (s == steps - 1) tc_commit_2sm(tfull_bar(acc));
            }
            if (++stage == NS) { stage = 0; phase ^= 1; }
          }
        }
        if (iter == 0) tg_stamp(p, 5);                             // first tile fully issued
      }
      tg_stamp(p, 6);
    }
    __syncwarp();
  } else if (warp < TG_EPI_WARPS) {
    // ================================ epilogue (both CTAs, own 128 rows) ================================
    const int row = (warp & 3) * 32 + lane;
    int rr = row;
    const int j1 = rr % p.box[0]; rr /= p.box[0];
    const int j2 = rr % p.box[1]; rr /= p.box[1];
    const int j3 = rr % p.box[2];
    const int j4 = rr / p.box[2];
    int iter = 0;
    for (int pt = cluster_id; pt < total_pairs; pt += num_clusters, ++iter) {
      const int acc = iter & 1, aphase = (iter >> 1) & 1;
      const TileCoord c = decode_pair(pt);
      epilogue_tile<T, LEAN>(p, &tmO, c, 2 * fast_div(pt, p.n_tiles, p.magic[0]) + static_cast<int>(rank), row, warp, j1, j2, j3, j4, acc, aphase,
                       tmem_base, s_bias, ostg, tfull_bar(acc), p.n_tiles > 1 || iter < 2, iter == 0 && threadIdx.x == 0);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(tempty_bar(acc), 0);
      if (iter == 0 && threadIdx.x == 0) tg_stamp(p, 9);                        // first tile stored
    }
    if (p.tma_out && lane == 0) bulk_wait_all();      // the store boxes live in this CTA's shared memory
    if (threadIdx.x == 0) tg_stamp(p, 10);
  }

  tc_fence_before();
  __syncthreads();
  if (threadIdx.x == 0) tg_stamp(p, 11);
  cluster_sync_all();                                   // nobody leaves (or frees TMEM) while the peer may still signal it
  if (warp == TG_EPI_WARPS + 1) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
    if (lane == 0) tg_stamp(p, 12);
  }
}

}  // namespace i2it
